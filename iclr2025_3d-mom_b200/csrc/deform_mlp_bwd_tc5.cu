// Deformation MLP backward on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a, F = 64.
//
// Maths (scene/deformation.py:55-65, :97-153 differentiated; see deform_mlp.cu for the forward):
//     dz_h   = (d_out_h W3_h) * [relu(z_h) > 0]                      h = pos, scales, rotations
//     d relu(hidden) = sum_h dz_h W2_h ;  dh = d relu(hidden) * [relu(hidden) > 0]
//     d feature = dh W1
//     dW3_h = d_out_h^T relu(z_h), dW2_h = dz_h^T relu(hidden), dW1 = dh^T feature, db = column sums
//
// One persistent CTA per SM (256 threads) walks 128-point tiles.
//   * SIMT side, thread = (4-column chunk q, 8 points): dz (the K <= 4 contraction with W3), the
//     ReLU masks, dW3 and every bias gradient are plain FP32 in registers (dW3 / biases accumulate in
//     registers over all tiles of the CTA).  Eight lanes cover one 128-byte row, so every global load
//     and every shared-memory store below is a full line / conflict free.
//   * dX chain on the tensor cores, SS mode, full three-term split (dY_lo W_hi + dY_hi W_lo + dY_hi W_hi, FP32-level
//     accuracy: its error would otherwise reach the per-point xyz gradients un-averaged):  D_RH[p][in] += dz[p][out]
//     W2_h[out][in], D_FE = dh W1.  A = the hi and lo dY planes of DYM read as a K-major operand (see below); B = the
//     transposed TF32 hi / lo weight images the forward left behind the stash, streamed in with cp.async.
//   * weight gradients on the tensor cores: D_W[out][in] += tf32(dY)^T tf32(X), contraction over the 128
//     points of the tile, with M = 128 rows = [dY_hi ; dY_lo] (the two halves are added at the flush, so
//     dY is exact and only X is rounded).  Both operands are MN-major; for TF32 the only MN-major shared-memory layout
//     tcgen05 accepts is SWIZZLE_128B_BASE32B (descriptor layout type 1): atoms of 4 k-rows x 128 B
//     (32 MN elements), the 32-byte granule index XORed with the row index (probed on hardware,
//     tools/probe/umma_probe.cu).  The accumulators D_W2[3], D_W1 stay in TMEM for the whole life of
//     the CTA and are flushed once per CTA at the end.
// Shared memory (~225 KB): W2 slot 32 K (hi|lo) | W1 32 K (hi|lo) | DYM 64 K | XH 32 K | DYK 2 x 33 K.
// TMEM columns: D_RH [0,64)  D_FE [64,128)  D_W2[h] [128 + 64 h, +64)  D_W1 [320,384).
#include "tc5_common.cuh"
#include "../../include/b200gs.h"

namespace b200gs {
namespace tc5 {

constexpr int BT = 256;                     // threads per CTA
constexpr u32 KCH = 2064;                   // DYK: bytes between 4-column chunks (2048 + 16 pad)
constexpr u32 KPLANE = 16 * KCH;            // one half of DYK (one TMA staging slot)
constexpr u64 DESC_SW128_32B = 1ull << 61;  // smem descriptor layout type SWIZZLE_128B_BASE32B

struct BwdArgs {
    b200gs_mlp_weights w;
    b200gs_mlp_grads gw;
    long long P;
    const float* feat; const float* saved;
    const float* d_pts; const float* d_scales; const float* d_rot;
    float* d_feat;
    u32 dy_sbo;                 // 512: byte stride between 8-point groups of the K-major view of the dY image (an argument,
                                // not a constant: folded into the code it makes ptxas spill in the TMA kernel)
};

__device__ __forceinline__ float4 tf32x4(float4 v)
{
    return make_float4(__uint_as_float(to_tf32(v.x)), __uint_as_float(to_tf32(v.y)), __uint_as_float(to_tf32(v.z)), __uint_as_float(to_tf32(v.w)));
}
__device__ __forceinline__ void split4(const float* x, float4& hi, float4& lo)
{
    hi = make_float4(x[0], x[1], x[2], x[3]);            // the tensor core truncates: see tf32_lo
    lo = make_float4(tf32_lo(x[0]), tf32_lo(x[1]), tf32_lo(x[2]), tf32_lo(x[3]));
}
__device__ __forceinline__ void sts128(u32 addr, float4 v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" :: "r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds128(u32 addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// Pipeline (same arithmetic, same operands and same TMEM map as the first generation, which measured 0.744 ms per 1M points):
//   * the two 32 KB weight slots alternate between consecutive MMA groups and the image of the NEXT group is streamed in
//     (cp.async) while the current phase computes, so no phase waits for its weights (W1 is re-streamed per tile from L2);
//   * MMAs are issued from a warp-uniform branch by the elected lane of warp 0 with the shared-memory descriptors formed by
//     adding constants to two hoisted bases: ~2 SASS instructions per tcgen05.mma instead of ~15 (the single issuing
//     thread sits on the critical path of every phase);
//   * the TMEM-resident weight gradients leave through a padded shared-memory transpose as hi + lo sums, one coalesced
//     128-bit RED per 4 elements (8x fewer atomics than one scalar atomic per hi / lo element, whole lines per warp);
//   * the upstream gradients d_out of the next phase are prefetched into L2 one phase ahead (loading them into registers
//     one phase ahead, or prefetching into L1, measured slower);
//   * ONE dY image: the dX chain reads its A operand dY from the MN-major SWIZZLE_128B_BASE32B image of the weight-gradient
//     MMAs, re-described as a K-major operand (rows = points, 128-byte rows of 32 out-features, 8-row group stride
//     BwdArgs::dy_sbo = 512 B -- the one combination that reproduces the product exactly on hardware, tools/probe/umma_probe2.cu,
//     profiles/r2a_umma_probe2.txt), so dY is stored to shared memory twice (hi, lo) instead of four times: 0.744 -> 0.686 ms
//     per 1M points (profiles/r2a_mlp_variant_check.txt).
// TMA (tiled feature layout only): the 66 KB of shared memory that frees become two 32 KB staging slots, and the stash / feature
// rows of a phase (one contiguous 32 KB tile each, tc5_common.cuh) arrive by ONE bulk copy (cp.async.bulk -> UBLKCP, the TMA
// engine) requested two phases ahead by the MMA-issuing thread and counted on the slot's mbarrier, instead of 8 LDG.128 per
// thread held in registers across a phase: 0.686 -> 0.597 ms (profiles/r2i_mlp_variant_check.txt; d_out in registers on top
// of it lost: 0.648).  Row-major features are read with the LDG.128 path (TMA = false).
template <bool TMA>
__global__ void __launch_bounds__(BT, 1) deform_mlp_bwd_tc5_kernel(const __grid_constant__ BwdArgs a)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* W2B = reinterpret_cast<float*>(smem_raw);                 // current head: hi [16 k-chunks][64 n][4] | lo  (32 KB)
    float* W1B = W2B + 2 * MW * MW;                                  // hi | lo                                      (32 KB)
    unsigned char* DYM = smem_raw + 4 * MW * MW * 4;        // 64 KB, MN-major swizzled  [out: 64 hi rows | 64 lo rows][p 128]
    unsigned char* XH = DYM + 65536;                                 // 32 KB, MN-major swizzled  [in 64][p 128]
    unsigned char* DYK = XH + 32768;              // 2 x 16 chunks x 2064 B: TMA staging slots / the D_RH bounce [p 128][in 64]
    u64* bar = reinterpret_cast<u64*>(DYK + 2 * KPLANE);
    u32* tmem_slot = reinterpret_cast<u32*>(bar + 3);          // bar[0]: MMA groups; bar[1], bar[2]: the two TMA staging slots
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // SIMT mapping: columns 32 c + 4 q + e, points 32 pg + 4 i + sub (i = 0..7)
    const int q = lane & 7, sub = lane >> 3, c = warp & 1, pg = warp >> 1;
    const int col0 = 32 * c + 4 * q;
    // TMEM mapping (tcgen05.ld 32x32b): lane = point, 32 consecutive columns
    const int pT = (warp & 3) * 32 + lane, cT = warp >> 2;
    const int kdim[3] = {3, 3, 4};

    // ---- one-time staging ----
    // transposed TF32 hi / lo weight images left behind the stash by the forward (tc5_common.cuh): W1 stays resident,
    // the current head's W2 pair is streamed in per head
    const float* images = reinterpret_cast<const float*>(a.saved) + 4 * stash_plane_floats(a.P);
    auto copy_image_pair = [&](float* dst, int m) {                   // 32 KB = 2048 16-byte pieces, 8 per thread
        const float4* src = reinterpret_cast<const float4*>(images + (size_t)(2 * m) * MW * MW);
#pragma unroll
        for (int i = 0; i < 8; ++i) cp_async16(reinterpret_cast<float4*>(dst) + tid + BT * i, src + tid + BT * i);
        cp_async_commit();
    };
    for (int i = tid; i < 98304 / 16; i += BT) reinterpret_cast<float4*>(DYM)[i] = make_float4(0.f, 0.f, 0.f, 0.f);   // DYM + XH
    if (tid == 0) {
        if (smem_u32(DYM) & 1023u) __trap();                          // the swizzle below assumes 1 KB aligned tiles
        mbar_init(bar, 1);
        if constexpr (TMA) { mbar_init(bar + 1, 1); mbar_init(bar + 2, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tbase = *tmem_slot;
    const u32 lane_addr = tbase + ((u32)((warp & 3) * 32) << 16);
    constexpr u32 C_RH = 0, C_FE = 64, C_W2 = 128, C_W1 = 320;
    const u32 id_kk = make_idesc(128, 64);
    const u32 id_mn = make_idesc(128, 64) | IDESC_A_MN | IDESC_B_MN;
    const u32 sDYM = smem_u32(DYM), sXH = smem_u32(XH), sDYK = smem_u32(DYK), sW2 = smem_u32(W2B), sW1 = smem_u32(W1B);
    // this thread's store offsets: MN tiles  c * 16 KB + p * 128 + (granule ^ (p & 3)) * 32 + half * 16 with p & 3 == sub
    const u32 mn_off = (u32)c * 16384u + (u32)((((q >> 1) ^ sub) << 5) | ((q & 1) << 4));
    const u32 k_off = (u32)(8 * c + q) * KCH;
    const int p0 = 32 * pg + sub;                                     // point of iteration i: p0 + 4 i
    bool first_tile = true;
    // One MMA group (dX chain into d_col, weight gradient into w_col) issued by the elected lane of warp 0.  Called by
    // every thread right after the block barrier, so warp 0 is converged; elect.sync picks the same lane every time, which
    // tcgen05.commit needs (it tracks the MMAs of the executing thread).  Descriptor start addresses are 14-bit fields of
    // (address >> 4) and shared memory ends below 256 KB, so adding (offset >> 4) to a hoisted base cannot carry out.
    auto issue_group = [&](u32 sW, u32 d_col, bool d_accumulate, u32 w_col, bool tma_go = false, const float* tma_src = nullptr, u32 tma_slot = 0) {
        if (warp == 0) {
            if (elect_one()) {
                tc_fence_after();
                const u64 dB = smem_desc(sW, MW * 16, 128);
                const u64 dA = smem_desc(sDYM, 16384, a.dy_sbo) | DESC_SW128_32B;
                const u64 dM = smem_desc(sDYM, 16384, 512) | DESC_SW128_32B, dX = smem_desc(sXH, 16384, 512) | DESC_SW128_32B;
#pragma unroll
                for (int j = 0; j < 8; ++j) {          // K = 64 out features, 8 per instruction; lo*hi + hi*lo + hi*hi
                    const u64 bh = dB + (u64)((j * 2 * (MW * 16)) >> 4), bl = bh + (u64)((MW * MW * 4) >> 4);
                    // 8 out-features = one 32-byte step inside the 128-byte row, 32 out-features per 16 KB half; lo plane +32 KB
                    const u64 ah = dA + (u64)(((j >> 2) * 16384 + (j & 3) * 32) >> 4);
                    const u64 al = ah + (u64)(32768u >> 4);
                    mma_ss(tbase + d_col, al, bh, id_kk, (d_accumulate || j > 0) ? 1u : 0u);
                    mma_ss(tbase + d_col, ah, bl, id_kk, 1u);
                    mma_ss(tbase + d_col, ah, bh, id_kk, 1u);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j)           // K = 128 points, 8 per instruction (two 4-row atoms)
                    mma_ss(tbase + w_col, dM + (u64)((j * 1024) >> 4), dX + (u64)((j * 1024) >> 4), id_mn, (first_tile && j == 0) ? 0u : 1u);
                tc_commit(bar);
                if constexpr (TMA) {
                    // the 32 KB tile of stash / feature rows that the phase after next will read: one bulk copy (TMA engine)
                    // into the staging slot this phase has just finished with, completion counted on the slot's mbarrier
                    if (tma_go) {
                        const u32 mb = smem_u32(bar + 1 + tma_slot), dst = sDYK + tma_slot * KPLANE;
                        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(32768u) : "memory");
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     :: "r"(dst), "l"(tma_src), "r"(32768u), "r"(mb) : "memory");
                    }
                }
            }
            __syncwarp();
        }
    };

    u32 phase = 0;
    u32 ngroup = 0;                  // MMA groups committed so far; group n reads the weight slot n & 1 (0 = W2B, 1 = W1B)
    bool pending = false;            // an MMA group has been committed and not yet waited for
    long long prev_row = -1;         // row (TMEM mapping) whose d_feature is still in D_FE
    float gW3[3][4][4], gB2[3][4], gB3[3][4], gB1[4];
#pragma unroll
    for (int h = 0; h < 3; ++h)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            gB2[h][k] = 0.f; gB3[h][k] = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) gW3[h][k][e] = 0.f;
        }
#pragma unroll
    for (int e = 0; e < 4; ++e) gB1[e] = 0.f;

    auto drain = [&]() {   // wait for the committed MMA group; then D_FE of the previous tile can be stored
        if (pending) {
            mbar_wait(bar, phase); phase ^= 1; pending = false;
            tc_fence_after();
        }
        if (prev_row >= 0) {
            u32 v[32];
            tmem_ld32(lane_addr + C_FE + 32 * cT, v);
            tmem_wait_ld();
            if (prev_row < a.P) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<float4*>(a.d_feat + (a.w.feat_tiled ? stash_off(prev_row, 32 * cT) + 16 * j : (size_t)prev_row * MW + 32 * cT + 4 * j)) =
                        make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            }
            prev_row = -1;
        }
    };

    // Global loads run one phase ahead of their use (phases of a tile: head 0, 1, 2, then the feature rows for dW1;
    // the relu(hidden) rows of the NEXT tile are fetched during the last phase), so their latency hides behind the
    // MMA drain + shared-memory stores of the phase before.
    const bool en0 = a.w.w2[0] != nullptr, en1 = a.w.w2[1] != nullptr, en2 = a.w.w2[2] != nullptr;
    auto next_phase = [&](int ph) { return (ph < 0 && en0) ? 0 : (ph < 1 && en1) ? 1 : (ph < 2 && en2) ? 2 : 3; };
    // TMA staging (TMA): the rows of phase n + 2 are requested at the end of phase n into slot (n & 1); every thread tracks the
    // (uniform) schedule: n_cons rows-tiles consumed so far, (iss_tile, iss_ph) = the next tile / phase to request
    u32 n_cons = 0, n_iss = 0;
    long long iss_tile = blockIdx.x;
    int iss_ph = next_phase(-1);
    auto tma_src_of = [&](long long tile, int ph) -> const float* {
        return (ph >= 3 ? a.feat : a.saved + (size_t)(1 + ph) * stash_plane_floats(a.P)) + (size_t)tile * (ROWS * MW);
    };
    auto iss_advance = [&]() {
        if (iss_ph >= 3) { iss_tile += gridDim.x; iss_ph = next_phase(-1); } else iss_ph = next_phase(iss_ph);
        ++n_iss;
    };
    auto stage_read = [&](float4* x, long long r0) {                         // this phase's rows out of its staging slot
        const u32 slot = n_cons & 1u;
        mbar_wait(bar + 1 + slot, (n_cons >> 1) & 1u);
        const u32 base = sDYK + slot * KPLANE + (u32)(((p0 >> 2) * 256 + (col0 >> 2) * 16 + (p0 & 3) * 4) * 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 v = lds128(base + (u32)i * 1024u);
            x[i] = r0 + 4 * i < a.P ? v : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        ++n_cons;
    };
    auto load_rows = [&](float4* x, const float* src, long long r0) {          // features: row-major [P][64] or stash-style tiles
        const float* base = src + (a.w.feat_tiled ? stash_off(r0, col0) : (size_t)r0 * MW + col0);
        const size_t step = a.w.feat_tiled ? 256 : 4 * MW;                       // rows r0 + 4 i
#pragma unroll
        for (int i = 0; i < 8; ++i)
            x[i] = r0 + 4 * i < a.P ? __ldg(reinterpret_cast<const float4*>(base + step * i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto load_stash = [&](float4* x, int plane, long long r0) {                  // tiled stash plane, see stash_off
        // r0 = tile * 128 + 32 pg + sub: the 8 rows r0 + 4 i are the same slot of 8 consecutive 4-point groups
        const float* src = a.saved + (size_t)plane * stash_plane_floats(a.P) + stash_off(r0, col0);
#pragma unroll
        for (int i = 0; i < 8; ++i)
            x[i] = r0 + 4 * i < a.P ? __ldg(reinterpret_cast<const float4*>(src + 256 * i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto load_phase_rows = [&](int ph, float4* x, long long r0) {
        if (ph >= 3) load_rows(x, a.feat, r0); else load_stash(x, 1 + ph, r0);
    };
    auto load_phase_dout = [&](int ph, float (*d)[4], long long r0) {
        if (ph >= 3) return;
        const float* dsrc = ph == 0 ? a.d_pts : (ph == 1 ? a.d_scales : a.d_rot);
        const int kd = ph == 2 ? 4 : 3;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const long long r = r0 + 4 * i;
#pragma unroll
            for (int k = 0; k < 4; ++k) d[i][k] = (r < a.P && dsrc && k < kd) ? __ldg(dsrc + (size_t)r * kd + k) : 0.f;
        }
    };

    // the d_out rows of one tile are one contiguous run of 128 * kd floats: one prefetch per 128-byte line, one line per thread
    auto prefetch_phase_dout = [&](int ph, long long tile) {
        if (ph >= 3) return;
        const float* dsrc = ph == 0 ? a.d_pts : (ph == 1 ? a.d_scales : a.d_rot);
        const int kd = ph == 2 ? 4 : 3;
        if (!dsrc || tid > 4 * kd) return;                                   // 128 * kd * 4 bytes = 4 kd lines (+1: unaligned base)
        const char* p = reinterpret_cast<const char*>(dsrc + (size_t)tile * ROWS * kd) + 128 * tid;
        if (p >= reinterpret_cast<const char*>(dsrc + (size_t)a.P * kd)) return;
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
    };
    const long long nblocks = (a.P + ROWS - 1) / ROWS;
    float4 hrow[8], xin[8];
    if ((long long)blockIdx.x < nblocks) {
        load_stash(hrow, 0, (long long)blockIdx.x * ROWS + p0);
        if constexpr (!TMA) load_phase_rows(next_phase(-1), xin, (long long)blockIdx.x * ROWS + p0);
    }
    if constexpr (TMA) {              // the first two row-tiles of this CTA's schedule -> slots 0 and 1
        for (int k = 0; k < 2; ++k) {
            if (iss_tile < nblocks && tid == 0) {
                const u32 mb = smem_u32(bar + 1 + (n_iss & 1u)), dst = sDYK + (n_iss & 1u) * KPLANE;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(32768u) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             :: "r"(dst), "l"(tma_src_of(iss_tile, iss_ph)), "r"(32768u), "r"(mb) : "memory");
            }
            iss_advance();
        }
    }
    copy_image_pair(W2B, next_phase(-1));            // group 0's weights -> slot 0 (waited for before its MMAs)
    for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const long long row0 = blk * ROWS + p0;
        // ---- relu(hidden): sign mask for dh + B operand of dW2 ----
        u32 hmask = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            hmask |= (hrow[i].x > 0.f ? 1u : 0u) << (4 * i) | (hrow[i].y > 0.f ? 1u : 0u) << (4 * i + 1) |
                     (hrow[i].z > 0.f ? 1u : 0u) << (4 * i + 2) | (hrow[i].w > 0.f ? 1u : 0u) << (4 * i + 3);
        bool h_staged = false, rh_started = false;
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            if (!a.w.w2[h]) continue;
            const int kd = kdim[h];
            if constexpr (TMA) stage_read(xin, row0);
            float4 w3[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) w3[k] = k < kd ? __ldg(reinterpret_cast<const float4*>(a.w.w3[h] + k * MW + col0)) : make_float4(0.f, 0.f, 0.f, 0.f);
            float din[8][4];
            load_phase_dout(h, din, row0);
            float dz[8][4];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float zz[4] = {xin[i].x, xin[i].y, xin[i].z, xin[i].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float wk[4] = {e == 0 ? w3[0].x : e == 1 ? w3[0].y : e == 2 ? w3[0].z : w3[0].w,
                                         e == 0 ? w3[1].x : e == 1 ? w3[1].y : e == 2 ? w3[1].z : w3[1].w,
                                         e == 0 ? w3[2].x : e == 1 ? w3[2].y : e == 2 ? w3[2].z : w3[2].w,
                                         e == 0 ? w3[3].x : e == 1 ? w3[3].y : e == 2 ? w3[3].z : w3[3].w};
                    float s = din[i][0] * wk[0];
                    s = fmaf(din[i][1], wk[1], s);
                    s = fmaf(din[i][2], wk[2], s);
                    if (kd > 3) s = fmaf(din[i][3], wk[3], s);
                    dz[i][e] = zz[e] > 0.f ? s : 0.f;
                    gB2[h][e] += dz[i][e];
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k < kd) gW3[h][k][e] = fmaf(din[i][k], zz[e], gW3[h][k][e]);
                }
                if (q == 0 && c == 0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) gB3[h][k] += din[i][k];
                }
            }
            if constexpr (!TMA) load_phase_rows(next_phase(h), xin, row0);          // next head's rows, or the feature rows
            prefetch_phase_dout(next_phase(h), blk);                                   // (nothing for the feature phase)
            drain();                 // the previous MMA group still reads DYK / DYM / XH and the W2 slot
            copy_image_pair((ngroup & 1u) ? W2B : W1B, next_phase(h));   // the NEXT group's image -> the slot the drained group used
            if (!h_staged) {
#pragma unroll
                for (int i = 0; i < 8; ++i) sts128(sXH + mn_off + (u32)(p0 + 4 * i) * 128u, tf32x4(hrow[i]));
                h_staged = true;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const u32 pp = (u32)(p0 + 4 * i);
                float4 hi, lo;
                split4(dz[i], hi, lo);
                sts128(sDYM + mn_off + pp * 128u, hi);
                sts128(sDYM + 32768u + mn_off + pp * 128u, lo);
            }
            cp_async_wait<1>();      // all but the next group's image
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            tc_fence_before();
            __syncthreads();
            const bool go = TMA && iss_tile < nblocks;
            issue_group((ngroup & 1u) ? sW1 : sW2, C_RH, rh_started, C_W2 + 64 * h, go, go ? tma_src_of(iss_tile, iss_ph) : nullptr, n_iss & 1u);
            if constexpr (TMA) iss_advance();
            ++ngroup;
            pending = true;
            rh_started = true;
        }
        // ---- dh = d relu(hidden) masked ; d feature = dh W1 ; dW1 += dh^T feature ----
        if constexpr (TMA) stage_read(xin, row0);
        else if (next_phase(-1) == 3) load_rows(xin, a.feat, row0);        // every head disabled: nothing was prefetched
        float4 frow[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) frow[i] = xin[i];
        if (blk + gridDim.x < nblocks) {                              // next tile: relu(hidden) rows and the first phase's inputs
            load_stash(hrow, 0, (blk + gridDim.x) * ROWS + p0);
            if constexpr (!TMA) load_phase_rows(next_phase(-1), xin, (blk + gridDim.x) * ROWS + p0);
            prefetch_phase_dout(next_phase(-1), blk + gridDim.x);
        }
        drain();
        // the next tile's first image -> the slot the drained group used (an empty group keeps the count)
        if (blk + gridDim.x < nblocks) copy_image_pair((ngroup & 1u) ? W2B : W1B, next_phase(-1));
        else cp_async_commit();
        // TMA: the bounce goes through the staging slot the feature rows were just read from (every thread has them in registers
        // once the barrier below has been passed); the next request for that slot is issued after this phase's last barrier
        const u32 sBounce = TMA ? sDYK + ((n_cons - 1u) & 1u) * KPLANE : sDYK;
        if constexpr (TMA) __syncthreads();
        {   // D_RH comes out of TMEM as (lane = point, 32 columns); bounce it through the DYK hi plane to reach the SIMT mapping
            u32 v[32];
            if (rh_started) {
                tmem_ld32(lane_addr + C_RH + 32 * cT, v);
                tmem_wait_ld();
            } else {
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = 0u;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                sts128(sBounce + (u32)(8 * cT + j) * KCH + (u32)pT * 16u,
                       make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])));
        }
        tc_fence_before();
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const u32 pp = (u32)(p0 + 4 * i);
            const float4 r4 = lds128(sBounce + k_off + pp * 16u);
            float x[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                x[e] = (hmask >> (4 * i + e)) & 1u ? x[e] : 0.f;
                gB1[e] += x[e];
            }
            float4 hi, lo;
            split4(x, hi, lo);
            sts128(sDYM + mn_off + pp * 128u, hi);
            sts128(sDYM + 32768u + mn_off + pp * 128u, lo);
            sts128(sXH + mn_off + pp * 128u, tf32x4(frow[i]));
        }
        cp_async_wait<1>();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        __syncthreads();
        const bool go = TMA && iss_tile < nblocks;
        issue_group((ngroup & 1u) ? sW1 : sW2, C_FE, false, C_W1, go, go ? tma_src_of(iss_tile, iss_ph) : nullptr, n_iss & 1u);
        if constexpr (TMA) iss_advance();
        ++ngroup;
        pending = true;
        prev_row = blk * ROWS + pT;
        first_tile = false;
    }
    drain();

    // ---- flush ----
    if (!first_tile) {
        // TMEM-resident weight gradients: lanes 0..63 = out feature from dY_hi, lanes 64..127 the same from dY_lo
        // through shared memory (DYM is free: every MMA has completed), rows padded to 68 floats so that both the
        // lane-per-row 128-bit stores and the row-contiguous 128-bit loads are conflict free; then hi + lo row pairs
        // leave as one 128-bit RED per 4 elements, 512 contiguous bytes per warp.  CTAs start at different matrices /
        // row blocks so that the 148 of them do not all hit the same lines at once.
        constexpr u32 SP = 68 * 4;
        for (int mi = 0; mi < 4; ++mi) {
            const int m = (mi + (int)blockIdx.x) & 3;
            if (m < 3 && !a.w.w2[m]) continue;
            float* dst = m < 3 ? a.gw.w2[m] : a.gw.w1;
            u32 v[32];
            tmem_ld32(lane_addr + (m < 3 ? C_W2 + 64 * m : C_W1) + 32 * cT, v);
            tmem_wait_ld();
            __syncthreads();                                  // the previous matrix has been read out of the staging rows
#pragma unroll
            for (int j = 0; j < 8; ++j)
                sts128(sDYM + (u32)pT * SP + (u32)(32 * cT + 4 * j) * 4u,
                       make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])));
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int idx = tid + BT * ((k + (int)(blockIdx.x >> 2)) & 3);      // 1024 float4 = 64 rows x 16
                const int r = idx >> 4, c4 = idx & 15;
                const float4 x = lds128(sDYM + (u32)r * SP + (u32)c4 * 16u), y = lds128(sDYM + (u32)(r + 64) * SP + (u32)c4 * 16u);
                red_add_v4(dst + r * MW + 4 * c4, x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
            }
        }
        // register-resident partial sums: fold the 4 `sub` lanes, then one atomic per column per warp
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            float s = gB1[e];
            s += __shfl_xor_sync(0xffffffffu, s, 8); s += __shfl_xor_sync(0xffffffffu, s, 16);
            if (sub == 0) atomicAdd(a.gw.b1 + col0 + e, s);
        }
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            if (!a.w.w2[h]) continue;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float s = gB2[h][e];
                s += __shfl_xor_sync(0xffffffffu, s, 8); s += __shfl_xor_sync(0xffffffffu, s, 16);
                if (sub == 0) atomicAdd(a.gw.b2[h] + col0 + e, s);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float t = gW3[h][k][e];
                    t += __shfl_xor_sync(0xffffffffu, t, 8); t += __shfl_xor_sync(0xffffffffu, t, 16);
                    if (sub == 0 && k < kdim[h]) atomicAdd(a.gw.w3[h] + k * MW + col0 + e, t);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float s = gB3[h][k];                     // non-zero only in lanes with q == 0 of the c == 0 warps
                s += __shfl_xor_sync(0xffffffffu, s, 8); s += __shfl_xor_sync(0xffffffffu, s, 16);
                if (lane == 0 && c == 0 && k < kdim[h]) atomicAdd(a.gw.b3[h] + k, s);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, 512);
}

size_t bwd_smem() { return (size_t)(2 * MW * MW + 2 * MW * MW) * 4 + 98304 + 2 * KPLANE + 64; }

}  // namespace tc5

int deform_mlp_backward_tc5(const b200gs_mlp_weights* w, const b200gs_mlp_grads* gw, long long P, const float* feat,
                            const float* saved, const float* d_pts, const float* d_scales, const float* d_rot,
                            float* d_feat, cudaStream_t stream)
{
    // the weight gradients leave as 128-bit REDs (see the flush above): W1 / W2 gradient rows must be 16-byte aligned
    bool aligned = ((uintptr_t)gw->w1 & 15) == 0;
    for (int h = 0; h < 3; ++h) aligned = aligned && (!w->w2[h] || ((uintptr_t)gw->w2[h] & 15) == 0);
    if (!aligned) { set_error("deform_mlp_backward: gw->w1 / gw->w2 must be 16-byte aligned"); return -1; }
    tc5::BwdArgs a;
    a.w = *w; a.gw = *gw; a.P = P; a.feat = feat; a.saved = saved; a.d_pts = d_pts; a.d_scales = d_scales; a.d_rot = d_rot;
    a.d_feat = d_feat; a.dy_sbo = 512u;
    const int grid = tc5::persistent_grid(P, g_opt_mlp_bwd_sms);
    const size_t smem = tc5::bwd_smem();
    // the TMA staging needs the tiled feature layout (one contiguous 32 KB tile per phase)
    void (*kern)(tc5::BwdArgs) = w->feat_tiled ? tc5::deform_mlp_bwd_tc5_kernel<true> : tc5::deform_mlp_bwd_tc5_kernel<false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, tc5::BT, smem, stream>>>(a);
    return check_launch("deform_mlp_backward(tcgen05)");
}

}  // namespace b200gs
