// Deformation MLP forward on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same function as the mma.sync forward it replaces (see deform_mlp.cu for the maths and the
// reference citations): hidden = Linear(F,64)(feature); three heads ReLU-Linear(64,64)-ReLU-Linear(64,k).
// One CTA (128 threads = one warpgroup) walks 128-point tiles:
//   * thread r of the CTA owns point r of the tile = TMEM lane r;
//   * activations live in TMEM as the A operand (lane = point, column = feature), written with
//     tcgen05.st after bias / ReLU / TF32 hi-lo split, so no activation ever touches shared memory;
//   * weights live in shared memory as K-major, un-swizzled UMMA operands (8-row x 16-byte core
//     matrices), pre-split into hi and lo TF32 copies once per CTA;
//   * every contraction is issued by ONE thread as 3 x (K/8) tcgen05.mma.kind::tf32 instructions
//     (lo*hi + hi*lo + hi*hi, FP32 accumulation in TMEM: ~FP32 accuracy, the reference computes in
//     true FP32), completion is signalled through tcgen05.commit -> mbarrier;
//   * the epilogue reads the accumulator with tcgen05.ld (32 lanes x 32 bit, 32 columns at a time).
// TMEM columns: [0, 2F) feature hi|lo, re-used as relu(hidden) hi [0,64) | lo [64,128);
//               [2F, 2F+128) relu(z) hi|lo; [2F+128, +64) accumulator; [2F+192, +16) head output.
#include "tc5_common.cuh"
#include "../../include/b200gs.h"

namespace b200gs {

namespace tc5 {

constexpr int NT = 128;            // threads per CTA

struct FwdArgs {
    b200gs_mlp_weights w;
    long long P;
    const float* feat; const float* xyz; const float* scales; const float* rot; const float* scene_flow;
    float frame_num, delta_scale;
    const float* frame_num_dev;
    float* pts_out; float* scales_out; float* rot_out;
    float* saved;                 // [4][P][64] row-major: relu(hidden), relu(z_pos), relu(z_scale), relu(z_rot)
};

template <int F>
__global__ void __launch_bounds__(NT, 1) deform_mlp_fwd_tc5_kernel(const __grid_constant__ FwdArgs a)
{
    extern __shared__ __align__(1024) float smem[];
    float* W1h = smem;                         // [F/4][64][4]
    float* W1l = W1h + MW * F;
    float* W2h = W1l + MW * F;                 // [3][16][64][4]
    float* W2l = W2h + 3 * MW * MW;
    float* W3h = W2l + 3 * MW * MW;            // [3][16][16][4]  (N padded to 16)
    float* W3l = W3h + 3 * 16 * MW;
    float* bias = W3l + 3 * 16 * MW;           // b1[64] b2[3][64] b3[3][16]
    u64* bar = reinterpret_cast<u64*>(bias + 4 * MW + 48);
    u32* tmem_slot = reinterpret_cast<u32*>(bar + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int kdim[3] = {3, 3, 4};

    stage_kmajor<NT>(W1h, W1l, a.w.w1, MW, MW, F);
    for (int i = tid; i < MW; i += NT) bias[i] = __ldg(a.w.b1 + i);
    for (int h = 0; h < 3; ++h) {
        if (!a.w.w2[h]) continue;
        stage_kmajor<NT>(W2h + h * MW * MW, W2l + h * MW * MW, a.w.w2[h], MW, MW, MW);
        stage_kmajor<NT>(W3h + h * 16 * MW, W3l + h * 16 * MW, a.w.w3[h], 16, kdim[h], MW);
        for (int i = tid; i < MW; i += NT) bias[MW + h * MW + i] = __ldg(a.w.b2[h] + i);
        if (tid < 16) bias[4 * MW + h * 16 + tid] = tid < kdim[h] ? __ldg(a.w.b3[h] + tid) : 0.f;
    }
    if (F == 64 && blockIdx.x == 0) {           // transposed TF32 weight images for the tcgen05 backward (see tc5_common.cuh)
        float* images = a.saved + 4 * stash_plane_floats(a.P);
        for (int h = 0; h < 3; ++h)
            if (a.w.w2[h]) write_bwd_weight_image(images, h, a.w.w2[h], NT);
        write_bwd_weight_image(images, 3, a.w.w1, NT);
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    // make the generic-proxy weight writes visible to the tensor-core (async) proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tbase = *tmem_slot;
    const u32 lane_addr = tbase + ((u32)(warp * 32) << 16);     // this warp's 32 TMEM lanes
    constexpr u32 C_H_HI = 0, C_H_LO = 64, C_FE_LO = F, C_Z_HI = 2 * F, C_Z_LO = 2 * F + 64, C_D = 2 * F + 128, C_D3 = 2 * F + 192;
    const u32 idesc64 = make_idesc(128, 64), idesc16 = make_idesc(128, 16);
    u32 phase = 0;

    const long long nblocks = (a.P + ROWS - 1) / ROWS;
    for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const long long r = blk * ROWS + tid;
        const bool valid = r < a.P;
        // ---- features -> TMEM (hi | lo) ----
#pragma unroll
        for (int c = 0; c < F / 32; ++c) {
            u32 hi[32], lo[32];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 v = valid ? __ldg(reinterpret_cast<const float4*>(a.feat + (a.w.feat_tiled ? stash_off(r, 32 * c + 4 * q) : (size_t)r * F + 32 * c + 4 * q))) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) { hi[4 * q + e] = to_tf32(x[e]); lo[4 * q + e] = to_tf32(x[e] - __uint_as_float(hi[4 * q + e])); }
            }
            tmem_st32(lane_addr + 32 * c, hi);
            tmem_st32(lane_addr + C_FE_LO + 32 * c, lo);
        }
        tmem_wait_st();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_layer(tbase + C_D, tbase, tbase + C_FE_LO, smem_u32(W1h), smem_u32(W1l), MW, F, idesc64);
            tc_commit(bar);
        }
        mbar_wait(bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- hidden: bias, ReLU, stash, split, back to TMEM as the next A operand ----
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            u32 v[32], lo[32];
            tmem_ld32(lane_addr + C_D + 32 * c, v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const float x = fmaxf(__uint_as_float(v[e]) + bias[32 * c + e], 0.f);
                v[e] = __float_as_uint(x);
            }
            if (valid) {
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    *reinterpret_cast<float4*>(a.saved + stash_off(r, 32 * c + 4 * q)) =
                        make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const float x = __uint_as_float(v[e]);
                v[e] = to_tf32(x);
                lo[e] = to_tf32(x - __uint_as_float(v[e]));
            }
            tmem_st32(lane_addr + C_H_HI + 32 * c, v);
            tmem_st32(lane_addr + C_H_LO + 32 * c, lo);
        }
        tmem_wait_st();
        tc_fence_before();
        __syncthreads();
        // ---- heads ----
        for (int h = 0; h < 3; ++h) {
            const int kd = kdim[h];
            if (!a.w.w2[h]) {            // head disabled (no_dx / no_ds / no_dr): pass through
                if (valid) {
                    const float* src = h == 0 ? a.xyz : (h == 1 ? a.scales : a.rot);
                    float* dst = h == 0 ? a.pts_out : (h == 1 ? a.scales_out : a.rot_out);
                    for (int c = 0; c < kd; ++c) dst[(size_t)r * kd + c] = __ldg(src + (size_t)r * kd + c);
                }
                continue;
            }
            if (tid == 0) {
                tc_fence_after();
                issue_layer(tbase + C_D, tbase + C_H_HI, tbase + C_H_LO, smem_u32(W2h + h * MW * MW), smem_u32(W2l + h * MW * MW), MW, MW, idesc64);
                tc_commit(bar);
            }
            mbar_wait(bar, phase); phase ^= 1;
            tc_fence_after();
            float* sv = a.saved + (size_t)(1 + h) * stash_plane_floats(a.P);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                u32 v[32], lo[32];
                tmem_ld32(lane_addr + C_D + 32 * c, v);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(fmaxf(__uint_as_float(v[e]) + bias[MW + h * MW + 32 * c + e], 0.f));
                if (valid) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<float4*>(sv + stash_off(r, 32 * c + 4 * q)) =
                            make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
                }
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const float x = __uint_as_float(v[e]);
                    v[e] = to_tf32(x);
                    lo[e] = to_tf32(x - __uint_as_float(v[e]));
                }
                tmem_st32(lane_addr + C_Z_HI + 32 * c, v);
                tmem_st32(lane_addr + C_Z_LO + 32 * c, lo);
            }
            tmem_wait_st();
            tc_fence_before();
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                issue_layer(tbase + C_D3, tbase + C_Z_HI, tbase + C_Z_LO, smem_u32(W3h + h * 16 * MW), smem_u32(W3l + h * 16 * MW), 16, MW, idesc16);
                tc_commit(bar);
            }
            mbar_wait(bar, phase); phase ^= 1;
            tc_fence_after();
            u32 o[16];
            tmem_ld16(lane_addr + C_D3, o);
            tmem_wait_ld();
            if (valid) {
                const float fn = a.frame_num_dev ? __ldg(a.frame_num_dev) : a.frame_num;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c >= kd) continue;
                    const float ov = __uint_as_float(o[c]) + bias[4 * MW + h * 16 + c];
                    if (h == 0) {
                        const float flow = __fmul_rn(a.delta_scale, __fmul_rn(fn, __ldg(a.scene_flow + 3 * r + c)));
                        a.pts_out[3 * r + c] = __fadd_rn(__fmul_rn(__ldg(a.xyz + 3 * r + c), 1.0f), __fadd_rn(ov, flow));
                    } else if (h == 1) {
                        a.scales_out[3 * r + c] = __fadd_rn(__fmul_rn(__ldg(a.scales + 3 * r + c), 1.0f), ov);
                    } else {
                        a.rot_out[4 * r + c] = __fadd_rn(__ldg(a.rot + 4 * r + c), ov);
                    }
                }
            }
            // all reads of this head's accumulators are done before the next MMA overwrites them
            tc_fence_before();
            __syncthreads();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, 512);
}

// ---------------------------------------------------------------------------------------------
// v2: same maths and TMEM / shared-memory operands as the kernel above, but pipelined inside a tile.
//   * 256 threads: warp w reads / writes the TMEM lanes of quarter w & 3 (lane = point) and the 32-column
//     half w >> 2 of every 64-wide accumulator, so each epilogue is half as long per thread;
//   * every MMA group has its own mbarrier (one completion per tile, parity = tile parity), so several
//     groups are in flight: the three heads' 64x64 layers are issued ahead of the epilogues
//     (L2_0, L2_1 | L3_0, L2_2 | L3_1 | L3_2), the tensor pipe works through them while the threads
//     run bias / ReLU / stash / split for the head before;
//   * the next tile's feature rows and this tile's xyz / scales / rotations / scene_flow are fetched into
//     registers while the first layer's MMAs run.
// Requires all three heads enabled (the reference's configuration); otherwise the kernel above is used.
// TMEM columns: A0 [0, 2F) feature hi|lo, then relu(hidden) hi [0,64) | lo [64,128); Z [128,256) relu(z) hi|lo
// (F = 128: the feature lo half overlaps Z, it is dead once layer 1 has completed); D2 [256,448) the three
// heads' accumulators (layer 1 accumulates into the first 64 of them); D3 [448,496) the head outputs.
constexpr int NT2 = 256;

// The MMAs are issued from a warp-uniform branch by the elected lane of warp 0 (tc5_common.cuh elect_one): `if (tid == 0)`
// makes the compiler wrap every tcgen05.mma in an ELECT / BRA.U.ANY loop.  The activation-stash stores of a layer are issued
// AFTER the next layer's MMAs have been started: they are not on the MMA -> epilogue -> MMA chain, the values just stay in
// registers a little longer.  Neither changes a computed value (same MMAs in the same order, the same stores later); for
// F = 128 they took the forward from 498 to 405 us per 1M points (B200, 1000 W power limit, tools/time_mlp.py MULTIRES=1,2,4,8).
template <int F>
__global__ void __launch_bounds__(NT2, 1) deform_mlp_fwd_tc5v2_kernel(const __grid_constant__ FwdArgs a)
{
    extern __shared__ __align__(1024) float smem[];
    float* W1h = smem;                         // [F/4][64][4]
    float* W1l = W1h + MW * F;
    float* W2h = W1l + MW * F;                 // [3][16][64][4]
    float* W2l = W2h + 3 * MW * MW;
    float* W3h = W2l + 3 * MW * MW;            // [3][16][16][4]  (N padded to 16)
    float* W3l = W3h + 3 * 16 * MW;
    float* bias = W3l + 3 * 16 * MW;           // b1[64] b2[3][64] b3[3][16]
    u64* bars = reinterpret_cast<u64*>(bias + 4 * MW + 48);     // [0] L1, [1..3] L2_h, [4..6] L3_h
    u32* tmem_slot = reinterpret_cast<u32*>(bars + 7);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int pT = (warp & 3) * 32 + lane, cT = warp >> 2;
    const int kdim[3] = {3, 3, 4};

    stage_kmajor<NT2>(W1h, W1l, a.w.w1, MW, MW, F);
    for (int i = tid; i < MW; i += NT2) bias[i] = __ldg(a.w.b1 + i);
    for (int h = 0; h < 3; ++h) {
        stage_kmajor<NT2>(W2h + h * MW * MW, W2l + h * MW * MW, a.w.w2[h], MW, MW, MW);
        stage_kmajor<NT2>(W3h + h * 16 * MW, W3l + h * 16 * MW, a.w.w3[h], 16, kdim[h], MW);
        for (int i = tid; i < MW; i += NT2) bias[MW + h * MW + i] = __ldg(a.w.b2[h] + i);
        if (tid < 16) bias[4 * MW + h * 16 + tid] = tid < kdim[h] ? __ldg(a.w.b3[h] + tid) : 0.f;
    }
    // a.saved == nullptr: inference (no backward will follow) -- nothing is stashed, 1 KB per point less HBM traffic
    const bool stash_on = a.saved != nullptr;
    if (F == 64 && blockIdx.x == 0 && stash_on) {           // transposed TF32 weight images for the tcgen05 backward (see tc5_common.cuh)
        float* images = a.saved + 4 * stash_plane_floats(a.P);
        for (int h = 0; h < 3; ++h) write_bwd_weight_image(images, h, a.w.w2[h], NT2);
        write_bwd_weight_image(images, 3, a.w.w1, NT2);
    }
    if (tid == 0) {
        for (int i = 0; i < 7; ++i) mbar_init(bars + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tbase = *tmem_slot;
    const u32 lane_addr = tbase + ((u32)((warp & 3) * 32) << 16);
    constexpr u32 C_H_HI = 0, C_H_LO = 64, C_FE_LO = F, C_Z_HI = 128, C_Z_LO = 192, C_D2 = 256, C_D3 = 448;
    constexpr int FH = F / 2;                  // feature columns per thread
    const u32 idesc64 = make_idesc(128, 64), idesc16 = make_idesc(128, 16);
    u32 parity = 0;

    auto sync_then = [&]() { tmem_wait_st(); tc_fence_before(); __syncthreads(); };
    // the thread that issues the MMAs; every call site follows a block barrier, so warp 0 is converged for elect.sync
    auto issuer = [&]() -> bool { return warp == 0 && elect_one(); };
    // epilogue of one 64-wide layer for this thread's 32 columns: bias, ReLU, split; returns hi / lo in v / lo
    auto layer_epilogue = [&](u32 d_col, const float* b, u32* v, u32* lo) {
        tmem_ld32(lane_addr + d_col + 32 * cT, v);
        tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(fmaxf(__uint_as_float(v[e]) + b[32 * cT + e], 0.f));
#pragma unroll
        for (int e = 0; e < 32; ++e) lo[e] = __float_as_uint(tf32_lo(__uint_as_float(v[e])));      // hi = the raw value (hardware truncates)
    };
    auto deferred_stash = [&](float* stash_plane, long long row, bool valid, const u32* v) {
        if (valid && stash_on) {
            float* dst = stash_plane + stash_off(row, 32 * cT);          // this thread's 8 chunks are 16 floats apart
#pragma unroll
            for (int j = 0; j < 8; ++j)
                *reinterpret_cast<float4*>(dst + 16 * j) =
                    make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
    };

    const long long nblocks = (a.P + ROWS - 1) / ROWS;
    float4 fr[FH / 4];                          // this thread's half of its point's feature row
    {
        const long long r = (long long)blockIdx.x * ROWS + pT;
#pragma unroll
        for (int j = 0; j < FH / 4; ++j)
            fr[j] = (blockIdx.x < nblocks && r < a.P) ? __ldg(reinterpret_cast<const float4*>(a.feat + (a.w.feat_tiled ? stash_off(r, FH * cT) + 16 * j : (size_t)r * F + FH * cT + 4 * j))) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const long long r = blk * ROWS + pT;
        const bool valid = r < a.P;
        // ---- features -> TMEM (hi | lo) ----
#pragma unroll
        for (int c = 0; c < FH / 32; ++c) {
            u32 hi[32], lo[32];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float x[4] = {fr[8 * c + j].x, fr[8 * c + j].y, fr[8 * c + j].z, fr[8 * c + j].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) { hi[4 * j + e] = __float_as_uint(x[e]); lo[4 * j + e] = __float_as_uint(tf32_lo(x[e])); }
            }
            tmem_st32(lane_addr + FH * cT + 32 * c, hi);
            tmem_st32(lane_addr + C_FE_LO + FH * cT + 32 * c, lo);
        }
        sync_then();
        if (issuer()) {
            tc_fence_after();
            issue_layer(tbase + C_D2, tbase, tbase + C_FE_LO, smem_u32(W1h), smem_u32(W1l), MW, F, idesc64);
            tc_commit(bars + 0);
        }
        // while layer 1 runs: next tile's features, this tile's pass-through inputs
        {
            const long long rn = (blk + gridDim.x) * ROWS + pT;
            const bool vn = blk + gridDim.x < nblocks && rn < a.P;
#pragma unroll
            for (int j = 0; j < FH / 4; ++j)
                fr[j] = vn ? __ldg(reinterpret_cast<const float4*>(a.feat + (a.w.feat_tiled ? stash_off(rn, FH * cT) + 16 * j : (size_t)rn * F + FH * cT + 4 * j))) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float in_x[3] = {0.f, 0.f, 0.f}, in_s[3] = {0.f, 0.f, 0.f}, in_r[4] = {0.f, 0.f, 0.f, 0.f}, in_f[3] = {0.f, 0.f, 0.f};
        if (valid && cT == 0) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                in_x[c] = __ldg(a.xyz + 3 * r + c); in_s[c] = __ldg(a.scales + 3 * r + c); in_f[c] = __ldg(a.scene_flow + 3 * r + c);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) in_r[c] = __ldg(a.rot + 4 * r + c);
        }
        u32 v[32], lo[32];
        // ---- hidden ----
        mbar_wait(bars + 0, parity);
        tc_fence_after();
        layer_epilogue(C_D2, bias, v, lo);
        tmem_st32(lane_addr + C_H_HI + 32 * cT, v);
        tmem_st32(lane_addr + C_H_LO + 32 * cT, lo);
        sync_then();
        if (issuer()) {
            tc_fence_after();
            issue_layer(tbase + C_D2, tbase + C_H_HI, tbase + C_H_LO, smem_u32(W2h), smem_u32(W2l), MW, MW, idesc64);
            tc_commit(bars + 1);
            issue_layer(tbase + C_D2 + 64, tbase + C_H_HI, tbase + C_H_LO, smem_u32(W2h + MW * MW), smem_u32(W2l + MW * MW), MW, MW, idesc64);
            tc_commit(bars + 2);
        }
        deferred_stash(a.saved, r, valid, v);
        // ---- heads ----
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            mbar_wait(bars + 1 + h, parity);
            tc_fence_after();
            layer_epilogue(C_D2 + 64 * h, bias + MW + h * MW, v, lo);
            if (h > 0) {                         // the previous head's last layer still reads Z
                mbar_wait(bars + 4 + (h - 1), parity);
                tc_fence_after();
            }
            tmem_st32(lane_addr + C_Z_HI + 32 * cT, v);
            tmem_st32(lane_addr + C_Z_LO + 32 * cT, lo);
            sync_then();
            if (issuer()) {
                tc_fence_after();
                issue_layer(tbase + C_D3 + 16 * h, tbase + C_Z_HI, tbase + C_Z_LO, smem_u32(W3h + h * 16 * MW), smem_u32(W3l + h * 16 * MW), 16, MW, idesc16);
                tc_commit(bars + 4 + h);
                if (h == 0) {
                    issue_layer(tbase + C_D2 + 128, tbase + C_H_HI, tbase + C_H_LO, smem_u32(W2h + 2 * MW * MW), smem_u32(W2l + 2 * MW * MW), MW, MW, idesc64);
                    tc_commit(bars + 3);
                }
            }
            deferred_stash(a.saved + (size_t)(1 + h) * stash_plane_floats(a.P), r, valid, v);
        }
        // ---- outputs ----
        mbar_wait(bars + 6, parity);
        tc_fence_after();
        if (cT == 0) {
            u32 o[16];
            const float fn = a.frame_num_dev ? __ldg(a.frame_num_dev) : a.frame_num;
            tmem_ld16(lane_addr + C_D3, o);
            tmem_wait_ld();
            if (valid) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float ov = __uint_as_float(o[c]) + bias[4 * MW + c];
                    const float flow = __fmul_rn(a.delta_scale, __fmul_rn(fn, in_f[c]));
                    a.pts_out[3 * r + c] = __fadd_rn(__fmul_rn(in_x[c], 1.0f), __fadd_rn(ov, flow));
                }
            }
            tmem_ld16(lane_addr + C_D3 + 16, o);
            tmem_wait_ld();
            if (valid) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    a.scales_out[3 * r + c] = __fadd_rn(__fmul_rn(in_s[c], 1.0f), __uint_as_float(o[c]) + bias[4 * MW + 16 + c]);
            }
            tmem_ld16(lane_addr + C_D3 + 32, o);
            tmem_wait_ld();
            if (valid) {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    a.rot_out[4 * r + c] = __fadd_rn(in_r[c], __uint_as_float(o[c]) + bias[4 * MW + 32 + c]);
            }
        }
        parity ^= 1;
        // the next tile's feature stores overwrite A0 / Z: every MMA of this tile has completed (bars[6] is the last
        // commit), and its D3 reads above are ordered before the next tile's layer-3 MMAs by the syncs in between
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, 512);
}

size_t fwd_smem(int F) { return (size_t)(2 * MW * F + 6 * MW * MW + 6 * 16 * MW + 4 * MW + 48) * sizeof(float) + 128; }

}  // namespace tc5

int deform_mlp_forward_tc5(const b200gs_mlp_weights* w, long long P, const float* feat, const float* xyz,
                           const float* scales, const float* rot, const float* scene_flow, float frame_num,
                           const float* frame_num_dev, float delta_scale, float* pts_out, float* scales_out,
                           float* rot_out, float* saved, cudaStream_t stream)
{
    tc5::FwdArgs a;
    a.w = *w; a.P = P; a.feat = feat; a.xyz = xyz; a.scales = scales; a.rot = rot; a.scene_flow = scene_flow;
    a.frame_num = frame_num; a.frame_num_dev = frame_num_dev; a.delta_scale = delta_scale; a.pts_out = pts_out;
    a.scales_out = scales_out; a.rot_out = rot_out; a.saved = saved;
    const int grid = tc5::persistent_grid(P, g_opt_mlp_fwd_sms);
    const size_t smem = tc5::fwd_smem(w->feat_dim);
    if (!saved && !(w->w2[0] && w->w2[1] && w->w2[2])) {
        set_error("deform_mlp_forward: saved == NULL (inference, nothing stashed) needs all three heads enabled");
        return -1;
    }
    if (w->w2[0] && w->w2[1] && w->w2[2]) {          // all heads on (the reference's configuration): pipelined kernel
        if (w->feat_dim == 64) {
            cudaFuncSetAttribute(tc5::deform_mlp_fwd_tc5v2_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            tc5::deform_mlp_fwd_tc5v2_kernel<64><<<grid, tc5::NT2, smem, stream>>>(a);
        } else {
            cudaFuncSetAttribute(tc5::deform_mlp_fwd_tc5v2_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            tc5::deform_mlp_fwd_tc5v2_kernel<128><<<grid, tc5::NT2, smem, stream>>>(a);
        }
        return check_launch("deform_mlp_forward(tcgen05 v2)");
    }
    if (w->feat_dim == 64) {
        cudaFuncSetAttribute(tc5::deform_mlp_fwd_tc5_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        tc5::deform_mlp_fwd_tc5_kernel<64><<<grid, tc5::NT, smem, stream>>>(a);
    } else {
        cudaFuncSetAttribute(tc5::deform_mlp_fwd_tc5_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        tc5::deform_mlp_fwd_tc5_kernel<128><<<grid, tc5::NT, smem, stream>>>(a);
    }
    return check_launch("deform_mlp_forward(tcgen05)");
}

}  // namespace b200gs
