// Opacity and SH deformation heads (no_do = False, no_dshs = False), sm_100a.
//
// scene/deformation.py:97-153 (forward_dynamic) with mask = ones:
//     opacity' = opacity[:, :1] * 1 + Linear(64,1)(ReLU(Linear(64,64)(ReLU(hidden))))
//     shs'     = shs * 1 + Linear(64,48)(ReLU(Linear(64,64)(ReLU(hidden)))).reshape(P, 16, 3)
// `hidden` is the same feature_out output the three geometry heads read.  These kernels run BESIDE the three-head kernels
// (deform_mlp_tc5.cu / deform_mlp_bwd_tc5.cu / deform_mlp.cu), which stay untouched: the forward reads relu(hidden) from
// plane 0 of the activation stash the three-head forward left, and the backward ADDS the two heads' share into the
// d_features / dW1 / db1 the three-head backward has just written (the ReLU mask of hidden is linear in the upstream
// gradient, so d_h = mask * (sum of every head's d relu(h)) splits into one term per group of heads).
//
// Forward: tcgen05, one CTA of 128 threads (thread = point = TMEM lane) per 128-point tile, both heads' layers issued
// together.  Every contraction is the three-term TF32 split (lo*hi + hi*lo + hi*hi) with FP32 accumulation in TMEM.
// TMEM columns: A = relu(hidden) hi [0,64) | lo [64,128), dead after layer 2 and re-used for the layer-3 accumulators
// (opacity [0,16), SH [64,112)); D2 [128,256) the two heads' layer-2 accumulators; Z [256,512) relu(z) hi|lo per head.
//
// Backward: the register-resident mma.sync structure of deform_mlp.cu's backward (each warp carries 16 points through the
// whole chain; weight gradients accumulate in fragments over every tile of a persistent CTA and are flushed once).  Same
// rounding rules as the three-head backwards: the dX chain runs the full three-term split, dY stays exact (hi + lo) in the
// weight gradients, X is rounded to TF32 once, bias gradients are FP32 sums.
#include "mma_tf32.cuh"
#include "../../include/b200gs.h"

namespace b200gs {
namespace heads {

using tc5::MW; using tc5::ROWS; using tc5::stash_off; using tc5::stash_plane_floats;
__host__ __device__ constexpr int KD(int h) { return h == 0 ? 1 : 48; }     // outputs of the opacity / SH head
__host__ __device__ constexpr int N3(int h) { return h == 0 ? 16 : 48; }    // their UMMA N (padded to a multiple of 16)

// ---------------------------------------------------------------------------------------------
// forward (tcgen05)
constexpr int FT = 128;

struct FwdArgs {
    b200gs_heads_weights w;
    long long P;
    const float* hidden;                  // plane 0 of the three-head stash: relu(hidden), tiled
    const float* opacity; const float* shs;
    float* opacity_out; float* shs_out;
    float* saved;                         // 2 planes: relu(z_opacity), relu(z_sh); null = inference
};

__global__ void __launch_bounds__(FT, 1) deform_heads_fwd_kernel(const __grid_constant__ FwdArgs a)
{
    using namespace tc5;
    extern __shared__ __align__(1024) float smem[];
    float* W2h = smem;                        // [2][16][64][4]
    float* W2l = W2h + 2 * MW * MW;
    float* W3h = W2l + 2 * MW * MW;           // [2][16][48][4] (opacity: N = 16)
    float* W3l = W3h + 2 * 48 * MW;
    float* bias = W3l + 2 * 48 * MW;          // b2[2][64], b3[2][48]
    u64* bar = reinterpret_cast<u64*>(bias + 2 * MW + 96);
    u32* tmem_slot = reinterpret_cast<u32*>(bar + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    const bool on[2] = {a.w.w2[0] != nullptr, a.w.w2[1] != nullptr};

    for (int h = 0; h < 2; ++h) {
        if (!on[h]) continue;
        stage_kmajor<FT>(W2h + h * MW * MW, W2l + h * MW * MW, a.w.w2[h], MW, MW, MW);
        stage_kmajor<FT>(W3h + h * 48 * MW, W3l + h * 48 * MW, a.w.w3[h], N3(h), KD(h), MW);
        for (int i = tid; i < MW; i += FT) bias[h * MW + i] = __ldg(a.w.b2[h] + i);
        for (int i = tid; i < KD(h); i += FT) bias[2 * MW + h * 48 + i] = __ldg(a.w.b3[h] + i);
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tbase = *tmem_slot;
    const u32 lane_addr = tbase + ((u32)(warp * 32) << 16);
    constexpr u32 C_A_LO = 64, C_D2 = 128, C_Z = 256;
    const u32 c_d3[2] = {0, 64};
    u32 phase = 0;
    auto sync_then = [&]() { tmem_wait_st(); tc_fence_before(); __syncthreads(); };
    auto issuer = [&]() -> bool { return warp == 0 && elect_one(); };

    const long long nblocks = (a.P + ROWS - 1) / ROWS;
    for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const long long r = blk * ROWS + tid;
        const bool valid = r < a.P;
        // ---- relu(hidden) -> TMEM (hi | lo) ----
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            u32 hi[32], lo[32];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 v = valid ? __ldg(reinterpret_cast<const float4*>(a.hidden + stash_off(r, 32 * c + 4 * q))) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) { hi[4 * q + e] = __float_as_uint(x[e]); lo[4 * q + e] = __float_as_uint(tf32_lo(x[e])); }
            }
            tmem_st32(lane_addr + 32 * c, hi);
            tmem_st32(lane_addr + C_A_LO + 32 * c, lo);
        }
        sync_then();
        if (issuer()) {
            tc_fence_after();
            for (int h = 0; h < 2; ++h)
                if (on[h]) issue_layer(tbase + C_D2 + 64 * h, tbase, tbase + C_A_LO, smem_u32(W2h + h * MW * MW), smem_u32(W2l + h * MW * MW), MW, MW, make_idesc(128, MW));
            tc_commit(bar);
        }
        mbar_wait(bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- relu(z): bias, ReLU, stash, split into Z ----
        for (int h = 0; h < 2; ++h) {
            if (!on[h]) continue;
            float* sv = a.saved ? a.saved + (size_t)h * stash_plane_floats(a.P) : nullptr;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                u32 v[32], lo[32];
                tmem_ld32(lane_addr + C_D2 + 64 * h + 32 * c, v);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const float x = fmaxf(__uint_as_float(v[e]) + bias[h * MW + 32 * c + e], 0.f);
                    v[e] = __float_as_uint(x);
                    lo[e] = __float_as_uint(tf32_lo(x));
                }
                tmem_st32(lane_addr + C_Z + 128 * h + 32 * c, v);
                tmem_st32(lane_addr + C_Z + 128 * h + 64 + 32 * c, lo);
                if (valid && sv) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<float4*>(sv + stash_off(r, 32 * c + 4 * q)) =
                            make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
                }
            }
        }
        sync_then();
        if (issuer()) {
            tc_fence_after();
            for (int h = 0; h < 2; ++h)
                if (on[h]) issue_layer(tbase + c_d3[h], tbase + C_Z + 128 * h, tbase + C_Z + 128 * h + 64,
                                       smem_u32(W3h + h * 48 * MW), smem_u32(W3l + h * 48 * MW), N3(h), MW, make_idesc(128, N3(h)));
            tc_commit(bar);
        }
        mbar_wait(bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- outputs: x * 1 + (head + b3) ----
        if (on[0]) {
            u32 o[16];
            tmem_ld16(lane_addr + c_d3[0], o);
            tmem_wait_ld();
            if (valid)
                a.opacity_out[r] = __fadd_rn(__fmul_rn(__ldg(a.opacity + r), 1.0f), __uint_as_float(o[0]) + bias[2 * MW]);
        }
        if (on[1]) {
            u32 o[48];
            tmem_ld32(lane_addr + c_d3[1], o);
            tmem_ld16(lane_addr + c_d3[1] + 32, o + 32);
            tmem_wait_ld();
            if (valid) {
                const float4* src = reinterpret_cast<const float4*>(a.shs + 48 * r);
                float4* dst = reinterpret_cast<float4*>(a.shs_out + 48 * r);
#pragma unroll
                for (int q = 0; q < 12; ++q) {
                    const float4 s = __ldg(src + q);
                    const float x[4] = {s.x, s.y, s.z, s.w};
                    float y[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        y[e] = __fadd_rn(__fmul_rn(x[e], 1.0f), __uint_as_float(o[4 * q + e]) + bias[2 * MW + 48 + 4 * q + e]);
                    dst[q] = make_float4(y[0], y[1], y[2], y[3]);
                }
            }
        }
        // the next tile's A stores overwrite the layer-3 accumulators read above
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, 512);
}

constexpr size_t FWD_SMEM = (size_t)(4 * MW * MW + 4 * 48 * MW + 2 * MW + 96) * sizeof(float) + 128;

// ---------------------------------------------------------------------------------------------
// backward (mma.sync)
constexpr int BT = 256;                   // 8 warps x 16 points
constexpr int LDS_T = MW + 8;             // row stride of the dz / d_h tile (conflict-free fragment loads)
constexpr int LDO = 48 + 8;               // row stride of the upstream-gradient tile
constexpr int RS2 = MW / 2 + 4;           // float4 row stride of a K = 64 operand
using tf32::split; using tf32::mma; using tf32::kstep;

// acc[m][n] (16 out x 8 in) += sum over the tile's rows of dY[row][16 (m0+m) + .] * tf32(X[row][8 (n0+n) + .]);
// dY from a row-major smem tile (stride lds; out rows >= n_out are zero), X from global memory (stash tiles or row-major).
template <int NM, int NN, bool TILED>
__device__ __forceinline__ void dw_accumulate(float (*acc)[NN][4], const float* __restrict__ dYs, int lds, int m0, int n_out,
                                              const float* __restrict__ X, size_t ldx, long long row0, long long P, int n0, int g, int t)
{
#pragma unroll 2
    for (int ks = 0; ks < ROWS / 8; ++ks) {
        const int r0 = 8 * ks + t, r1 = r0 + 4;
        const bool v0 = row0 + r0 < P, v1 = row0 + r1 < P;
        u32 b0[NN], b1[NN];
#pragma unroll
        for (int n = 0; n < NN; ++n) {
            const int col = 8 * (n0 + n) + g;
            b0[n] = tc5::to_tf32(v0 ? __ldg(X + (TILED ? stash_off(row0 + r0, col) : (size_t)(row0 + r0) * ldx + col)) : 0.f);
            b1[n] = tc5::to_tf32(v1 ? __ldg(X + (TILED ? stash_off(row0 + r1, col) : (size_t)(row0 + r1) * ldx + col)) : 0.f);
        }
#pragma unroll
        for (int m = 0; m < NM; ++m) {
            const int o = 16 * (m0 + m) + g;
            const bool hi_ok = o + 8 < n_out;
            const float af[4] = {dYs[r0 * lds + o], hi_ok ? dYs[r0 * lds + o + 8] : 0.f,
                                 dYs[r1 * lds + o], hi_ok ? dYs[r1 * lds + o + 8] : 0.f};
            u32 ahi[4], alo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) split(af[i], ahi[i], alo[i]);
#pragma unroll
            for (int n = 0; n < NN; ++n) mma(acc[m][n], alo, b0[n], b1[n]);
#pragma unroll
            for (int n = 0; n < NN; ++n) mma(acc[m][n], ahi, b0[n], b1[n]);
        }
    }
}

// flush one accumulator fragment (rows 16 m + g, g + 8; columns c0 = 8 n + 2t, +1) into a row-major [.., ld] gradient with
// one 128-bit reduction per lane: lanes t, t^1 swap halves so that each holds four consecutive columns of one row
__device__ __forceinline__ void flush_v4(float* __restrict__ gw, int ld, const float c[4], int row_g, int col0, int t)
{
    const float o0 = __shfl_xor_sync(0xffffffffu, c[0], 1), o1 = __shfl_xor_sync(0xffffffffu, c[1], 1);
    const float o2 = __shfl_xor_sync(0xffffffffu, c[2], 1), o3 = __shfl_xor_sync(0xffffffffu, c[3], 1);
    if ((t & 1) == 0) red_add_v4(gw + (size_t)row_g * ld + col0, c[0], c[1], o0, o1);
    else red_add_v4(gw + (size_t)(row_g + 8) * ld + col0 - 2, o2, o3, c[2], c[3]);
}

struct BwdArgs {
    b200gs_heads_weights w;
    b200gs_heads_grads gw;
    long long P;
    const float* feat; const float* hidden; const float* saved;
    const float* d_opacity; const float* d_shs;
    float* d_feat;
    float* sh_grad; int sh_overwrite;
};

template <int F>
__global__ void __launch_bounds__(BT, 1) deform_heads_bwd_kernel(const __grid_constant__ BwdArgs a)
{
    extern __shared__ __align__(16) float4 smem4[];
    constexpr bool RESIDENT = (F == 64);      // F = 128: one W2 slot, re-staged per head (shared-memory budget)
    constexpr int NT1 = F / 8;
    constexpr int RS3[2] = {4, 48 / 2 + 4};   // W3 operands: K = 8 (padded) and 48
    float4* W3b[2] = {smem4, smem4 + MW * RS3[0]};
    float4* W2b = W3b[1] + MW * RS3[1];
    float4* W1b = W2b + (RESIDENT ? 2 : 1) * MW * RS2;
    float* Ds = reinterpret_cast<float*>(W1b + F * RS2);    // [ROWS][LDS_T] dz, then d_h
    float* Dout = Ds + ROWS * LDS_T;                          // [ROWS][LDO]   upstream gradient of the head
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const bool on[2] = {a.w.w2[0] != nullptr, a.w.w2[1] != nullptr};

    tf32::stage_weight<BT>(W1b, a.w.w1, MW, F, MW, F, RS2);
    for (int h = 0; h < 2; ++h) {
        if (!on[h]) continue;
        if (RESIDENT) tf32::stage_weight<BT>(W2b + h * MW * RS2, a.w.w2[h], MW, MW, MW, MW, RS2);
        tf32::stage_weight<BT>(W3b[h], a.w.w3[h], h == 0 ? 8 : 48, MW, KD(h), MW, RS3[h]);
    }
    __syncthreads();

    const int mt = warp >> 1, ntb = (warp & 1) * 4;
    float gW2[2][1][4][4], gW1[1][NT1 / 2][4], gW3o[1][1][4], gW3s[3][1][4];
    float gB2[2] = {0.f, 0.f}, gB1 = 0.f, gB3[2] = {0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        gW3o[0][0][i] = 0.f;
#pragma unroll
        for (int m = 0; m < 3; ++m) gW3s[m][0][i] = 0.f;
#pragma unroll
        for (int n = 0; n < 4; ++n) gW2[0][0][n][i] = gW2[1][0][n][i] = 0.f;
#pragma unroll
        for (int n = 0; n < NT1 / 2; ++n) gW1[0][n][i] = 0.f;
    }

    const long long nblocks = (a.P + ROWS - 1) / ROWS;
    for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const long long row0 = blk * ROWS;
        const int lr_lo = warp * 16 + g, lr_hi = lr_lo + 8;
        const long long r_lo = row0 + lr_lo, r_hi = row0 + lr_hi;
        const bool v_lo = r_lo < a.P, v_hi = r_hi < a.P;
        float dRh[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) dRh[nt][i] = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (!on[h]) continue;
            const int kd = KD(h), ksteps = h == 0 ? 1 : 6;
            const float* dsrc = h == 0 ? a.d_opacity : a.d_shs;
            const float* zsv = a.saved + (size_t)h * stash_plane_floats(a.P);
            const float4* W2h = W2b + (RESIDENT ? h : 0) * MW * RS2;
            if (!RESIDENT) {                  // every warp is past the previous head's use of the slot (trailing barrier below)
                tf32::stage_weight<BT>(W2b, a.w.w2[h], MW, MW, MW, MW, RS2);
                __syncthreads();
            }
            // dz = (d_out W3) masked by relu(z) > 0; d_out also goes to the smem tile (dW3, db3) and, for the SH head, into the
            // step's SH gradient (d shs = d shs': the identity path)
            float dz[8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int i = 0; i < 4; ++i) dz[nt][i] = 0.f;
            for (int j = 0; j < ksteps; ++j) {
                const int c0 = 8 * j + 2 * t;
                float df[4];
                if (h == 0) {
                    df[0] = (v_lo && dsrc && c0 < kd) ? __ldg(dsrc + r_lo) : 0.f;
                    df[1] = (v_hi && dsrc && c0 < kd) ? __ldg(dsrc + r_hi) : 0.f;
                    df[2] = 0.f; df[3] = 0.f;
                } else {
                    const float2 x = (v_lo && dsrc) ? __ldg(reinterpret_cast<const float2*>(dsrc + 48 * r_lo + c0)) : make_float2(0.f, 0.f);
                    const float2 y = (v_hi && dsrc) ? __ldg(reinterpret_cast<const float2*>(dsrc + 48 * r_hi + c0)) : make_float2(0.f, 0.f);
                    df[0] = x.x; df[2] = x.y; df[1] = y.x; df[3] = y.y;
                    if (a.sh_grad) {
                        float2* gl = reinterpret_cast<float2*>(a.sh_grad + 48 * r_lo + c0);
                        float2* gh = reinterpret_cast<float2*>(a.sh_grad + 48 * r_hi + c0);
                        if (a.sh_overwrite) {
                            if (v_lo) *gl = x;
                            if (v_hi) *gh = y;
                        } else {
                            if (v_lo) { const float2 o = *gl; *gl = make_float2(o.x + x.x, o.y + x.y); }
                            if (v_hi) { const float2 o = *gh; *gh = make_float2(o.x + y.x, o.y + y.y); }
                        }
                    }
                }
                *reinterpret_cast<float2*>(Dout + lr_lo * LDO + c0) = make_float2(df[0], df[2]);
                *reinterpret_cast<float2*>(Dout + lr_hi * LDO + c0) = make_float2(df[1], df[3]);
                kstep<8>(dz, df, W3b[h], RS3[h], j, g, t);
            }
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const float2 x = v_lo ? __ldg(reinterpret_cast<const float2*>(zsv + stash_off(r_lo, 8 * nt + 2 * t))) : make_float2(0.f, 0.f);
                const float2 y = v_hi ? __ldg(reinterpret_cast<const float2*>(zsv + stash_off(r_hi, 8 * nt + 2 * t))) : make_float2(0.f, 0.f);
                dz[nt][0] = x.x > 0.f ? dz[nt][0] : 0.f; dz[nt][1] = x.y > 0.f ? dz[nt][1] : 0.f;
                dz[nt][2] = y.x > 0.f ? dz[nt][2] : 0.f; dz[nt][3] = y.y > 0.f ? dz[nt][3] : 0.f;
                *reinterpret_cast<float2*>(Ds + lr_lo * LDS_T + 8 * nt + 2 * t) = make_float2(dz[nt][0], dz[nt][1]);
                *reinterpret_cast<float2*>(Ds + lr_hi * LDS_T + 8 * nt + 2 * t) = make_float2(dz[nt][2], dz[nt][3]);
            }
            // d relu(h) += dz W2
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float af[4] = {dz[j][0], dz[j][2], dz[j][1], dz[j][3]};
                kstep<8>(dRh, af, W2h, RS2, j, g, t);
            }
            __syncthreads();                                              // dz and d_out tiles complete
            dw_accumulate<1, 4, true>(gW2[h], Ds, LDS_T, mt, MW, a.hidden, MW, row0, a.P, ntb, g, t);     // dW2 += dz^T relu(h)
            if (h == 0) dw_accumulate<1, 1, true>(gW3o, Dout, LDO, 0, 1, zsv, MW, row0, a.P, warp, g, t);  // dW3 += d_out^T relu(z)
            else dw_accumulate<3, 1, true>(gW3s, Dout, LDO, 0, 48, zsv, MW, row0, a.P, warp, g, t);
            if (tid < MW) {
                float s = 0.f;
#pragma unroll 8
                for (int r = 0; r < ROWS; ++r) s += Ds[r * LDS_T + tid];
                gB2[h] += s;
            } else if (tid < MW + kd) {
                float s = 0.f;
                for (int r = 0; r < ROWS; ++r) s += Dout[r * LDO + (tid - MW)];
                gB3[h] += s;
            }
            __syncthreads();                                              // before the next head overwrites the tiles
        }
        // d_h = d relu(h) masked by hidden > 0; d_features += d_h W1
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const float2 x = v_lo ? __ldg(reinterpret_cast<const float2*>(a.hidden + stash_off(r_lo, 8 * nt + 2 * t))) : make_float2(0.f, 0.f);
            const float2 y = v_hi ? __ldg(reinterpret_cast<const float2*>(a.hidden + stash_off(r_hi, 8 * nt + 2 * t))) : make_float2(0.f, 0.f);
            dRh[nt][0] = x.x > 0.f ? dRh[nt][0] : 0.f; dRh[nt][1] = x.y > 0.f ? dRh[nt][1] : 0.f;
            dRh[nt][2] = y.x > 0.f ? dRh[nt][2] : 0.f; dRh[nt][3] = y.y > 0.f ? dRh[nt][3] : 0.f;
            *reinterpret_cast<float2*>(Ds + lr_lo * LDS_T + 8 * nt + 2 * t) = make_float2(dRh[nt][0], dRh[nt][1]);
            *reinterpret_cast<float2*>(Ds + lr_hi * LDS_T + 8 * nt + 2 * t) = make_float2(dRh[nt][2], dRh[nt][3]);
        }
        // (in 64-column halves: a whole F = 128 row of accumulators next to the weight-gradient fragments would spill)
        const bool tiled = F == 64 && a.w.feat_tiled;
#pragma unroll
        for (int half = 0; half < F / 64; ++half) {
            float dF[8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int i = 0; i < 4; ++i) dF[nt][i] = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float af[4] = {dRh[j][0], dRh[j][2], dRh[j][1], dRh[j][3]};
                kstep<8>(dF, af, W1b + half * MW * RS2, RS2, j, g, t);
            }
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int c = 64 * half + 8 * nt + 2 * t;
                if (v_lo) {
                    float2* p = reinterpret_cast<float2*>(a.d_feat + (tiled ? stash_off(r_lo, c) : (size_t)r_lo * F + c));
                    const float2 o = *p;
                    *p = make_float2(o.x + dF[nt][0], o.y + dF[nt][1]);
                }
                if (v_hi) {
                    float2* p = reinterpret_cast<float2*>(a.d_feat + (tiled ? stash_off(r_hi, c) : (size_t)r_hi * F + c));
                    const float2 o = *p;
                    *p = make_float2(o.x + dF[nt][2], o.y + dF[nt][3]);
                }
            }
        }
        __syncthreads();
        if (F == 64 && a.w.feat_tiled)
            dw_accumulate<1, NT1 / 2, true>(gW1, Ds, LDS_T, mt, MW, a.feat, F, row0, a.P, (warp & 1) * (NT1 / 2), g, t);
        else
            dw_accumulate<1, NT1 / 2, false>(gW1, Ds, LDS_T, mt, MW, a.feat, F, row0, a.P, (warp & 1) * (NT1 / 2), g, t);
        if (tid < MW) {
            float s = 0.f;
#pragma unroll 8
            for (int r = 0; r < ROWS; ++r) s += Ds[r * LDS_T + tid];
            gB1 += s;
        }
        __syncthreads();
    }

    // flush: one reduction per element per CTA
#pragma unroll
    for (int n = 0; n < NT1 / 2; ++n)
        flush_v4(a.gw.w1, F, gW1[0][n], 16 * mt + g, 8 * ((warp & 1) * (NT1 / 2) + n) + 2 * t, t);
    if (tid < MW) atomicAdd(a.gw.b1 + tid, gB1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (!on[h]) continue;
#pragma unroll
        for (int n = 0; n < 4; ++n) flush_v4(a.gw.w2[h], MW, gW2[h][0][n], 16 * mt + g, 8 * (ntb + n) + 2 * t, t);
        if (tid < MW) atomicAdd(a.gw.b2[h] + tid, gB2[h]);
        else if (tid < MW + KD(h)) atomicAdd(a.gw.b3[h] + (tid - MW), gB3[h]);
    }
    if (on[0] && g == 0) {            // out row 0 of the padded m-tile; columns 8 warp + 2t (+1)
        atomicAdd(a.gw.w3[0] + 8 * warp + 2 * t, gW3o[0][0][0]);
        atomicAdd(a.gw.w3[0] + 8 * warp + 2 * t + 1, gW3o[0][0][1]);
    }
    if (on[1]) {
#pragma unroll
        for (int m = 0; m < 3; ++m) flush_v4(a.gw.w3[1], MW, gW3s[m][0], 16 * m + g, 8 * warp + 2 * t, t);
    }
}

size_t bwd_smem(int F)
{
    return (size_t)(MW * 4 + MW * 28 + (F == 64 ? 2 : 1) * MW * RS2 + F * RS2) * sizeof(float4) +
           (size_t)(ROWS * LDS_T + ROWS * LDO) * sizeof(float);
}

int check(const b200gs_heads_weights* w, int sh_coeffs, const char* what)
{
    if (!w) { set_error("%s: null weights", what); return -1; }
    if (w->width != MW) { set_error("%s: net_width=%d unsupported (need %d)", what, w->width, MW); return -1; }
    if (w->feat_dim != 64 && w->feat_dim != 128) { set_error("%s: feature dim %d unsupported (64 or 128)", what, w->feat_dim); return -1; }
    if (w->feat_tiled && w->feat_dim != 64) { set_error("%s: tiled features need feature dim 64", what); return -1; }
    if (!w->w2[0] && !w->w2[1]) { set_error("%s: both heads are off", what); return -1; }
    for (int h = 0; h < 2; ++h)
        if (w->w2[h] && (!w->b2[h] || !w->w3[h] || !w->b3[h])) { set_error("%s: head %d incomplete", what, h); return -1; }
    if (w->w2[1] && sh_coeffs != 16) { set_error("%s: %d SH coefficients per point (the SH head needs 16)", what, sh_coeffs); return -1; }
    return 0;
}

}  // namespace heads
}  // namespace b200gs

using namespace b200gs;

extern "C" {

size_t b200gs_deform_heads_saved_floats(long long P) { return P > 0 ? 2 * tc5::stash_plane_floats(P) : 0; }

int b200gs_deform_heads_forward(const b200gs_heads_weights* w, long long P, int sh_coeffs, const float* mlp_saved,
                                const float* opacity, const float* shs, float* opacity_out, float* shs_out, float* heads_saved,
                                b200gs_stream_t stream)
{
    if (heads::check(w, sh_coeffs, "deform_heads_forward")) return -1;
    if (P <= 0) return 0;
    heads::FwdArgs a;
    a.w = *w; a.P = P; a.hidden = mlp_saved; a.opacity = opacity; a.shs = shs; a.opacity_out = opacity_out;
    a.shs_out = shs_out; a.saved = heads_saved;
    const int grid = tc5::persistent_grid(P, g_opt_mlp_fwd_sms);
    cudaFuncSetAttribute(heads::deform_heads_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)heads::FWD_SMEM);
    heads::deform_heads_fwd_kernel<<<grid, heads::FT, heads::FWD_SMEM, (cudaStream_t)stream>>>(a);
    return check_launch("deform_heads_forward");
}

int b200gs_deform_heads_backward(const b200gs_heads_weights* w, const b200gs_heads_grads* gw, long long P, int sh_coeffs,
                                 const float* features, const float* mlp_saved, const float* heads_saved,
                                 const float* d_opacity, const float* d_shs, float* d_features, float* sh_grad,
                                 int sh_grad_overwrite, b200gs_stream_t stream)
{
    if (heads::check(w, sh_coeffs, "deform_heads_backward")) return -1;
    if (!gw) { set_error("deform_heads_backward: null gradient table"); return -1; }
    const auto misaligned = [](const void* p) { return ((uintptr_t)p & 15) != 0; };
    if (!gw->w1 || !gw->b1 || misaligned(gw->w1)) { set_error("deform_heads_backward: dW1 / db1 missing or dW1 not 16-byte aligned"); return -1; }
    for (int h = 0; h < 2; ++h) {
        if (!w->w2[h]) continue;
        if (!gw->w2[h] || !gw->b2[h] || !gw->w3[h] || !gw->b3[h]) { set_error("deform_heads_backward: head %d gradient missing", h); return -1; }
        if (misaligned(gw->w2[h]) || (h == 1 && misaligned(gw->w3[h]))) {
            set_error("deform_heads_backward: head %d weight gradient not 16-byte aligned", h); return -1;
        }
    }
    if (P <= 0) return 0;
    heads::BwdArgs a;
    a.w = *w; a.gw = *gw; a.P = P; a.feat = features; a.hidden = mlp_saved; a.saved = heads_saved;
    a.d_opacity = d_opacity; a.d_shs = d_shs; a.d_feat = d_features;
    a.sh_grad = w->w2[1] ? sh_grad : nullptr; a.sh_overwrite = sh_grad_overwrite;
    const int grid = tc5::persistent_grid(P, g_opt_mlp_bwd_sms);
    const size_t smem = heads::bwd_smem(w->feat_dim);
    if (w->feat_dim == 64) {
        cudaFuncSetAttribute(heads::deform_heads_bwd_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        heads::deform_heads_bwd_kernel<64><<<grid, heads::BT, smem, (cudaStream_t)stream>>>(a);
    } else {
        cudaFuncSetAttribute(heads::deform_heads_bwd_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        heads::deform_heads_bwd_kernel<128><<<grid, heads::BT, smem, (cudaStream_t)stream>>>(a);
    }
    return check_launch("deform_heads_backward");
}

}  // extern "C"
