// m16n8k8 TF32 mma.sync helpers shared by the register-resident deformation-MLP backwards (deform_mlp.cu, deform_heads.cu).
// Every dX contraction runs the error-compensated split x = hi + lo, issued as lo*hi + hi*lo + hi*hi with FP32
// accumulation (~FP32 accuracy).  An accumulator fragment is re-used as the A fragment of the next layer by permuting
// the K index (fragment slot t <-> column 2t, slot t+4 <-> column 2t+1); the weights are laid out to match.
#pragma once
#include "tc5_common.cuh"

namespace b200gs {
namespace tf32 {

__device__ __forceinline__ void split(float x, u32& hi, u32& lo)
{
    hi = tc5::to_tf32(x);
    lo = tc5::to_tf32(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma(float c[4], const u32 a[4], u32 b0, u32 b1)
{
    asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Pre-split weight operand for  Y[rows][n] = sum_k X[rows][k] Wm[k][n],  Wm[k][n] = w[k * sk + n] (zero for k >= K_real),
// staged by a block of NTHREADS: entry (n, j, t) = {hi Wm[8j+2t][n], hi Wm[8j+2t+1][n], lo ..., lo ...} at float4 index
// n * rs + 4j + t.  rs = K/2 + 4 (== 4 mod 8) puts the 8 lanes of an LDS.128 phase on disjoint banks; a K = 8 operand
// (rs = 4, rows contiguous) is conflict free as it is.
template <int NTHREADS>
__device__ __forceinline__ void stage_weight(float4* __restrict__ dst, const float* __restrict__ w, int K, int N, int K_real, int sk, int rs)
{
    for (int i = threadIdx.x; i < N * (K / 2); i += NTHREADS) {
        const int n = i / (K / 2), kk = i - n * (K / 2);      // kk = 4j + t
        const int k0 = 2 * kk, k1 = k0 + 1;
        const float v0 = k0 < K_real ? __ldg(w + (size_t)k0 * sk + n) : 0.f;
        const float v1 = k1 < K_real ? __ldg(w + (size_t)k1 * sk + n) : 0.f;
        u32 h0, l0, h1, l1;
        split(v0, h0, l0); split(v1, h1, l1);
        dst[n * rs + kk] = make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
    }
}

// acc[nt] += A(k-step j) * B[:, n-tile nt]  for nt in [0, NT); A given as its 4 fragment values.
// The three passes of the split are issued pass-major over groups of four n-tiles, so that back-to-back
// MMAs never depend on each other (a dependent HMMA would wait out the full pipe latency).
template <int NT>
__device__ __forceinline__ void kstep(float (*acc)[4], const float a[4], const float4* __restrict__ Bq, int rs, int j,
                                      int g, int t)
{
    u32 ahi[4], alo[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split(a[i], ahi[i], alo[i]);
    constexpr int G = NT < 4 ? NT : 4;
#pragma unroll
    for (int n0 = 0; n0 < NT; n0 += G) {
        float4 b[G];
#pragma unroll
        for (int q = 0; q < G; ++q) b[q] = Bq[(8 * (n0 + q) + g) * rs + 4 * j + t];
#pragma unroll
        for (int q = 0; q < G; ++q) mma(acc[n0 + q], alo, __float_as_uint(b[q].x), __float_as_uint(b[q].y));
#pragma unroll
        for (int q = 0; q < G; ++q) mma(acc[n0 + q], ahi, __float_as_uint(b[q].z), __float_as_uint(b[q].w));
#pragma unroll
        for (int q = 0; q < G; ++q) mma(acc[n0 + q], ahi, __float_as_uint(b[q].x), __float_as_uint(b[q].y));
    }
}

}  // namespace tf32
}  // namespace b200gs
