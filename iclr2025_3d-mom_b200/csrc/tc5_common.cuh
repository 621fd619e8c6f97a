// tcgen05 / TMEM / mbarrier helpers shared by the deformation-MLP tensor-core kernels (sm_100a).
#pragma once
#include "common.cuh"

namespace b200gs {
namespace tc5 {

constexpr int MW = 64;
constexpr int ROWS = 128;

__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u32 to_tf32(float x) { u32 r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return r; }
// Exact two-term split for tcgen05.mma.kind::tf32. The tensor core TRUNCATES an FP32 container to TF32 (it ignores the low
// 13 mantissa bits; measured with tools/probe/umma_probe.cu), so the "hi" operand can be the raw value itself and
// lo = x - trunc(x) is exact (13 significant bits, of which the hardware keeps 10): hi + lo reproduces x to 2^-21 relative
// with two instructions instead of the five of a round / subtract / round split.
__device__ __forceinline__ float tf32_lo(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

// Activation stash layout (forward -> backward, opaque to callers): 4 planes (relu(hidden), relu(z_pos),
// relu(z_scale), relu(z_rot)) of ceil(P/128) tiles; a tile is [32 groups of 4 points][16 column chunks][4 points]
// [4 floats].  The backward reads 8 chunks x 4 points per warp instruction = one contiguous 512-byte run; the
// forward (one lane per point) writes 64-byte runs, 8 lines per instruction instead of the 32 of a row-major stash.
__host__ __device__ __forceinline__ size_t stash_plane_floats(long long P) { return (size_t)((P + ROWS - 1) / ROWS) * ROWS * MW; }
__host__ __device__ __forceinline__ size_t stash_off(long long row, int col)
{
    return (size_t)(row >> 7) * (ROWS * MW) + (size_t)((row & 127) >> 2) * 256 + (size_t)(col >> 2) * 16 + (size_t)(row & 3) * 4 + (col & 3);
}

// Grid of a persistent kernel walking the ceil(P/128) tiles: one CTA per SM, at most `cap` when 0 < cap < NUM_SMS (the
// b200gs_set_option CTA caps, which leave SMs to a concurrent stream), never more CTAs than tiles.
inline int persistent_grid(long long P, int cap)
{
    const long long nblocks = (P + ROWS - 1) / ROWS;
    const int sms = cap > 0 && cap < NUM_SMS ? cap : NUM_SMS;
    return (int)(nblocks < sms ? nblocks : sms);
}

// Behind the four stash planes the forward leaves, for the tcgen05 backward (feature dim 64), the transposed weights as
// ready-to-copy K-major UMMA B operands [N = in][K = out] in TF32 hi / lo pairs: W2^T of the three heads, then W1^T
// (8 images of 64 x 64 floats). The backward streams the current head's pair into shared memory with cp.async instead
// of keeping single-precision-rounded copies of all of them resident, which is what lets its dX chain run the full
// three-term split (a rounded weight operand left up to 2 % error on a few per-point xyz gradients at 1M points).
constexpr size_t BWD_W_IMAGE_FLOATS = 8 * MW * MW;
__host__ __device__ __forceinline__ size_t stash_total_floats(long long P) { return 4 * stash_plane_floats(P) + BWD_W_IMAGE_FLOATS; }
// image m (0..2: W2 of head m, 3: W1), plane 0 = hi, 1 = lo; w = torch [out 64][in 64] row-major
__device__ __forceinline__ void write_bwd_weight_image(float* __restrict__ images, int m, const float* __restrict__ w, int nthreads)
{
    float* hi = images + (size_t)(2 * m) * MW * MW;
    float* lo = hi + MW * MW;
    for (int i = threadIdx.x; i < MW * MW; i += nthreads) {
        const int k = i >> 6, n = i & 63;                      // k = out row, n = in column: B[n][k] = W[k][n]
        const float v = __ldg(w + i);
        const float h = __uint_as_float(to_tf32(v));
        const int off = (k >> 2) * (MW * 4) + n * 4 + (k & 3);
        hi[off] = h;
        lo[off] = __uint_as_float(to_tf32(v - h));
    }
}

__device__ __forceinline__ void mbar_init(u64* bar, u32 count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity)
{
    u32 ok = 0, spins = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (ok) break;
        if (++spins > (1u << 24)) __trap();      // never hang the GPU on a protocol error
    }
}
// One lane of a converged warp (the same lane on every call): the issuer of tcgen05.mma / tcgen05.commit.  Used inside a
// warp-uniform branch this compiles to plain straight-line UTCHMMA sequences, where `if (threadIdx.x == 0)` makes the
// compiler wrap every MMA in an ELECT / BRA.U.ANY loop.
__device__ __forceinline__ bool elect_one()
{
    u32 pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(u64* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(u32 d_tmem, u32 a_tmem, u64 b_desc, u32 idesc, u32 accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
                 :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}

// K-major, no swizzle: element (n, k) of an [N x K] operand at byte (k/4)*(N*16) + n*16 + (k%4)*4
// -> core matrix = 8 rows x 16 B contiguous (SBO = 128 B), next 16-byte K chunk at LBO = N*16 B.
__device__ __forceinline__ u64 kmajor_desc(u32 smem_addr, int N)
{
    const u64 lbo = (u64)((N * 16) >> 4), sbo = (u64)(128 >> 4);
    return (u64)((smem_addr >> 4) & 0x3FFF) | (lbo << 16) | (sbo << 32) | (1ull << 46);
}
__device__ __forceinline__ u32 make_idesc(int M, int N)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((u32)(N >> 3) << 17) | ((u32)(M >> 4) << 24);   // F32 accum, TF32 x TF32, K-major A and B
}

#define R8(v, o) "=r"(v[o]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), "=r"(v[o + 7])
#define W8(v, o) "r"(v[o]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3]), "r"(v[o + 4]), "r"(v[o + 5]), "r"(v[o + 6]), "r"(v[o + 7])
__device__ __forceinline__ void tmem_ld32(u32 addr, u32* v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : R8(v, 0), R8(v, 8), R8(v, 16), R8(v, 24) : "r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(u32 addr, u32* v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : R8(v, 0), R8(v, 8) : "r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_ld8(u32 addr, u32* v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : R8(v, 0) : "r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_st32(u32 addr, const u32* v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
                 :: "r"(addr), W8(v, 0), W8(v, 8), W8(v, 16), W8(v, 24) : "memory");
}
// Warp-collective: `cols` TMEM columns, base address written to *slot; the allocation permit is given up at once so that
// the CTA never blocks another one's allocation on the same SM.  Freed by tmem_dealloc from one warp before the CTA exits.
__device__ __forceinline__ void tmem_alloc(u32* slot, u32 cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(u32 base, u32 cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(base), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }


// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void mma_ss(u32 d_tmem, u64 a_desc, u64 b_desc, u32 idesc, u32 accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// Un-swizzled shared-memory operand descriptor. The operand is made of 128-byte core matrices
// (8 rows of 16 bytes). K-major: rows = 8 consecutive M/N indices, 16 bytes = 4 consecutive K;
// SBO = stride between 8-row groups, LBO = stride between 16-byte K chunks. MN-major: rows = 8
// consecutive K indices, 16 bytes = 4 consecutive M/N; SBO = stride between 16-byte M/N chunks,
// LBO = stride between 8-row K groups.
__device__ __forceinline__ u64 smem_desc(u32 smem_addr, u32 lbo_bytes, u32 sbo_bytes)
{
    return (u64)((smem_addr >> 4) & 0x3FFF) | ((u64)(lbo_bytes >> 4) << 16) | ((u64)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
constexpr u32 IDESC_A_MN = 1u << 15, IDESC_B_MN = 1u << 16;

// weights: torch [N_real x K] row-major -> hi / lo K-major UMMA operands with N rows (zero padded), by a block of NTHREADS
template <int NTHREADS>
__device__ __forceinline__ void stage_kmajor(float* __restrict__ hi, float* __restrict__ lo, const float* __restrict__ w,
                                             int N, int N_real, int K)
{
    for (int i = threadIdx.x; i < N * K; i += NTHREADS) {
        const int n = i / K, k = i - n * K;
        const float v = n < N_real ? __ldg(w + (size_t)n * K + k) : 0.f;
        const u32 h = to_tf32(v), l = to_tf32(v - __uint_as_float(h));
        const int off = (k >> 2) * (N * 4) + n * 4 + (k & 3);
        hi[off] = __uint_as_float(h);
        lo[off] = __uint_as_float(l);
    }
}

// 3 x (K/8) MMAs: D = (Ahi + Alo) (Bhi + Blo) without lo*lo, small terms first
__device__ __forceinline__ void issue_layer(u32 d_tmem, u32 a_hi, u32 a_lo, u32 b_hi_smem, u32 b_lo_smem, int N, int K, u32 idesc)
{
    const u64 dh = kmajor_desc(b_hi_smem, N), dl = kmajor_desc(b_lo_smem, N);
    const u64 step = (u64)((2 * N * 16) >> 4);         // two 16-byte K chunks per instruction
    for (int j = 0; j < K / 8; ++j) {
        mma_ts(d_tmem, a_lo + 8 * j, dh + step * j, idesc, j > 0);
        mma_ts(d_tmem, a_hi + 8 * j, dl + step * j, idesc, 1u);
        mma_ts(d_tmem, a_hi + 8 * j, dh + step * j, idesc, 1u);
    }
}

}  // namespace tc5
}  // namespace b200gs
