// Rasterizer forward: projection + SH, binning, compositing.
//
// Behaviour follows the reference's forward pass
//   RAST/cuda_rasterizer/forward.cu:155-256  (per-Gaussian preprocess)
//   RAST/cuda_rasterizer/rasterizer_impl.cu:70-138, 198-339 (binning, orchestration)
//   RAST/cuda_rasterizer/forward.cu:261-379  (per-tile compositing)
// with a different pipeline: Gaussians are depth-sorted once (P keys), (tile, gaussian)
// instances are emitted in that order by a load-balanced kernel, and a stable radix sort
// on the tile id alone produces the same (tile, depth, index) order as the reference's
// 64-bit key sort at a fraction of the traffic.
#include "rast_state.cuh"
#include <cmath>
#include <cstdio>

namespace b200gs {

namespace {

constexpr float SH0 = 0.28209479177387814f;
constexpr float SH1 = 0.4886025119029199f;
__constant__ float SH2c[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                              -1.0925484305920792f, 0.5462742152960396f};
__constant__ float SH3c[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f,
                              0.3731763325901154f, -0.4570457994644658f, 1.445305721320277f,
                              -0.5900435899266435f};

constexpr int PRE_THREADS = 128;
constexpr int PRE_WARPS = PRE_THREADS / 32;

// The bit-exact part of the projection (radii, tile rectangles and depth keys must equal the
// reference's to the last bit) is written with explicit round-to-nearest intrinsics, so no
// compiler contraction choice can change a rounding.  The operation order restates what the
// reference's expressions compile to under nvcc's default -fmad=true (verified against its
// SASS): a*b + c*d + e*f  ->  fma(e, f, fma(a, b, c*d)).
__device__ __forceinline__ float dot3(float a0, float b0, float a1, float b1, float a2, float b2) {
    return __fmaf_rn(a2, b2, __fmaf_rn(a0, b0, __fmul_rn(a1, b1)));
}
// matrix[0]*x + matrix[4]*y + matrix[8]*z + matrix[12]  (auxiliary.h:58-76)
__device__ __forceinline__ float affine3(float x, float y, float z, float m0, float m1, float m2, float m3) {
    return __fadd_rn(dot3(x, m0, y, m1, z, m2), m3);
}
__device__ __forceinline__ float3 xform43(const float3 p, const float* m) {
    return make_float3(affine3(p.x, p.y, p.z, m[0], m[4], m[8], m[12]),
                       affine3(p.x, p.y, p.z, m[1], m[5], m[9], m[13]),
                       affine3(p.x, p.y, p.z, m[2], m[6], m[10], m[14]));
}
__device__ __forceinline__ float4 xform44(const float3 p, const float* m) {
    return make_float4(affine3(p.x, p.y, p.z, m[0], m[4], m[8], m[12]),
                       affine3(p.x, p.y, p.z, m[1], m[5], m[9], m[13]),
                       affine3(p.x, p.y, p.z, m[2], m[6], m[10], m[14]),
                       affine3(p.x, p.y, p.z, m[3], m[7], m[11], m[15]));
}

// NDC -> pixel; evaluated in double exactly like the reference (auxiliary.h:41-44).
__device__ __forceinline__ float ndc_to_pix(float v, int S) {
    return (float)__dmul_rn(__fma_rn(__dadd_rn((double)v, 1.0), (double)S, -1.0), 0.5);
}

// World-space covariance from scale and (already normalised) quaternion, forward.cu:118-152.
// M = S*R has exactly one non-zero term per entry, so M[c][r] = s_r * R[c][r]; Sigma = M^T M.
__device__ __forceinline__ void cov3d_from_scale_rot(const float3 scale, float mod, const float4 q, float* cov)
{
    const float s[3] = {__fmul_rn(mod, scale.x), __fmul_rn(mod, scale.y), __fmul_rn(mod, scale.z)};
    const float r = q.x, x = q.y, y = q.z, z = q.w;
    const float xz = __fmul_rn(x, z), rx = __fmul_rn(r, x), rz = __fmul_rn(r, z);
    const float yy = __fmul_rn(y, y), zz = __fmul_rn(z, z);
    auto dbl = [](float v) { return __fadd_rn(v, v); };
    float R[3][3];   // R[c][r], column-major like the reference's matrix type
    R[0][0] = __fsub_rn(1.f, dbl(__fadd_rn(yy, zz)));
    R[0][1] = dbl(__fmaf_rn(x, y, -rz));
    R[0][2] = dbl(__fmaf_rn(r, y, xz));
    R[1][0] = dbl(__fmaf_rn(x, y, rz));
    R[1][1] = __fsub_rn(1.f, dbl(__fmaf_rn(x, x, zz)));
    R[1][2] = dbl(__fmaf_rn(y, z, -rx));
    R[2][0] = dbl(__fmaf_rn(-r, y, xz));
    R[2][1] = dbl(__fmaf_rn(y, z, rx));
    R[2][2] = __fsub_rn(1.f, dbl(__fmaf_rn(x, x, yy)));
    float M[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int rr = 0; rr < 3; ++rr) M[c][rr] = __fmul_rn(s[rr], R[c][rr]);
    auto sig = [&](int c, int rr) { return dot3(M[rr][0], M[c][0], M[rr][1], M[c][1], M[rr][2], M[c][2]); };
    cov[0] = sig(0, 0); cov[1] = sig(0, 1); cov[2] = sig(0, 2);
    cov[3] = sig(1, 1); cov[4] = sig(1, 2); cov[5] = sig(2, 2);
}

// EWA projection of the 3D covariance, forward.cu:74-113: cov2D = T^T Vrk^T T with T = W J,
// the third column of J being zero.
__device__ __forceinline__ float3 cov2d_project(const float3 mean, float fx, float fy, float tanx, float tany,
                                                const float* c, const float* vm)
{
    const float3 t0 = xform43(mean, vm);
    const float tz = t0.z;
    const float limx = __fmul_rn(1.3f, tanx), limy = __fmul_rn(1.3f, tany);
    const float txtz = __fdiv_rn(t0.x, tz), tytz = __fdiv_rn(t0.y, tz);
    const float tx = __fmul_rn(fminf(limx, fmaxf(-limx, txtz)), tz);
    const float ty = __fmul_rn(fminf(limy, fmaxf(-limy, tytz)), tz);
    const float tz2 = __fmul_rn(tz, tz);
    const float J00 = __fdiv_rn(fx, tz), J02 = __fdiv_rn(-__fmul_rn(fx, tx), tz2);
    const float J11 = __fdiv_rn(fy, tz), J12 = __fdiv_rn(-__fmul_rn(fy, ty), tz2);
    // T[0][r] = W[0][r]*J00 + W[2][r]*J02 ; T[1][r] = W[1][r]*J11 + W[2][r]*J12 ; W[k][r] = vm[4r + k]
    float T0[3], T1[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        T0[r] = __fmaf_rn(vm[4 * r + 2], J02, __fmul_rn(vm[4 * r + 0], J00));
        T1[r] = __fmaf_rn(vm[4 * r + 2], J12, __fmul_rn(vm[4 * r + 1], J11));
    }
    // A[k][0] = T0 . Vrk column k, A[k][1] = T1 . Vrk column k (Vrk symmetric: c0 c1 c2 / c1 c3 c4 / c2 c4 c5)
    const float A00 = dot3(T0[0], c[0], T0[1], c[1], T0[2], c[2]);
    const float A10 = dot3(T0[0], c[1], T0[1], c[3], T0[2], c[4]);
    const float A20 = dot3(T0[0], c[2], T0[1], c[4], T0[2], c[5]);
    const float A01 = dot3(T1[0], c[0], T1[1], c[1], T1[2], c[2]);
    const float A11 = dot3(T1[0], c[1], T1[1], c[3], T1[2], c[4]);
    const float A21 = dot3(T1[0], c[2], T1[1], c[4], T1[2], c[5]);
    const float c00 = __fadd_rn(dot3(A00, T0[0], A10, T0[1], A20, T0[2]), 0.3f);
    const float c01 = dot3(A01, T0[0], A11, T0[1], A21, T0[2]);
    const float c11 = __fadd_rn(dot3(A01, T1[0], A11, T1[1], A21, T1[2]), 0.3f);
    return make_float3(c00, c01, c11);
}

struct PreArgs {
    int P, D, M, W, H;
    const float* means; const float* scales; const float* rots; const float* opac;
    const float* shs; const float* cov3d_pre; const float* colors_pre;
    const float* view; const float* proj; const float* campos;
    float scale_mod, tanx, tany, fx, fy;
    int grid_x, grid_y;
    int prefiltered;
    int* radii;
    GeomState g;
};

// One thread per Gaussian. SH coefficients (the bulk of the bytes: 192 of 236 per
// Gaussian at degree 3) are pulled in by whole warps with 128-bit coalesced loads and
// handed to their owner lanes through padded shared memory.
__global__ void __launch_bounds__(PRE_THREADS) preprocess_fwd_kernel(const PreArgs a)
{
    extern __shared__ float s_sh[];            // [PRE_WARPS][32][3M+1]
    __shared__ float s_cam[36];                // view[16] proj[16] campos[3]
    __shared__ unsigned long long s_sum[PRE_WARPS * 2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 16) s_cam[tid] = __ldg(a.view + tid);
    else if (tid < 32) s_cam[tid] = __ldg(a.proj + (tid - 16));
    else if (tid < 35) s_cam[tid] = __ldg(a.campos + (tid - 32));
    __syncthreads();
    const float* vm = s_cam; const float* pm = s_cam + 16;

    const int idx = blockIdx.x * PRE_THREADS + tid;
    const bool in_range = idx < a.P;
    bool alive = in_range;
    float3 p = make_float3(0.f, 0.f, 0.f);
    float3 p_view = p;
    if (in_range) {
        p = make_float3(__ldg(a.means + 3 * idx), __ldg(a.means + 3 * idx + 1), __ldg(a.means + 3 * idx + 2));
        p_view = xform43(p, vm);
        // near cull, auxiliary.h:139-164 (the lateral test is disabled there)
        if (p_view.z <= 0.2f) {
            alive = false;
            if (a.prefiltered) { printf("Point is filtered although prefiltered is set. This shouldn't happen!"); __trap(); }
        }
    }
    float3 conic = make_float3(0.f, 0.f, 0.f);
    float2 pix = make_float2(0.f, 0.f);
    float radius = 0.f;
    u32 xmin = 0, xmax = 0, ymin = 0, ymax = 0;
    if (alive) {
        float4 ph = xform44(p, pm);
        const float pw = __fdiv_rn(1.0f, __fadd_rn(ph.w, 0.0000001f));
        const float3 pp = make_float3(__fmul_rn(ph.x, pw), __fmul_rn(ph.y, pw), __fmul_rn(ph.z, pw));
        float cov_local[6];
        const float* cov3 = cov_local;
        if (a.cov3d_pre) {
#pragma unroll
            for (int k = 0; k < 6; ++k) cov_local[k] = __ldg(a.cov3d_pre + 6 * (size_t)idx + k);
        } else {
            float3 sc = make_float3(__ldg(a.scales + 3 * idx), __ldg(a.scales + 3 * idx + 1), __ldg(a.scales + 3 * idx + 2));
            float4 q = __ldg(reinterpret_cast<const float4*>(a.rots) + idx);
            cov3d_from_scale_rot(sc, a.scale_mod, q, cov_local);
#pragma unroll
            for (int k = 0; k < 6; ++k) a.g.cov3D[6 * (size_t)idx + k] = cov_local[k];
        }
        float3 cov = cov2d_project(p, a.fx, a.fy, a.tanx, a.tany, cov3, vm);
        const float det = __fmaf_rn(cov.x, cov.z, -__fmul_rn(cov.y, cov.y));
        if (det == 0.0f) alive = false;
        else {
            const float det_inv = __fdiv_rn(1.f, det);
            conic = make_float3(__fmul_rn(cov.z, det_inv), -__fmul_rn(cov.y, det_inv), __fmul_rn(cov.x, det_inv));
            const float mid = __fmul_rn(0.5f, __fadd_rn(cov.x, cov.z));
            const float disc = __fsqrt_rn(fmaxf(0.1f, __fmaf_rn(mid, mid, -det)));
            const float lambda1 = __fadd_rn(mid, disc), lambda2 = __fsub_rn(mid, disc);
            radius = ceilf(__fmul_rn(3.f, __fsqrt_rn(fmaxf(lambda1, lambda2))));
            pix = make_float2(ndc_to_pix(pp.x, a.W), ndc_to_pix(pp.y, a.H));
            // tile rectangle, auxiliary.h:46-56
            const int ri = (int)radius;
            const float rf = (float)ri, tw = (float)TILE_X, th = (float)TILE_Y;
            xmin = min((u32)a.grid_x, (u32)max(0, (int)__fdiv_rn(__fsub_rn(pix.x, rf), tw)));
            ymin = min((u32)a.grid_y, (u32)max(0, (int)__fdiv_rn(__fsub_rn(pix.y, rf), th)));
            xmax = min((u32)a.grid_x, (u32)max(0, (int)__fdiv_rn(__fsub_rn(__fadd_rn(__fadd_rn(pix.x, rf), tw), 1.f), tw)));
            ymax = min((u32)a.grid_y, (u32)max(0, (int)__fdiv_rn(__fsub_rn(__fadd_rn(__fadd_rn(pix.y, rf), th), 1.f), th)));
            if ((xmax - xmin) * (ymax - ymin) == 0) alive = false;
        }
    }

    // ---- colour: SH -> RGB (forward.cu:20-71) or precomputed --------------------------
    float3 rgb = make_float3(0.f, 0.f, 0.f);
    unsigned char clampbits = 0;
    if (a.colors_pre == nullptr) {
        const int nco = (a.D + 1) * (a.D + 1);
        const int nact = 3 * nco;                 // floats actually used per Gaussian
        const int stride = 3 * a.M + 1;           // odd => conflict-free owner reads
        float* ws = s_sh + (size_t)warp * 32 * stride;
        const bool any_alive = __any_sync(0xffffffffu, alive);
        if (any_alive) {
            const int g0 = blockIdx.x * PRE_THREADS + warp * 32;
            const int ng = min(32, a.P - g0);
            const float* src = a.shs + (size_t)g0 * 3 * a.M;
            if (nco == a.M && ((3 * a.M) & 3) == 0) {
                const int total4 = ng * 3 * a.M / 4;
                const float4* src4 = reinterpret_cast<const float4*>(src);
                for (int e = lane; e < total4; e += 32) {
                    float4 v = __ldg(src4 + e);
                    int f = e * 4;
                    int gg = f / (3 * a.M), k = f - gg * 3 * a.M;   // 3M % 4 == 0: never straddles
                    float* d = ws + gg * stride + k;
                    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
                }
            } else {
                const int total = ng * nact;
                for (int e = lane; e < total; e += 32) {
                    int gg = e / nact, k = e - gg * nact;
                    ws[gg * stride + k] = __ldg(src + (size_t)gg * 3 * a.M + k);
                }
            }
        }
        __syncwarp();
        if (alive) {
            const float* sh = ws + lane * stride;
            const float3 cam = make_float3(s_cam[32], s_cam[33], s_cam[34]);
            float3 dir = make_float3(p.x - cam.x, p.y - cam.y, p.z - cam.z);
            float len = sqrtf(dir.x * dir.x + dir.y * dir.y + dir.z * dir.z);
            dir.x = dir.x / len; dir.y = dir.y / len; dir.z = dir.z / len;
            float res[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) res[c] = SH0 * sh[c];
            if (a.D > 0) {
                const float x = dir.x, y = dir.y, z = dir.z;
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    res[c] = res[c] - SH1 * y * sh[3 + c] + SH1 * z * sh[6 + c] - SH1 * x * sh[9 + c];
                if (a.D > 1) {
                    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        res[c] = res[c] + SH2c[0] * xy * sh[12 + c] + SH2c[1] * yz * sh[15 + c] +
                                 SH2c[2] * (2.0f * zz - xx - yy) * sh[18 + c] + SH2c[3] * xz * sh[21 + c] +
                                 SH2c[4] * (xx - yy) * sh[24 + c];
                    if (a.D > 2) {
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            res[c] = res[c] + SH3c[0] * y * (3.0f * xx - yy) * sh[27 + c] +
                                     SH3c[1] * xy * z * sh[30 + c] +
                                     SH3c[2] * y * (4.0f * zz - xx - yy) * sh[33 + c] +
                                     SH3c[3] * z * (2.0f * zz - 3.0f * xx - 3.0f * yy) * sh[36 + c] +
                                     SH3c[4] * x * (4.0f * zz - xx - yy) * sh[39 + c] +
                                     SH3c[5] * z * (xx - yy) * sh[42 + c] +
                                     SH3c[6] * x * (xx - 3.0f * yy) * sh[45 + c];
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                res[c] += 0.5f;
                if (res[c] < 0.f) clampbits |= (unsigned char)(1u << c);
                res[c] = fmaxf(res[c], 0.f);
            }
            rgb = make_float3(res[0], res[1], res[2]);
        }
    } else if (alive) {
        rgb = make_float3(__ldg(a.colors_pre + 3 * (size_t)idx), __ldg(a.colors_pre + 3 * (size_t)idx + 1),
                          __ldg(a.colors_pre + 3 * (size_t)idx + 2));
    }

    // ---- write-out -----------------------------------------------------------------------
    u32 touched = 0;
    if (in_range) {
        a.g.order_iota[idx] = (u32)idx;
        if (alive) {
            touched = (ymax - ymin) * (xmax - xmin);
            const float op = __ldg(a.opac + idx);
            // Pairs whose exponent lies below this bound are certain to fail the reference's
            // alpha >= 1/255 test (margin 1e-4 >> the few-ulp error of expf/logf), so the
            // compositing kernels skip them without evaluating the exponential.
            const float reject = (op > 0.f) ? (-logf(255.f * op) - 1e-4f) : 1.f;
            a.radii[idx] = (int)radius;
            a.g.depth_key[idx] = __float_as_uint(p_view.z);
            a.g.rect[idx] = make_uint2(xmin | (xmax << 16), ymin | (ymax << 16));
            a.g.recA[idx] = make_float4(pix.x, pix.y, conic.x, conic.y);
            a.g.recB[idx] = make_float4(conic.z, op, p_view.z, reject);
            a.g.recC[idx] = make_float4(rgb.x, rgb.y, rgb.z, 0.f);
            a.g.clamped[idx] = clampbits;
        } else {
            a.radii[idx] = 0;
            a.g.depth_key[idx] = 0xFFFFFFFFu;
        }
        a.g.tiles_touched[idx] = touched;
    }
    // block totals -> two global atomics per block
    unsigned long long tsum = touched, vsum = alive ? 1ull : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
        vsum += __shfl_xor_sync(0xffffffffu, vsum, o);
    }
    if (lane == 0) { s_sum[warp] = tsum; s_sum[PRE_WARPS + warp] = vsum; }
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0, v = 0;
#pragma unroll
        for (int w = 0; w < PRE_WARPS; ++w) { t += s_sum[w]; v += s_sum[PRE_WARPS + w]; }
        if (t) atomicAdd(a.g.counters + 0, t);
        if (v) atomicAdd(a.g.counters + 1, v);
    }
}

// ---- instance emission ----------------------------------------------------------------
// Walks the depth-sorted Gaussian list; a chained scan (decoupled look-back) of the
// per-Gaussian tile counts gives each block its output window, and the block then writes
// its instances with one thread per *instance* (binary search over the 256 local
// offsets), so large splats do not serialise a thread as in rasterizer_impl.cu:70-111.
// (2 / 4 Gaussians per thread -- a 2 / 4 times shorter look-back chain -- were measured: stage 2 0.405 / 0.412 vs 0.409 ms, not kept.)
constexpr u64 EM_AGG = 1ull << 62, EM_INCL = 1ull << 63, EM_VALUE = (1ull << 62) - 1;

// Warp 0 looks back over 32 predecessors per step (ballots over their states, one shuffle reduction) instead of thread 0
// walking them one dependent L2 round trip at a time.  Same prefix, same output.
__global__ void __launch_bounds__(256)
emit_instances_kernel(const u32* __restrict__ sorted_idx, u32 n_vis, const u32* __restrict__ tiles_touched,
                      const uint2* __restrict__ rect, int grid_x, u32* __restrict__ out_tile,
                      u32* __restrict__ out_gid, u64* status, u32* ticket)
{
    __shared__ u32 s_off[257];
    __shared__ uint2 s_rect[256];
    __shared__ u32 s_gid[256];
    __shared__ u32 s_scan[8];
    __shared__ u32 s_tile;
    __shared__ u64 s_base;
    const u32 tid = threadIdx.x;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const u32 i = tile * 256 + tid;
    u32 cnt = 0, gid = 0;
    uint2 rc = make_uint2(0, 0);
    if (i < n_vis) {
        gid = __ldg(sorted_idx + i);
        cnt = __ldg(tiles_touched + gid);
        rc = __ldg(rect + gid);
    }
    u32 total;
    const u32 off = block_exclusive_scan_256(cnt, s_scan, &total);
    s_off[tid] = off; s_rect[tid] = rc; s_gid[tid] = gid;
    if (tid < 32) {
        const u32 lane = tid;
        u64 prefix = 0;
        if (lane == 0) {
            s_off[256] = total;
            st_volatile_u64(status + tile, (u64)total | (tile == 0 ? EM_INCL : EM_AGG));
        }
        long long t = (long long)tile - 1;          // nearest predecessor not yet taken
        bool done = tile == 0;
        while (!done) {
            const long long idx = t - (long long)lane;
            const u64 v = idx >= 0 ? ld_volatile_u64(status + idx) : EM_INCL;       // before tile 0: an inclusive 0
            const u32 m_ready = __ballot_sync(0xffffffffu, (v & (EM_AGG | EM_INCL)) != 0);
            const u32 m_incl = __ballot_sync(0xffffffffu, (v & EM_INCL) != 0);
            const u32 n_ready = m_ready == 0xffffffffu ? 32u : (u32)__ffs((int)~m_ready) - 1u;    // published states, nearest first, without a gap
            const u32 incl_in = m_incl & (n_ready == 32u ? 0xffffffffu : ((1u << n_ready) - 1u));
            const u32 take = incl_in ? (u32)__ffs((int)incl_in) : n_ready;          // up to and including the first inclusive one
            u64 contrib = lane < take ? (v & EM_VALUE) : 0ull;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
            prefix += contrib;
            if (incl_in) done = true; else t -= (long long)take;
        }
        if (lane == 0) {
            if (tile != 0) st_volatile_u64(status + tile, (prefix + total) | EM_INCL);
            s_base = prefix;
        }
    }
    __syncthreads();
    const u64 base = s_base;
    for (u32 j = tid; j < total; j += 256) {
        // largest k with s_off[k] <= j (zero-count entries share their successor's offset)
        u32 lo = 0, hi = 256;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            u32 mid = (lo + hi) >> 1;
            if (s_off[mid] <= j) lo = mid; else hi = mid;
        }
        const uint2 r = s_rect[lo];
        const u32 x0 = r.x & 0xFFFFu, x1 = r.x >> 16, y0 = r.y & 0xFFFFu;
        const u32 w = x1 - x0;
        const u32 t = j - s_off[lo];
        const u32 ty = t / w, tx = t - ty * w;
        out_tile[base + j] = (y0 + ty) * (u32)grid_x + x0 + tx;
        out_gid[base + j] = s_gid[lo];
    }
}

// Tile boundaries in the sorted instance list (rasterizer_impl.cu:116-138).
__global__ void __launch_bounds__(256)
tile_ranges_kernel(const u32* __restrict__ tile_sorted, u32 R, uint2* __restrict__ ranges)
{
    const u32 i = blockIdx.x * 256 + threadIdx.x;
    if (i >= R) return;
    const u32 cur = tile_sorted[i];
    if (i == 0) ranges[cur].x = 0;
    else {
        const u32 prev = tile_sorted[i - 1];
        if (cur != prev) { ranges[prev].y = i; ranges[cur].x = i; }
    }
    if (i == R - 1) ranges[cur].y = R;
}

// ---- compositing ------------------------------------------------------------------------
// One 16x16 tile per block, one pixel per thread (each warp covers an 8x4 pixel patch so
// that rejection is coherent within a warp). Batches of 256 splat records are staged in
// shared memory with cp.async, double-buffered so the gather of batch i+1 overlaps the
// blending of batch i.
constexpr int CB = 256;   // batch size

struct __align__(16) Stage { float4 A[CB]; float4 B[CB]; float4 C[CB]; };

__device__ __forceinline__ void stage_fill(Stage& st, const u32* __restrict__ list, u32 begin, u32 end,
                                           u32 first, bool reverse, const float4* __restrict__ recA,
                                           const float4* __restrict__ recB, const float4* __restrict__ recC)
{
    const u32 t = threadIdx.x;
    const u32 pos = first + t;
    if (pos < end - begin) {
        const u32 g = __ldg(list + (reverse ? (end - 1 - pos) : (begin + pos)));
        cp_async16(&st.A[t], recA + g);
        cp_async16(&st.B[t], recB + g);
        cp_async16(&st.C[t], recC + g);
    }
}

__global__ void __launch_bounds__(TILE_PIXELS)
composite_fwd_kernel(const uint2* __restrict__ ranges, const u32* __restrict__ list, int W, int H, int grid_x,
                     const float4* __restrict__ recA, const float4* __restrict__ recB,
                     const float4* __restrict__ recC, const float* __restrict__ bg,
                     float* __restrict__ final_T, u32* __restrict__ n_contrib,
                     float* __restrict__ out_color, float* __restrict__ out_depth)
{
    __shared__ Stage stage[2];
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 tile = blockIdx.x;
    const u32 tx = tile % (u32)grid_x, ty = tile / (u32)grid_x;
    const u32 px = tx * TILE_X + (warp & 1) * 8 + (lane & 7);
    const u32 py = ty * TILE_Y + (warp >> 1) * 4 + (lane >> 3);
    const bool inside = px < (u32)W && py < (u32)H;
    const float fxp = (float)px, fyp = (float)py;
    const float patch_x = (float)(tx * TILE_X + (warp & 1) * 8), patch_y = (float)(ty * TILE_Y + (warp >> 1) * 4);
    const uint2 range = ranges[tile];
    const u32 n = range.y - range.x;
    const int rounds = (int)((n + CB - 1) / CB);

    bool done = !inside;
    float T = 1.0f, C0 = 0.f, C1 = 0.f, C2 = 0.f, Dp = 0.f;
    u32 last = 0;

    if (rounds > 0) stage_fill(stage[0], list, range.x, range.y, 0, false, recA, recB, recC);
    cp_async_commit();
    for (int r = 0; r < rounds; ++r) {
        if (r + 1 < rounds) stage_fill(stage[(r + 1) & 1], list, range.x, range.y, (u32)(r + 1) * CB, false, recA, recB, recC);
        cp_async_commit();
        cp_async_wait<1>();
        // all threads see batch r; also the block-wide early-out vote of forward.cu:312
        if (__syncthreads_count(done) == TILE_PIXELS) break;
        const Stage& st = stage[r & 1];
        const int cnt = (int)min((u32)CB, n - (u32)r * CB);
        // Each warp first tests the 256 staged splats against its own 8x4 pixel patch (one splat per
        // lane and round, conservative ellipse-vs-box bound) and then walks only the survivors, all 32
        // lanes in lock-step (finished pixels are predicated off).  Rejected (patch, splat) pairs thus
        // cost ~1.6 instructions instead of a full per-pixel evaluation, and the warp-uniform loop keeps
        // the lanes converged, which the data-dependent `continue`s of forward.cu:328-366 do not.
        u32 masks[CB / 32];
#pragma unroll
        for (int q = 0; q < CB / 32; ++q) {
            const int j = q * 32 + (int)lane;
            const bool keep = j < cnt && splat_may_touch_patch(st.A[j], st.B[j], patch_x, patch_y);
            masks[q] = __ballot_sync(0xffffffffu, keep);
        }
        bool all_done = __all_sync(0xffffffffu, done);
#pragma unroll
        for (int q = 0; q < CB / 32; ++q) {
            u32 m = masks[q];
            while (m != 0 && !all_done) {
                const int j = q * 32 + __ffs(m) - 1;
                m &= m - 1;
                const float4 A = st.A[j];
                const float4 B = st.B[j];
                const float dx = A.x - fxp, dy = A.y - fyp;
                const float power = -0.5f * (A.z * dx * dx + B.x * dy * dy) - A.w * dx * dy;
                if (!done && !(power > 0.0f) && !(power < B.w)) {
                    const float alpha = fminf(0.99f, B.y * expf(power));
                    if (!(alpha < 1.0f / 255.0f)) {
                        const float test_T = T * (1 - alpha);
                        if (test_T < 0.0001f) {
                            done = true;
                        } else {
                            const float4 Cc = st.C[j];
                            C0 += Cc.x * alpha * T;
                            C1 += Cc.y * alpha * T;
                            C2 += Cc.z * alpha * T;
                            Dp += B.z * alpha * T;
                            T = test_T;
                            last = (u32)r * CB + (u32)j + 1u;
                        }
                    }
                }
                all_done = __all_sync(0xffffffffu, done);
            }
        }
        __syncthreads();   // batch r fully consumed before its buffer is refilled
    }
    cp_async_wait<0>();
    if (inside) {
        const size_t pid = (size_t)py * W + px;
        const size_t HW = (size_t)H * W;
        final_T[pid] = T;
        n_contrib[pid] = last;
        out_color[pid] = C0 + T * bg[0];
        out_color[HW + pid] = C1 + T * bg[1];
        out_color[2 * HW + pid] = C2 + T * bg[2];
        out_depth[pid] = Dp;
    }
}


// (A two-pixels-per-lane variant with packed FP32 pairs, as in composite_bwd2_kernel, was built and measured: bit-identical
// outputs, 0.436 vs 0.425 ms for stage 2 at 1M / 1280x720 -- the forward has no reduction to amortise and its two accurate expf
// per lane do not pack -- so it was not kept.)

__global__ void mark_visible_kernel(int P, const float* __restrict__ means, const float* __restrict__ view,
                                    unsigned char* __restrict__ present)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P) return;
    float3 p = make_float3(means[3 * idx], means[3 * idx + 1], means[3 * idx + 2]);
    float3 pv = xform43(p, view);
    present[idx] = (pv.z <= 0.2f) ? 0 : 1;   // auxiliary.h:154
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host-side orchestration
// ---------------------------------------------------------------------------------------------
struct RastDims { int grid_x, grid_y; size_t tiles, npix; int tile_bits; };
static RastDims dims_of(int W, int H) {
    RastDims d;
    d.grid_x = (W + TILE_X - 1) / TILE_X; d.grid_y = (H + TILE_Y - 1) / TILE_Y;
    d.tiles = (size_t)d.grid_x * d.grid_y; d.npix = (size_t)W * H;
    d.tile_bits = tile_bits_for(d.tiles);
    return d;
}

int rast_buffer_sizes(int P, long long R, int W, int H, size_t out[3])
{
    if (P < 0 || R < 0 || W <= 0 || H <= 0) { set_error("rast_buffer_sizes: bad arguments"); return -1; }
    RastDims d = dims_of(W, H);
    GeomState::carve(nullptr, (size_t)P, &out[0]);
    BinState::carve(nullptr, (size_t)P, (size_t)R, d.tile_bits, &out[1]);
    ImgState::carve(nullptr, d.npix, d.tiles, &out[2]);
    return 0;
}

int rast_forward_stage1(int P, int D, int M, int W, int H, const float* means3D, const float* shs,
                        const float* colors_precomp, const float* opacities, const float* scales,
                        float scale_modifier, const float* rotations, const float* cov3D_precomp,
                        const float* viewmatrix, const float* projmatrix, const float* campos,
                        float tan_fovx, float tan_fovy, int prefiltered, int* radii, void* geom_buf,
                        size_t geom_bytes, unsigned long long* host_counters, cudaStream_t stream)
{
    if (P <= 0) { if (host_counters) host_counters[0] = host_counters[1] = 0; return 0; }
    if (!colors_precomp && !shs) { set_error("rast_forward: need SHs or precomputed colours"); return -1; }
    if (!cov3D_precomp && (!scales || !rotations)) { set_error("rast_forward: need scales+rotations or cov3D"); return -1; }
    if (!colors_precomp && (D < 0 || (D + 1) * (D + 1) > M)) { set_error("rast_forward: sh degree %d needs %d coefficients, have %d", D, (D + 1) * (D + 1), M); return -1; }
    if (!colors_precomp && D > 3) { set_error("rast_forward: sh degree > 3 unsupported"); return -1; }
    RastDims d = dims_of(W, H);
    if (d.grid_x > 65535 || d.grid_y > 65535) { set_error("rast_forward: image too large"); return -1; }
    size_t need;
    GeomState g = GeomState::carve(geom_buf, (size_t)P, &need);
    if (geom_bytes < need) { set_error("rast_forward: geometry buffer too small (%zu < %zu)", geom_bytes, need); return -1; }
    cudaMemsetAsync(g.counters, 0, 4 * sizeof(unsigned long long), stream);
    PreArgs a;
    a.P = P; a.D = D; a.M = M; a.W = W; a.H = H;
    a.means = means3D; a.scales = scales; a.rots = rotations; a.opac = opacities; a.shs = shs;
    a.cov3d_pre = cov3D_precomp; a.colors_pre = colors_precomp;
    a.view = viewmatrix; a.proj = projmatrix; a.campos = campos;
    a.scale_mod = scale_modifier; a.tanx = tan_fovx; a.tany = tan_fovy;
    a.fx = W / (2.0f * tan_fovx); a.fy = H / (2.0f * tan_fovy);
    a.grid_x = d.grid_x; a.grid_y = d.grid_y; a.prefiltered = prefiltered; a.radii = radii; a.g = g;
    const size_t smem = colors_precomp ? 0 : (size_t)PRE_WARPS * 32 * (3 * M + 1) * sizeof(float);
    if (smem > 48 * 1024) {
        if (smem > 200 * 1024) { set_error("rast_forward: too many SH coefficients"); return -1; }
        cudaFuncSetAttribute(preprocess_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    {
        ProfScope prof(PROF_PREPROCESS_FWD, stream);
        preprocess_fwd_kernel<<<(P + PRE_THREADS - 1) / PRE_THREADS, PRE_THREADS, smem, stream>>>(a);
    }
    if (check_launch("preprocess_fwd")) return -1;
    // The one device->host read of the forward pass (the reference does the same blocking
    // 4-byte copy at rasterizer_impl.cu:282): the caller sizes the binning buffer from it.
    // The depth sort of the Gaussians does not depend on that count, so it is queued BEHIND the copy and the host waits on an
    // event recorded between the two: the GPU sorts while the host reads the counters, allocates and launches stage 2.
    static thread_local cudaEvent_t ev_read = nullptr;
    if (host_counters) {
        if (!ev_read && cudaEventCreateWithFlags(&ev_read, cudaEventDisableTiming) != cudaSuccess) { check_launch("rast_forward_stage1 event"); return -1; }
        if (cudaMemcpyAsync(host_counters, g.counters, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
            cudaEventRecord(ev_read, stream) != cudaSuccess) {
            check_launch("rast_forward_stage1 readback");
            return -1;
        }
    }
    // depth order of the Gaussians (stable; culled ones carry key 0xFFFFFFFF and sink); which side holds the result depends
    // on P only (stage 2 recomputes it)
    {
        ProfScope prof(PROF_DEPTH_SORT, stream);
        if (radix_sort_pairs(g.depth_key, g.order_iota, g.gkeys_b, g.gvals_b, (size_t)P, 0, 32, g.sort_temp, g.sort_temp_bytes, stream) < 0) return -1;
    }
    if (host_counters) {
        if (cudaEventSynchronize(ev_read) != cudaSuccess) { check_launch("rast_forward_stage1 readback"); return -1; }
        if (host_counters[0] >= (1ull << 30)) { set_error("rast_forward: %llu instances exceed the 2^30 limit", host_counters[0]); return -1; }
    }
    return 0;
}

int rast_forward_stage2(int P, long long R, long long n_visible, int W, int H, const float* bg,
                        void* geom_buf, void* bin_buf, size_t bin_bytes, void* img_buf, size_t img_bytes,
                        float* out_color, float* out_depth, cudaStream_t stream)
{
    RastDims d = dims_of(W, H);
    size_t need_img, need_bin, tmp;
    ImgState img = ImgState::carve(img_buf, d.npix, d.tiles, &need_img);
    if (img_bytes < need_img) { set_error("rast_forward: image buffer too small"); return -1; }
    GeomState g = GeomState::carve(geom_buf, (size_t)(P > 0 ? P : 0), &tmp);
    BinState b = BinState::carve(bin_buf, (size_t)(P > 0 ? P : 0), (size_t)R, d.tile_bits, &need_bin);
    if (bin_bytes < need_bin) { set_error("rast_forward: binning buffer too small (%zu < %zu)", bin_bytes, need_bin); return -1; }
    cudaMemsetAsync(img.ranges, 0, d.tiles * sizeof(uint2), stream);
    const u32* sorted_list = b.ivals_a;
    if (P > 0 && R > 0) {
        // 1. depth order of the Gaussians: sorted by stage 1 (queued behind its counter read-back)
        int side = radix_plan((size_t)P, 0, 32).passes & 1;
        const u32* sorted_gid = side ? g.gvals_b : g.order_iota;
        // 2. (tile, gaussian) instances in depth order
        const u32 nblk = (u32)((n_visible + 255) / 256);
        {
        ProfScope prof(PROF_EMIT, stream);
        cudaMemsetAsync(b.emit_status, 0, ((size_t)nblk + 1) * sizeof(u64), stream);
        cudaMemsetAsync(b.emit_ticket, 0, 64 * sizeof(u32), stream);
        emit_instances_kernel<<<nblk, 256, 0, stream>>>(sorted_gid, (u32)n_visible, g.tiles_touched, g.rect,
                                                        d.grid_x, b.ikeys_a, b.ivals_a, b.emit_status, b.emit_ticket);
        }
        // 3. stable sort by tile id => (tile, depth, index) order
        {
            ProfScope prof(PROF_TILE_SORT, stream);
            side = radix_sort_pairs(b.ikeys_a, b.ivals_a, b.ikeys_b, b.ivals_b, (size_t)R, 0, d.tile_bits,
                                    b.sort_temp, b.sort_temp_bytes, stream);
        }
        if (side < 0) return -1;
        const u32* sorted_tile = side ? b.ikeys_b : b.ikeys_a;
        sorted_list = side ? b.ivals_b : b.ivals_a;
        // 4. per-tile ranges
        ProfScope prof(PROF_TILE_RANGES, stream);
        tile_ranges_kernel<<<(unsigned)((R + 255) / 256), 256, 0, stream>>>(sorted_tile, (u32)R, img.ranges);
    }
    ProfScope prof(PROF_COMPOSITE_FWD, stream);
    // 5. compositing (runs for empty scenes too: background only)
    composite_fwd_kernel<<<(unsigned)d.tiles, TILE_PIXELS, 0, stream>>>(
        img.ranges, sorted_list, W, H, d.grid_x, g.recA, g.recB, g.recC, bg, img.final_T, img.n_contrib,
        out_color, out_depth);
    return check_launch("rast_forward_stage2");
}

int mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                 unsigned char* present, cudaStream_t stream)
{
    (void)projmatrix;
    if (P <= 0) return 0;
    mark_visible_kernel<<<(P + 255) / 256, 256, 0, stream>>>(P, means3D, viewmatrix, present);
    return check_launch("mark_visible");
}

}  // namespace b200gs
