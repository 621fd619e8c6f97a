// HexPlane multi-resolution feature sampling, forward and backward.
//
// Replaces, per call, the 6*levels F.grid_sample launches + 5*levels multiplies + cat of
// scene/hexplane.py:73-106 (interpolate_ms_features) and the normalisation of :19-20,
// :153-164 with one kernel each way.  Semantics restated from there and from ATen's
// grid_sampler_2d (bilinear, align_corners=True, padding_mode='border'):
//   n      = (xyz - aabb[0]) * (2 / (aabb[1] - aabb[0])) - 1       aabb[0] = max, aabb[1] = min
//   c      = (n.x, n.y, n.z, t)                                      t used raw
//   plane k of a level pairs coordinates (a,b) in (0,1)(0,2)(0,3)(1,2)(1,3)(2,3); x = c[a]
//            indexes the plane's width (resolution of a), y = c[b] its height
//   ix     = clamp(((x + 1) / 2) * (W - 1), 0, W - 1)               same for iy
//   value  = nw*w_nw + ne*w_ne + sw*w_sw + se*w_se                   corner order of ATen
//   feature[level] = 1 * v0 * v1 * v2 * v3 * v4 * v5                 (left to right), levels concatenated
// Planes are read CHANNELS-LAST ([H][W][C] in memory, C = 16 or 32; the nn.Parameter keeps its
// [1,C,H,W] shape with torch.channels_last strides): C/4 lanes serve one point with four channels
// each, so every texel fetch is one coalesced line of C floats (128 bytes at C = 32, 64 at C = 16).
#include "common.cuh"
#include "radix_sort.cuh"
#include "tc5_common.cuh"
#include "../../include/b200gs.h"

namespace b200gs {

namespace {

constexpr int HP_MAXL = B200GS_HEXPLANE_MAX_LEVELS;
constexpr int TR_C = 32;                 // channels of the pre-blended time-row kernels (32-channel planes only)

// Channel layout of the six-plane kernels: a point slot is C/4 lanes x 4 channels, so one LDG.128 per lane fetches a whole
// texel; C = 32: 8 lanes, 4 slots per warp; C = 16: 4 lanes, 8 slots per warp.
template <int C> struct Lanes {
    static_assert(C == 16 || C == 32, "HexPlane planes have 16 or 32 channels");
    static constexpr int per_slot = C / 4, slots = 32 / per_slot;
};


struct Bilinear {
    int o_nw, o_ne, o_sw, o_se;          // texel offsets (in texels), -1 if out of bounds
    float w_nw, w_ne, w_sw, w_se;
    float ix, iy;                        // clamped pixel coordinates
    float gx_mult, gy_mult;              // d(ix)/d(coord), zero where the border clamp is active
    int ix_nw, iy_nw;
};

__device__ __forceinline__ float unnormalize_clip(float coord, int size, float& mult)
{
    // ATen grid_sampler_compute_source_index_set_grad, align_corners = true, border padding
    float v = ((coord + 1.f) / 2) * (size - 1);
    mult = (float)(size - 1) / 2;
    const float hi = (float)(size - 1);
    if (v <= 0.f) { v = 0.f; mult = 0.f; }          // clip_coordinates_set_grad: gradient 0 at/below 0
    else if (v >= hi) { v = hi; mult = 0.f; }       // and at/above size-1
    return v;
}

__device__ __forceinline__ Bilinear bilinear_setup(float x, float y, int W, int H)
{
    Bilinear b;
    b.ix = unnormalize_clip(x, W, b.gx_mult);
    b.iy = unnormalize_clip(y, H, b.gy_mult);
    const float fx = floorf(b.ix), fy = floorf(b.iy);
    b.ix_nw = (int)fx; b.iy_nw = (int)fy;
    const float ix_ne = fx + 1.f, iy_sw = fy + 1.f;
    b.w_nw = (ix_ne - b.ix) * (iy_sw - b.iy);
    b.w_ne = (b.ix - fx) * (iy_sw - b.iy);
    b.w_sw = (ix_ne - b.ix) * (b.iy - fy);
    b.w_se = (b.ix - fx) * (b.iy - fy);
    const bool x0 = b.ix_nw >= 0 && b.ix_nw < W, x1 = b.ix_nw + 1 >= 0 && b.ix_nw + 1 < W;
    const bool y0 = b.iy_nw >= 0 && b.iy_nw < H, y1 = b.iy_nw + 1 >= 0 && b.iy_nw + 1 < H;
    b.o_nw = (x0 && y0) ? b.iy_nw * W + b.ix_nw : -1;
    b.o_ne = (x1 && y0) ? b.iy_nw * W + b.ix_nw + 1 : -1;
    b.o_sw = (x0 && y1) ? (b.iy_nw + 1) * W + b.ix_nw : -1;
    b.o_se = (x1 && y1) ? (b.iy_nw + 1) * W + b.ix_nw + 1 : -1;
    return b;
}

// ---- 128-bit path: a warp serves 32/(C/4) points at once (4 at C = 32, 8 at C = 16); the C/4 lanes of a point slot own 4
// channels each, so one LDG.128 per lane fetches a whole texel per slot. Points are visited in
// `order` (a cell-sorted permutation, see hexplane_order below) so that neighbouring warps touch
// the same few texels and the gathers are served by L1 instead of L2.
template <int C>
__device__ __forceinline__ float4 ld4(const float* __restrict__ plane, int texel, int cg)
{
    return texel >= 0 ? __ldg(reinterpret_cast<const float4*>(plane + (size_t)texel * C) + cg)
                      : make_float4(0.f, 0.f, 0.f, 0.f);
}

__device__ __forceinline__ float interp1(float nw, float ne, float sw, float se, const Bilinear& b)
{
    float acc = __fmul_rn(nw, b.w_nw);
    acc = __fmaf_rn(ne, b.w_ne, acc);
    acc = __fmaf_rn(sw, b.w_sw, acc);
    acc = __fmaf_rn(se, b.w_se, acc);
    return acc;
}

__device__ __forceinline__ float4 interp4(const float4 nw, const float4 ne, const float4 sw, const float4 se, const Bilinear& b)
{
    return make_float4(interp1(nw.x, ne.x, sw.x, se.x, b), interp1(nw.y, ne.y, sw.y, se.y, b),
                       interp1(nw.z, ne.z, sw.z, se.z, b), interp1(nw.w, ne.w, sw.w, se.w, b));
}

// The aabb is the same for every point: its three IEEE divisions are done once per thread, not once per point.
struct AabbNorm { float a0[3], scale[3]; };
__device__ __forceinline__ AabbNorm aabb_norm(const float* __restrict__ aabb)
{
    AabbNorm n;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float a1 = __ldg(aabb + 3 + a);
        n.a0[a] = __ldg(aabb + a);
        n.scale[a] = __fdiv_rn(2.0f, __fsub_rn(a1, n.a0[a]));
    }
    return n;
}
__device__ __forceinline__ void normalized_coords(const float* __restrict__ pts, const float* __restrict__ times,
                                                  float time_scalar, const AabbNorm& n, size_t g,
                                                  float c[4], float scale[3])
{
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        scale[a] = n.scale[a];
        c[a] = __fsub_rn(__fmul_rn(__fsub_rn(__ldg(pts + 3 * g + a), n.a0[a]), n.scale[a]), 1.0f);
    }
    c[3] = times ? __ldg(times + g) : time_scalar;
}

template <int K> struct Pair;
template <> struct Pair<0> { static constexpr int a = 0, b = 1; };
template <> struct Pair<1> { static constexpr int a = 0, b = 2; };
template <> struct Pair<2> { static constexpr int a = 0, b = 3; };
template <> struct Pair<3> { static constexpr int a = 1, b = 2; };
template <> struct Pair<4> { static constexpr int a = 1, b = 3; };
template <> struct Pair<5> { static constexpr int a = 2, b = 3; };

template <int C, int K>
__device__ __forceinline__ float4 sample_plane(const b200gs_hexplane_desc& d, int l, const float c[4], int cg, Bilinear& b)
{
    b = bilinear_setup(c[Pair<K>::a], c[Pair<K>::b], d.res[l][Pair<K>::a], d.res[l][Pair<K>::b]);
    const float* plane = d.plane[l][K];
    return interp4(ld4<C>(plane, b.o_nw, cg), ld4<C>(plane, b.o_ne, cg), ld4<C>(plane, b.o_sw, cg), ld4<C>(plane, b.o_se, cg), b);
}

__device__ __forceinline__ float4 mul4(const float4 a, const float4 b)
{
    return make_float4(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y), __fmul_rn(a.z, b.z), __fmul_rn(a.w, b.w));
}

// C = 16: five resident CTAs requested explicitly; without the bound ptxas keeps the same 48 registers but spills the aabb
// origin to the stack and reloads it per point.  C = 32 keeps the plain bound (its code is unchanged by the 16-channel layout).
template <int C>
__global__ void __launch_bounds__(256, C == 16 ? 5 : 0)
hexplane_fwd_kernel(const __grid_constant__ b200gs_hexplane_desc d, long long P, const float* __restrict__ pts,
                    const unsigned int* __restrict__ order, const float* __restrict__ times, float time_scalar,
                    int mask, const float* __restrict__ factor, float* __restrict__ feat)
{
    constexpr int LPS = Lanes<C>::per_slot, SPW = Lanes<C>::slots;
    const int lane = threadIdx.x & 31, slot = lane / LPS, cg = lane % LPS;
    const AabbNorm an = aabb_norm(d.aabb);
    const int F = d.levels * C;
    // blocked assignment: a CTA walks ONE contiguous run of the (cell-sorted) order, so the texels of a small 3-D
    // region stay in its SM's L1 from one iteration to the next (a grid-stride walk re-fetched them from L2)
    const long long ppi = (long long)(blockDim.x >> 5) * SPW;                    // points per CTA iteration
    const long long chunk = ((P + gridDim.x - 1) / gridDim.x + ppi - 1) / ppi * ppi;
    const long long begin = (long long)blockIdx.x * chunk, end = begin + chunk < P ? begin + chunk : P;
    for (long long base = begin + (long long)(threadIdx.x >> 5) * SPW; base < end; base += ppi) {
        const long long i = base + slot;
        if (i >= end) continue;
        const size_t g = order ? (size_t)__ldg(order + i) : (size_t)i;
        float c[4], scale[3];
        normalized_coords(pts, times, time_scalar, an, g, c, scale);
        for (int l = 0; l < d.levels; ++l) {
            Bilinear b;
            // feature = factor * prod_{k in mask} plane_k; mask = all six planes and no factor is the reference's
            // left-to-right product (hexplane.py:87-96)
            float4 f = factor ? __ldg(reinterpret_cast<const float4*>(factor + g * F + l * C + cg * 4)) : make_float4(1.f, 1.f, 1.f, 1.f);
            if (mask & 1) f = mul4(f, sample_plane<C, 0>(d, l, c, cg, b));
            if (mask & 2) f = mul4(f, sample_plane<C, 1>(d, l, c, cg, b));
            if (mask & 4) f = mul4(f, sample_plane<C, 2>(d, l, c, cg, b));
            if (mask & 8) f = mul4(f, sample_plane<C, 3>(d, l, c, cg, b));
            if (mask & 16) f = mul4(f, sample_plane<C, 4>(d, l, c, cg, b));
            if (mask & 32) f = mul4(f, sample_plane<C, 5>(d, l, c, cg, b));
            *reinterpret_cast<float4*>(feat + g * F + l * C + cg * 4) = f;
        }
    }
}

// Backward, pass A: sample one plane ONCE and keep, per lane (4 channels), the value and its derivatives with respect
// to the two pixel coordinates -- v, dv/dix, dv/diy -- plus the clamped pixel coordinates.  Pass B (after the product
// rule has turned d_feature into the plane's upstream gradient gv) rebuilds offsets and weights from (ix, iy) alone,
// scatters gv into the four texels with 128-bit vector reductions and finishes the coordinate gradient as two dot
// products.  Compared with re-sampling the plane in pass B this halves the texel gathers (6.1 KB instead of 12.3 KB
// per point) and drops the second bilinear set-up.
struct PlaneSample { float4 v, dx, dy; float ix, iy; };

template <int C, int K>
__device__ __forceinline__ void sample_plane_full(const b200gs_hexplane_desc& d, int l, const float c[4], int cg, PlaneSample& s)
{
    const int W = d.res[l][Pair<K>::a], H = d.res[l][Pair<K>::b];
    const Bilinear b = bilinear_setup(c[Pair<K>::a], c[Pair<K>::b], W, H);
    const float* plane = d.plane[l][K];
    const float4 nw = ld4<C>(plane, b.o_nw, cg), ne = ld4<C>(plane, b.o_ne, cg), sw = ld4<C>(plane, b.o_sw, cg), se = ld4<C>(plane, b.o_se, cg);
    s.v = interp4(nw, ne, sw, se, b);
    const float fx = (float)b.ix_nw, fy = (float)b.iy_nw;
    const float wx1 = (fx + 1.f) - b.ix, wx0 = b.ix - fx, wy1 = (fy + 1.f) - b.iy, wy0 = b.iy - fy;
    s.dx = make_float4((ne.x - nw.x) * wy1 + (se.x - sw.x) * wy0, (ne.y - nw.y) * wy1 + (se.y - sw.y) * wy0,
                       (ne.z - nw.z) * wy1 + (se.z - sw.z) * wy0, (ne.w - nw.w) * wy1 + (se.w - sw.w) * wy0);
    if (Pair<K>::b < 3)
        s.dy = make_float4((sw.x - nw.x) * wx1 + (se.x - ne.x) * wx0, (sw.y - nw.y) * wx1 + (se.y - ne.y) * wx0,
                           (sw.z - nw.z) * wx1 + (se.z - ne.z) * wx0, (sw.w - nw.w) * wx1 + (se.w - ne.w) * wx0);
    s.ix = b.ix; s.iy = b.iy;
}

// Offset (floats) of the 1-D gradient row of time plane (a, t) of level l inside one replica of the row scratch.
template <int C>
__device__ __host__ __forceinline__ size_t time_row_offset(const b200gs_hexplane_desc& d, int l, int a)
{
    size_t o = 0;
    for (int ll = 0; ll < l; ++ll) o += (size_t)(d.res[ll][0] + d.res[ll][1] + d.res[ll][2]);
    for (int aa = 0; aa < a; ++aa) o += (size_t)d.res[l][aa];
    return o * C;
}
template <int C>
__device__ __host__ __forceinline__ size_t time_row_floats(const b200gs_hexplane_desc& d) { return time_row_offset<C>(d, d.levels, 0); }

template <int C, int K>
__device__ __forceinline__ void plane_backward_full(const b200gs_hexplane_desc& d, int l, int cg, const PlaneSample& s,
                                                    const float4 gv, float gc[3], float* __restrict__ rows)
{
    const int W = d.res[l][Pair<K>::a], H = d.res[l][Pair<K>::b];
    float* gp = d.grad_plane[l][K];
    const float fx = floorf(s.ix), fy = floorf(s.iy);
    const int ixn = (int)fx, iyn = (int)fy;
    if (Pair<K>::b == 3 && rows != nullptr) {
        // The whole launch shares one timestamp, so every point hits the same two rows of this plane: 4 M reductions onto
        // a few hundred 128-byte lines serialise in L2.  Reduce along x only, into this CTA's replica of a 1-D row
        // (weights wx1 / wx0); hexplane_time_rows_flush then adds wy1 / wy0 times the replica sum to the two plane rows.
        if (gp != nullptr && (gv.x != 0.f || gv.y != 0.f || gv.z != 0.f || gv.w != 0.f)) {
            const float wx1 = (fx + 1.f) - s.ix, wx0 = s.ix - fx;
            float* base = rows + time_row_offset<C>(d, l, Pair<K>::a) + (size_t)ixn * C + cg * 4;
            red_add_v4(base, gv.x * wx1, gv.y * wx1, gv.z * wx1, gv.w * wx1);
            if (ixn + 1 < W) red_add_v4(base + C, gv.x * wx0, gv.y * wx0, gv.z * wx0, gv.w * wx0);
        }
    } else
    if (gp != nullptr && (gv.x != 0.f || gv.y != 0.f || gv.z != 0.f || gv.w != 0.f)) {
        const float wx1 = (fx + 1.f) - s.ix, wx0 = s.ix - fx, wy1 = (fy + 1.f) - s.iy, wy0 = s.iy - fy;
        const float w_nw = wx1 * wy1, w_ne = wx0 * wy1, w_sw = wx1 * wy0, w_se = wx0 * wy0;
        const bool x1 = ixn + 1 < W, y1 = iyn + 1 < H;            // (ixn, iyn) itself is always inside: the coordinates are clamped
        float* base = gp + ((size_t)iyn * W + ixn) * C + cg * 4;
        red_add_v4(base, gv.x * w_nw, gv.y * w_nw, gv.z * w_nw, gv.w * w_nw);
        if (x1) red_add_v4(base + C, gv.x * w_ne, gv.y * w_ne, gv.z * w_ne, gv.w * w_ne);
        if (y1) red_add_v4(base + (size_t)W * C, gv.x * w_sw, gv.y * w_sw, gv.z * w_sw, gv.w * w_sw);
        if (x1 && y1) red_add_v4(base + (size_t)(W + 1) * C, gv.x * w_se, gv.y * w_se, gv.z * w_se, gv.w * w_se);
    }
    // clip_coordinates_set_grad: the coordinate gradient vanishes where the border clamp is active
    if (Pair<K>::a < 3) {
        const float mult = (s.ix <= 0.f || s.ix >= (float)(W - 1)) ? 0.f : (float)(W - 1) / 2;
        gc[Pair<K>::a] += mult * (gv.x * s.dx.x + gv.y * s.dx.y + gv.z * s.dx.z + gv.w * s.dx.w);
    }
    if (Pair<K>::b < 3) {
        const float mult = (s.iy <= 0.f || s.iy >= (float)(H - 1)) ? 0.f : (float)(H - 1) / 2;
        gc[Pair<K>::b] += mult * (gv.x * s.dy.x + gv.y * s.dy.y + gv.z * s.dy.z + gv.w * s.dy.w);
    }
}

template <int C>
__global__ void __launch_bounds__(128, 3)
hexplane_bwd_kernel(const __grid_constant__ b200gs_hexplane_desc d, long long P, const float* __restrict__ pts,
                    const unsigned int* __restrict__ order, const float* __restrict__ times, float time_scalar,
                    int mask, const float* __restrict__ factor, float* __restrict__ dfactor /* [P,F], accumulated, or null */,
                    const float* __restrict__ dfeat, float* __restrict__ dpts /* [P,3], written */,
                    float* __restrict__ time_rows /* [replicas][time_row_floats], or null */, int replicas)
{
    constexpr int LPS = Lanes<C>::per_slot, SPW = Lanes<C>::slots;
    float* rows = time_rows ? time_rows + (size_t)(blockIdx.x % replicas) * time_row_floats<C>(d) : nullptr;
    const int lane = threadIdx.x & 31, slot = lane / LPS, cg = lane % LPS;
    const AabbNorm an = aabb_norm(d.aabb);
    const int F = d.levels * C;
    const long long ppi = (long long)(blockDim.x >> 5) * SPW;                    // blocked assignment, see the forward
    const long long chunk = ((P + gridDim.x - 1) / gridDim.x + ppi - 1) / ppi * ppi;
    const long long begin = (long long)blockIdx.x * chunk, end = begin + chunk < P ? begin + chunk : P;
    for (long long base = begin + (long long)(threadIdx.x >> 5) * SPW; base < end; base += ppi) {
        const long long i = base + slot;
        const bool valid = i < end;
        const size_t g = valid ? (order ? (size_t)__ldg(order + i) : (size_t)i) : 0;
        float c[4], scale[3];
        normalized_coords(pts, times, time_scalar, an, g, c, scale);
        float gc[3] = {0.f, 0.f, 0.f};
        if (valid) {
            for (int l = 0; l < d.levels; ++l) {
                const float4 gout = __ldg(reinterpret_cast<const float4*>(dfeat + g * F + l * C + cg * 4));
                auto mul = [](const float4 a, const float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); };
                // planes outside `mask` count as the constant 1 (their factor arrives through `factor` instead)
                const float4 ones = make_float4(1.f, 1.f, 1.f, 1.f);
                PlaneSample s0, s1, s2, s3, s4, s5;
                s0.v = s1.v = s2.v = s3.v = s4.v = s5.v = ones;
                if (mask & 1) sample_plane_full<C, 0>(d, l, c, cg, s0);
                if (mask & 2) sample_plane_full<C, 1>(d, l, c, cg, s1);
                if (mask & 4) sample_plane_full<C, 2>(d, l, c, cg, s2);
                if (mask & 8) sample_plane_full<C, 3>(d, l, c, cg, s3);
                if (mask & 16) sample_plane_full<C, 4>(d, l, c, cg, s4);
                if (mask & 32) sample_plane_full<C, 5>(d, l, c, cg, s5);
                const float4 go = factor ? mul(gout, __ldg(reinterpret_cast<const float4*>(factor + g * F + l * C + cg * 4))) : gout;
                // prefix / suffix products of the six factors (the forward multiplies left to right)
                const float4 p1 = s0.v, p2 = mul(p1, s1.v), p3 = mul(p2, s2.v), p4 = mul(p3, s3.v), p5 = mul(p4, s4.v);
                const float4 q4 = s5.v, q3 = mul(q4, s4.v), q2 = mul(q3, s3.v), q1 = mul(q2, s2.v), q0 = mul(q1, s1.v);
                if (mask & 1) plane_backward_full<C, 0>(d, l, cg, s0, mul(go, q0), gc, rows);
                if (mask & 2) plane_backward_full<C, 1>(d, l, cg, s1, mul(go, mul(p1, q1)), gc, rows);
                if (mask & 4) plane_backward_full<C, 2>(d, l, cg, s2, mul(go, mul(p2, q2)), gc, rows);
                if (mask & 8) plane_backward_full<C, 3>(d, l, cg, s3, mul(go, mul(p3, q3)), gc, rows);
                if (mask & 16) plane_backward_full<C, 4>(d, l, cg, s4, mul(go, mul(p4, q4)), gc, rows);
                if (mask & 32) plane_backward_full<C, 5>(d, l, cg, s5, mul(go, p5), gc, rows);
                if (dfactor) {                       // d factor += d feature * prod_{k in mask} plane_k
                    float4* da = reinterpret_cast<float4*>(dfactor + g * F + l * C + cg * 4);
                    const float4 prod = mul(p5, s5.v), old = *da;
                    *da = make_float4(old.x + gout.x * prod.x, old.y + gout.y * prod.y, old.z + gout.z * prod.z, old.w + gout.w * prod.w);
                }
            }
        }
        if (dpts != nullptr) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                float s = gc[a];
#pragma unroll
                for (int o = 1; o < LPS; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                gc[a] = s * scale[a];
            }
            if (valid && cg < 3) dpts[3 * g + cg] = cg == 0 ? gc[0] : (cg == 1 ? gc[1] : gc[2]);
        }
    }
}

// Adds the replica-summed 1-D rows to the two time rows of every time plane: G[t0][x] += wy1 * r[x], G[t1][x] += wy0 * r[x].
template <int C>
__global__ void __launch_bounds__(256)
hexplane_time_rows_flush_kernel(const __grid_constant__ b200gs_hexplane_desc d, float time_scalar, const float* __restrict__ rows, int replicas)
{
    const size_t total = time_row_floats<C>(d);
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    int l = 0, a = 0;
    size_t rem = i / C;                                      // texel index over all (level, axis) rows
    for (;; ) {
        const size_t n = (size_t)d.res[l][a];
        if (rem < n) break;
        rem -= n;
        if (++a == 3) { a = 0; ++l; }
    }
    const int K = a == 0 ? 2 : (a == 1 ? 4 : 5), ch = (int)(i % C), x = (int)rem;
    float* gp = d.grad_plane[l][K];
    if (gp == nullptr) return;
    float sum = 0.f;
    for (int r = 0; r < replicas; ++r) sum += rows[(size_t)r * total + i];
    const int W = d.res[l][a], H = d.res[l][3];
    float mult;
    const float iy = unnormalize_clip(time_scalar, H, mult);
    const float fy = floorf(iy);
    const int iyn = (int)fy;
    const float wy1 = (fy + 1.f) - iy, wy0 = iy - fy;
    gp[((size_t)iyn * W + x) * C + ch] += sum * wy1;
    if (iyn + 1 < H) gp[((size_t)(iyn + 1) * W + x) * C + ch] += sum * wy0;
}


// ---- time planes of a one-timestamp launch, served from shared memory ------------------------------------------------
// With the spatial-plane product S shared by the views of a step (see the *_masked variants), a view only needs the
// three time planes (x,t), (y,t), (z,t) of every level -- and the whole view has ONE t.  Each CTA therefore pre-blends
// the two touched time rows of every time plane into a 1-D row  R[x] = wy1 G[t0][x] + wy0 G[t1][x]  in shared memory
// (73.7 KB for the reference's 2-level / 64-128 resolution field).  Sampling becomes a 1-D lerp with no global texel
// traffic at all; the backward accumulates the row gradient in shared memory and adds it to the two plane rows once per
// CTA.  Per point the kernels move only xyz, S, the feature / its gradient and d(S): they are HBM-bound.
struct TimeRowSetup { int off[HP_MAXL][3]; int total; };     // float offsets of row (level, axis) inside the row buffer

__device__ __forceinline__ void time_rows_prepare(const b200gs_hexplane_desc& d, float t, float* __restrict__ R, const TimeRowSetup& ts)
{
    for (int l = 0; l < d.levels; ++l) {
        float mult;
        const int H = d.res[l][3];
        const float iy = unnormalize_clip(t, H, mult);
        const float fy = floorf(iy);
        const int iyn = (int)fy;
        const float wy1 = (fy + 1.f) - iy, wy0 = iy - fy;
        const bool y1 = iyn + 1 < H;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int K = a == 0 ? 2 : (a == 1 ? 4 : 5), W = d.res[l][a];
            const float* g0 = d.plane[l][K] + (size_t)iyn * W * TR_C;
            const float* g1 = g0 + (size_t)W * TR_C;
            // 128-bit loads, four in flight per thread: this runs before every CTA's main loop, so its latency is exposed
#pragma unroll 4
            for (int i = threadIdx.x; i < W * (TR_C / 4); i += blockDim.x) {
                const float4 p0 = __ldg(reinterpret_cast<const float4*>(g0) + i);
                const float4 p1 = y1 ? __ldg(reinterpret_cast<const float4*>(g1) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                reinterpret_cast<float4*>(R + ts.off[l][a])[i] =
                    make_float4(__fmaf_rn(p1.x, wy0, __fmul_rn(p0.x, wy1)), __fmaf_rn(p1.y, wy0, __fmul_rn(p0.y, wy1)),
                                __fmaf_rn(p1.z, wy0, __fmul_rn(p0.z, wy1)), __fmaf_rn(p1.w, wy0, __fmul_rn(p0.w, wy1)));
            }
        }
    }
}

struct RowSample { float4 v, dv; float wx0, wx1, mult; int x0, x1; };

__device__ __forceinline__ RowSample row_sample(const float* __restrict__ row, float coord, int W, int cg)
{
    RowSample r;
    const float ix = unnormalize_clip(coord, W, r.mult);
    const float fx = floorf(ix);
    r.x0 = (int)fx;
    r.x1 = r.x0 + 1 < W ? r.x0 + 1 : r.x0;          // out of range on the right edge: its weight is exactly 0
    r.wx1 = (fx + 1.f) - ix; r.wx0 = ix - fx;
    const float4 a = *reinterpret_cast<const float4*>(row + r.x0 * TR_C + cg * 4);
    const float4 b = *reinterpret_cast<const float4*>(row + r.x1 * TR_C + cg * 4);
    r.v = make_float4(__fmaf_rn(b.x, r.wx0, __fmul_rn(a.x, r.wx1)), __fmaf_rn(b.y, r.wx0, __fmul_rn(a.y, r.wx1)),
                      __fmaf_rn(b.z, r.wx0, __fmul_rn(a.z, r.wx1)), __fmaf_rn(b.w, r.wx0, __fmul_rn(a.w, r.wx1)));
    r.dv = make_float4(b.x - a.x, b.y - a.y, b.z - a.z, b.w - a.w);
    return r;
}

__global__ void __launch_bounds__(512)
hexplane_time_fwd_kernel(const __grid_constant__ b200gs_hexplane_desc d, const __grid_constant__ TimeRowSetup ts, long long P,
                         const float* __restrict__ pts, const unsigned int* __restrict__ order, float t,
                         const float* __restrict__ factor, float* __restrict__ feat, int tiled)
{
    extern __shared__ float R[];
    time_rows_prepare(d, t, R, ts);
    __syncthreads();
    const int lane = threadIdx.x & 31, slot = lane >> 3, cg = lane & 7;
    const AabbNorm an = aabb_norm(d.aabb);
    const int F = d.levels * TR_C;
    const long long ppi = (long long)(blockDim.x >> 5) * 4;
    const long long chunk = ((P + gridDim.x - 1) / gridDim.x + ppi - 1) / ppi * ppi;
    const long long begin = (long long)blockIdx.x * chunk, end = begin + chunk < P ? begin + chunk : P;
    for (long long base = begin + (long long)(threadIdx.x >> 5) * 4; base < end; base += ppi) {
        const long long i = base + slot;
        if (i >= end) continue;
        const size_t g = order ? (size_t)__ldg(order + i) : (size_t)i;
        float c[4], scale[3];
        normalized_coords(pts, nullptr, t, an, g, c, scale);
        for (int l = 0; l < d.levels; ++l) {
            float4 f = factor ? __ldg(reinterpret_cast<const float4*>(factor + g * F + l * TR_C + cg * 4)) : make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
            for (int a = 0; a < 3; ++a) f = mul4(f, row_sample(R + ts.off[l][a], c[a], d.res[l][a], cg).v);
            *reinterpret_cast<float4*>(feat + (tiled ? tc5::stash_off((long long)g, l * TR_C + cg * 4) : g * F + l * TR_C + cg * 4)) = f;
        }
    }
}

// 2 levels (the reference's configuration): compile-time level count, both levels' factor rows requested before the first is
// used, both feature rows stored at the end; same arithmetic per element as the kernel above, bit-identical features.  The
// register budget is set for 2 resident CTAs per SM (the kernel above is capped at 42 registers for 3):
// 0.134 -> 0.112 ms (profiles/r2a_hexplane_time_check.txt).
__global__ void __launch_bounds__(512, 2)
hexplane_time_fwd2_kernel(const __grid_constant__ b200gs_hexplane_desc d, const __grid_constant__ TimeRowSetup ts, long long P,
                          const float* __restrict__ pts, const unsigned int* __restrict__ order, float t,
                          const float* __restrict__ factor, float* __restrict__ feat, int tiled)
{
    constexpr int L = 2, F = L * TR_C;
    extern __shared__ float R[];
    time_rows_prepare(d, t, R, ts);
    __syncthreads();
    const int lane = threadIdx.x & 31, slot = lane >> 3, cg = lane & 7;
    const AabbNorm an = aabb_norm(d.aabb);
    const long long ppi = (long long)(blockDim.x >> 5) * 4;
    const long long chunk = ((P + gridDim.x - 1) / gridDim.x + ppi - 1) / ppi * ppi;
    const long long begin = (long long)blockIdx.x * chunk, end = begin + chunk < P ? begin + chunk : P;
    for (long long base = begin + (long long)(threadIdx.x >> 5) * 4; base < end; base += ppi) {
        const long long i = base + slot;
        if (i >= end) continue;
        const size_t g = order ? (size_t)__ldg(order + i) : (size_t)i;
        float4 f[L];
#pragma unroll
        for (int l = 0; l < L; ++l)
            f[l] = factor ? __ldg(reinterpret_cast<const float4*>(factor + g * F + l * TR_C + cg * 4)) : make_float4(1.f, 1.f, 1.f, 1.f);
        float c[4], scale[3];
        normalized_coords(pts, nullptr, t, an, g, c, scale);
#pragma unroll
        for (int l = 0; l < L; ++l) {
#pragma unroll
            for (int a = 0; a < 3; ++a) f[l] = mul4(f[l], row_sample(R + ts.off[l][a], c[a], d.res[l][a], cg).v);
        }
#pragma unroll
        for (int l = 0; l < L; ++l)
            *reinterpret_cast<float4*>(feat + (tiled ? tc5::stash_off((long long)g, l * TR_C + cg * 4) : g * F + l * TR_C + cg * 4)) = f[l];
    }
}

__global__ void __launch_bounds__(256, 3)
hexplane_time_bwd_kernel(const __grid_constant__ b200gs_hexplane_desc d, const __grid_constant__ TimeRowSetup ts, long long P,
                         const float* __restrict__ pts, const unsigned int* __restrict__ order, float t,
                         const float* __restrict__ factor, float* __restrict__ dfactor, const float* __restrict__ dfeat,
                         float* __restrict__ dpts, float* __restrict__ time_rows /* [replicas][ts.total], zeroed */, int replicas,
                         int tiled_flags)
{
    const int tiled = tiled_flags & 1;
    const bool overwrite = (tiled_flags & 2) != 0;
    extern __shared__ float R[];
    float* rows = time_rows + (size_t)(blockIdx.x % replicas) * ts.total;      // row gradients: this CTA's replica
    time_rows_prepare(d, t, R, ts);
    __syncthreads();
    const int lane = threadIdx.x & 31, slot = lane >> 3, cg = lane & 7;
    const AabbNorm an = aabb_norm(d.aabb);
    const int F = d.levels * TR_C;
    const long long ppi = (long long)(blockDim.x >> 5) * 4;
    const long long chunk = ((P + gridDim.x - 1) / gridDim.x + ppi - 1) / ppi * ppi;
    const long long begin = (long long)blockIdx.x * chunk, end = begin + chunk < P ? begin + chunk : P;
    for (long long base = begin + (long long)(threadIdx.x >> 5) * 4; base < end; base += ppi) {
        const long long i = base + slot;
        const bool valid = i < end;
        const size_t g = valid ? (order ? (size_t)__ldg(order + i) : (size_t)i) : 0;
        float c[4], scale[3];
        normalized_coords(pts, nullptr, t, an, g, c, scale);
        float gc[3] = {0.f, 0.f, 0.f};
        if (valid) {
            for (int l = 0; l < d.levels; ++l) {
                const float4 gout = __ldg(reinterpret_cast<const float4*>(dfeat + (tiled ? tc5::stash_off((long long)g, l * TR_C + cg * 4) : g * F + l * TR_C + cg * 4)));
                const float4 fac = factor ? __ldg(reinterpret_cast<const float4*>(factor + g * F + l * TR_C + cg * 4)) : make_float4(1.f, 1.f, 1.f, 1.f);
                RowSample r[3];
#pragma unroll
                for (int a = 0; a < 3; ++a) r[a] = row_sample(R + ts.off[l][a], c[a], d.res[l][a], cg);
                const float4 go = mul4(gout, fac);
                if (dfactor) {                       // d S += d feature * T
                    float4* da = reinterpret_cast<float4*>(dfactor + g * F + l * TR_C + cg * 4);
                    const float4 T = mul4(mul4(r[0].v, r[1].v), r[2].v), old = overwrite ? make_float4(0.f, 0.f, 0.f, 0.f) : *da;
                    *da = make_float4(old.x + gout.x * T.x, old.y + gout.y * T.y, old.z + gout.z * T.z, old.w + gout.w * T.w);
                }
                if (go.x != 0.f || go.y != 0.f || go.z != 0.f || go.w != 0.f) {
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        const float4 oth = mul4(r[(a + 1) % 3].v, r[(a + 2) % 3].v);
                        const float4 gv = mul4(go, oth);
                        // (shared-memory float atomics are compare-and-swap loops on this architecture; the vector reductions to
                        //  this CTA's replica of the global row buffer are native and four channels wide)
                        float* g0 = rows + ts.off[l][a] + r[a].x0 * TR_C + cg * 4;
                        red_add_v4(g0, gv.x * r[a].wx1, gv.y * r[a].wx1, gv.z * r[a].wx1, gv.w * r[a].wx1);
                        if (r[a].x1 != r[a].x0) {
                            float* g1 = rows + ts.off[l][a] + r[a].x1 * TR_C + cg * 4;
                            red_add_v4(g1, gv.x * r[a].wx0, gv.y * r[a].wx0, gv.z * r[a].wx0, gv.w * r[a].wx0);
                        }
                        gc[a] += r[a].mult * (gv.x * r[a].dv.x + gv.y * r[a].dv.y + gv.z * r[a].dv.z + gv.w * r[a].dv.w);
                    }
                }
            }
        }
        if (dpts != nullptr) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                float s = gc[a];
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                s += __shfl_xor_sync(0xffffffffu, s, 4);
                gc[a] = s * scale[a];
            }
            if (valid && cg < 3) dpts[3 * g + cg] = cg == 0 ? gc[0] : (cg == 1 ? gc[1] : gc[2]);
        }
    }
}

// 2 levels (the reference's configuration): same arithmetic per element as the kernel above, but the level count is a
// compile-time 2, so both levels' d_feature / factor / d_factor rows of a point group are requested before the first one is
// used (the kernel above waits for one level's rows, works, then requests the next: two exposed memory latencies per
// iteration -- 66 % of its stall samples are the first use of a load).  The register budget is set for 2 resident CTAs per
// SM (128 registers and a third fewer warps than 3 at 85 registers): 0.417 -> 0.354 ms (profiles/r2a_hexplane_time_check.txt).
__global__ void __launch_bounds__(256, 2)
hexplane_time_bwd2_kernel(const __grid_constant__ b200gs_hexplane_desc d, const __grid_constant__ TimeRowSetup ts, long long P,
                          const float* __restrict__ pts, const unsigned int* __restrict__ order, float t,
                          const float* __restrict__ factor, float* __restrict__ dfactor, const float* __restrict__ dfeat,
                          float* __restrict__ dpts, float* __restrict__ time_rows, int replicas, int tiled_flags)
{
    constexpr int L = 2, F = L * TR_C;
    const int tiled = tiled_flags & 1;
    const bool overwrite = (tiled_flags & 2) != 0;          // d_factor is WRITTEN, not accumulated (a fresh buffer: no read, no memset)
    extern __shared__ float R[];
    float* rows = time_rows + (size_t)(blockIdx.x % replicas) * ts.total;
    time_rows_prepare(d, t, R, ts);
    __syncthreads();
    const int lane = threadIdx.x & 31, slot = lane >> 3, cg = lane & 7;
    const AabbNorm an = aabb_norm(d.aabb);
    const long long ppi = (long long)(blockDim.x >> 5) * 4;
    const long long chunk = ((P + gridDim.x - 1) / gridDim.x + ppi - 1) / ppi * ppi;
    const long long begin = (long long)blockIdx.x * chunk, end = begin + chunk < P ? begin + chunk : P;
    for (long long base = begin + (long long)(threadIdx.x >> 5) * 4; base < end; base += ppi) {
        const long long i = base + slot;
        const bool valid = i < end;
        const size_t g = valid ? (order ? (size_t)__ldg(order + i) : (size_t)i) : 0;
        // (prefetching the next iteration's rows into L1 was measured: 0.365 vs 0.353 ms, not kept)
        float4 gout[L], fac[L], old[L];
        if (valid) {
#pragma unroll
            for (int l = 0; l < L; ++l) {
                gout[l] = __ldg(reinterpret_cast<const float4*>(dfeat + (tiled ? tc5::stash_off((long long)g, l * TR_C + cg * 4) : g * F + l * TR_C + cg * 4)));
                fac[l] = factor ? __ldg(reinterpret_cast<const float4*>(factor + g * F + l * TR_C + cg * 4)) : make_float4(1.f, 1.f, 1.f, 1.f);
                old[l] = (dfactor && !overwrite) ? *reinterpret_cast<const float4*>(dfactor + g * F + l * TR_C + cg * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        float c[4], scale[3];
        normalized_coords(pts, nullptr, t, an, g, c, scale);
        float gc[3] = {0.f, 0.f, 0.f};
        if (valid) {
#pragma unroll
            for (int l = 0; l < L; ++l) {
                RowSample r[3];
#pragma unroll
                for (int a = 0; a < 3; ++a) r[a] = row_sample(R + ts.off[l][a], c[a], d.res[l][a], cg);
                const float4 go = mul4(gout[l], fac[l]);
                if (dfactor) {                       // d S += d feature * T
                    const float4 T = mul4(mul4(r[0].v, r[1].v), r[2].v);
                    *reinterpret_cast<float4*>(dfactor + g * F + l * TR_C + cg * 4) =
                        make_float4(old[l].x + gout[l].x * T.x, old[l].y + gout[l].y * T.y, old[l].z + gout[l].z * T.z, old[l].w + gout[l].w * T.w);
                }
                if (go.x != 0.f || go.y != 0.f || go.z != 0.f || go.w != 0.f) {
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        const float4 oth = mul4(r[(a + 1) % 3].v, r[(a + 2) % 3].v);
                        const float4 gv = mul4(go, oth);
                        float* g0 = rows + ts.off[l][a] + r[a].x0 * TR_C + cg * 4;
                        red_add_v4(g0, gv.x * r[a].wx1, gv.y * r[a].wx1, gv.z * r[a].wx1, gv.w * r[a].wx1);
                        if (r[a].x1 != r[a].x0) {
                            float* g1 = rows + ts.off[l][a] + r[a].x1 * TR_C + cg * 4;
                            red_add_v4(g1, gv.x * r[a].wx0, gv.y * r[a].wx0, gv.z * r[a].wx0, gv.w * r[a].wx0);
                        }
                        gc[a] += r[a].mult * (gv.x * r[a].dv.x + gv.y * r[a].dv.y + gv.z * r[a].dv.z + gv.w * r[a].dv.w);
                    }
                }
            }
        }
        if (dpts != nullptr) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                float s = gc[a];
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                s += __shfl_xor_sync(0xffffffffu, s, 4);
                gc[a] = s * scale[a];
            }
            if (valid && cg < 3) dpts[3 * g + cg] = cg == 0 ? gc[0] : (cg == 1 ? gc[1] : gc[2]);
        }
    }
}

bool time_rows_setup(const b200gs_hexplane_desc& d, TimeRowSetup& ts)
{
    int o = 0;
    for (int l = 0; l < d.levels; ++l)
        for (int a = 0; a < 3; ++a) { ts.off[l][a] = o; o += d.res[l][a] * TR_C; }
    ts.total = o;
    return (size_t)o * sizeof(float) <= 200 * 1024;             // the pre-blended rows must fit one CTA's shared memory
}

// ---- cell order: a permutation of the points sorted by an 8-bit-per-axis Morton code of their
// normalised position (a pure performance hint: any permutation gives the same results).
__device__ __forceinline__ unsigned int spread8(unsigned int x)
{
    x = (x | (x << 16)) & 0x0300000Fu;
    x = (x | (x << 8)) & 0x0300F00Fu;
    x = (x | (x << 4)) & 0x030C30C3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}

__global__ void __launch_bounds__(256)
hexplane_cellkey_kernel(long long P, const float* __restrict__ pts, const float* __restrict__ aabb,
                        unsigned int* __restrict__ keys, unsigned int* __restrict__ ids)
{
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= P) return;
    unsigned int key = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float a0 = __ldg(aabb + a), a1 = __ldg(aabb + 3 + a);
        float n = ((__ldg(pts + 3 * (size_t)i + a) - a0) / (a1 - a0));          // 0..1 inside the box
        n = fminf(fmaxf(n, 0.f), 1.f);
        key |= spread8((unsigned int)(n * 255.f)) << a;
    }
    keys[i] = key;
    ids[i] = (unsigned int)i;
}


// ---- plane regulariser (scene/gaussian_model.py:730-769 compute_regulation; scene/regulation.py:22-28) ----------
// per level:  w_plane * sum_{k in 0,1,3} S(G_k) + w_time * sum_{k in 2,4,5} S(G_k) + w_l1 * sum_{k in 2,4,5} mean|1 - G_k|
// S(G) = mean over [C, H-2, W] of (G[y+2] - 2 G[y+1] + G[y])^2  (second difference along the plane's HEIGHT).
// One thread owns one (x, 4-channel) column of a channels-last plane and walks it top to bottom with the three
// live second differences in registers: value and gradient in one pass, 8 B/parameter (+4 when the L1 term reads it
// anyway).  dS/dG[j] = (2/N) (d[j] - 2 d[j-1] + d[j-2]),  d[i] defined for 0 <= i <= H-3.
template <int C>
__global__ void __launch_bounds__(128)
hexplane_regulation_kernel(const __grid_constant__ b200gs_hexplane_desc d, float w_plane, float w_time, float w_l1,
                           float* __restrict__ loss)
{
    const int l = blockIdx.y / 6, k = blockIdx.y % 6;
    constexpr int pa[6] = {0, 0, 0, 1, 1, 2}, pb[6] = {1, 2, 3, 2, 3, 3};
    const int W = d.res[l][pa[k]], H = d.res[l][pb[k]];
    const bool is_time = pb[k] == 3;
    const float w_s = is_time ? w_time : w_plane;
    const float* __restrict__ G = d.plane[l][k];
    float* __restrict__ gG = d.grad_plane[l][k];
    const int col = blockIdx.x * 128 + threadIdx.x;            // (x, channel quad)
    float acc = 0.f;
    if (col < W * (C / 4)) {
        const size_t stride = (size_t)W * (C / 4);             // float4 units per row
        const float4* g4 = reinterpret_cast<const float4*>(G) + col;
        float4* o4 = gG ? reinterpret_cast<float4*>(gG) + col : nullptr;
        const float cs = H > 2 ? w_s * 2.f / ((float)C * (float)(H - 2) * (float)W) : 0.f;        // 2 w / N
        const float cl = is_time ? w_l1 / ((float)C * (float)H * (float)W) : 0.f;
        float sq = 0.f, l1 = 0.f;
        float4 t0 = H > 0 ? __ldg(g4) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 t1 = H > 1 ? __ldg(g4 + stride) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 dm1 = make_float4(0.f, 0.f, 0.f, 0.f), dm2 = dm1;            // d[j-1], d[j-2]
        for (int j = 0; j < H; ++j) {
            const float4 t2 = j + 2 < H ? __ldg(g4 + (size_t)(j + 2) * stride) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 dj = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j + 2 < H) {
                dj = make_float4(t2.x - 2.f * t1.x + t0.x, t2.y - 2.f * t1.y + t0.y, t2.z - 2.f * t1.z + t0.z, t2.w - 2.f * t1.w + t0.w);
                sq += dj.x * dj.x + dj.y * dj.y + dj.z * dj.z + dj.w * dj.w;
            }
            float4 g = make_float4(cs * (dj.x - 2.f * dm1.x + dm2.x), cs * (dj.y - 2.f * dm1.y + dm2.y),
                                   cs * (dj.z - 2.f * dm1.z + dm2.z), cs * (dj.w - 2.f * dm1.w + dm2.w));
            if (is_time) {                                     // d/dG mean|1 - G| = -sign(1 - G) / M
                const float e[4] = {1.f - t0.x, 1.f - t0.y, 1.f - t0.z, 1.f - t0.w};
                l1 += fabsf(e[0]) + fabsf(e[1]) + fabsf(e[2]) + fabsf(e[3]);
                g.x -= e[0] > 0.f ? cl : (e[0] < 0.f ? -cl : 0.f); g.y -= e[1] > 0.f ? cl : (e[1] < 0.f ? -cl : 0.f);
                g.z -= e[2] > 0.f ? cl : (e[2] < 0.f ? -cl : 0.f); g.w -= e[3] > 0.f ? cl : (e[3] < 0.f ? -cl : 0.f);
            }
            if (o4) {
                float4* o = o4 + (size_t)j * stride;
                const float4 prev = *o;
                *o = make_float4(prev.x + g.x, prev.y + g.y, prev.z + g.z, prev.w + g.w);
            }
            dm2 = dm1; dm1 = dj; t0 = t1; t1 = t2;
        }
        acc = 0.5f * cs * sq + cl * l1;                        // w * mean(d^2) = (cs / 2) * sum d^2
    }
    if (loss) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        __shared__ float part[4];
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) atomicAdd(loss, part[0] + part[1] + part[2] + part[3]);
    }
}

// Channel counts an entry point accepts (a set of these bits): 16 and 32 are the only layouts compiled.
constexpr unsigned CH16 = 1, CH32 = 2;

int validate(const b200gs_hexplane_desc* d, unsigned channels)
{
    if (!d) { set_error("hexplane: null descriptor"); return -1; }
    if (d->levels < 1 || d->levels > HP_MAXL) { set_error("hexplane: levels=%d unsupported (1..%d)", d->levels, HP_MAXL); return -1; }
    if (!((d->channels == 16 && (channels & CH16)) || (d->channels == 32 && (channels & CH32)))) {
        set_error("hexplane: %d channels per plane unsupported (this entry point takes %s)", d->channels,
                  channels == CH32 ? "32" : "16 or 32");
        return -1;
    }
    if (!d->aabb) { set_error("hexplane: aabb is null"); return -1; }
    for (int l = 0; l < d->levels; ++l) {
        for (int a = 0; a < 4; ++a) if (d->res[l][a] < 1) { set_error("hexplane: bad resolution"); return -1; }
        for (int k = 0; k < 6; ++k) if (!d->plane[l][k]) { set_error("hexplane: plane pointer is null"); return -1; }
    }
    return 0;
}

template <int C>
int grid_for(long long P)
{
    constexpr long long per_block = 8 * Lanes<C>::slots;
    long long blocks = (P + per_block - 1) / per_block;     // 8 warps x 4 (C = 32) or 8 (C = 16) point slots per block
    const long long cap = (long long)NUM_SMS * 8;    // persistent-style cap: 8 resident blocks per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

// The six-plane backward of b200gs_hexplane_backward_masked for C channels (desc validated, P > 0).
template <int C>
int backward_masked(const b200gs_hexplane_desc& d, long long P, const float* pts, const unsigned int* order, const float* times,
                    float time_scalar, int plane_mask, const float* factor, float* d_factor_accum, const float* d_features, float* d_pts,
                    void* time_row_scratch, size_t time_row_scratch_bytes, cudaStream_t stream)
{
    // uniform-time fast path for the time planes' gradient: needs one shared timestamp (times == null) and scratch
    float* rows = nullptr;
    int replicas = 0;
    if (times == nullptr && time_row_scratch != nullptr && (plane_mask & 0x34)) {
        const size_t per = time_row_floats<C>(d) * sizeof(float);
        replicas = (int)(time_row_scratch_bytes / per);
        if (replicas > 64) replicas = 64;
        if (replicas >= 1) {
            rows = (float*)time_row_scratch;
            cudaMemsetAsync(rows, 0, per * replicas, stream);
        }
    }
    // 4 warps x 4 (C = 32) or 8 (C = 16) point slots per block, 3 blocks resident per SM (170 registers)
    constexpr long long per_block = 4 * Lanes<C>::slots;
    long long blocks = (P + per_block - 1) / per_block;
    if (blocks > (long long)NUM_SMS * 12) blocks = (long long)NUM_SMS * 12;
    hexplane_bwd_kernel<C><<<(unsigned)blocks, 128, 0, stream>>>(d, P, pts, order, times, time_scalar, plane_mask & 63, factor,
                                                                 d_factor_accum, d_features, d_pts, rows, replicas);
    if (rows) {
        const size_t total = time_row_floats<C>(d);
        hexplane_time_rows_flush_kernel<C><<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(d, time_scalar, rows, replicas);
    }
    return check_launch("hexplane_backward");
}

}  // namespace
}  // namespace b200gs

using namespace b200gs;

extern "C" {

size_t b200gs_hexplane_order_scratch_bytes(long long P)
{
    const size_t n = P > 0 ? (size_t)P : 0;
    return 3 * align_up(n * sizeof(u32), 256) + radix_plan(n, 0, 24).temp_bytes + 256;
}

int b200gs_hexplane_order(long long P, const float* pts, const float* aabb, unsigned int* order, void* scratch,
                          size_t scratch_bytes, b200gs_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (P <= 0) return 0;
    if (scratch_bytes < b200gs_hexplane_order_scratch_bytes(P)) { set_error("hexplane_order: scratch too small"); return -1; }
    Carver c(scratch);
    u32* keys_a = c.take<u32>((size_t)P); u32* keys_b = c.take<u32>((size_t)P); u32* ids_b = c.take<u32>((size_t)P);
    const size_t tb = radix_plan((size_t)P, 0, 24).temp_bytes;
    void* temp = c.take<char>(tb);
    hexplane_cellkey_kernel<<<(unsigned)((P + 255) / 256), 256, 0, stream>>>(P, pts, aabb, keys_a, order);
    const int side = radix_sort_pairs(keys_a, order, keys_b, ids_b, (size_t)P, 0, 24, temp, tb, stream);
    if (side < 0) return -1;
    if (side == 1) cudaMemcpyAsync(order, ids_b, (size_t)P * sizeof(u32), cudaMemcpyDeviceToDevice, stream);
    return check_launch("hexplane_order");
}

int b200gs_hexplane_forward_masked(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                   const float* times, float time_scalar, int plane_mask, const float* factor, float* features,
                                   b200gs_stream_t stream)
{
    if (validate(desc, CH16 | CH32)) return -1;
    if (P <= 0) return 0;
    if (desc->channels == 16)
        hexplane_fwd_kernel<16><<<grid_for<16>(P), 256, 0, (cudaStream_t)stream>>>(*desc, P, pts, order, times, time_scalar, plane_mask & 63, factor, features);
    else
        hexplane_fwd_kernel<32><<<grid_for<32>(P), 256, 0, (cudaStream_t)stream>>>(*desc, P, pts, order, times, time_scalar, plane_mask & 63, factor, features);
    return check_launch("hexplane_forward");
}

int b200gs_hexplane_forward(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                            const float* times, float time_scalar, float* features, b200gs_stream_t stream)
{
    return b200gs_hexplane_forward_masked(desc, P, pts, order, times, time_scalar, 63, nullptr, features, stream);
}

int b200gs_hexplane_backward_masked(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                    const float* times, float time_scalar, int plane_mask, const float* factor, float* d_factor_accum,
                                    const float* d_features, float* d_pts, void* time_row_scratch, size_t time_row_scratch_bytes,
                                    b200gs_stream_t stream)
{
    if (validate(desc, CH16 | CH32)) return -1;
    if (P <= 0) return 0;
    return desc->channels == 16
        ? backward_masked<16>(*desc, P, pts, order, times, time_scalar, plane_mask, factor, d_factor_accum, d_features, d_pts,
                              time_row_scratch, time_row_scratch_bytes, (cudaStream_t)stream)
        : backward_masked<32>(*desc, P, pts, order, times, time_scalar, plane_mask, factor, d_factor_accum, d_features, d_pts,
                              time_row_scratch, time_row_scratch_bytes, (cudaStream_t)stream);
}

size_t b200gs_hexplane_time_row_scratch_bytes(const b200gs_hexplane_desc* desc, int replicas)
{
    if (!desc || desc->levels < 1 || desc->levels > HP_MAXL || replicas < 1) return 0;
    if (desc->channels == 16) return time_row_floats<16>(*desc) * sizeof(float) * (size_t)replicas;
    if (desc->channels == 32) return time_row_floats<32>(*desc) * sizeof(float) * (size_t)replicas;
    return 0;
}

int b200gs_hexplane_backward(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                             const float* times, float time_scalar, const float* d_features, float* d_pts,
                             b200gs_stream_t stream)
{
    return b200gs_hexplane_backward_masked(desc, P, pts, order, times, time_scalar, 63, nullptr, nullptr, d_features, d_pts, nullptr, 0, stream);
}

int b200gs_hexplane_regulation(const b200gs_hexplane_desc* desc, float plane_tv_weight, float time_smoothness_weight,
                               float l1_time_planes_weight, float* loss_accum, b200gs_stream_t stream)
{
    if (validate(desc, CH16 | CH32)) return -1;
    int wmax = 1;
    for (int l = 0; l < desc->levels; ++l)
        for (int a = 0; a < 3; ++a) wmax = desc->res[l][a] > wmax ? desc->res[l][a] : wmax;
    const int quads = desc->channels / 4;            // one thread per (x, 4-channel) column
    dim3 grid((unsigned)((wmax * quads + 127) / 128), (unsigned)(desc->levels * 6));
    if (desc->channels == 16)
        hexplane_regulation_kernel<16><<<grid, 128, 0, (cudaStream_t)stream>>>(*desc, plane_tv_weight, time_smoothness_weight,
                                                                                l1_time_planes_weight, loss_accum);
    else
        hexplane_regulation_kernel<32><<<grid, 128, 0, (cudaStream_t)stream>>>(*desc, plane_tv_weight, time_smoothness_weight,
                                                                                l1_time_planes_weight, loss_accum);
    return check_launch("hexplane_regulation");
}

int b200gs_hexplane_time_supported(const b200gs_hexplane_desc* desc)
{
    if (validate(desc, CH32)) return 0;
    TimeRowSetup ts;
    return time_rows_setup(*desc, ts) ? 1 : 0;
}

int b200gs_hexplane_time_forward(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                 float time_scalar, const float* factor, float* features, int features_tiled, b200gs_stream_t stream)
{
    if (validate(desc, CH32)) return -1;
    if (features_tiled && desc->levels != 2) { set_error("hexplane_time_forward: tiled features need 2 levels (64 columns)"); return -1; }
    TimeRowSetup ts;
    if (!time_rows_setup(*desc, ts)) { set_error("hexplane_time_forward: time rows do not fit shared memory"); return -1; }
    if (P <= 0) return 0;
    const size_t smem = (size_t)ts.total * sizeof(float);
    long long blocks = (P + 63) / 64;                // 16 warps x 4 point slots per block; the kernels are latency bound, so as many warps as fit
    const long long cap = (long long)NUM_SMS * (smem * 3 <= 220 * 1024 ? 3 : (smem * 2 <= 220 * 1024 ? 2 : 1));
    if (blocks > cap) blocks = cap;
    if (desc->levels == 2) {                         // see hexplane_time_fwd2_kernel: 2 resident CTAs per SM
        cudaFuncSetAttribute(hexplane_time_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (blocks > (long long)NUM_SMS * 2) blocks = (long long)NUM_SMS * 2;
        hexplane_time_fwd2_kernel<<<(unsigned)blocks, 512, smem, (cudaStream_t)stream>>>(*desc, ts, P, pts, order, time_scalar, factor, features, features_tiled);
    } else {
        cudaFuncSetAttribute(hexplane_time_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        hexplane_time_fwd_kernel<<<(unsigned)blocks, 512, smem, (cudaStream_t)stream>>>(*desc, ts, P, pts, order, time_scalar, factor, features, features_tiled);
    }
    return check_launch("hexplane_time_forward");
}

int b200gs_hexplane_time_backward(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                  float time_scalar, const float* factor, float* d_factor_accum, const float* d_features,
                                  float* d_pts, void* time_row_scratch, size_t time_row_scratch_bytes, int d_features_tiled,
                                  b200gs_stream_t stream)
{
    if (validate(desc, CH32)) return -1;
    if ((d_features_tiled & 1) && desc->levels != 2) { set_error("hexplane_time_backward: tiled d_features need 2 levels (64 columns)"); return -1; }
    TimeRowSetup ts;
    if (!time_rows_setup(*desc, ts)) { set_error("hexplane_time_backward: time rows do not fit shared memory"); return -1; }
    if (P <= 0) return 0;
    const size_t per = (size_t)ts.total * sizeof(float);
    int replicas = time_row_scratch ? (int)(time_row_scratch_bytes / per) : 0;
    if (replicas > 64) replicas = 64;
    if (replicas < 1) { set_error("hexplane_time_backward: scratch for at least one row replica is required"); return -1; }
    float* rows = (float*)time_row_scratch;
    cudaMemsetAsync(rows, 0, per * replicas, (cudaStream_t)stream);
    long long blocks = (P + 31) / 32;
    const long long cap = (long long)NUM_SMS * (per * 3 <= 220 * 1024 ? 3 : (per * 2 <= 220 * 1024 ? 2 : 1));
    if (blocks > cap) blocks = cap;
    if (desc->levels == 2) {                         // see hexplane_time_bwd2_kernel: 2 resident CTAs per SM
        cudaFuncSetAttribute(hexplane_time_bwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)per);
        if (blocks > (long long)NUM_SMS * 2) blocks = (long long)NUM_SMS * 2;
        hexplane_time_bwd2_kernel<<<(unsigned)blocks, 256, per, (cudaStream_t)stream>>>(*desc, ts, P, pts, order, time_scalar, factor, d_factor_accum,
                                                                                        d_features, d_pts, rows, replicas, d_features_tiled);
    } else {
        cudaFuncSetAttribute(hexplane_time_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)per);
        hexplane_time_bwd_kernel<<<(unsigned)blocks, 256, per, (cudaStream_t)stream>>>(*desc, ts, P, pts, order, time_scalar, factor, d_factor_accum,
                                                                                       d_features, d_pts, rows, replicas, d_features_tiled);
    }
    hexplane_time_rows_flush_kernel<TR_C><<<(unsigned)((ts.total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*desc, time_scalar, rows, replicas);
    return check_launch("hexplane_time_backward");
}

}  // extern "C"
