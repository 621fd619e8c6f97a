// Deformation MLP (feature decoder + position / scale / rotation heads): C-ABI entry points, and the
// register-resident mma.sync BACKWARD that serves the 4-level (feature dim 128) configuration. The forward
// (deform_mlp_tc5.cu) and the 2-level backward (deform_mlp_bwd_tc5.cu) run on tcgen05 / TMEM.
//
// Restates scene/deformation.py:55-65 (create_net), :68-85 (query_time) and :97-153
// (forward_dynamic) for the configuration the reference trains with (SURVEY.md §8 a17):
//     hidden = Linear(F, 64)(feature)                                   feature_out, defor_depth <= 1
//     d{x,s,r} = Linear(64, k)(ReLU(Linear(64, 64)(ReLU(hidden))))      k = 3, 3, 4
//     pts   = xyz * 1 + (dx + delta_scale * (frame_num * scene_flow))
//     scale = scales * 1 + ds ;  rot = rotations + dr
// The reference runs seven true-FP32 cuBLAS SGEMMs (TF32 is off by default in torch) with every
// [P,64] intermediate round-tripping HBM.  Here each warp owns 16 points and carries them through
// the whole chain in REGISTERS: every contraction is an m16n8k8 TF32 tensor-core MMA issued three
// times on an error-compensated split (x = hi + lo; hi*hi + lo*hi + hi*lo), which restores ~FP32
// accuracy (2^-21 relative) while the accumulation stays FP32.  The accumulator fragment of one
// layer is re-used directly as the A fragment of the next by permuting the K index (fragment slot t
// <-> column 2t, slot t+4 <-> column 2t+1; the weights are laid out in shared memory to match), so
// no shuffle or shared-memory transpose sits between layers.  Weights are split once per CTA into
// {hi_k, hi_k+1, lo_k, lo_k+1} float4s (one conflict-free LDS.128 per k-step and n-tile).  Only the
// ReLU'd activations the backward needs (4 x 256 B per point, plain row-major) leave the SM.
// The backward accumulates all weight gradients in register fragments across every tile a
// persistent CTA processes and flushes them with one atomic per element per CTA.
#include "mma_tf32.cuh"
#include "../../include/b200gs.h"

namespace b200gs {

namespace {

using tc5::MW;                     // net_width
using tc5::stash_off; using tc5::stash_plane_floats; using tc5::to_tf32;
using tf32::split; using tf32::mma; using tf32::kstep; using tf32::stage_weight;
constexpr int MT = 256;            // threads per CTA (8 warps x 16 points)
using tc5::ROWS;                   // points per CTA iteration
constexpr int LDS_T = MW + 8;      // row stride (floats) of the row-major smem tiles: conflict-free fragment loads

// ---------------------------------------------------------------------------------------------
struct BwdArgs {
    b200gs_mlp_weights w;
    b200gs_mlp_grads gw;
    long long P;
    const float* feat; const float* saved;
    const float* d_pts; const float* d_scales; const float* d_rot;
    float* d_feat;
};

// dW tile accumulation: acc[nt] (16 out x 8 in) += sum over the CTA tile's rows of
// dY[row][16*mt + .] * X[row][8*(nt0+nt) + .]; dY from the row-major smem tile (stride LDS_T),
// X from global row-major memory (stride ldx).  Weight gradients are sums over up to millions of
// rows accumulated in FP32: dY is kept exact (hi + lo split, 2 MMAs), X is rounded to TF32 once
// (relative 2^-12 per term, random sign), well inside the 1e-3 gradient tolerance; the full 3-pass
// split is kept for the dX chain, whose errors would compound through the layers.
template <int NT, bool TILED>
__device__ __forceinline__ void dw_accumulate(float (*acc)[4], const float* __restrict__ dYs, int mt,
                                              const float* __restrict__ X, size_t ldx, long long row0, long long P,
                                              int nt0, int g, int t)
{
#pragma unroll 4
    for (int ks = 0; ks < ROWS / 8; ++ks) {
        const int r0 = 8 * ks + t, r1 = r0 + 4;
        const bool v0 = row0 + r0 < P, v1 = row0 + r1 < P;
        float x0[NT], x1[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            x0[nt] = v0 ? __ldg(X + (TILED ? stash_off(row0 + r0, 8 * (nt0 + nt) + g) : (size_t)(row0 + r0) * ldx + 8 * (nt0 + nt) + g)) : 0.f;
            x1[nt] = v1 ? __ldg(X + (TILED ? stash_off(row0 + r1, 8 * (nt0 + nt) + g) : (size_t)(row0 + r1) * ldx + 8 * (nt0 + nt) + g)) : 0.f;
        }
        const float af[4] = {dYs[r0 * LDS_T + 16 * mt + g], dYs[r0 * LDS_T + 16 * mt + g + 8],
                             dYs[r1 * LDS_T + 16 * mt + g], dYs[r1 * LDS_T + 16 * mt + g + 8]};
        u32 ahi[4], alo[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) split(af[i], ahi[i], alo[i]);
        u32 b0[NT], b1[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) { b0[nt] = to_tf32(x0[nt]); b1[nt] = to_tf32(x1[nt]); }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) mma(acc[nt], alo, b0[nt], b1[nt]);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) mma(acc[nt], ahi, b0[nt], b1[nt]);
    }
}

template <int F>      // F = 128 (feature dim 64 runs the tcgen05 backward)
__global__ void __launch_bounds__(MT, 1) deform_mlp_bwd_kernel(const __grid_constant__ BwdArgs a)
{
    extern __shared__ __align__(16) float4 smem4[];
    constexpr int RS2 = MW / 2 + 4;            // K = 64 operands
    constexpr int RS3 = 4;                     // K = 8 operand (W3): 4 float4 per row, contiguous -> conflict-free
    constexpr int NT1 = F / 8;                 // n-tiles of d_feature / in-features of W1
    float4* W3b = smem4;                       // [3][64][RS3]   Wm[k=out(pad 8)][n=in 64]  = W3[k][n]
    float4* W2b = W3b + 3 * MW * RS3;          // [64][RS2]      Wm[k=out][n=in]            = W2[k][n], one slot re-staged per head
    float4* W1b = W2b + MW * RS2;              // [F][RS2]       Wm[k=out 64][n=in F]       = W1[k][n]
    float* Ds = reinterpret_cast<float*>(W1b + F * RS2);          // [ROWS][LDS_T]  dz / d hidden, row-major
    float* Dout = Ds + ROWS * LDS_T;                              // [ROWS][8]      upstream gradient of the head
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int kdim[3] = {3, 3, 4};

    // backward dX = dY W: Wm[k][n] = W_torch[k][n] -> sk = row length
    stage_weight<MT>(W1b, a.w.w1, MW, F, MW, F, RS2);
    for (int h = 0; h < 3; ++h) {
        if (!a.w.w2[h]) continue;
        for (int i = tid; i < MW * 4; i += MT) {                     // K = 8 (padded outputs), rs = 4
            const int n = i >> 2, kk = i & 3, k0 = 2 * kk, k1 = k0 + 1;
            const float v0 = k0 < kdim[h] ? __ldg(a.w.w3[h] + k0 * MW + n) : 0.f;
            const float v1 = k1 < kdim[h] ? __ldg(a.w.w3[h] + k1 * MW + n) : 0.f;
            u32 h0, l0, h1, l1;
            split(v0, h0, l0); split(v1, h1, l1);
            W3b[h * MW * RS3 + n * RS3 + kk] = make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
        }
    }
    __syncthreads();

    // weight-gradient fragments owned by this warp (persist over all tiles of the CTA)
    const int mt = warp >> 1;                  // 16-row block of `out` features
    const int ntb = (warp & 1) * 4;            // first of 4 n-tiles of `in` features (W2)
    float gW2[3][4][4], gW1[NT1 / 2][4], gW3[3][4];
    float gB2[3] = {0.f, 0.f, 0.f}, gB1 = 0.f, gB3[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int h = 0; h < 3; ++h) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            gW3[h][i] = 0.f;
#pragma unroll
            for (int n = 0; n < 4; ++n) gW2[h][n][i] = 0.f;
        }
    }
#pragma unroll
    for (int n = 0; n < NT1 / 2; ++n)
#pragma unroll
        for (int i = 0; i < 4; ++i) gW1[n][i] = 0.f;

    const long long nblocks = (a.P + ROWS - 1) / ROWS;
    for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const long long row0 = blk * ROWS;
        const int lr_lo = warp * 16 + g, lr_hi = lr_lo + 8;          // local rows of this lane
        const long long r_lo = row0 + lr_lo, r_hi = row0 + lr_hi;
        const bool v_lo = r_lo < a.P, v_hi = r_hi < a.P;
        float hC[8][4], dRh[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const float2 x = v_lo ? __ldg(reinterpret_cast<const float2*>(a.saved + stash_off(r_lo, 8 * nt + 2 * t))) : make_float2(0.f, 0.f);
            const float2 y = v_hi ? __ldg(reinterpret_cast<const float2*>(a.saved + stash_off(r_hi, 8 * nt + 2 * t))) : make_float2(0.f, 0.f);
            hC[nt][0] = x.x; hC[nt][1] = x.y; hC[nt][2] = y.x; hC[nt][3] = y.y;
#pragma unroll
            for (int i = 0; i < 4; ++i) dRh[nt][i] = 0.f;
        }
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            if (!a.w.w2[h]) continue;
            const int kd = kdim[h];
            const float* dsrc = h == 0 ? a.d_pts : (h == 1 ? a.d_scales : a.d_rot);
            const float* zsv = a.saved + (size_t)(1 + h) * stash_plane_floats(a.P);
            // every warp is past the previous head's use of the slot (trailing barrier below)
            stage_weight<MT>(W2b, a.w.w2[h], MW, MW, MW, MW, RS2);
            __syncthreads();
            // upstream gradient as an A fragment (one k-step, columns >= kd are zero) and as a smem tile
            float df[4];
            {
                const int c0 = 2 * t, c1 = c0 + 1;
                df[0] = (v_lo && dsrc && c0 < kd) ? __ldg(dsrc + (size_t)r_lo * kd + c0) : 0.f;
                df[1] = (v_hi && dsrc && c0 < kd) ? __ldg(dsrc + (size_t)r_hi * kd + c0) : 0.f;
                df[2] = (v_lo && dsrc && c1 < kd) ? __ldg(dsrc + (size_t)r_lo * kd + c1) : 0.f;
                df[3] = (v_hi && dsrc && c1 < kd) ? __ldg(dsrc + (size_t)r_hi * kd + c1) : 0.f;
                *reinterpret_cast<float2*>(Dout + lr_lo * 8 + c0) = make_float2(df[0], df[2]);
                *reinterpret_cast<float2*>(Dout + lr_hi * 8 + c0) = make_float2(df[1], df[3]);
            }
            // dz = (d_out W3) masked by relu(z) > 0
            float dz[8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int i = 0; i < 4; ++i) dz[nt][i] = 0.f;
            kstep<8>(dz, df, W3b + h * MW * RS3, RS3, 0, g, t);
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
                kstep<8>(dRh, af, W2b, RS2, j, g, t);
            }
            __syncthreads();                                             // dz and d_out tiles complete
            dw_accumulate<4, true>(gW2[h], Ds, mt, a.saved, MW, row0, a.P, ntb, g, t);            // dW2 += dz^T relu(h)
            // dW3 (out padded to one 16-row m-tile; n-tile `warp` of the 64 in-features) += d_out^T relu(z)
#pragma unroll 4
            for (int ks = 0; ks < ROWS / 8; ++ks) {
                const int r0 = 8 * ks + t, r1 = r0 + 4;
                const float x0 = row0 + r0 < a.P ? __ldg(zsv + stash_off(row0 + r0, 8 * warp + g)) : 0.f;
                const float x1 = row0 + r1 < a.P ? __ldg(zsv + stash_off(row0 + r1, 8 * warp + g)) : 0.f;
                u32 ahi[4] = {0u, 0u, 0u, 0u}, alo[4] = {0u, 0u, 0u, 0u};      // rows g+8 of the m-tile are padding
                split(Dout[r0 * 8 + g], ahi[0], alo[0]);
                split(Dout[r1 * 8 + g], ahi[2], alo[2]);
                const u32 b0 = to_tf32(x0), b1 = to_tf32(x1);
                mma(gW3[h], alo, b0, b1);
                mma(gW3[h], ahi, b0, b1);
            }
            if (tid < MW) {
                float s = 0.f;
#pragma unroll 8
                for (int r = 0; r < ROWS; ++r) s += Ds[r * LDS_T + tid];
                gB2[h] += s;
            } else if (tid < MW + 8) {
                float s = 0.f;
                for (int r = 0; r < ROWS; ++r) s += Dout[r * 8 + (tid - MW)];
                gB3[h] += s;
            }
            __syncthreads();                                             // before the next head overwrites the tiles
        }
        // d hidden = d relu(h) masked; tile for dW1; d feature = dh W1
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int i = 0; i < 4; ++i) dRh[nt][i] = hC[nt][i] > 0.f ? dRh[nt][i] : 0.f;
            *reinterpret_cast<float2*>(Ds + lr_lo * LDS_T + 8 * nt + 2 * t) = make_float2(dRh[nt][0], dRh[nt][1]);
            *reinterpret_cast<float2*>(Ds + lr_hi * LDS_T + 8 * nt + 2 * t) = make_float2(dRh[nt][2], dRh[nt][3]);
        }
        {
            float dF[NT1][4];
#pragma unroll
            for (int nt = 0; nt < NT1; ++nt)
#pragma unroll
                for (int i = 0; i < 4; ++i) dF[nt][i] = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float af[4] = {dRh[j][0], dRh[j][2], dRh[j][1], dRh[j][3]};
                kstep<NT1>(dF, af, W1b, RS2, j, g, t);
            }
#pragma unroll
            for (int nt = 0; nt < NT1; ++nt) {
                if (v_lo) *reinterpret_cast<float2*>(a.d_feat + (size_t)r_lo * F + 8 * nt + 2 * t) = make_float2(dF[nt][0], dF[nt][1]);
                if (v_hi) *reinterpret_cast<float2*>(a.d_feat + (size_t)r_hi * F + 8 * nt + 2 * t) = make_float2(dF[nt][2], dF[nt][3]);
            }
        }
        __syncthreads();
        dw_accumulate<NT1 / 2, false>(gW1, Ds, mt, a.feat, F, row0, a.P, (warp & 1) * (NT1 / 2), g, t);     // dW1 += dh^T feature
        if (tid < MW) {
            float s = 0.f;
#pragma unroll 8
            for (int r = 0; r < ROWS; ++r) s += Ds[r * LDS_T + tid];
            gB1 += s;
        }
        __syncthreads();
    }

    // flush: C fragment (16 x 8): c0 (g, 2t) c1 (g, 2t+1) c2 (g+8, 2t) c3 (g+8, 2t+1)
#pragma unroll
    for (int n = 0; n < NT1 / 2; ++n) {
        const int in0 = 8 * ((warp & 1) * (NT1 / 2) + n) + 2 * t;
        atomicAdd(a.gw.w1 + (size_t)(16 * mt + g) * F + in0, gW1[n][0]);
        atomicAdd(a.gw.w1 + (size_t)(16 * mt + g) * F + in0 + 1, gW1[n][1]);
        atomicAdd(a.gw.w1 + (size_t)(16 * mt + g + 8) * F + in0, gW1[n][2]);
        atomicAdd(a.gw.w1 + (size_t)(16 * mt + g + 8) * F + in0 + 1, gW1[n][3]);
    }
    if (tid < MW) atomicAdd(a.gw.b1 + tid, gB1);
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        if (!a.w.w2[h]) continue;
#pragma unroll
        for (int n = 0; n < 4; ++n) {
            const int in0 = 8 * (ntb + n) + 2 * t;
            atomicAdd(a.gw.w2[h] + (16 * mt + g) * MW + in0, gW2[h][n][0]);
            atomicAdd(a.gw.w2[h] + (16 * mt + g) * MW + in0 + 1, gW2[h][n][1]);
            atomicAdd(a.gw.w2[h] + (16 * mt + g + 8) * MW + in0, gW2[h][n][2]);
            atomicAdd(a.gw.w2[h] + (16 * mt + g + 8) * MW + in0 + 1, gW2[h][n][3]);
        }
        if (g < kdim[h]) {           // row g of the padded m-tile = out feature; columns 8*warp + 2t (+1)
            atomicAdd(a.gw.w3[h] + g * MW + 8 * warp + 2 * t, gW3[h][0]);
            atomicAdd(a.gw.w3[h] + g * MW + 8 * warp + 2 * t + 1, gW3[h][1]);
        }
        if (tid < MW) atomicAdd(a.gw.b2[h] + tid, gB2[h]);
        else if (tid < MW + 8 && tid - MW < kdim[h]) atomicAdd(a.gw.b3[h] + (tid - MW), gB3[h]);
    }
}

constexpr size_t BWD_SMEM = (size_t)(3 * MW * 4 + MW * (MW / 2 + 4) + 128 * (MW / 2 + 4)) * sizeof(float4) +
                            (size_t)(ROWS * LDS_T + ROWS * 8) * sizeof(float);

int check_weights(const b200gs_mlp_weights* w)
{
    if (!w) { set_error("deform_mlp: null weights"); return -1; }
    if (w->width != MW) { set_error("deform_mlp: net_width=%d unsupported (need %d)", w->width, MW); return -1; }
    if (w->feat_dim != 64 && w->feat_dim != 128) { set_error("deform_mlp: feature dim %d unsupported (64 or 128: 2 or 4 HexPlane levels)", w->feat_dim); return -1; }
    if (w->feat_tiled && w->feat_dim != 64) { set_error("deform_mlp: tiled features need feature dim 64"); return -1; }
    if (!w->w1 || !w->b1) { set_error("deform_mlp: feature_out weights missing"); return -1; }
    for (int h = 0; h < 3; ++h)
        if (w->w2[h] && (!w->b2[h] || !w->w3[h] || !w->b3[h])) { set_error("deform_mlp: head %d incomplete", h); return -1; }
    return 0;
}

}  // namespace
}  // namespace b200gs

namespace b200gs {
int deform_mlp_forward_tc5(const b200gs_mlp_weights* w, long long P, const float* feat, const float* xyz,
                           const float* scales, const float* rot, const float* scene_flow, float frame_num,
                           const float* frame_num_dev, float delta_scale, float* pts_out, float* scales_out,
                           float* rot_out, float* saved, cudaStream_t stream);
int deform_mlp_backward_tc5(const b200gs_mlp_weights* w, const b200gs_mlp_grads* gw, long long P, const float* feat,
                            const float* saved, const float* d_pts, const float* d_scales, const float* d_rot,
                            float* d_feat, cudaStream_t stream);
}

using namespace b200gs;

extern "C" {

size_t b200gs_deform_mlp_saved_floats(long long P) { return P > 0 ? tc5::stash_total_floats(P) : 0; }

int b200gs_deform_mlp_forward(const b200gs_mlp_weights* w, long long P, const float* feat, const float* xyz,
                              const float* scales, const float* rot, const float* scene_flow, float frame_num,
                              const float* frame_num_dev, float delta_scale, float* pts_out, float* scales_out,
                              float* rot_out, float* saved, b200gs_stream_t stream)
{
    if (check_weights(w)) return -1;
    if (P <= 0) return 0;
    return deform_mlp_forward_tc5(w, P, feat, xyz, scales, rot, scene_flow, frame_num, frame_num_dev, delta_scale,
                                  pts_out, scales_out, rot_out, saved, (cudaStream_t)stream);
}

int b200gs_deform_mlp_backward(const b200gs_mlp_weights* w, const b200gs_mlp_grads* gw, long long P, const float* feat,
                               const float* saved, const float* d_pts, const float* d_scales, const float* d_rot,
                               float* d_feat, b200gs_stream_t stream)
{
    if (check_weights(w)) return -1;
    if (!gw) { set_error("deform_mlp_backward: null gradient table"); return -1; }
    if (P <= 0) return 0;
    if (w->feat_dim == 64)
        return deform_mlp_backward_tc5(w, gw, P, feat, saved, d_pts, d_scales, d_rot, d_feat, (cudaStream_t)stream);
    BwdArgs a;
    a.w = *w; a.gw = *gw; a.P = P; a.feat = feat; a.saved = saved; a.d_pts = d_pts; a.d_scales = d_scales;
    a.d_rot = d_rot; a.d_feat = d_feat;
    const int grid = tc5::persistent_grid(P, 0);       // no CTA cap: this kernel does not take mlp_bwd_sms
    cudaFuncSetAttribute(deform_mlp_bwd_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BWD_SMEM);
    deform_mlp_bwd_kernel<128><<<grid, MT, BWD_SMEM, (cudaStream_t)stream>>>(a);
    return check_launch("deform_mlp_backward");
}

}  // extern "C"
