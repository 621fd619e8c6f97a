// Rasterizer backward: reverse-order compositing gradients, then the per-Gaussian chain
// back to means / scales / rotations / SH.
//
// Behaviour follows RAST/cuda_rasterizer/backward.cu:415-590 (compositing),
// :144-274 (cov2D), :346-412 (projection, depth), :20-139 (SH), :278-341 (cov3D).
// The compositing kernel does not issue one global atomic per (pixel, Gaussian, value)
// like the reference (10 REDG per pair): the 64 pixels of a warp visit the same splat in
// lock-step, so their 10 partial gradients are folded with a transposed butterfly
// (14 shuffles), accumulated per batch slot in shared memory, and leave the SM as three
// 128-bit vector reductions per (tile, splat) instance.
#include "rast_state.cuh"
#include "f32x2.cuh"

namespace b200gs {

namespace {

constexpr int ACC = 12;   // floats per Gaussian in the accumulation arena (3 x float4)

// ---- compositing backward: TWO pixels per lane and packed FP32 pairs ----------------------------------------------------------
// One pixel per lane is issue-slot bound (ncu: 75 % of issue slots busy, FMA pipe 34 %; 88 instructions per (warp, splat) of which
// ~44 are the butterfly).  Here a warp covers an 8x8 patch: lane (lx, ly) owns pixels (lx, ly) and (lx, ly + 4) and carries their
// state as f32x2 pairs, so the per-pixel arithmetic is issued once for both (FFMA2 / FMUL2 / FADD2, splat constants as
// scalar-broadcast operands) and the 10-value butterfly is paid once per 64 pixels instead of once per 32: 0.765 -> 0.608 ms per
// 1M-Gaussian 1280x720 view.
//   * A pixel for which the splat is inactive takes part with alpha = G = 0: T / (1 - 0), w = 0 and every partial gradient are
//     exact no-ops, and the "previous colour" recurrence  rec = la * lc + (1 - la) * rec  evaluated one splat early gives the same
//     value one splat later (0 * C + 1 * rec), so no per-pixel selects are needed and the previous colour is warp-uniform.
//   * 1 / (1 - alpha) uses MUFU.RCP (relative error ~1e-7 per pair, 1e-5 over a chain of 100 contributors; the bar for these
//     gradients is 1e-3); exp stays the accurate sequence (see below).
constexpr int CB2_THREADS = 128;
// CB2 = splats per batch, with the register budget set for 6 CTAs per SM (34 KB of shared memory per CTA, <= 85 registers).
// Measured at 1M / 1280x720 and 200k / 512^2 (profiles/r2y_composite_pairs_occupancy.txt), whole rasterizer backward:
// 256 / 5 CTAs: 0.612 / 0.322 ms, 224 / 6: 0.594 / 0.298 ms, 192 / 7: 0.582 / 0.321 ms.
constexpr int CB2 = 224;
struct __align__(16) BStage2 { float4 A[CB2]; float4 B[CB2]; float4 C[CB2]; u32 gid[CB2]; };

__global__ void __launch_bounds__(CB2_THREADS, 6)
composite_bwd2_kernel(const uint2* __restrict__ ranges, const u32* __restrict__ list, int W, int H, int grid_x,
                      const float4* __restrict__ recA, const float4* __restrict__ recB,
                      const float4* __restrict__ recC, const float* __restrict__ bg,
                      const float* __restrict__ final_T, const u32* __restrict__ n_contrib,
                      const float* __restrict__ dL_dpix, const float* __restrict__ dL_dpix_depth,
                      float* __restrict__ acc)
{
    __shared__ BStage2 stage[2];
    __shared__ __align__(16) float s_acc[CB2 * ACC];
    __shared__ u32 s_max[4];
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 tile = blockIdx.x;
    const u32 tx = tile % (u32)grid_x, ty = tile / (u32)grid_x;
    const u32 px = tx * TILE_X + (warp & 1) * 8 + (lane & 7);
    const u32 pyA = ty * TILE_Y + (warp >> 1) * 8 + (lane >> 3), pyB = pyA + 4;
    const bool inA = px < (u32)W && pyA < (u32)H, inB = px < (u32)W && pyB < (u32)H;
    const float fxp = (float)px;
    const f2 fyp = pk((float)pyA, (float)pyB);
    const uint2 range = ranges[tile];
    const size_t pidA = (size_t)pyA * W + px, pidB = (size_t)pyB * W + px;
    const size_t HW = (size_t)H * W;
    const u32 lastA = inA ? n_contrib[pidA] : 0, lastB = inB ? n_contrib[pidB] : 0;
    const float patch_x = (float)(tx * TILE_X + (warp & 1) * 8), patch_y = (float)(ty * TILE_Y + (warp >> 1) * 8);
    u32 m = max(lastA, lastB);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    const u32 warp_last = m;
    if (lane == 0) s_max[warp] = m;
    for (u32 i = tid; i < CB2 * ACC; i += CB2_THREADS) s_acc[i] = 0.f;
    __syncthreads();
    u32 n_eff = max(max(s_max[0], s_max[1]), max(s_max[2], s_max[3]));
    n_eff = min(n_eff, range.y - range.x);
    if (n_eff == 0) return;
    const int rounds = (int)((n_eff + CB2 - 1) / CB2);

    const f2 T_final = pk(inA ? final_T[pidA] : 0.f, inB ? final_T[pidB] : 0.f);
    f2 T = T_final;
    const f2 dLp0 = pk(inA ? dL_dpix[pidA] : 0.f, inB ? dL_dpix[pidB] : 0.f);
    const f2 dLp1 = pk(inA ? dL_dpix[HW + pidA] : 0.f, inB ? dL_dpix[HW + pidB] : 0.f);
    const f2 dLp2 = pk(inA ? dL_dpix[2 * HW + pidA] : 0.f, inB ? dL_dpix[2 * HW + pidB] : 0.f);
    const f2 dLd = pk((inA && dL_dpix_depth) ? dL_dpix_depth[pidA] : 0.f, (inB && dL_dpix_depth) ? dL_dpix_depth[pidB] : 0.f);
    // -T_final * (bg . dL_dpixel): the background term of dL_dalpha before its 1 / (1 - alpha)
    const f2 nTb = mul2(sub2(pk1(0.f), T_final), fma2(pk1(bg[2]), dLp2, fma2(pk1(bg[1]), dLp1, mul2(pk1(bg[0]), dLp0))));
    f2 rec0 = pk1(0.f), rec1 = pk1(0.f), rec2 = pk1(0.f), recd = pk1(0.f), last_alpha = pk1(0.f);
    float lc0 = 0.f, lc1 = 0.f, lc2 = 0.f, ld = 0.f;          // colour / depth of the previous splat this warp processed
    const float ddelx_dx = 0.5f * W, ddely_dy = 0.5f * H;

    auto fill = [&](BStage2& st, u32 first) {
#pragma unroll
        for (int h = 0; h < (CB2 + CB2_THREADS - 1) / CB2_THREADS; ++h) {
            const u32 t = tid + h * CB2_THREADS, pos = first + t;
            if (t < (u32)CB2 && pos < n_eff) {
                const u32 g = __ldg(list + (range.x + n_eff - 1 - pos));
                st.gid[t] = g;
                cp_async16(&st.A[t], recA + g);
                cp_async16(&st.B[t], recB + g);
                cp_async16(&st.C[t], recC + g);
            }
        }
    };
    fill(stage[0], 0);
    cp_async_commit();
    for (int r = 0; r < rounds; ++r) {
        if (r + 1 < rounds) fill(stage[(r + 1) & 1], (u32)(r + 1) * CB2);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const BStage2& st = stage[r & 1];
        const int cnt = (int)min((u32)CB2, n_eff - (u32)r * CB2);
        u32 masks[CB2 / 32];
#pragma unroll
        for (int q = 0; q < CB2 / 32; ++q) {
            const int j = q * 32 + (int)lane;
            const u32 p = n_eff - 1u - ((u32)r * CB2 + (u32)j);
            const bool keep = j < cnt && p < warp_last && splat_may_touch_patch(st.A[j], st.B[j], patch_x, patch_y, 7.f);
            masks[q] = __ballot_sync(0xffffffffu, keep);
        }
#pragma unroll
        for (int q = 0; q < CB2 / 32; ++q) {
          u32 mq = masks[q];
          while (mq != 0) {
            const int j = q * 32 + __ffs(mq) - 1;
            mq &= mq - 1;
            const u32 contributor = n_eff - 1u - ((u32)r * CB2 + (u32)j);
            const float4 A = st.A[j];
            const float4 B = st.B[j];
            const float dx = A.x - fxp;
            const f2 dy = sub2(pk1(A.y), fyp);
            // power = -0.5 (a dx^2 + c dy^2) - b dx dy
            const float adx2 = A.z * dx * dx, bdx = A.w * dx;
            const f2 quad = fma2(mul2(pk1(B.x), dy), dy, pk1(adx2));
            const f2 power = fma2(quad, pk1(-0.5f), mul2(pk1(-bdx), dy));
            const float pwA = lo(power), pwB = hi(power);
            bool actA = contributor < lastA && !(pwA > 0.0f) && !(pwA < B.w);
            bool actB = contributor < lastB && !(pwB > 0.0f) && !(pwB < B.w);
            // the accurate expf, as in the forward and in the reference's backward: T is recovered as T_final / prod (1 - alpha), so
            // an alpha that differs from the forward's by 3e-7 (ex2.approx) is amplified by 1 / (1 - alpha) along the chain
            const float GA = expf(pwA), GB = expf(pwB);
            float aA = fminf(0.99f, B.y * GA), aB = fminf(0.99f, B.y * GB);
            actA = actA && !(aA < 1.0f / 255.0f);
            actB = actB && !(aB < 1.0f / 255.0f);
            if (!__any_sync(0xffffffffu, actA || actB)) continue;
            // an inactive pixel takes part with alpha = G = 0 (see the kernel comment)
            const f2 G = pk(actA ? GA : 0.f, actB ? GB : 0.f);
            const f2 alpha = pk(actA ? aA : 0.f, actB ? aB : 0.f);
            const float4 Cc = st.C[j];
            const f2 oma = sub2(pk1(1.f), alpha);
            float qA, qB;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(qA) : "f"(lo(oma)));
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(qB) : "f"(hi(oma)));
            const f2 q1 = pk(qA, qB);                     // 1 / (1 - alpha)
            T = mul2(T, q1);
            const f2 w = mul2(alpha, T);
            const f2 omla = sub2(pk1(1.f), last_alpha);
            rec0 = fma2(last_alpha, pk1(lc0), mul2(omla, rec0));
            rec1 = fma2(last_alpha, pk1(lc1), mul2(omla, rec1));
            rec2 = fma2(last_alpha, pk1(lc2), mul2(omla, rec2));
            recd = fma2(last_alpha, pk1(ld), mul2(omla, recd));
            lc0 = Cc.x; lc1 = Cc.y; lc2 = Cc.z; ld = B.z;
            last_alpha = alpha;
            f2 dLa = mul2(sub2(pk1(Cc.x), rec0), dLp0);
            dLa = fma2(sub2(pk1(Cc.y), rec1), dLp1, dLa);
            dLa = fma2(sub2(pk1(Cc.z), rec2), dLp2, dLa);
            dLa = fma2(sub2(pk1(B.z), recd), dLd, dLa);
            dLa = fma2(nTb, q1, mul2(dLa, T));            // * T  +  (-T_final / (1 - alpha)) * (bg . dL_dpixel)
            const f2 dL_dG = mul2(pk1(B.y), dLa);
            const f2 gdx = mul2(G, pk1(dx)), gdy = mul2(G, dy);
            const f2 dGx = fma2(gdy, pk1(-A.w), mul2(gdx, pk1(-A.z)));
            const f2 dGy = fma2(gdx, pk1(-A.w), mul2(gdy, pk1(-B.x)));
            const f2 hx = mul2(gdx, dL_dG), hy = mul2(gdy, dL_dG);
            const f2 mhdy = mul2(dy, pk1(-0.5f));
            const f2 p0 = mul2(mul2(dL_dG, dGx), pk1(ddelx_dx));      // d mean2D.x
            const f2 p1 = mul2(mul2(dL_dG, dGy), pk1(ddely_dy));      // d mean2D.y
            const f2 p2 = mul2(hx, pk1(-0.5f * dx));                  // d conic.a
            const f2 p3 = mul2(hx, mhdy);                             // d conic.b
            const f2 p4 = mul2(hy, mhdy);                             // d conic.c
            const f2 p5 = mul2(G, dLa);                               // d opacity
            const f2 p6 = mul2(w, dLd);                               // d depth
            const f2 p7 = mul2(w, dLp0), p8 = mul2(w, dLp1), p9 = mul2(w, dLp2);   // d colour
            const float v0 = lo(p0) + hi(p0), v1 = lo(p1) + hi(p1), v2 = lo(p2) + hi(p2), v3 = lo(p3) + hi(p3), v4 = lo(p4) + hi(p4),
                        v5 = lo(p5) + hi(p5), v6 = lo(p6) + hi(p6), v7 = lo(p7) + hi(p7), v8 = lo(p8) + hi(p8), v9 = lo(p9) + hi(p9);
            // transposed butterfly: 8 values (v0..v7) -> lane>>2 owns value (lane>>2); v8,v9 -> lanes 0/16
            {
                const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
                float u0 = (h16 ? v4 : v0) + __shfl_xor_sync(0xffffffffu, h16 ? v0 : v4, 16);
                float u1 = (h16 ? v5 : v1) + __shfl_xor_sync(0xffffffffu, h16 ? v1 : v5, 16);
                float u2 = (h16 ? v6 : v2) + __shfl_xor_sync(0xffffffffu, h16 ? v2 : v6, 16);
                float u3 = (h16 ? v7 : v3) + __shfl_xor_sync(0xffffffffu, h16 ? v3 : v7, 16);
                float y = (h16 ? v9 : v8) + __shfl_xor_sync(0xffffffffu, h16 ? v8 : v9, 16);
                float w0 = (h8 ? u2 : u0) + __shfl_xor_sync(0xffffffffu, h8 ? u0 : u2, 8);
                float w1 = (h8 ? u3 : u1) + __shfl_xor_sync(0xffffffffu, h8 ? u1 : u3, 8);
                y += __shfl_xor_sync(0xffffffffu, y, 8);
                float x = (h4 ? w1 : w0) + __shfl_xor_sync(0xffffffffu, h4 ? w0 : w1, 4);
                y += __shfl_xor_sync(0xffffffffu, y, 4);
                x += __shfl_xor_sync(0xffffffffu, x, 2);
                y += __shfl_xor_sync(0xffffffffu, y, 2);
                x += __shfl_xor_sync(0xffffffffu, x, 1);
                y += __shfl_xor_sync(0xffffffffu, y, 1);
                if ((lane & 3) == 0) {
                    const int k = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                    const int slot = (k == 7) ? 8 : k;
                    if (x != 0.f) atomicAdd(&s_acc[j * ACC + slot], x);
                }
                if ((lane & 15) == 0) {
                    const int slot = (lane & 16) ? 10 : 9;
                    if (y != 0.f) atomicAdd(&s_acc[j * ACC + slot], y);
                }
            }
          }
        }
        __syncthreads();
        // flush this batch: one thread per instance, three 128-bit reductions
#pragma unroll
        for (int h = 0; h < (CB2 + CB2_THREADS - 1) / CB2_THREADS; ++h) {
            const int t = (int)tid + h * CB2_THREADS;
            if (t < cnt) {
                float4* sa = reinterpret_cast<float4*>(&s_acc[t * ACC]);
                const float4 a0 = sa[0], a1 = sa[1], a2 = sa[2];
                float* dst = acc + (size_t)st.gid[t] * ACC;
                if (a0.x != 0.f || a0.y != 0.f || a0.z != 0.f || a0.w != 0.f) red_add_v4(dst, a0.x, a0.y, a0.z, a0.w);
                if (a1.x != 0.f || a1.y != 0.f || a1.z != 0.f) red_add_v4(dst + 4, a1.x, a1.y, a1.z, 0.f);
                if (a2.x != 0.f || a2.y != 0.f || a2.z != 0.f) red_add_v4(dst + 8, a2.x, a2.y, a2.z, 0.f);
                const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                sa[0] = z; sa[1] = z; sa[2] = z;
            }
        }
        __syncthreads();
    }
    cp_async_wait<0>();
}

// -----------------------------------------------------------------------------------------
// per-Gaussian backward
// -----------------------------------------------------------------------------------------
constexpr float SH0 = 0.28209479177387814f;
constexpr float SH1 = 0.4886025119029199f;
__constant__ float SH2b[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                              -1.0925484305920792f, 0.5462742152960396f};
__constant__ float SH3b[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f,
                              0.3731763325901154f, -0.4570457994644658f, 1.445305721320277f,
                              -0.5900435899266435f};

constexpr int PB_THREADS = 128;
constexpr int PB_WARPS = PB_THREADS / 32;

struct PreBwdArgs {
    int P, D, M, W, H;
    const float* means; const float* scales; const float* rots; const float* shs;
    const float* cov3d;            // precomputed or the forward's own
    const float* view; const float* proj; const float* campos;
    float scale_mod, tanx, tany, fx, fy;
    const int* radii; const unsigned char* clamped;
    const float* acc;              // [P][12] from the compositing backward
    int has_colors_precomp;
    float* dL_dmean2D;             // [P,3]
    float* dL_dcolor;              // [P,3]
    float* dL_dopacity;            // [P]
    float* dL_dmean3D;             // [P,3]
    float* dL_dcov3D;              // [P,6]
    float* dL_dsh;                 // [P,M,3] or null
    int accumulate_sh;             // 1: dL_dsh += (rows of invisible Gaussians are left alone); 0: every row is written
    float* dL_dscale;              // [P,3]
    float* dL_drot;                // [P,4]
};

__global__ void __launch_bounds__(PB_THREADS) preprocess_bwd_kernel(const PreBwdArgs a)
{
    extern __shared__ float s_sh[];     // [PB_WARPS][32][3M+1] (SH in, SH gradient out)
    __shared__ float s_cam[36];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 16) s_cam[tid] = __ldg(a.view + tid);
    else if (tid < 32) s_cam[tid] = __ldg(a.proj + (tid - 16));
    else if (tid < 35) s_cam[tid] = __ldg(a.campos + (tid - 32));
    __syncthreads();
    const float* vm = s_cam; const float* pm = s_cam + 16;

    const int idx = blockIdx.x * PB_THREADS + tid;
    const bool in_range = idx < a.P;
    const bool vis = in_range && (__ldg(a.radii + idx) > 0);
    const bool use_sh = a.shs != nullptr && a.dL_dsh != nullptr;
    const int stride = 3 * a.M + 1;
    float* ws = s_sh + (size_t)warp * 32 * stride;
    const int g0 = blockIdx.x * PB_THREADS + warp * 32;
    const int ng = max(0, min(32, a.P - g0));
    const bool any_vis = __any_sync(0xffffffffu, vis);

    // stage SH coefficients (coalesced), as in the forward
    if (use_sh && any_vis) {
        const float* src = a.shs + (size_t)g0 * 3 * a.M;
        const int per = 3 * a.M;
        if ((per & 3) == 0) {
            const float4* src4 = reinterpret_cast<const float4*>(src);
            for (int e = lane; e < ng * per / 4; e += 32) {
                float4 v = __ldg(src4 + e);
                int f = e * 4, gg = f / per, k = f - gg * per;
                float* d = ws + gg * stride + k;
                d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
            }
        } else {
            for (int e = lane; e < ng * per; e += 32) { int gg = e / per, k = e - gg * per; ws[gg * stride + k] = __ldg(src + e); }
        }
    }
    __syncwarp();

    float3 dmean = make_float3(0.f, 0.f, 0.f);
    float dcov[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float3 dscale = make_float3(0.f, 0.f, 0.f);
    float4 drot = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0;
    if (vis) {
        const float4* accv = reinterpret_cast<const float4*>(a.acc + (size_t)idx * ACC);
        a0 = __ldg(accv); a1 = __ldg(accv + 1); a2 = __ldg(accv + 2);
        const float3 mean = make_float3(__ldg(a.means + 3 * idx), __ldg(a.means + 3 * idx + 1), __ldg(a.means + 3 * idx + 2));
        float c3[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) c3[k] = __ldg(a.cov3d + 6 * (size_t)idx + k);

        // ---- conic -> cov2D -> cov3D and mean (backward.cu:144-274) ----
        float3 t = make_float3(vm[0] * mean.x + vm[4] * mean.y + vm[8] * mean.z + vm[12],
                               vm[1] * mean.x + vm[5] * mean.y + vm[9] * mean.z + vm[13],
                               vm[2] * mean.x + vm[6] * mean.y + vm[10] * mean.z + vm[14]);
        const float limx = 1.3f * a.tanx, limy = 1.3f * a.tany;
        const float txtz = t.x / t.z, tytz = t.y / t.z;
        t.x = fminf(limx, fmaxf(-limx, txtz)) * t.z;
        t.y = fminf(limy, fmaxf(-limy, tytz)) * t.z;
        const float xgm = (txtz < -limx || txtz > limx) ? 0.f : 1.f;
        const float ygm = (tytz < -limy || tytz > limy) ? 0.f : 1.f;
        const float J00 = a.fx / t.z, J02 = -(a.fx * t.x) / (t.z * t.z);
        const float J11 = a.fy / t.z, J12 = -(a.fy * t.y) / (t.z * t.z);
        // Wc[c][r]: column c of the view rotation as the reference arranges it
        const float W00 = vm[0], W01 = vm[4], W02 = vm[8];
        const float W10 = vm[1], W11 = vm[5], W12 = vm[9];
        const float W20 = vm[2], W21 = vm[6], W22 = vm[10];
        // T = W * J (third column is zero)
        const float T00 = W00 * J00 + W20 * J02, T01 = W01 * J00 + W21 * J02, T02 = W02 * J00 + W22 * J02;
        const float T10 = W10 * J11 + W20 * J12, T11 = W11 * J11 + W21 * J12, T12 = W12 * J11 + W22 * J12;
        const float V00 = c3[0], V01 = c3[1], V02 = c3[2], V11 = c3[3], V12 = c3[4], V22 = c3[5];
        // rows of V*T^T needed for cov2D and for dL/dT
        const float p00 = T00 * V00 + T01 * V01 + T02 * V02;   // (T0 . V0)
        const float p01 = T00 * V01 + T01 * V11 + T02 * V12;   // (T0 . V1)
        const float p02 = T00 * V02 + T01 * V12 + T02 * V22;   // (T0 . V2)
        const float p10 = T10 * V00 + T11 * V01 + T12 * V02;
        const float p11 = T10 * V01 + T11 * V11 + T12 * V12;
        const float p12 = T10 * V02 + T11 * V12 + T12 * V22;
        const float ca = p00 * T00 + p01 * T01 + p02 * T02 + 0.3f;
        const float cb = p00 * T10 + p01 * T11 + p02 * T12;
        const float cc = p10 * T10 + p11 * T11 + p12 * T12 + 0.3f;
        const float dca = a0.z, dcb = a0.w, dcc = a1.x;
        const float denom = ca * cc - cb * cb;
        const float d2i = 1.0f / ((denom * denom) + 0.0000001f);
        float dL_da = 0.f, dL_db = 0.f, dL_dc = 0.f;
        if (d2i != 0.f) {
            dL_da = d2i * (-cc * cc * dca + 2 * cb * cc * dcb + (denom - ca * cc) * dcc);
            dL_dc = d2i * (-ca * ca * dcc + 2 * ca * cb * dcb + (denom - ca * cc) * dca);
            dL_db = d2i * 2 * (cb * cc * dca - (denom + 2 * cb * cb) * dcb + ca * cb * dcc);
            dcov[0] = T00 * T00 * dL_da + T00 * T10 * dL_db + T10 * T10 * dL_dc;
            dcov[3] = T01 * T01 * dL_da + T01 * T11 * dL_db + T11 * T11 * dL_dc;
            dcov[5] = T02 * T02 * dL_da + T02 * T12 * dL_db + T12 * T12 * dL_dc;
            dcov[1] = 2 * T00 * T01 * dL_da + (T00 * T11 + T01 * T10) * dL_db + 2 * T10 * T11 * dL_dc;
            dcov[2] = 2 * T00 * T02 * dL_da + (T00 * T12 + T02 * T10) * dL_db + 2 * T10 * T12 * dL_dc;
            dcov[4] = 2 * T02 * T01 * dL_da + (T01 * T12 + T02 * T11) * dL_db + 2 * T11 * T12 * dL_dc;
        }
        const float dT00 = 2 * p00 * dL_da + p10 * dL_db, dT01 = 2 * p01 * dL_da + p11 * dL_db, dT02 = 2 * p02 * dL_da + p12 * dL_db;
        const float dT10 = 2 * p10 * dL_dc + p00 * dL_db, dT11 = 2 * p11 * dL_dc + p01 * dL_db, dT12 = 2 * p12 * dL_dc + p02 * dL_db;
        const float dJ00 = W00 * dT00 + W01 * dT01 + W02 * dT02;
        const float dJ02 = W20 * dT00 + W21 * dT01 + W22 * dT02;
        const float dJ11 = W10 * dT10 + W11 * dT11 + W12 * dT12;
        const float dJ12 = W20 * dT10 + W21 * dT11 + W22 * dT12;
        const float tz = 1.f / t.z, tz2 = tz * tz, tz3 = tz2 * tz;
        const float dtx = xgm * -a.fx * tz2 * dJ02;
        const float dty = ygm * -a.fy * tz2 * dJ12;
        const float dtz = -a.fx * tz2 * dJ00 - a.fy * tz2 * dJ11 + (2 * a.fx * t.x) * tz3 * dJ02 + (2 * a.fy * t.y) * tz3 * dJ12;
        dmean.x = vm[0] * dtx + vm[1] * dty + vm[2] * dtz;
        dmean.y = vm[4] * dtx + vm[5] * dty + vm[6] * dtz;
        dmean.z = vm[8] * dtx + vm[9] * dty + vm[10] * dtz;

        // ---- screen-space mean and depth -> mean (backward.cu:366-403) ----
        const float hw = pm[3] * mean.x + pm[7] * mean.y + pm[11] * mean.z + pm[15];
        const float m_w = 1.0f / (hw + 0.0000001f);
        const float mul1 = (pm[0] * mean.x + pm[4] * mean.y + pm[8] * mean.z + pm[12]) * m_w * m_w;
        const float mul2 = (pm[1] * mean.x + pm[5] * mean.y + pm[9] * mean.z + pm[13]) * m_w * m_w;
        const float g2x = a0.x, g2y = a0.y;
        dmean.x += (pm[0] * m_w - pm[3] * mul1) * g2x + (pm[1] * m_w - pm[3] * mul2) * g2y;
        dmean.y += (pm[4] * m_w - pm[7] * mul1) * g2x + (pm[5] * m_w - pm[7] * mul2) * g2y;
        dmean.z += (pm[8] * m_w - pm[11] * mul1) * g2x + (pm[9] * m_w - pm[11] * mul2) * g2y;
        const float mul3 = vm[2] * mean.x + vm[6] * mean.y + vm[10] * mean.z + vm[14];
        const float gdep = a1.z;
        dmean.x += (vm[2] - vm[3] * mul3) * gdep;
        dmean.y += (vm[6] - vm[7] * mul3) * gdep;
        dmean.z += (vm[10] - vm[11] * mul3) * gdep;

        // ---- colour -> SH and view direction -> mean (backward.cu:20-139) ----
        if (use_sh) {
            float* sh = ws + lane * stride;      // read coefficients, then overwrite with their gradient
            const unsigned char cl = __ldg(a.clamped + idx);
            const float gr = (cl & 1) ? 0.f : a2.x, gg = (cl & 2) ? 0.f : a2.y, gb = (cl & 4) ? 0.f : a2.z;
            const float3 cam = make_float3(s_cam[32], s_cam[33], s_cam[34]);
            const float3 d0 = make_float3(mean.x - cam.x, mean.y - cam.y, mean.z - cam.z);
            const float len = sqrtf(d0.x * d0.x + d0.y * d0.y + d0.z * d0.z);
            const float x = d0.x / len, y = d0.y / len, z = d0.z / len;
            float3 dx_ = make_float3(0.f, 0.f, 0.f), dy_ = dx_, dz_ = dx_;   // dRGB/d{x,y,z} per channel
            auto coef = [&](int k) { return make_float3(sh[3 * k], sh[3 * k + 1], sh[3 * k + 2]); };
            auto put = [&](int k, float w) { sh[3 * k] = w * gr; sh[3 * k + 1] = w * gg; sh[3 * k + 2] = w * gb; };
            auto axpy = [&](float3& acc3, float w, const float3 v) { acc3.x += w * v.x; acc3.y += w * v.y; acc3.z += w * v.z; };
            const int D = a.D;
            float3 s1, s2, s3;
            if (D > 0) { s1 = coef(1); s2 = coef(2); s3 = coef(3); }
            put(0, SH0);
            if (D > 0) {
                put(1, -SH1 * y); put(2, SH1 * z); put(3, -SH1 * x);
                axpy(dx_, -SH1, s3); axpy(dy_, -SH1, s1); axpy(dz_, SH1, s2);
                if (D > 1) {
                    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
                    const float3 s4 = coef(4), s5 = coef(5), s6 = coef(6), s7 = coef(7), s8 = coef(8);
                    put(4, SH2b[0] * xy); put(5, SH2b[1] * yz); put(6, SH2b[2] * (2.f * zz - xx - yy));
                    put(7, SH2b[3] * xz); put(8, SH2b[4] * (xx - yy));
                    axpy(dx_, SH2b[0] * y, s4); axpy(dx_, SH2b[2] * 2.f * -x, s6); axpy(dx_, SH2b[3] * z, s7); axpy(dx_, SH2b[4] * 2.f * x, s8);
                    axpy(dy_, SH2b[0] * x, s4); axpy(dy_, SH2b[1] * z, s5); axpy(dy_, SH2b[2] * 2.f * -y, s6); axpy(dy_, SH2b[4] * 2.f * -y, s8);
                    axpy(dz_, SH2b[1] * y, s5); axpy(dz_, SH2b[2] * 2.f * 2.f * z, s6); axpy(dz_, SH2b[3] * x, s7);
                    if (D > 2) {
                        const float3 s9 = coef(9), s10 = coef(10), s11 = coef(11), s12 = coef(12), s13 = coef(13), s14 = coef(14), s15 = coef(15);
                        put(9, SH3b[0] * y * (3.f * xx - yy)); put(10, SH3b[1] * xy * z);
                        put(11, SH3b[2] * y * (4.f * zz - xx - yy)); put(12, SH3b[3] * z * (2.f * zz - 3.f * xx - 3.f * yy));
                        put(13, SH3b[4] * x * (4.f * zz - xx - yy)); put(14, SH3b[5] * z * (xx - yy));
                        put(15, SH3b[6] * x * (xx - 3.f * yy));
                        axpy(dx_, SH3b[0] * 3.f * 2.f * xy, s9); axpy(dx_, SH3b[1] * yz, s10); axpy(dx_, SH3b[2] * -2.f * xy, s11);
                        axpy(dx_, SH3b[3] * -3.f * 2.f * xz, s12); axpy(dx_, SH3b[4] * (-3.f * xx + 4.f * zz - yy), s13);
                        axpy(dx_, SH3b[5] * 2.f * xz, s14); axpy(dx_, SH3b[6] * 3.f * (xx - yy), s15);
                        axpy(dy_, SH3b[0] * 3.f * (xx - yy), s9); axpy(dy_, SH3b[1] * xz, s10);
                        axpy(dy_, SH3b[2] * (-3.f * yy + 4.f * zz - xx), s11); axpy(dy_, SH3b[3] * -3.f * 2.f * yz, s12);
                        axpy(dy_, SH3b[4] * -2.f * xy, s13); axpy(dy_, SH3b[5] * -2.f * yz, s14); axpy(dy_, SH3b[6] * -3.f * 2.f * xy, s15);
                        axpy(dz_, SH3b[1] * xy, s10); axpy(dz_, SH3b[2] * 4.f * 2.f * yz, s11);
                        axpy(dz_, SH3b[3] * 3.f * (2.f * zz - xx - yy), s12); axpy(dz_, SH3b[4] * 4.f * 2.f * xz, s13);
                        axpy(dz_, SH3b[5] * (xx - yy), s14);
                    }
                }
            }
            const int nco = (D + 1) * (D + 1);
            for (int k = 3 * nco; k < 3 * a.M; ++k) sh[k] = 0.f;
            const float3 ddir = make_float3(dx_.x * gr + dx_.y * gg + dx_.z * gb,
                                            dy_.x * gr + dy_.y * gg + dy_.z * gb,
                                            dz_.x * gr + dz_.y * gg + dz_.z * gb);
            // Jacobian of v/|v| (auxiliary.h:107-117)
            const float sum2 = d0.x * d0.x + d0.y * d0.y + d0.z * d0.z;
            const float inv32 = 1.0f / sqrtf(sum2 * sum2 * sum2);
            dmean.x += ((sum2 - d0.x * d0.x) * ddir.x - d0.y * d0.x * ddir.y - d0.z * d0.x * ddir.z) * inv32;
            dmean.y += (-d0.x * d0.y * ddir.x + (sum2 - d0.y * d0.y) * ddir.y - d0.z * d0.y * ddir.z) * inv32;
            dmean.z += (-d0.x * d0.z * ddir.x - d0.y * d0.z * ddir.y + (sum2 - d0.z * d0.z) * ddir.z) * inv32;
        }

        // ---- cov3D -> scale, rotation (backward.cu:278-341) ----
        if (a.scales != nullptr) {
            const float3 sc = make_float3(__ldg(a.scales + 3 * idx), __ldg(a.scales + 3 * idx + 1), __ldg(a.scales + 3 * idx + 2));
            const float4 q = __ldg(reinterpret_cast<const float4*>(a.rots) + idx);
            const float r = q.x, x = q.y, y = q.z, z = q.w;
            float R[3][3];    // R[c][r], same arrangement as the forward
            R[0][0] = 1.f - 2.f * (y * y + z * z); R[0][1] = 2.f * (x * y - r * z); R[0][2] = 2.f * (x * z + r * y);
            R[1][0] = 2.f * (x * y + r * z); R[1][1] = 1.f - 2.f * (x * x + z * z); R[1][2] = 2.f * (y * z - r * x);
            R[2][0] = 2.f * (x * z - r * y); R[2][1] = 2.f * (y * z + r * x); R[2][2] = 1.f - 2.f * (x * x + y * y);
            const float s[3] = {a.scale_mod * sc.x, a.scale_mod * sc.y, a.scale_mod * sc.z};
            float Mm[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int rr = 0; rr < 3; ++rr) Mm[c][rr] = s[rr] * R[c][rr];
            float dS[3][3];   // symmetric dL/dSigma
            dS[0][0] = dcov[0]; dS[1][1] = dcov[3]; dS[2][2] = dcov[5];
            dS[0][1] = dS[1][0] = 0.5f * dcov[1]; dS[0][2] = dS[2][0] = 0.5f * dcov[2]; dS[1][2] = dS[2][1] = 0.5f * dcov[4];
            // dL/dM = 2 M dSigma  (column-major product: out[c][r] = sum_k M[k][r] * dS[c][k])
            float dM[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int rr = 0; rr < 3; ++rr)
                    dM[c][rr] = 2.f * (Mm[0][rr] * dS[c][0] + Mm[1][rr] * dS[c][1] + Mm[2][rr] * dS[c][2]);
            // dMt[c][r] = dM[r][c];  Rt[c][r] = R[r][c]
            float dMt[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int rr = 0; rr < 3; ++rr) dMt[c][rr] = dM[rr][c];
            dscale.x = R[0][0] * dMt[0][0] + R[1][0] * dMt[0][1] + R[2][0] * dMt[0][2];
            dscale.y = R[0][1] * dMt[1][0] + R[1][1] * dMt[1][1] + R[2][1] * dMt[1][2];
            dscale.z = R[0][2] * dMt[2][0] + R[1][2] * dMt[2][1] + R[2][2] * dMt[2][2];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int rr = 0; rr < 3; ++rr) dMt[c][rr] *= s[c];
            drot.x = 2 * z * (dMt[0][1] - dMt[1][0]) + 2 * y * (dMt[2][0] - dMt[0][2]) + 2 * x * (dMt[1][2] - dMt[2][1]);
            drot.y = 2 * y * (dMt[1][0] + dMt[0][1]) + 2 * z * (dMt[2][0] + dMt[0][2]) + 2 * r * (dMt[1][2] - dMt[2][1]) - 4 * x * (dMt[2][2] + dMt[1][1]);
            drot.z = 2 * x * (dMt[1][0] + dMt[0][1]) + 2 * r * (dMt[2][0] - dMt[0][2]) + 2 * z * (dMt[1][2] + dMt[2][1]) - 4 * y * (dMt[2][2] + dMt[0][0]);
            drot.w = 2 * r * (dMt[0][1] - dMt[1][0]) + 2 * x * (dMt[2][0] + dMt[0][2]) + 2 * y * (dMt[1][2] + dMt[2][1]) - 4 * z * (dMt[1][1] + dMt[0][0]);
        }
    } else if (use_sh && any_vis && in_range) {
        float* sh = ws + lane * stride;
        for (int k = 0; k < 3 * a.M; ++k) sh[k] = 0.f;
    }

    // ---- write-out: every row is written (zeros for culled Gaussians), so the caller can
    // hand in uninitialised tensors instead of the reference's ten torch::zeros fills ----
    if (in_range) {
        a.dL_dmean2D[3 * idx] = a0.x; a.dL_dmean2D[3 * idx + 1] = a0.y; a.dL_dmean2D[3 * idx + 2] = 0.f;
        a.dL_dcolor[3 * idx] = a2.x; a.dL_dcolor[3 * idx + 1] = a2.y; a.dL_dcolor[3 * idx + 2] = a2.z;
        a.dL_dopacity[idx] = a1.y;
        a.dL_dmean3D[3 * idx] = dmean.x; a.dL_dmean3D[3 * idx + 1] = dmean.y; a.dL_dmean3D[3 * idx + 2] = dmean.z;
#pragma unroll
        for (int k = 0; k < 6; ++k) a.dL_dcov3D[6 * (size_t)idx + k] = dcov[k];
        a.dL_dscale[3 * idx] = dscale.x; a.dL_dscale[3 * idx + 1] = dscale.y; a.dL_dscale[3 * idx + 2] = dscale.z;
        reinterpret_cast<float4*>(a.dL_drot)[idx] = drot;
    }
    if (use_sh) {
        __syncwarp();
        float* dst = a.dL_dsh + (size_t)g0 * 3 * a.M;
        const int per = 3 * a.M;
        if (!any_vis) {
            if (a.accumulate_sh) {
                // nothing to add
            } else if ((per & 3) == 0) {
                float4* d4 = reinterpret_cast<float4*>(dst);
                for (int e = lane; e < ng * per / 4; e += 32) d4[e] = make_float4(0.f, 0.f, 0.f, 0.f);
            } else for (int e = lane; e < ng * per; e += 32) dst[e] = 0.f;
        } else if ((per & 3) == 0) {
            float4* d4 = reinterpret_cast<float4*>(dst);
            for (int e = lane; e < ng * per / 4; e += 32) {
                int f = e * 4, gg = f / per, k = f - gg * per;
                const float* s = ws + gg * stride + k;
                float4 v = make_float4(s[0], s[1], s[2], s[3]);
                if (a.accumulate_sh) { const float4 o = d4[e]; v = make_float4(o.x + v.x, o.y + v.y, o.z + v.z, o.w + v.w); }
                d4[e] = v;
            }
        } else {
            for (int e = lane; e < ng * per; e += 32) {
                int gg = e / per, k = e - gg * per;
                dst[e] = (a.accumulate_sh ? dst[e] : 0.f) + ws[gg * stride + k];
            }
        }
    }
}

}  // namespace

int rast_backward(int P, int D, int M, long long R, int W, int H, const float* bg, const float* means3D,
                  const float* shs, const float* colors_precomp, const float* scales, float scale_modifier,
                  const float* rotations, const float* cov3D_precomp, const float* viewmatrix,
                  const float* projmatrix, const float* campos, float tan_fovx, float tan_fovy,
                  const int* radii, void* geom_buf, void* bin_buf, void* img_buf, const float* dL_dpix,
                  const float* dL_dpix_depth, float* grad_arena, float* dL_dmean2D, float* dL_dcolor,
                  float* dL_dopacity, float* dL_dmean3D, float* dL_dcov3D, float* dL_dsh, float* dL_dscale,
                  float* dL_drot, int accumulate_sh, cudaStream_t stream)
{
    if (P <= 0) return 0;
    const int grid_x = (W + TILE_X - 1) / TILE_X, grid_y = (H + TILE_Y - 1) / TILE_Y;
    const size_t tiles = (size_t)grid_x * grid_y, npix = (size_t)W * H;
    const int tile_bits = tile_bits_for(tiles);
    size_t tmp;
    GeomState g = GeomState::carve(geom_buf, (size_t)P, &tmp);
    BinState b = BinState::carve(bin_buf, (size_t)P, (size_t)R, tile_bits, &tmp);
    ImgState img = ImgState::carve(img_buf, npix, tiles, &tmp);
    const int passes = radix_plan((size_t)R, 0, tile_bits).passes;
    const u32* sorted_list = (R > 0 && (passes & 1)) ? b.ivals_b : b.ivals_a;

    {
        ProfScope prof(PROF_COMPOSITE_BWD, stream);
        cudaMemsetAsync(grad_arena, 0, (size_t)P * ACC * sizeof(float), stream);
        if (R > 0)
            composite_bwd2_kernel<<<(unsigned)tiles, CB2_THREADS, 0, stream>>>(
                img.ranges, sorted_list, W, H, grid_x, g.recA, g.recB, g.recC, bg, img.final_T, img.n_contrib,
                dL_dpix, dL_dpix_depth, grad_arena);
    }

    PreBwdArgs a;
    a.P = P; a.D = D; a.M = M; a.W = W; a.H = H;
    a.means = means3D; a.scales = scales; a.rots = rotations;
    a.shs = colors_precomp ? nullptr : shs;
    a.cov3d = cov3D_precomp ? cov3D_precomp : g.cov3D;
    a.view = viewmatrix; a.proj = projmatrix; a.campos = campos;
    a.scale_mod = scale_modifier; a.tanx = tan_fovx; a.tany = tan_fovy;
    a.fx = W / (2.0f * tan_fovx); a.fy = H / (2.0f * tan_fovy);
    a.radii = radii; a.clamped = g.clamped; a.acc = grad_arena;
    a.has_colors_precomp = colors_precomp != nullptr;
    a.dL_dmean2D = dL_dmean2D; a.dL_dcolor = dL_dcolor; a.dL_dopacity = dL_dopacity; a.dL_dmean3D = dL_dmean3D;
    a.dL_dcov3D = dL_dcov3D; a.dL_dsh = (colors_precomp || M == 0) ? nullptr : dL_dsh; a.accumulate_sh = accumulate_sh;
    a.dL_dscale = dL_dscale; a.dL_drot = dL_drot;
    const size_t smem = a.dL_dsh ? (size_t)PB_WARPS * 32 * (3 * M + 1) * sizeof(float) : 0;
    if (smem > 48 * 1024) cudaFuncSetAttribute(preprocess_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    ProfScope prof(PROF_PREPROCESS_BWD, stream);
    preprocess_bwd_kernel<<<(P + PB_THREADS - 1) / PB_THREADS, PB_THREADS, smem, stream>>>(a);
    return check_launch("rast_backward");
}

}  // namespace b200gs
