// D-SSIM loss term: utils/loss_utils.py:ssim (the 3DGS formulation, SURVEY.md §2 row 11) as a value + gradient pair of
// launches.  Per image plane, with w the 11x11 Gaussian window (sigma 1.5) and zero padding:
//   mu1 = w*x, mu2 = w*y, s11 = w*(x x) - mu1^2, s22 = w*(y y) - mu2^2, s12 = w*(x y) - mu1 mu2
//   map = ((2 mu1 mu2 + C1)(2 s12 + C2)) / ((mu1^2 + mu2^2 + C1)(s11 + s22 + C2)),   C1 = 0.01^2, C2 = 0.03^2
// and for L = sum map:  dL/dx = w*A + 2 x (w*B) + y (w*Cc),  B = dmap/ds11, Cc = dmap/ds12, A = dmap/dmu1 - 2 mu1 B - mu2 Cc
// (the window is symmetric; A, B, Cc are zero outside the image, which is what zero padding implies).
//   ssim_fwd_kernel  loads a 32x32 output tile plus a 5-pixel halo of x and y into shared memory, blurs the five moments
//                    separably (11 taps along x, then 11 along y), evaluates the map, reduces it per CTA (one FP64 atomic per
//                    CTA into the caller's scratch) and, when a gradient is wanted, writes A, B, Cc to the caller's scratch;
//   ssim_bwd_kernel  blurs A, B, Cc the same way and ADDS weight * dL/dx into the caller's gradient buffer;
//   ssim_sum_kernel  adds value_offset + value_scale * (the image's map sum) into ssim_sum[n].
// The blurs accumulate in FP64 (inputs and taps are FP32; products of two FP32 values are exact in FP64): s11 = w*(x x) - mu1^2
// cancels catastrophically where an image is flat: with FP32 blurs a constant 64x64 pair's SSIM was off by 6e-6 (relative) on a
// B200, and the backward's w*A + 2 x (w*B) terms, which cancel the same way, by 1e-4 of the gradient's maximum in an FP32
// emulation (FP64 blurs: 3e-6).  Everything pointwise
// (the map, A, B, Cc, the gradient's scaling) is FP32.  B200: FP64 FMAs issue at half the FP32 rate, the kernels stay
// memory / shared-memory bound.  Traffic per pixel and channel: 8 B read (forward) + 12 B written (A, B, Cc),
// 12 B + 8 B + 4 B read and 4 B written (backward) -> 48 B; arithmetic 5 x 22 + 3 x 22 FP64 FMAs plus the pointwise terms.
#include <cmath>

#include "common.cuh"
#include "../../include/b200gs.h"

namespace b200gs {
namespace {

constexpr int SS_R = 5;                          // window radius: 11 taps
constexpr int SS_K = 2 * SS_R + 1;
constexpr int SS_TX = 32, SS_TY = 32;            // outputs per CTA
constexpr int SS_HX = SS_TX + 2 * SS_R, SS_HY = SS_TY + 2 * SS_R;      // 42 x 42 halo tile
constexpr int SS_THREADS = 256;                  // vertical pass: 32 columns x 8 groups of 4 consecutive rows
constexpr int SS_ROWS = SS_TY / (SS_THREADS / SS_TX);                   // 4
// the reference's Python constants, rounded to float as torch does when it adds them to a float32 tensor
constexpr float SS_C1 = (float)(0.01 * 0.01), SS_C2 = (float)(0.03 * 0.03);

struct Taps { float g[SS_K]; };

// float(u8) / 255.0f (IEEE division) = utils/general_utils.py:PILtoTorch, like the u8 L1 kernel
template <bool U8>
__device__ __forceinline__ float load_target(const void* __restrict__ y, long long plane_off, long long pix, int c)
{
    if (U8) return __fdiv_rn((float)__ldg(reinterpret_cast<const unsigned char*>(y) + 3 * pix + c), 255.0f);
    return __ldg(reinterpret_cast<const float*>(y) + plane_off + pix);
}

// Separable blur of the planes loaded into shared memory (halo included) -> out[m][o] for the SS_ROWS outputs of this
// thread: rows SS_ROWS*ty .. +SS_ROWS-1 of column tx.  `prod` forms the NB blurred quantities at a halo position (the forward
// blurs x, y, x x, y y, x y out of two loaded planes).  s_h is the horizontal result [NB][SS_HY][SS_TX].  FP64 accumulation.
template <int NB, typename F>
__device__ __forceinline__ void blur_tile(const Taps& t, double (*s_h)[SS_HY][SS_TX], F prod, double (&out)[NB][SS_ROWS])
{
    for (int i = threadIdx.x; i < SS_HY * SS_TX; i += SS_THREADS) {
        const int r = i / SS_TX, q = i % SS_TX;
        double h[NB];
#pragma unroll
        for (int m = 0; m < NB; ++m) h[m] = 0.0;
#pragma unroll
        for (int k = 0; k < SS_K; ++k) {
            double v[NB];
            prod(r, q + k, v);
#pragma unroll
            for (int m = 0; m < NB; ++m) h[m] = fma((double)t.g[k], v[m], h[m]);
        }
#pragma unroll
        for (int m = 0; m < NB; ++m) s_h[m][r][q] = h[m];
    }
    __syncthreads();
    const int tx = threadIdx.x % SS_TX, r0 = (threadIdx.x / SS_TX) * SS_ROWS;
#pragma unroll
    for (int m = 0; m < NB; ++m)
#pragma unroll
        for (int o = 0; o < SS_ROWS; ++o) out[m][o] = 0.0;
    // sliding window: SS_ROWS + 10 loads per plane instead of 11 * SS_ROWS; taps applied in order k = 0..10 for every output
#pragma unroll
    for (int j = 0; j < SS_ROWS + 2 * SS_R; ++j) {
#pragma unroll
        for (int m = 0; m < NB; ++m) {
            const double h = s_h[m][r0 + j][tx];
#pragma unroll
            for (int o = 0; o < SS_ROWS; ++o)
                if (j - o >= 0 && j - o < SS_K) out[m][o] = fma((double)t.g[j - o], h, out[m][o]);
        }
    }
}

template <bool U8, bool GRAD>
__global__ void __launch_bounds__(SS_THREADS) ssim_fwd_kernel(int C, int H, int W, const float* __restrict__ x, const void* __restrict__ y,
                                                              Taps t, double* __restrict__ map_sum, float* __restrict__ abc, long long total)
{
    extern __shared__ __align__(16) unsigned char ss_smem[];
    auto s_h = reinterpret_cast<double (*)[SS_HY][SS_TX]>(ss_smem);                              // [5]: 53.8 KB
    auto s_in = reinterpret_cast<float (*)[SS_HY][SS_HX]>(ss_smem + 5 * sizeof(double) * SS_HY * SS_TX);   // [2]: 14.1 KB
    __shared__ float s_part[SS_THREADS / 32];
    const int plane = blockIdx.z, n = plane / C, c = plane - n * C;
    const long long HW = (long long)H * W, off = (long long)plane * HW;
    const int x0 = blockIdx.x * SS_TX, y0 = blockIdx.y * SS_TY;
    for (int i = threadIdx.x; i < SS_HX * SS_HY; i += SS_THREADS) {
        const int r = i / SS_HX, q = i % SS_HX, gy = y0 - SS_R + r, gx = x0 - SS_R + q;
        float a = 0.f, b = 0.f;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            const long long pix = (long long)gy * W + gx;
            a = __ldg(x + off + pix);
            b = load_target<U8>(y, off, pix, c);
        }
        s_in[0][r][q] = a; s_in[1][r][q] = b;
    }
    __syncthreads();
    double mom[5][SS_ROWS];
    blur_tile<5>(t, s_h, [&](int r, int q, double (&v)[5]) {
        const double a = s_in[0][r][q], b = s_in[1][r][q];
        v[0] = a; v[1] = b; v[2] = a * a; v[3] = b * b; v[4] = a * b;
    }, mom);
    const int gx = x0 + threadIdx.x % SS_TX, gy0 = y0 + (threadIdx.x / SS_TX) * SS_ROWS;
    float acc = 0.f;
#pragma unroll
    for (int o = 0; o < SS_ROWS; ++o) {
        if (gx >= W || gy0 + o >= H) continue;
        const float mu1 = (float)mom[0][o], mu2 = (float)mom[1][o];
        const float mu1_sq = mu1 * mu1, mu2_sq = mu2 * mu2, mu1_mu2 = mu1 * mu2;
        const float s11 = (float)(mom[2][o] - mom[0][o] * mom[0][o]), s22 = (float)(mom[3][o] - mom[1][o] * mom[1][o]);
        const float s12 = (float)(mom[4][o] - mom[0][o] * mom[1][o]);
        const float n1 = 2.f * mu1_mu2 + SS_C1, n2 = 2.f * s12 + SS_C2;
        const float d1 = mu1_sq + mu2_sq + SS_C1, d2 = s11 + s22 + SS_C2;
        const float map = (n1 * n2) / (d1 * d2);
        acc += map;
        if (GRAD) {
            const float dd = d1 * d2;
            const float gB = -map / d2;                                   // dmap/ds11 (= dmap/ds22)
            const float gC = 2.f * n1 / dd;                               // dmap/ds12
            const float gmu1 = 2.f * mu2 * n2 / dd - 2.f * mu1 * map / d1;  // dmap/dmu1 with s11, s12 held
            const float gA = gmu1 - 2.f * mu1 * gB - mu2 * gC;            // s11, s12 depend on mu1 too
            const long long idx = off + (long long)(gy0 + o) * W + gx;
            abc[idx] = gA; abc[total + idx] = gB; abc[2 * total + idx] = gC;
        }
    }
    if (!map_sum) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < SS_THREADS / 32; ++w) s += s_part[w];
        atomicAdd(map_sum + n, (double)s);
    }
}

template <bool U8>
__global__ void __launch_bounds__(SS_THREADS) ssim_bwd_kernel(int C, int H, int W, const float* __restrict__ x, const void* __restrict__ y,
                                                              Taps t, float weight, const float* __restrict__ abc, long long total,
                                                              float* __restrict__ d_x)
{
    extern __shared__ __align__(16) unsigned char ss_smem[];
    auto s_h = reinterpret_cast<double (*)[SS_HY][SS_TX]>(ss_smem);                              // [3]: 32.3 KB
    auto s_in = reinterpret_cast<float (*)[SS_HY][SS_HX]>(ss_smem + 3 * sizeof(double) * SS_HY * SS_TX);   // [3]: 21.2 KB
    const int plane = blockIdx.z, c = plane % C;
    const long long HW = (long long)H * W, off = (long long)plane * HW;
    const int x0 = blockIdx.x * SS_TX, y0 = blockIdx.y * SS_TY;
    for (int i = threadIdx.x; i < SS_HX * SS_HY; i += SS_THREADS) {
        const int r = i / SS_HX, q = i % SS_HX, gy = y0 - SS_R + r, gx = x0 - SS_R + q;
        float a = 0.f, b = 0.f, cc = 0.f;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            const long long idx = off + (long long)gy * W + gx;
            a = __ldg(abc + idx); b = __ldg(abc + total + idx); cc = __ldg(abc + 2 * total + idx);
        }
        s_in[0][r][q] = a; s_in[1][r][q] = b; s_in[2][r][q] = cc;
    }
    __syncthreads();
    double bl[3][SS_ROWS];
    blur_tile<3>(t, s_h, [&](int r, int q, double (&v)[3]) { v[0] = s_in[0][r][q]; v[1] = s_in[1][r][q]; v[2] = s_in[2][r][q]; }, bl);
    const int gx = x0 + threadIdx.x % SS_TX, gy0 = y0 + (threadIdx.x / SS_TX) * SS_ROWS;
#pragma unroll
    for (int o = 0; o < SS_ROWS; ++o) {
        if (gx >= W || gy0 + o >= H) continue;
        const long long pix = (long long)(gy0 + o) * W + gx;
        const float xv = __ldg(x + off + pix), yv = load_target<U8>(y, off, pix, c);
        const float g = (float)(bl[0][o] + 2.0 * xv * bl[1][o] + (double)yv * bl[2][o]);
        d_x[off + pix] += weight * g;
    }
}

__global__ void __launch_bounds__(256) ssim_sum_kernel(int N, const double* __restrict__ map_sum, double value_offset, double value_scale,
                                                       float* __restrict__ ssim_sum)
{
    const int n = blockIdx.x * 256 + threadIdx.x;
    if (n < N) ssim_sum[n] += (float)(value_offset + value_scale * map_sum[n]);
}

constexpr size_t SS_FWD_SMEM = 5 * sizeof(double) * SS_HY * SS_TX + 2 * sizeof(float) * SS_HY * SS_HX;
constexpr size_t SS_BWD_SMEM = 3 * sizeof(double) * SS_HY * SS_TX + 3 * sizeof(float) * SS_HY * SS_HX;

// utils/loss_utils.py:gaussian(11, 1.5): exp in double (Python floats), rounded to a float32 tensor, divided by its float32 sum
Taps make_taps()
{
    Taps t;
    float raw[SS_K];
    double sum = 0.0;
    for (int k = 0; k < SS_K; ++k) {
        raw[k] = (float)std::exp(-(double)((k - SS_R) * (k - SS_R)) / (2.0 * 1.5 * 1.5));
        sum += raw[k];
    }
    const float s = (float)sum;
    for (int k = 0; k < SS_K; ++k) t.g[k] = raw[k] / s;
    return t;
}

// scratch = [N FP64 map sums | A, B, Cc: 3 * N*C*H*W floats when a gradient is wanted]
size_t scratch_layout(int N, int C, int H, int W, bool grad, void* base, double** map_sum, float** abc)
{
    Carver cv(base);
    double* ms = cv.take<double>((size_t)N);
    float* p = grad ? cv.take<float>(3 * (size_t)N * C * H * W) : nullptr;
    if (map_sum) *map_sum = ms;
    if (abc) *abc = p;
    return cv.used();
}

template <bool U8>
int ssim_launch(const char* what, int N, int C, int H, int W, const float* x, const void* y, float value_offset, float value_scale,
                float* ssim_sum, float weight, float* d_x, void* scratch, size_t scratch_bytes, cudaStream_t st)
{
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || (!ssim_sum && !d_x)) return 0;
    if (!x || !y) { set_error("%s: null pointer", what); return -1; }
    if ((long long)N * C > 65535) { set_error("%s: N * C = %lld exceeds 65535 image planes", what, (long long)N * C); return -1; }
    const size_t need = scratch_layout(N, C, H, W, d_x != nullptr, nullptr, nullptr, nullptr);
    if (!scratch || scratch_bytes < need) {
        set_error("%s: needs %zu bytes of scratch (b200gs_ssim_scratch_bytes), got %zu", what, need, scratch ? scratch_bytes : (size_t)0);
        return -1;
    }
    double* map_sum;
    float* abc;
    scratch_layout(N, C, H, W, d_x != nullptr, scratch, &map_sum, &abc);
    static const Taps taps = make_taps();
    static const bool smem_ok = cudaFuncSetAttribute(ssim_fwd_kernel<U8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SS_FWD_SMEM) == cudaSuccess
        && cudaFuncSetAttribute(ssim_fwd_kernel<U8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SS_FWD_SMEM) == cudaSuccess
        && cudaFuncSetAttribute(ssim_bwd_kernel<U8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SS_BWD_SMEM) == cudaSuccess;
    if (!smem_ok) { (void)cudaGetLastError(); set_error("%s: cannot enable %zu bytes of shared memory per CTA", what, SS_FWD_SMEM); return -1; }
    const long long total = (long long)N * C * H * W;
    const dim3 grid((unsigned)((W + SS_TX - 1) / SS_TX), (unsigned)((H + SS_TY - 1) / SS_TY), (unsigned)(N * C));
    if (ssim_sum) {
        const cudaError_t e = cudaMemsetAsync(map_sum, 0, sizeof(double) * N, st);
        if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return -1; }
    }
    double* ms = ssim_sum ? map_sum : nullptr;
    if (d_x) {
        ssim_fwd_kernel<U8, true><<<grid, SS_THREADS, SS_FWD_SMEM, st>>>(C, H, W, x, y, taps, ms, abc, total);
        ssim_bwd_kernel<U8><<<grid, SS_THREADS, SS_BWD_SMEM, st>>>(C, H, W, x, y, taps, weight, abc, total, d_x);
    } else {
        ssim_fwd_kernel<U8, false><<<grid, SS_THREADS, SS_FWD_SMEM, st>>>(C, H, W, x, y, taps, ms, nullptr, total);
    }
    if (ssim_sum) ssim_sum_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, map_sum, (double)value_offset, (double)value_scale, ssim_sum);
    return check_launch(what);
}

}  // namespace
}  // namespace b200gs

using namespace b200gs;

extern "C" {

size_t b200gs_ssim_scratch_bytes(int N, int C, int H, int W, int with_grad)
{
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
    return scratch_layout(N, C, H, W, with_grad != 0, nullptr, nullptr, nullptr);
}

int b200gs_ssim_fwd_bwd(int N, int C, int H, int W, const float* x, const float* y, float value_offset, float value_scale,
                        float* ssim_sum, float weight, float* d_x, void* scratch, size_t scratch_bytes, b200gs_stream_t stream)
{
    return ssim_launch<false>("ssim", N, C, H, W, x, y, value_offset, value_scale, ssim_sum, weight, d_x, scratch, scratch_bytes,
                              (cudaStream_t)stream);
}

int b200gs_ssim_fwd_bwd_u8(int H, int W, const float* x_chw, const unsigned char* y_hwc, float value_offset, float value_scale,
                           float* ssim_sum, float weight, float* d_x_chw, void* scratch, size_t scratch_bytes, b200gs_stream_t stream)
{
    return ssim_launch<true>("ssim_u8", 1, 3, H, W, x_chw, y_hwc, value_offset, value_scale, ssim_sum, weight, d_x_chw, scratch,
                             scratch_bytes, (cudaStream_t)stream);
}

}  // extern "C"
