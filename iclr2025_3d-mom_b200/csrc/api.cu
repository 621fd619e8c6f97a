// extern "C" surface of libb200gs.so (declared in include/b200gs.h).
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "rast_state.cuh"
#include "../../include/b200gs.h"

namespace b200gs {

static thread_local char g_err[512] = "";

// CTA caps of the persistent MLP kernels (b200gs_set_option); 0 = every SM
int g_opt_mlp_fwd_sms = 0;
int g_opt_mlp_bwd_sms = 0;

// ---- opt-in phase timing ---------------------------------------------------------------------------------------------
int g_prof_enabled = 0;
static const char* const PROF_NAMES[PROF_SLOTS] = {"preprocess_fwd", "depth_sort", "emit_instances", "tile_sort", "tile_ranges",
                                                   "composite_fwd", "composite_bwd", "preprocess_bwd"};
struct ProfPair { cudaEvent_t a, b; };
static std::vector<ProfPair> g_prof[PROF_SLOTS];          // recorded pairs per slot (only touched while profiling is enabled)
static std::vector<ProfPair> g_prof_pool;
void prof_mark(int slot, bool begin, cudaStream_t stream)
{
    if (slot < 0 || slot >= PROF_SLOTS) return;
    if (begin) {
        ProfPair p;
        if (!g_prof_pool.empty()) { p = g_prof_pool.back(); g_prof_pool.pop_back(); }
        else if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) return;
        cudaEventRecord(p.a, stream);
        g_prof[slot].push_back(p);
    } else if (!g_prof[slot].empty()) {
        cudaEventRecord(g_prof[slot].back().b, stream);
    }
}

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return -1; }
    return 0;
}

// implemented in the kernel translation units
int rast_buffer_sizes(int P, long long R, int W, int H, size_t out[3]);
int rast_forward_stage1(int P, int D, int M, int W, int H, const float* means3D, const float* shs,
                        const float* colors_precomp, const float* opacities, const float* scales,
                        float scale_modifier, const float* rotations, const float* cov3D_precomp,
                        const float* viewmatrix, const float* projmatrix, const float* campos,
                        float tan_fovx, float tan_fovy, int prefiltered, int* radii, void* geom_buf,
                        size_t geom_bytes, unsigned long long* host_counters, cudaStream_t stream);
int rast_forward_stage2(int P, long long R, long long n_visible, int W, int H, const float* bg,
                        void* geom_buf, void* bin_buf, size_t bin_bytes, void* img_buf, size_t img_bytes,
                        float* out_color, float* out_depth, cudaStream_t stream);
int rast_backward(int P, int D, int M, long long R, int W, int H, const float* bg, const float* means3D,
                  const float* shs, const float* colors_precomp, const float* scales, float scale_modifier,
                  const float* rotations, const float* cov3D_precomp, const float* viewmatrix,
                  const float* projmatrix, const float* campos, float tan_fovx, float tan_fovy,
                  const int* radii, void* geom_buf, void* bin_buf, void* img_buf, const float* dL_dpix,
                  const float* dL_dpix_depth, float* grad_arena, float* dL_dmean2D, float* dL_dcolor,
                  float* dL_dopacity, float* dL_dmean3D, float* dL_dcov3D, float* dL_dsh, float* dL_dscale,
                  float* dL_drot, int accumulate_sh, cudaStream_t stream);
int mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                 unsigned char* present, cudaStream_t stream);

size_t dist2_scratch_bytes(size_t P);
int dist2(int P, const float* points, float* mean_dists, void* scratch, size_t scratch_bytes, cudaStream_t stream);

// ---- export of internal state in the reference's layout (parity tests only) -------------
enum ExportField { F_DEPTHS, F_MEANS2D, F_CONIC_OPACITY, F_RGB, F_CLAMPED, F_KEYS };

__global__ void export_geom_kernel(int field, int P, const int* __restrict__ unused, const float4* __restrict__ recA,
                                   const float4* __restrict__ recB, const float4* __restrict__ recC,
                                   const unsigned char* __restrict__ clamped, const u32* __restrict__ touched,
                                   void* __restrict__ dst)
{
    (void)unused;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const bool vis = touched[i] > 0;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 A = vis ? recA[i] : z, B = vis ? recB[i] : z, C = vis ? recC[i] : z;
    switch (field) {
        case F_DEPTHS: ((float*)dst)[i] = B.z; break;
        case F_MEANS2D: ((float2*)dst)[i] = make_float2(A.x, A.y); break;
        case F_CONIC_OPACITY: ((float4*)dst)[i] = make_float4(A.z, A.w, B.x, B.y); break;
        case F_RGB: ((float*)dst)[3 * i] = C.x; ((float*)dst)[3 * i + 1] = C.y; ((float*)dst)[3 * i + 2] = C.z; break;
        case F_CLAMPED: {
            unsigned char c = vis ? clamped[i] : 0;
            ((unsigned char*)dst)[3 * i] = c & 1; ((unsigned char*)dst)[3 * i + 1] = (c >> 1) & 1; ((unsigned char*)dst)[3 * i + 2] = (c >> 2) & 1;
        } break;
    }
}

__global__ void export_keys_kernel(u32 R, const u32* __restrict__ tile_sorted, const u32* __restrict__ list,
                                   const float4* __restrict__ recB, u64* __restrict__ dst)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    dst[i] = ((u64)tile_sorted[i] << 32) | (u64)__float_as_uint(recB[list[i]].z);
}

}  // namespace b200gs

using namespace b200gs;

extern "C" {

const char* b200gs_last_error(void) { return g_err; }
int b200gs_version(void) { return 100; }

int b200gs_set_option(const char* name, int value)
{
    if (name && !strcmp(name, "mlp_fwd_sms")) { b200gs::g_opt_mlp_fwd_sms = value; return 0; }
    if (name && !strcmp(name, "mlp_bwd_sms")) { b200gs::g_opt_mlp_bwd_sms = value; return 0; }
    set_error("b200gs_set_option: unknown option '%s'", name ? name : "(null)");
    return -1;
}
int b200gs_get_option(const char* name)
{
    if (name && !strcmp(name, "mlp_fwd_sms")) return b200gs::g_opt_mlp_fwd_sms;
    if (name && !strcmp(name, "mlp_bwd_sms")) return b200gs::g_opt_mlp_bwd_sms;
    return -1;
}

int b200gs_profile_enable(int enable)
{
    for (int s = 0; s < PROF_SLOTS; ++s) {               // (re)start from an empty record either way
        for (auto& p : b200gs::g_prof[s]) b200gs::g_prof_pool.push_back(p);
        b200gs::g_prof[s].clear();
    }
    b200gs::g_prof_enabled = enable != 0;
    return 0;
}

int b200gs_profile_read(const char* phase, int* calls, float* total_ms)
{
    for (int s = 0; s < PROF_SLOTS; ++s) {
        if (!phase || strcmp(phase, b200gs::PROF_NAMES[s])) continue;
        float total = 0.f; int n = 0;
        for (auto& p : b200gs::g_prof[s]) {
            float ms = 0.f;
            if (cudaEventSynchronize(p.b) != cudaSuccess || cudaEventElapsedTime(&ms, p.a, p.b) != cudaSuccess) {
                cudaGetLastError(); continue;
            }
            total += ms; ++n;
        }
        if (calls) *calls = n;
        if (total_ms) *total_ms = total;
        return 0;
    }
    set_error("b200gs_profile_read: unknown phase '%s'", phase ? phase : "(null)");
    return -1;
}

int b200gs_rast_buffer_sizes(int P, long long R, int W, int H, size_t out_bytes[3])
{
    return rast_buffer_sizes(P, R, W, H, out_bytes);
}

int b200gs_rast_forward_stage1(int P, int D, int M, int W, int H, const float* means3D, const float* shs,
                               const float* colors_precomp, const float* opacities, const float* scales,
                               float scale_modifier, const float* rotations, const float* cov3D_precomp,
                               const float* viewmatrix, const float* projmatrix, const float* campos,
                               float tan_fovx, float tan_fovy, int prefiltered, int* radii, void* geom_buf,
                               size_t geom_bytes, unsigned long long* host_counters, b200gs_stream_t stream)
{
    return rast_forward_stage1(P, D, M, W, H, means3D, shs, colors_precomp, opacities, scales, scale_modifier,
                               rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx, tan_fovy,
                               prefiltered, radii, geom_buf, geom_bytes, host_counters, (cudaStream_t)stream);
}

int b200gs_rast_forward_stage2(int P, long long num_rendered, long long num_visible, int W, int H,
                               const float* background, void* geom_buf, void* bin_buf, size_t bin_bytes,
                               void* img_buf, size_t img_bytes, float* out_color, float* out_depth,
                               b200gs_stream_t stream)
{
    return rast_forward_stage2(P, num_rendered, num_visible, W, H, background, geom_buf, bin_buf, bin_bytes,
                               img_buf, img_bytes, out_color, out_depth, (cudaStream_t)stream);
}

int b200gs_rast_backward(int P, int D, int M, long long num_rendered, int W, int H, const float* background,
                         const float* means3D, const float* shs, const float* colors_precomp,
                         const float* scales, float scale_modifier, const float* rotations,
                         const float* cov3D_precomp, const float* viewmatrix, const float* projmatrix,
                         const float* campos, float tan_fovx, float tan_fovy, const int* radii, void* geom_buf,
                         void* bin_buf, void* img_buf, const float* dL_dpix, const float* dL_dpix_depth,
                         float* grad_arena, float* dL_dmean2D, float* dL_dcolor, float* dL_dopacity,
                         float* dL_dmean3D, float* dL_dcov3D, float* dL_dsh, float* dL_dscale, float* dL_drot,
                         b200gs_stream_t stream)
{
    return rast_backward(P, D, M, num_rendered, W, H, background, means3D, shs, colors_precomp, scales,
                         scale_modifier, rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx,
                         tan_fovy, radii, geom_buf, bin_buf, img_buf, dL_dpix, dL_dpix_depth, grad_arena,
                         dL_dmean2D, dL_dcolor, dL_dopacity, dL_dmean3D, dL_dcov3D, dL_dsh, dL_dscale, dL_drot, 0,
                         (cudaStream_t)stream);
}

int b200gs_rast_backward_accumulate_sh(int P, int D, int M, long long num_rendered, int W, int H, const float* background,
                                       const float* means3D, const float* shs, const float* colors_precomp,
                                       const float* scales, float scale_modifier, const float* rotations,
                                       const float* cov3D_precomp, const float* viewmatrix, const float* projmatrix,
                                       const float* campos, float tan_fovx, float tan_fovy, const int* radii, void* geom_buf,
                                       void* bin_buf, void* img_buf, const float* dL_dpix, const float* dL_dpix_depth,
                                       float* grad_arena, float* dL_dmean2D, float* dL_dcolor, float* dL_dopacity,
                                       float* dL_dmean3D, float* dL_dcov3D, float* dL_dsh_accum, float* dL_dscale, float* dL_drot,
                                       b200gs_stream_t stream)
{
    return rast_backward(P, D, M, num_rendered, W, H, background, means3D, shs, colors_precomp, scales,
                         scale_modifier, rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx,
                         tan_fovy, radii, geom_buf, bin_buf, img_buf, dL_dpix, dL_dpix_depth, grad_arena,
                         dL_dmean2D, dL_dcolor, dL_dopacity, dL_dmean3D, dL_dcov3D, dL_dsh_accum, dL_dscale, dL_drot, 1,
                         (cudaStream_t)stream);
}

int b200gs_mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                        unsigned char* present, b200gs_stream_t stream)
{
    return mark_visible(P, means3D, viewmatrix, projmatrix, present, (cudaStream_t)stream);
}

long long b200gs_rast_export(const char* field, int P, long long R, int W, int H, void* geom_buf,
                             void* bin_buf, void* img_buf, void* dst, long long dst_bytes,
                             b200gs_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    const int grid_x = (W + TILE_X - 1) / TILE_X, grid_y = (H + TILE_Y - 1) / TILE_Y;
    const size_t tiles = (size_t)grid_x * grid_y, npix = (size_t)W * H;
    const int tile_bits = tile_bits_for(tiles);
    size_t tmp;
    GeomState g = GeomState::carve(geom_buf, (size_t)P, &tmp);
    BinState b = BinState::carve(bin_buf, (size_t)P, (size_t)R, tile_bits, &tmp);
    ImgState img = ImgState::carve(img_buf, npix, tiles, &tmp);
    const int passes = radix_plan((size_t)R, 0, tile_bits).passes;
    const bool side_b = R > 0 && (passes & 1);
    const u32* list = side_b ? b.ivals_b : b.ivals_a;
    const u32* tile_sorted = side_b ? b.ikeys_b : b.ikeys_a;
    const std::string f(field);
    size_t n = 0;
    int gf = -1;
    const void* src = nullptr;
    if (f == "depths") { n = (size_t)P * 4; gf = F_DEPTHS; }
    else if (f == "means2D") { n = (size_t)P * 8; gf = F_MEANS2D; }
    else if (f == "conic_opacity") { n = (size_t)P * 16; gf = F_CONIC_OPACITY; }
    else if (f == "rgb") { n = (size_t)P * 12; gf = F_RGB; }
    else if (f == "clamped") { n = (size_t)P * 3; gf = F_CLAMPED; }
    else if (f == "cov3D") { n = (size_t)P * 24; src = g.cov3D; }
    else if (f == "tiles_touched") { n = (size_t)P * 4; src = g.tiles_touched; }
    else if (f == "point_list") { n = (size_t)R * 4; src = list; }
    else if (f == "keys") { n = (size_t)R * 8; gf = F_KEYS; }
    else if (f == "ranges") { n = tiles * 8; src = img.ranges; }
    else if (f == "n_contrib") { n = npix * 4; src = img.n_contrib; }
    else if (f == "accum_alpha") { n = npix * 4; src = img.final_T; }
    else { set_error("rast_export: unknown field '%s'", field); return -1; }
    if (!dst) return (long long)n;
    if ((size_t)dst_bytes < n) { set_error("rast_export: destination too small"); return -1; }
    if (n == 0) return 0;
    if (src) cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToDevice, stream);
    else if (gf == F_KEYS)
        export_keys_kernel<<<(unsigned)((R + 255) / 256), 256, 0, stream>>>((u32)R, tile_sorted, list, g.recB, (u64*)dst);
    else
        export_geom_kernel<<<(P + 255) / 256, 256, 0, stream>>>(gf, P, nullptr, g.recA, g.recB, g.recC, g.clamped,
                                                                g.tiles_touched, dst);
    if (check_launch("rast_export")) return -1;
    return (long long)n;
}

size_t b200gs_sort_temp_bytes(size_t n, int begin_bit, int end_bit)
{
    return radix_plan(n, begin_bit, end_bit).temp_bytes;
}

int b200gs_sort_pairs_u32(uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b, size_t n,
                          int begin_bit, int end_bit, void* temp, size_t temp_bytes, b200gs_stream_t stream)
{
    return radix_sort_pairs(keys_a, vals_a, keys_b, vals_b, n, begin_bit, end_bit, temp, temp_bytes,
                            (cudaStream_t)stream);
}

size_t b200gs_dist2_scratch_bytes(size_t P) { return dist2_scratch_bytes(P); }
int b200gs_dist2(int P, const float* points, float* mean_dists, void* scratch, size_t scratch_bytes,
                 b200gs_stream_t stream)
{
    return dist2(P, points, mean_dists, scratch, scratch_bytes, (cudaStream_t)stream);
}

}  // extern "C"
