// One training VIEW of the hot path through the C ABI, in the trainer's order and without Python (SURVEY.md 8d, C3 shape):
//   time-row HexPlane forward (spatial product shared by the step) -> deformation MLP forward -> activations -> rasterizer
//   forward (stage 1 + 2) -> L1 loss + gradient -> rasterizer backward (SH gradient accumulated) -> activations backward ->
//   deformation MLP backward -> time-row HexPlane backward
// plus the per-step pieces once (spatial HexPlane forward / backward, plane regulariser).  Device time per entry point (CUDA
// events on the launching stream) and per view, so that two builds or launch settings can be A/B'd end to end in seconds:
//     tools/native/view_check 1000000 1280 720 0.01 8
//     tools/native/view_check 1000000 1280 720 0.01 8 mlp_fwd_sms=120 mlp_bwd_sms=120
// Synthetic inputs with the distributions of b200gs/synthetic.py (not the same random stream), random-init field.  This is a
// timing tool: results are summarised by checksums only (the parity tests live in tests/).
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "b200gs.h"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)
#define BK(x) do { if ((x) != 0) { printf("b200gs error: %s (%s:%d)\n", b200gs_last_error(), __FILE__, __LINE__); exit(3); } } while (0)

static unsigned long long rng_state = 6666ull * 0x9E3779B97F4A7C15ull + 1;
static double urand() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (double)(rng_state >> 11) * (1.0 / 9007199254740992.0); }
static double nrand() { double u = urand(), v = urand(); if (u < 1e-300) u = 1e-300; return sqrt(-2.0 * log(u)) * cos(6.283185307179586 * v); }
static float* dev_fill(size_t n, double (*gen)(), double scale, double shift)
{
    std::vector<float> h(n);
    for (auto& v : h) v = (float)(gen() * scale + shift);
    float* d; CK(cudaMalloc(&d, (n ? n : 1) * sizeof(float))); CK(cudaMemcpy(d, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    return d;
}
static float* dev_zero(size_t n) { float* d; CK(cudaMalloc(&d, (n ? n : 1) * sizeof(float))); CK(cudaMemset(d, 0, (n ? n : 1) * sizeof(float))); return d; }
static double dev_sum(const float* d, size_t n)
{
    std::vector<float> h(n); CK(cudaMemcpy(h.data(), d, n * sizeof(float), cudaMemcpyDeviceToHost));
    double s = 0; for (float v : h) s += v; return s;
}
static void mat_mul4(const float* A, const float* B, float* C) { for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) { double s = 0; for (int k = 0; k < 4; ++k) s += (double)A[4 * i + k] * B[4 * k + j]; C[4 * i + j] = (float)s; } }

struct Timer {
    std::vector<std::string> names; std::vector<double> ms; std::vector<int> calls;
    cudaEvent_t e0, e1; cudaStream_t st;
    explicit Timer(cudaStream_t s) : st(s) { CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); }
    int slot(const char* n) { for (size_t i = 0; i < names.size(); ++i) if (names[i] == n) return (int)i; names.push_back(n); ms.push_back(0); calls.push_back(0); return (int)names.size() - 1; }
    void begin() { CK(cudaEventRecord(e0, st)); }
    void end(const char* n, bool count) { CK(cudaEventRecord(e1, st)); CK(cudaEventSynchronize(e1)); float t; CK(cudaEventElapsedTime(&t, e0, e1)); if (count) { int i = slot(n); ms[i] += t; calls[i]++; } }
};

int main(int argc, char** argv)
{
    const int P = argc > 1 ? atoi(argv[1]) : 1000000, W = argc > 2 ? atoi(argv[2]) : 1280, H = argc > 3 ? atoi(argv[3]) : 720;
    const double mu = argc > 4 ? atof(argv[4]) : 0.01;
    const int views = argc > 5 ? atoi(argv[5]) : 8;
    for (int i = 6; i < argc; ++i) {
        char* eq = strchr(argv[i], '=');
        if (!eq) continue;
        *eq = 0;
        BK(b200gs_set_option(argv[i], atoi(eq + 1)));
        printf("option %s = %d\n", argv[i], b200gs_get_option(argv[i]));
    }
    printf("b200gs %d: P = %d, %d x %d, scale_mu = %g, %d views after 2 warm-up views\n", b200gs_version(), P, W, H, mu, views);
    const int D = 3, M = 16, F = 64;
    const size_t rowsP = (size_t)((P + 127) / 128) * 128;
    cudaStream_t st; CK(cudaStreamCreate(&st));
    // ---- model ----
    float* xyz = dev_fill((size_t)P * 3, urand, 3.0, -1.5);
    float* log_scale = dev_fill((size_t)P * 3, nrand, 0.6, log(mu));
    float* rot_raw = dev_fill((size_t)P * 4, nrand, 1.0, 0.0);
    float* opac_raw = dev_fill(P, nrand, 1.5, 0.0);
    float* flow = dev_fill((size_t)P * 3, nrand, 1e-3, 0.0);
    float* shs; { std::vector<float> h((size_t)P * M * 3); for (int i = 0; i < P; ++i) { for (int c = 0; c < 3; ++c) h[(size_t)i * 48 + c] = (float)(urand() * 3.0 - 1.5); for (int k = 3; k < 48; ++k) h[(size_t)i * 48 + k] = (float)(nrand() * 0.05); }
                  CK(cudaMalloc(&shs, h.size() * 4)); CK(cudaMemcpy(shs, h.data(), h.size() * 4, cudaMemcpyHostToDevice)); }
    b200gs_hexplane_desc hd; memset(&hd, 0, sizeof(hd));
    hd.levels = 2; hd.channels = 32;
    const int pa[6] = {0, 0, 0, 1, 1, 2}, pb[6] = {1, 2, 3, 2, 3, 3};
    size_t plane_floats[2][6];
    for (int l = 0; l < 2; ++l) {
        const int r = l == 0 ? 64 : 128;
        hd.res[l][0] = hd.res[l][1] = hd.res[l][2] = r; hd.res[l][3] = 50;
        for (int k = 0; k < 6; ++k) {
            plane_floats[l][k] = (size_t)hd.res[l][pb[k]] * hd.res[l][pa[k]] * 32;
            const bool is_time = k == 2 || k == 4 || k == 5;                      // reference init: U(0.1, 0.5) spatial, ones temporal (+ noise)
            hd.plane[l][k] = is_time ? dev_fill(plane_floats[l][k], nrand, 0.01, 1.0) : dev_fill(plane_floats[l][k], urand, 0.4, 0.1);
            hd.grad_plane[l][k] = dev_zero(plane_floats[l][k]);
        }
    }
    { std::vector<float> aabb = {1.5f, 1.5f, 1.5f, -1.5f, -1.5f, -1.5f}; float* d; CK(cudaMalloc(&d, 24)); CK(cudaMemcpy(d, aabb.data(), 24, cudaMemcpyHostToDevice)); hd.aabb = d; }
    if (b200gs_hexplane_time_supported(&hd) != 1) { printf("time-row kernels unsupported\n"); return 3; }
    b200gs_mlp_weights mw; memset(&mw, 0, sizeof(mw));
    const int kd[3] = {3, 3, 4};
    mw.feat_dim = F; mw.width = 64; mw.feat_tiled = 1;
    mw.w1 = dev_fill(64 * F, nrand, 0.15, 0.0); mw.b1 = dev_fill(64, nrand, 0.05, 0.0);
    float* gbuf = dev_zero(64 * F + 64 + 3 * (64 * 64 + 64 + 4 * 64 + 16));
    b200gs_mlp_grads mg; { float* g = gbuf; mg.w1 = g; g += 64 * F; mg.b1 = g; g += 64;
        for (int h = 0; h < 3; ++h) { mg.w2[h] = g; g += 64 * 64; mg.b2[h] = g; g += 64; mg.w3[h] = g; g += 4 * 64; mg.b3[h] = g; g += 16; } }
    for (int h = 0; h < 3; ++h) {
        mw.w2[h] = dev_fill(64 * 64, nrand, 0.15, 0.0); mw.b2[h] = dev_fill(64, nrand, 0.05, 0.0);
        mw.w3[h] = dev_fill((size_t)kd[h] * 64, nrand, 0.001, 0.0); mw.b3[h] = dev_fill(kd[h], nrand, 0.0001, 0.0);   // small heads: deformations stay small
    }
    // ---- per-view buffers ----
    float* S = dev_zero((size_t)P * F), *A = dev_zero((size_t)P * F), *feat = dev_zero(rowsP * F), *dfeat = dev_zero(rowsP * F);
    float* saved = dev_zero(b200gs_deform_mlp_saved_floats(P));
    float *pts_o = dev_zero((size_t)P * 3), *sc_o = dev_zero((size_t)P * 3), *rt_o = dev_zero((size_t)P * 4);
    float *sc_a = dev_zero((size_t)P * 3), *rt_a = dev_zero((size_t)P * 4), *op_a = dev_zero(P);
    int* radii; CK(cudaMalloc(&radii, (size_t)P * 4));
    float *color = dev_zero((size_t)3 * H * W), *depth = dev_zero((size_t)H * W), *gt = dev_fill((size_t)3 * H * W, urand, 1.0, 0.0), *dimg = dev_zero((size_t)3 * H * W);
    float* loss = dev_zero(1);
    float *g_arena = dev_zero((size_t)12 * P), *g_m2d = dev_zero((size_t)3 * P), *g_col = dev_zero((size_t)3 * P), *g_op = dev_zero(P), *g_m3d = dev_zero((size_t)3 * P),
          *g_cov = dev_zero((size_t)6 * P), *g_sh = dev_zero((size_t)P * M * 3), *g_sc = dev_zero((size_t)3 * P), *g_rot = dev_zero((size_t)4 * P);
    float *d_sc_raw = dev_zero((size_t)3 * P), *d_rt_raw = dev_zero((size_t)4 * P), *d_op_raw = dev_zero(P), *d_xyz_t = dev_zero((size_t)3 * P), *d_xyz_s = dev_zero((size_t)3 * P);
    const size_t sb = b200gs_hexplane_time_row_scratch_bytes(&hd, 64);
    void* scratch; CK(cudaMalloc(&scratch, sb));
    size_t sz[3]; BK(b200gs_rast_buffer_sizes(P, 0, W, H, sz));
    void *geom, *img, *bin = nullptr; size_t bin_cap = 0;
    CK(cudaMalloc(&geom, sz[0])); CK(cudaMalloc(&img, sz[2]));
    // camera: quarter orbit of synthetic.orbit_cameras around the cube, 4.5 units away
    const double focal = 582.69 * (H / 512.0), tanx = W / (2 * focal), tany = H / (2 * focal), zn = 0.01, zf = 100.0;
    float projT[16] = {0}; projT[0] = (float)(1.0 / tanx); projT[5] = (float)(1.0 / tany); projT[10] = (float)(zf / (zf - zn)); projT[14] = (float)(-(zf * zn) / (zf - zn)); projT[11] = 1.f;
    float *d_view, *d_full, *d_campos, *d_bg; CK(cudaMalloc(&d_view, 64)); CK(cudaMalloc(&d_full, 64)); CK(cudaMalloc(&d_campos, 12)); CK(cudaMalloc(&d_bg, 12)); CK(cudaMemset(d_bg, 0, 12));
    Timer tm(st);
    unsigned long long cnt[2] = {0, 0};
    double view_ms = 0;
    cudaEvent_t v0, v1; CK(cudaEventCreate(&v0)); CK(cudaEventCreate(&v1));
    // ---- per-step: spatial product ----
    tm.begin(); BK(b200gs_hexplane_forward_masked(&hd, P, xyz, nullptr, nullptr, 0.f, 0x0B, nullptr, S, st)); tm.end("step: hexplane spatial forward", true);
    for (int v = -2; v < views; ++v) {
        const bool count = v >= 0;
        const int k = (v + 2) % 8;
        const double ang = 2 * M_PI * k / 8.0 * 0.25 - 0.3, c = cos(ang), s = sin(ang);
        // world-to-view (row-vector convention): [R 0; t 1] with R = camera-to-world rotation about y, t = (0, 0, 4.5)
        float view[16] = {(float)c, 0, (float)s, 0, 0, 1, 0, 0, (float)-s, 0, (float)c, 0, 0, 0, 4.5f, 1};
        float full[16]; mat_mul4(view, projT, full);
        float campos[3] = {(float)(-(view[2] * 4.5f)), 0.f, (float)(-(view[10] * 4.5f))};      // -t R^T
        CK(cudaMemcpyAsync(d_view, view, 64, cudaMemcpyHostToDevice, st)); CK(cudaMemcpyAsync(d_full, full, 64, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_campos, campos, 12, cudaMemcpyHostToDevice, st)); CK(cudaStreamSynchronize(st));
        const float t = (float)k / 7.f, frame = (float)k;
        CK(cudaEventRecord(v0, st));
        tm.begin(); BK(b200gs_hexplane_time_forward(&hd, P, xyz, nullptr, t, S, feat, 1, st)); tm.end("hexplane_time_forward", count);
        tm.begin(); BK(b200gs_deform_mlp_forward(&mw, P, feat, xyz, log_scale, rot_raw, flow, frame, nullptr, 1.f, pts_o, sc_o, rt_o, saved, st)); tm.end("deform_mlp_forward", count);
        tm.begin(); BK(b200gs_activations_forward(P, sc_o, rt_o, opac_raw, sc_a, rt_a, op_a, st)); tm.end("activations_forward", count);
        tm.begin();
        BK(b200gs_rast_forward_stage1(P, D, M, W, H, pts_o, shs, nullptr, op_a, sc_a, 1.f, rt_a, nullptr, d_view, d_full, d_campos, (float)tanx, (float)tany, 0, radii, geom, sz[0], cnt, st));
        tm.end("rast_forward_stage1 (+ host read-back)", count);
        BK(b200gs_rast_buffer_sizes(P, (long long)cnt[0], W, H, sz));
        if (sz[1] > bin_cap) { if (bin) CK(cudaFree(bin)); bin_cap = sz[1] + sz[1] / 8; CK(cudaMalloc(&bin, bin_cap)); }
        tm.begin(); BK(b200gs_rast_forward_stage2(P, (long long)cnt[0], (long long)cnt[1], W, H, d_bg, geom, bin, bin_cap, img, sz[2], color, depth, st)); tm.end("rast_forward_stage2", count);
        tm.begin(); BK(b200gs_l1_loss_fwd_bwd((long long)3 * H * W, color, gt, 1.f / (3.f * H * W * 8.f), loss, nullptr, dimg, st)); tm.end("l1_loss_fwd_bwd", count);
        tm.begin();
        BK(b200gs_rast_backward_accumulate_sh(P, D, M, (long long)cnt[0], W, H, d_bg, pts_o, shs, nullptr, sc_a, 1.f, rt_a, nullptr, d_view, d_full, d_campos, (float)tanx, (float)tany,
                                              radii, geom, bin, img, dimg, nullptr, g_arena, g_m2d, g_col, g_op, g_m3d, g_cov, g_sh, g_sc, g_rot, st));
        tm.end("rast_backward_accumulate_sh", count);
        tm.begin(); BK(b200gs_activations_backward(P, sc_a, rt_o, op_a, g_sc, g_rot, g_op, d_sc_raw, d_rt_raw, d_op_raw, st)); tm.end("activations_backward", count);
        tm.begin(); BK(b200gs_deform_mlp_backward(&mw, &mg, P, feat, saved, g_m3d, d_sc_raw, d_rt_raw, dfeat, st)); tm.end("deform_mlp_backward", count);
        tm.begin(); BK(b200gs_hexplane_time_backward(&hd, P, xyz, nullptr, t, S, A, dfeat, d_xyz_t, scratch, sb, 1, st)); tm.end("hexplane_time_backward", count);
        CK(cudaEventRecord(v1, st)); CK(cudaEventSynchronize(v1));
        if (count) { float ms; CK(cudaEventElapsedTime(&ms, v0, v1)); view_ms += ms; }
    }
    tm.begin(); BK(b200gs_hexplane_backward_masked(&hd, P, xyz, nullptr, nullptr, 0.f, 0x0B, nullptr, nullptr, A, d_xyz_s, nullptr, 0, st)); tm.end("step: hexplane spatial backward", true);
    tm.begin(); BK(b200gs_hexplane_regulation(&hd, 0.0001f, 0.01f, 0.0001f, loss, st)); tm.end("step: plane regulariser", true);
    CK(cudaStreamSynchronize(st));
    printf("instances R = %llu, visible = %llu (last view)\n", cnt[0], cnt[1]);
    double sum_entries = 0;
    for (size_t i = 0; i < tm.names.size(); ++i) {
        const bool step = tm.names[i].rfind("step:", 0) == 0;
        printf("  %-42s %8.3f ms %s\n", tm.names[i].c_str(), tm.ms[i] / tm.calls[i], step ? "per step" : "per view");
        if (!step) sum_entries += tm.ms[i] / tm.calls[i];
    }
    printf("per view: %.3f ms between the first and last event (entries sum to %.3f ms; each entry is synchronised here, so launch gaps are included)\n", view_ms / views, sum_entries);
    printf("checksums: loss %.6e, sum(colour) %.6e, sum(dW1) %.6e, sum(d_xyz time) %.6e, sum(dL_dsh) %.6e\n", dev_sum(loss, 1), dev_sum(color, (size_t)3 * H * W),
           dev_sum(mg.w1, 64 * F), dev_sum(d_xyz_t, (size_t)3 * P), dev_sum(g_sh, (size_t)P * M * 3));
    return 0;
}
