// Standalone check of the radix sort through the C ABI: b200gs_sort_pairs_u32 on random (key, value) pairs must equal
// std::stable_sort (the sort is stable, so the output is unique), with its device time (CUDA events, 10 sorts after one warm-up).
// run: tools/native/sort_check [n = 1000000] [bits = 32]
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <vector>
#include <cuda_runtime.h>
#include "b200gs.h"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)

int main(int argc, char** argv)
{
    const size_t n = argc > 1 ? (size_t)atoll(argv[1]) : 1000000;
    const int bits = argc > 2 ? atoi(argv[2]) : 32;
    std::vector<uint32_t> keys(n), vals(n);
    uint64_t s = 88172645463325252ull;
    for (size_t i = 0; i < n; ++i) { s ^= s << 13; s ^= s >> 7; s ^= s << 17; keys[i] = (uint32_t)(s >> 20) & (bits >= 32 ? 0xFFFFFFFFu : ((1u << bits) - 1)); vals[i] = (uint32_t)i; }
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    uint32_t *ka, *va, *kb, *vb, *k0, *v0; void* temp;
    const size_t tb = b200gs_sort_temp_bytes(n, 0, bits);
    CK(cudaMalloc(&ka, n * 4)); CK(cudaMalloc(&va, n * 4)); CK(cudaMalloc(&kb, n * 4)); CK(cudaMalloc(&vb, n * 4)); CK(cudaMalloc(&k0, n * 4)); CK(cudaMalloc(&v0, n * 4));
    CK(cudaMalloc(&temp, tb));
    CK(cudaMemcpy(k0, keys.data(), n * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(v0, vals.data(), n * 4, cudaMemcpyHostToDevice));
    cudaStream_t st; CK(cudaStreamCreate(&st));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float total = 0; int side = 0;
    for (int rep = -1; rep < 10; ++rep) {
        CK(cudaMemcpyAsync(ka, k0, n * 4, cudaMemcpyDeviceToDevice, st)); CK(cudaMemcpyAsync(va, v0, n * 4, cudaMemcpyDeviceToDevice, st));
        CK(cudaEventRecord(e0, st));
        side = b200gs_sort_pairs_u32(ka, va, kb, vb, n, 0, bits, temp, tb, st);
        CK(cudaEventRecord(e1, st)); CK(cudaStreamSynchronize(st));
        if (side < 0) { printf("sort failed: %s\n", b200gs_last_error()); return 3; }
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); if (rep >= 0) total += ms;
    }
    std::vector<uint32_t> ok_k(n), ok_v(n);
    CK(cudaMemcpy(ok_k.data(), side ? kb : ka, n * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(ok_v.data(), side ? vb : va, n * 4, cudaMemcpyDeviceToHost));
    size_t bad = 0;
    for (size_t i = 0; i < n; ++i) bad += ok_v[i] != order[i] || ok_k[i] != keys[order[i]];
    printf("%.1f us per sort of %zu pairs on %d bits, %zu mismatches against std::stable_sort\n", 100.f * total, n, bits, bad);
    const bool ok = bad == 0;
    printf("RESULT: %s\n", ok ? "PASS" : "FAIL");
    return ok ? 0 : 1;
}
