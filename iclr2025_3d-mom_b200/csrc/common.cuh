// Shared helpers for the b200gs kernels (sm_100a only).
#pragma once
#include <cstdint>
#include <cstddef>
#include <cuda_runtime.h>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "b200gs kernels are written for sm_100a (Blackwell B200) only"
#endif

namespace b200gs {

constexpr int TILE_X = 16;          // reference: config.h:15-16 (BLOCK_X/BLOCK_Y)
constexpr int TILE_Y = 16;
constexpr int TILE_PIXELS = TILE_X * TILE_Y;
constexpr int NUM_SMS = 148;        // B200: 2 dies x 74 SMs

typedef uint32_t u32;
typedef uint64_t u64;

// Per-thread last error text (the library keeps no other global state).
void set_error(const char* fmt, ...);
int check_launch(const char* what);   // returns 0 or sets error and returns -1
// CTA caps of the persistent MLP kernels, see b200gs_set_option (api.cu)
extern int g_opt_mlp_fwd_sms, g_opt_mlp_bwd_sms;

// Opt-in phase timing (b200gs_profile_enable / b200gs_profile_read, api.cu): CUDA events recorded on the launching stream around
// the kernels of one phase of a multi-kernel entry point, so that bench.py can report each kernel family's live duration
// (preprocess, depth sort, emission, tile sort, compositing ...).  Disabled (the default): one predictable branch, no events.
enum ProfSlot { PROF_PREPROCESS_FWD = 0, PROF_DEPTH_SORT, PROF_EMIT, PROF_TILE_SORT, PROF_TILE_RANGES, PROF_COMPOSITE_FWD,
                PROF_COMPOSITE_BWD, PROF_PREPROCESS_BWD, PROF_SLOTS };
extern int g_prof_enabled;
void prof_mark(int slot, bool begin, cudaStream_t stream);
struct ProfScope {
    int slot; cudaStream_t stream;
    ProfScope(int s, cudaStream_t st) : slot(s), stream(st) { if (g_prof_enabled) prof_mark(slot, true, stream); }
    ~ProfScope() { if (g_prof_enabled) prof_mark(slot, false, stream); }
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-owned byte buffer. 256-B alignment keeps every
// array usable by 128-bit vector loads and by bulk async copies.
struct Carver {
    char* base; size_t off;
    explicit Carver(void* p) : base((char*)p), off(0) {}
    template <typename T> T* take(size_t count) {
        off = align_up(off, 256);
        T* r = base ? (T*)(base + off) : nullptr;
        off += count * sizeof(T);
        return r;
    }
    size_t used() const { return align_up(off, 256); }
};

__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 lanemask_lt() { u32 m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

__device__ __forceinline__ u32 ld_volatile_u32(const u32* p) {
    u32 v; asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ u64 ld_volatile_u64(const u64* p) {
    u64 v; asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_volatile_u32(u32* p, u32 v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_volatile_u64(u64* p, u64 v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// ---- cp.async (LDGSTS) helpers -------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    u32 s = (u32)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    u32 s = (u32)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory");
}

// sm_90+: 128-bit vector float reduction to global memory (one RED for 4 floats).
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" :: "l"(addr), "f"(a), "f"(b) : "memory");
}

// Exclusive scan of one u32 per thread over a 256-thread block (s_warp: 8 words of smem).
__device__ __forceinline__ u32 block_exclusive_scan_256(u32 v, u32* s_warp, u32* total = nullptr)
{
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (u32)o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    u32 woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        u32 t = s_warp[w];
        if ((u32)w < warp) woff += t;
        tot += t;
    }
    if (total) *total = tot;
    __syncthreads();
    return woff + inc - v;
}

}  // namespace b200gs
