// Onesweep LSD radix sort, see radix_sort.cuh.
#include "radix_sort.cuh"

namespace b200gs {

namespace {

constexpr u32 LB_AGG = 1u << 30;     // tile aggregate published
constexpr u32 LB_INCL = 1u << 31;    // inclusive prefix published
constexpr u32 LB_VALUE = (1u << 30) - 1;

struct DigitSpec { int shift[RS_MAX_PASSES]; u32 mask[RS_MAX_PASSES]; };

// One read of the keys builds the digit histogram of every pass.
__global__ void __launch_bounds__(256)
rs_histogram(const u32* __restrict__ keys, u32 n, int passes, DigitSpec spec, u32* __restrict__ g_hist)
{
    __shared__ u32 s_hist[RS_MAX_PASSES * RS_RADIX];
    for (int i = threadIdx.x; i < passes * RS_RADIX; i += 256) s_hist[i] = 0;
    __syncthreads();
    const u32 stride = gridDim.x * 256;
    const u32 gtid = blockIdx.x * 256 + threadIdx.x;
    const u32 n4 = n >> 2;
    const uint4* k4 = reinterpret_cast<const uint4*>(keys);
    auto add = [&](u32 k) {
#pragma unroll
        for (int p = 0; p < RS_MAX_PASSES; ++p)
            if (p < passes) atomicAdd(&s_hist[p * RS_RADIX + ((k >> spec.shift[p]) & spec.mask[p])], 1u);
    };
    for (u32 i = gtid; i < n4; i += stride) {
        uint4 k = __ldg(k4 + i);
        add(k.x); add(k.y); add(k.z); add(k.w);
    }
    for (u32 i = (n4 << 2) + gtid; i < n; i += stride) add(keys[i]);
    __syncthreads();
    for (int i = threadIdx.x; i < passes * RS_RADIX; i += 256) {
        u32 c = s_hist[i];
        if (c) atomicAdd(&g_hist[i], c);
    }
}

// Turns each pass's histogram into exclusive digit bases.
__global__ void __launch_bounds__(256) rs_scan_hist(u32* __restrict__ g_hist)
{
    __shared__ u32 s_warp[8];
    u32* h = g_hist + blockIdx.x * RS_RADIX;
    u32 v = h[threadIdx.x];
    h[threadIdx.x] = block_exclusive_scan_256(v, s_warp);
}

// LB_BATCH (8 while every tile is resident at once: 111 -> 103 us per 1M-pair 32-bit sort, profiles/r2a_sort_check.txt): the
// decoupled look-back of a digit walks its predecessors' states LB_BATCH at a
// time (independent volatile loads in flight together) instead of one dependent L2 round trip per predecessor -- with a
// few hundred tiles resident at once the serial walk is what a pass on ~1M keys spends its time in.  Same sums, same result.
template <bool HAS_VALS, int IPT, int LB_BATCH, int BALLOT>
__global__ void __launch_bounds__(RS_THREADS)
rs_onesweep_pass(const u32* __restrict__ keys_in, const u32* __restrict__ vals_in,
                 u32* __restrict__ keys_out, u32* __restrict__ vals_out, u32 n, int shift, u32 mask,
                 const u32* __restrict__ g_base, u32* lookback, u32* ticket)
{
    __shared__ u32 s_warp_hist[RS_WARPS][RS_RADIX];
    constexpr int TILE = RS_THREADS * IPT;
    __shared__ u32 s_keys[TILE];
    __shared__ u32 s_vals[HAS_VALS ? TILE : 1];
    __shared__ u32 s_digit_off[RS_RADIX];
    __shared__ u32 s_scan[8];
    __shared__ u32 s_tile;

    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) s_warp_hist[w][tid] = 0;
    __syncthreads();
    const u32 tile = s_tile;
    const u32 base = tile * TILE;
    const u32 wbase = base + warp * (32 * IPT);

    u32 key[IPT];
    unsigned short rank[IPT];
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
        u32 idx = wbase + i * 32 + lane;
        key[i] = idx < n ? __ldg(keys_in + idx) : 0xFFFFFFFFu;
    }
    // Stable in-warp ranking: items are visited in index order (i-major, then lane).  The lanes that hold the same digit are found
    // with one ballot per digit bit (VOTE + LOP3, a few cycles each and independent across the IPT items) rather than MATCH.ANY
    // (one instruction, but its latency was the top stall of this kernel, profiles/r2w_stalls_rs_onesweep_pass.txt): 103 -> 87 us
    // per 1M-pair 32-bit sort, 96 -> 79 us per 2.4M-pair 12-bit sort (profiles/r3h_sort_check.txt).
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
        u32 d = (key[i] >> shift) & mask;
        u32 peers = 0xffffffffu;
#pragma unroll
        for (int b = 0; b < BALLOT; ++b) {   // BALLOT = how many digit bits this pass can have set (4 or 8)
            const u32 vote = __ballot_sync(0xffffffffu, (d >> b) & 1u);
            peers &= ((d >> b) & 1u) ? vote : ~vote;
        }
        u32 before = s_warp_hist[warp][d];
        rank[i] = (unsigned short)(before + __popc(peers & lt));
        __syncwarp();
        if ((peers & lt) == 0) s_warp_hist[warp][d] = before + __popc(peers);
        __syncwarp();
    }
    __syncthreads();

    // Thread d owns digit d: exclusive scan over warps, then chain with earlier tiles.
    u32 count = 0;
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
        u32 t = s_warp_hist[w][tid];
        s_warp_hist[w][tid] = count;
        count += t;
    }
    u32 prefix = 0;
    u32* lb = lookback + (size_t)tile * RS_RADIX + tid;
    if (tile == 0) {
        st_volatile_u32(lb, count | LB_INCL);
    } else {
        st_volatile_u32(lb, count | LB_AGG);
        if constexpr (LB_BATCH <= 1) {
            for (u32 t = tile; t-- > 0;) {
                const u32* p = lookback + (size_t)t * RS_RADIX + tid;
                u32 v;
                do { v = ld_volatile_u32(p); } while ((v & (LB_AGG | LB_INCL)) == 0);
                prefix += v & LB_VALUE;
                if (v & LB_INCL) break;
            }
        } else {
            int t = (int)tile - 1;                  // next predecessor to take
            bool done = false;
            while (!done) {
                u32 v[LB_BATCH];
#pragma unroll
                for (int k = 0; k < LB_BATCH; ++k)  // before tile 0: an inclusive 0 (never reached: tile 0 publishes INCL)
                    v[k] = t - k >= 0 ? ld_volatile_u32(lookback + (size_t)(t - k) * RS_RADIX + tid) : LB_INCL;
                int consumed = 0;                   // taken strictly in order; the first unpublished state ends the batch
#pragma unroll
                for (int k = 0; k < LB_BATCH; ++k) {
                    if (!done && consumed == k && (v[k] & (LB_AGG | LB_INCL)) != 0) {
                        prefix += v[k] & LB_VALUE;
                        done = (v[k] & LB_INCL) != 0;
                        consumed = k + 1;
                    }
                }
                t -= consumed;                      // an unpublished predecessor is simply fetched again
            }
        }
        st_volatile_u32(lb, ((prefix + count) & LB_VALUE) | LB_INCL);
    }
    const u32 local_start = block_exclusive_scan_256(count, s_scan);
    s_digit_off[tid] = g_base[tid] + prefix - local_start;
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) s_warp_hist[w][tid] += local_start;
    __syncthreads();

#pragma unroll
    for (int i = 0; i < IPT; ++i) {
        u32 d = (key[i] >> shift) & mask;
        u32 pos = s_warp_hist[warp][d] + rank[i];
        s_keys[pos] = key[i];
        if (HAS_VALS) {
            u32 idx = wbase + i * 32 + lane;
            s_vals[pos] = idx < n ? __ldg(vals_in + idx) : 0u;
        }
    }
    __syncthreads();
    const u32 valid = min((u32)TILE, n - base);
    for (u32 j = tid; j < valid; j += RS_THREADS) {
        u32 k = s_keys[j];
        u32 out = s_digit_off[(k >> shift) & mask] + j;
        keys_out[out] = k;
        if (HAS_VALS) vals_out[out] = s_vals[j];
    }
}

}  // namespace

int radix_sort_pairs(u32* keys_a, u32* vals_a, u32* keys_b, u32* vals_b, size_t n,
                     int begin_bit, int end_bit, void* temp, size_t temp_bytes,
                     cudaStream_t stream)
{
    if (n == 0) return 0;
    if (n >= (size_t)LB_VALUE) { set_error("radix_sort_pairs: n=%zu exceeds 2^30-1", n); return -1; }
    RadixPlan plan = radix_plan(n, begin_bit, end_bit);
    if (plan.passes > RS_MAX_PASSES) { set_error("radix_sort_pairs: more than %d passes", RS_MAX_PASSES); return -1; }
    if (temp_bytes < plan.temp_bytes) { set_error("radix_sort_pairs: temp too small"); return -1; }
    u32* g_hist = (u32*)temp;
    u32* tickets = g_hist + (size_t)plan.passes * RS_RADIX;
    u32* lookback = tickets + 256;
    const size_t tiles = plan.tiles;
    // clear what this call uses: digit bases, tickets, look-back state of `tiles` tiles per pass
    cudaMemsetAsync(temp, 0, ((size_t)plan.passes * RS_RADIX + 256 + (size_t)plan.passes * tiles * RS_RADIX) * sizeof(u32), stream);

    DigitSpec spec;
    const int per = RS_RADIX_BITS;       // (an even 6 + 6 split of the tile-id bits was measured: no gain, profiles/r2a_sort_check.txt)
    for (int p = 0; p < RS_MAX_PASSES; ++p) {
        int lo = begin_bit + p * per;
        int nb = end_bit - lo; if (nb > per) nb = per; if (nb < 1) nb = 1;
        spec.shift[p] = lo < 32 ? lo : 31;
        spec.mask[p] = (1u << nb) - 1;
    }
    int hgrid = (int)((n / 4 + 255) / 256); if (hgrid < 1) hgrid = 1;
    if (hgrid > NUM_SMS * 8) hgrid = NUM_SMS * 8;
    rs_histogram<<<hgrid, 256, 0, stream>>>(keys_a, (u32)n, plan.passes, spec, g_hist);
    rs_scan_hist<<<plan.passes, 256, 0, stream>>>(g_hist);

    u32 *kin = keys_a, *kout = keys_b, *vin = vals_a, *vout = vals_b;
    for (int p = 0; p < plan.passes; ++p) {
        u32* lb = lookback + (size_t)p * tiles * RS_RADIX;
#define RS_LAUNCH(HV, IPTV, LBV) rs_onesweep_pass<HV, IPTV, LBV, BL><<<(unsigned)tiles, RS_THREADS, 0, stream>>>( \
            kin, HV ? vin : nullptr, kout, HV ? vout : nullptr, (u32)n, spec.shift[p], spec.mask[p], g_hist + p * RS_RADIX, lb, tickets + p)
        // batched look-back pays while every tile is resident at once (3 CTAs per SM: 80 registers); beyond one wave the tiles of
        // the next wave find inclusive prefixes waiting and the plain walk is shorter (2.4M pairs / 12 bits: 79 vs 85 us)
        const bool hv = vals_a != nullptr, par = tiles <= (size_t)3 * NUM_SMS;
        // (32 states per round trip for single-wave inputs was measured too: 112 vs 103 us per 1M-pair sort, not kept;
        //  so was __launch_bounds__(256, 4): 64 registers with 20-36 B of spills, 87 -> 95 us per 1M-pair sort, 79 -> 76 us at 2.4M)
#define RS_PICK(BLV) do { constexpr int BL = BLV; \
        if (hv && par) RS_LAUNCH(true, RS_IPT, 8); \
        else if (hv) RS_LAUNCH(true, RS_IPT, 1); \
        else if (par) RS_LAUNCH(false, RS_IPT, 8); \
        else RS_LAUNCH(false, RS_IPT, 1); } while (0)
        if (spec.mask[p] < 16u) RS_PICK(4); else RS_PICK(8);
#undef RS_PICK
#undef RS_LAUNCH
        u32* t = kin; kin = kout; kout = t;
        t = vin; vin = vout; vout = t;
    }
    if (check_launch("radix_sort_pairs")) return -1;
    return (plan.passes & 1) ? 1 : 0;
}

}  // namespace b200gs
