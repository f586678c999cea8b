// libdsa device primitives: exclusive scan, min/max reduction, iota — hand-written, stream-ordered.
#pragma once
#include "common.cuh"

namespace dsa {

// ---------------------------------------------------------------------------------------------
// Exclusive prefix sum of int32 in one launch (chained scan with decoupled look-back).
// Tile = 256 threads x 16 items.  out may alias in.
// ---------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;   // 4096 items per tile: the look-back chain of a 1M-item scan is 245 tiles long
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// Tiles are handed out by an atomic ticket (so a tile's predecessors have always started: forward progress), every
// tile publishes one 64-bit word {epoch:30 | flag:2 | sum:32} (aggregate first, inclusive prefix once known); a tile adds up its
// predecessors' words back to the nearest inclusive one.  The epoch makes stale words of earlier calls invisible, so the state
// array needs no clearing between calls; the tile that draws the last ticket resets the ticket counter.
constexpr unsigned long long SCAN_FLAG_AGG = 1ull, SCAN_FLAG_INCL = 2ull;
__device__ __forceinline__ unsigned long long scan_word(uint32_t epoch, unsigned long long flag, int32_t v) {
    return ((unsigned long long)epoch << 34) | (flag << 32) | (unsigned long long)(uint32_t)v;
}

template <typename InT>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_onepass(const InT* __restrict__ in, int32_t* __restrict__ out, int64_t n, int64_t ntiles,
                                                                 unsigned long long* __restrict__ state, uint32_t* __restrict__ ticket,
                                                                 uint32_t epoch, int64_t* __restrict__ total_out) {
    __shared__ int32_t warp_tot[SCAN_THREADS / 32];
    __shared__ int64_t s_tile;
    __shared__ int32_t s_prefix;
    if (threadIdx.x == 0) {
        const uint32_t t = atomicAdd(ticket, 1u);
        if ((int64_t)t == ntiles - 1) *ticket = 0;   // every ticket of this call has been drawn
        s_tile = (int64_t)t;
    }
    __syncthreads();
    const int64_t tile = s_tile;
    const int64_t base = tile * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int32_t v[SCAN_ITEMS];
    int32_t s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        const int64_t idx = base + i;
        v[i] = idx < n ? (int32_t)in[idx] : 0;
        s += v[i];
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int32_t incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    int32_t woff = 0, agg = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; ++w) {
        if (w < wid) woff += warp_tot[w];
        agg += warp_tot[w];
    }
    volatile unsigned long long* vstate = state;
    if (wid == 0) {   // warp 0: publish, look back, publish the inclusive prefix
        int32_t prefix = 0;
        if (tile == 0) {
            if (lane == 0) vstate[0] = scan_word(epoch, SCAN_FLAG_INCL, agg);
        } else {
            if (lane == 0) vstate[tile] = scan_word(epoch, SCAN_FLAG_AGG, agg);
            int64_t hi = tile - 1;   // nearest predecessor not summed yet
            while (true) {
                const int64_t j = hi - lane;
                unsigned long long w = 0;
                bool valid;
                do {   // wait until the 32 predecessors hi, hi-1, ... (those that exist) have published something in this epoch
                    w = j >= 0 ? vstate[j] : scan_word(epoch, SCAN_FLAG_INCL, 0);
                    valid = (uint32_t)(w >> 34) == epoch && ((w >> 32) & 3ull) != 0;
                } while (!__all_sync(0xffffffffu, valid));
                const bool is_incl = ((w >> 32) & 3ull) == SCAN_FLAG_INCL;
                const unsigned im = __ballot_sync(0xffffffffu, is_incl);
                const int stop = im ? __ffs(im) - 1 : 31;   // nearest inclusive word (lane 0 = nearest predecessor)
                int32_t part = lane <= stop ? (int32_t)(uint32_t)w : 0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                prefix += part;
                if (im) break;
                hi -= 32;
            }
            if (lane == 0) vstate[tile] = scan_word(epoch, SCAN_FLAG_INCL, prefix + agg);
        }
        if (lane == 0) {
            s_prefix = prefix;
            if (tile == ntiles - 1 && total_out) *total_out = (int64_t)prefix + (int64_t)agg;
        }
    }
    __syncthreads();
    int32_t run = s_prefix + woff + incl - s;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        const int64_t idx = base + i;
        if (idx < n) out[idx] = run;
        run += v[i];
    }
}

struct ScanWorkspace {
    DBuf<unsigned long long> state;   // tile words + (last element) the ticket counter
    size_t state_cap = 0;
    uint32_t epoch = 0;
};

// out[i] = sum_{j<i} in[j]; *d_total (device int64, may be null) = sum of all
template <typename InT>
inline void exclusive_scan_i32(ScanWorkspace& ws, const InT* d_in, int32_t* d_out, int64_t n, int64_t* d_total, cudaStream_t st) {
    if (n <= 0) {
        if (d_total) DSA_CUDA(cudaMemsetAsync(d_total, 0, sizeof(int64_t), st));
        return;
    }
    const int64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    ws.state.ensure((size_t)ntiles + 1);
    if (ws.state.cap != ws.state_cap || ws.epoch >= (1u << 30) - 1) {   // new block (or epoch wrap): clear words + ticket once
        DSA_CUDA(cudaMemsetAsync(ws.state.p, 0, ws.state.cap * sizeof(unsigned long long), st));
        ws.state_cap = ws.state.cap;
        ws.epoch = 0;
    }
    ws.epoch += 1;
    uint32_t* ticket = reinterpret_cast<uint32_t*>(ws.state.p + (ws.state.cap - 1));
    DSA_LAUNCH("scan_onepass", (k_scan_onepass<InT>), (unsigned)ntiles, SCAN_THREADS, 0, st, d_in, d_out, n, ntiles, ws.state.p, ticket,
               ws.epoch, d_total);
}

// ---------------------------------------------------------------------------------------------
// min / max of int64 (for radix bit ranges and dimension tracking)
// ---------------------------------------------------------------------------------------------
__global__ void k_minmax_init(int64_t* mm) {
    mm[0] = INT64_MAX;
    mm[1] = INT64_MIN;
}
__global__ void __launch_bounds__(256) k_minmax_i64(const int64_t* __restrict__ a, int64_t n, int64_t* __restrict__ mm) {
    int64_t lo = INT64_MAX, hi = INT64_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t v = a[i];
        lo = v < lo ? v : lo;
        hi = v > hi ? v : hi;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t l2 = __shfl_down_sync(0xffffffffu, lo, o), h2 = __shfl_down_sync(0xffffffffu, hi, o);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin((long long*)&mm[0], (long long)lo);
        atomicMax((long long*)&mm[1], (long long)hi);
    }
}
inline void minmax_i64(const int64_t* d_a, int64_t n, int64_t* d_mm2, cudaStream_t st) {
    DSA_LAUNCH("minmax_init", k_minmax_init, 1, 1, 0, st, d_mm2);
    if (n > 0) {
        unsigned g = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8);
        DSA_LAUNCH("minmax_i64", k_minmax_i64, g, 256, 0, st, d_a, n, d_mm2);
    }
}

}  // namespace dsa
