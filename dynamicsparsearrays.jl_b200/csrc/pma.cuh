// libdsa — the packed memory array on the device: layout, bulk build (K4), finds (K6), batched merge with
// density tree / window selection (K2, K3) and redistribute (K4).  Shared by the vector and both PCSR orientations.
//
// HBM layout (SoA, all 8-byte lanes so a warp streams 256 B per load):
//   keys[capacity]  int64   GAP_KEY = `nothing`; 0 = semaphore key (pcsr.jl:23); >= 1 user keys
//   vals[capacity]  double  value, or the partition id of a semaphore cell (pcsr.jl:39-40)
//   leafcnt[nb_segments] int32   stored cells per segment (what _nbcells, utils.jl:48, recounts every time)
//   post[2*nb_segments]  int32   implicit tree of post-batch counts, level h at off[h] (pma.jl:105-141 walks it leaf->root)
#pragma once
#include "common.cuh"
#include "hostlogic.hpp"
#include "primitives.cuh"
#include "spread.cuh"

namespace dsa {

struct Levels {
    int64_t off[MAX_LEVELS];   // offset of level h in the tree arrays
    int64_t mn[MAX_LEVELS];    // accept iff mn[h] <= count <= mx[h]   (pma.jl:119-123)
    int64_t mx[MAX_LEVELS];
    int64_t nsegs;
    int H;
    int lgS;
    int hsmall;                // windows with h <= hsmall hold <= SMALL_CELLS cells: one CTA re-lays them in shared memory
    uint32_t leafmask[33];     // leafmask[m] = cells a leaf of S cells occupies when spread! lays m elements over it
};
constexpr int SMALL_CELLS = 2048;

enum : uint8_t { FL_OVERWRITE = 1, FL_DELETE = 2, FL_INSERT = 4 };
enum { ST_OVER = 0, ST_UNDER = 1, ST_NINS = 2, ST_ROOT = 3, ST_NHIGH = 4, ST_ANYBIG = 5, ST_NACT = 6, ST_ANYHIGH = 7, ST_TICKET = 8, ST_NPEND = 9,
       ST_NBIG = 10, ST_MAXBIGH = 11, ST_MAXSMALLH = 12, ST_WORDS = 16 };

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
// bits 0..x (x >= 31: all 32)
__device__ __forceinline__ unsigned mask_le(int x) { return x >= 31 ? 0xffffffffu : ((2u << x) - 1u); }
// bits 0..n-1, n <= 32 (the cells of a leaf of n cells)
__host__ __device__ __forceinline__ constexpr unsigned low_bits(int n) { return n >= 32 ? 0xffffffffu : ((1u << n) - 1u); }
__device__ __forceinline__ int64_t warp_sum_i64(int64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// K4 bulk layout: destination-driven spread of n sorted elements over `cap` cells (pma.jl:27-55 + moves.jl:120).
// One thread per cell: rank via the closed form, coalesced gather + coalesced store, leaf counts by ballot,
// semaphores[id] = position for key-0 cells (pcsr.jl:55-61).  If src == nullptr only gaps are written and cells that
// already hold an element are left alone (used after a scatter into a fresh array).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_layout(int64_t* __restrict__ keys, double* __restrict__ vals, int64_t cap, int64_t n,
                                                 const int64_t* __restrict__ src_k, const double* __restrict__ src_v,
                                                 int32_t* __restrict__ leafcnt, int64_t* __restrict__ sem, int lgS) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const Spread sp = spread_make(cap, n);
    int64_t r = -1;
    if (p < cap) r = spread_rank_at(sp, p);
    const bool live = r >= 0;
    if (p < cap) {
        if (src_k) {
            if (live) {
                int64_t k = src_k[r];
                double v = src_v[r];
                keys[p] = k;
                vals[p] = v;
                if (sem && k == 0) sem[(int64_t)v - 1] = p;
            } else {
                keys[p] = GAP_KEY;
                vals[p] = 0.0;
            }
        } else if (!live) {
            keys[p] = GAP_KEY;
            vals[p] = 0.0;
        }
    }
    const unsigned b = __ballot_sync(0xffffffffu, live);
    const int S = 1 << lgS;
    if (p < cap && (p & (S - 1)) == 0) leafcnt[p >> lgS] = __popc((b >> lane) & low_bits(S));
}

// ---------------------------------------------------------------------------------------------
// K6 find: the reference's gapped binary search (finds.jl:29-57), 0-based, one thread per query.
// Returns the position of the exact hit or of the predecessor (-1 = none); *hit tells which.
// (An 8-ary variant — 7 independent probes per round, 3 dependent rounds instead of 8 on a partition span — returned the same
// positions and was slower: 79 us against 55 us for the bucket kernel at config 2, 13 M against 142 M finds/s on the 2^21-cell
// vector: three times the loads at half the occupancy cost more than the shorter dependency chain saves.)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t gapped_find(const int64_t* __restrict__ keys, int64_t key, int64_t from, int64_t to, bool* hit) {
    int64_t lo = from, hi = to;
    while (lo <= hi) {
        const int64_t mid = (lo + hi) >> 1;
        int64_t i = mid;
        int64_t k = keys[i];
        while (k == GAP_KEY && i > lo) {   // walk left to the nearest element (finds.jl:33-35)
            --i;
            k = keys[i];
        }
        if (k == GAP_KEY) {
            lo = mid + 1;
        } else if (k > key) {
            hi = i - 1;
        } else if (k < key) {
            lo = mid + 1;
        } else {
            *hit = true;
            return i;
        }
    }
    *hit = false;
    int64_t i = hi;
    while (i >= 0 && keys[i] == GAP_KEY) --i;   // finds.jl:49-56
    return i;
}

// exclusive end of the span of partition `s`: the position of the next placed semaphore, or the capacity
// (pcsr.jl:177-186 _pos_of_partition_end + 1).  next_slot[s] = next live, already placed slot (-1 = none).
__device__ __forceinline__ int64_t span_end(const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot, int32_t s, int64_t cap) {
    const int32_t ns = next_slot[s];
    return ns >= 0 ? sem[ns] : cap;
}

// Locate every (sorted, unique) op.  pid == nullptr: plain PMA, search the whole array.  Otherwise the partition span is
// [sem[pid], next_sem[pid]) and, like pcsr.jl:305-307, inserts search (sem, end] while deletes search [sem, end].
// sem[pid] < 0 marks a partition created by this batch: everything goes right before the next live semaphore.
// one op: position of the hit or of the predecessor, and what the op turns into
__device__ __forceinline__ uint8_t locate_one(const int64_t* __restrict__ keys, int64_t cap, bool partitioned, int32_t pid, int64_t key,
                                              bool is_set, const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot,
                                              int64_t* pos_out) {
    int64_t pos;
    bool hit = false;
    if (partitioned) {
        const int64_t s = sem[pid];
        const int64_t e = span_end(sem, next_slot, pid, cap);
        if (s < 0 || key == 0) {
            pos = e - 1;   // new partition (or its semaphore): before the next live semaphore (pcsr.jl:121-126,101)
        } else {
            pos = gapped_find(keys, key, is_set ? s + 1 : s, e - 1, &hit);
        }
    } else {
        pos = gapped_find(keys, key, 0, cap - 1, &hit);
    }
    *pos_out = pos;
    return hit ? (is_set ? FL_OVERWRITE : FL_DELETE) : ((is_set || (partitioned && key == 0)) ? FL_INSERT : 0);
}

__global__ void __launch_bounds__(256) k_locate(const int64_t* __restrict__ keys, int64_t cap, const int32_t* __restrict__ op_pid,
                                                 const int64_t* __restrict__ op_key, const double* __restrict__ op_val, int64_t nops,
                                                 const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot,
                                                 int64_t* __restrict__ op_pos, uint8_t* __restrict__ op_flag,
                                                 const int64_t* __restrict__ n_dev, int32_t* __restrict__ ins_flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nops) return;
    if (i >= (n_dev ? *n_dev : nops)) {   // beyond the unique ops
        op_flag[i] = 0;
        ins_flag[i] = 0;
        return;
    }
    int64_t pos;
    const uint8_t f = locate_one(keys, cap, op_pid != nullptr, op_pid ? op_pid[i] : 0, op_key[i], op_val[i] != 0.0 /* pma.jl:197, pcsr.jl:301 */,
                                 sem, next_slot, &pos);
    op_pos[i] = pos;
    op_flag[i] = f;
    ins_flag[i] = f == FL_INSERT ? 1 : 0;
}

// batched getindex (pma.jl:189-193 / pcsr.jl:228-232): value or 0.0.  pid < 0 = column absent (pcsr.jl:263-265).
__global__ void __launch_bounds__(256) k_get(const int64_t* __restrict__ keys, const double* __restrict__ vals, int64_t cap,
                                              const int32_t* __restrict__ q_pid, const int64_t* __restrict__ q_key, int64_t nq,
                                              const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot,
                                              double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    bool hit = false;
    int64_t pos = -1;
    if (q_pid) {
        const int32_t pid = q_pid[i];
        if (pid >= 0 && sem[pid] >= 0) pos = gapped_find(keys, q_key[i], sem[pid], span_end(sem, next_slot, pid, cap) - 1, &hit);
    } else {
        pos = gapped_find(keys, q_key[i], 0, cap - 1, &hit);
    }
    out[i] = hit ? vals[pos] : 0.0;
}

// Located ops -> effects, one kernel: hits overwrite in place (writes.jl:16-19) or blank the cell (writes.jl:65-68; leaf count
// and touched flag follow); misses with a value are compacted, order-preserving, into the insert arrays (ins_idx = exclusive
// scan of the insert flags).  Runs after ALL ops are located: a delete must not change what another op's search sees.
// OVERWRITES = false when the locating kernel already stored the new values (bucket path).
template <bool OVERWRITES>
__global__ void __launch_bounds__(256) k_apply_compact(int64_t* __restrict__ keys, double* __restrict__ vals,
                                                        const int64_t* __restrict__ op_key, const double* __restrict__ op_val,
                                                        const int64_t* __restrict__ op_pos, const uint8_t* __restrict__ op_flag,
                                                        const int32_t* __restrict__ ins_idx, int64_t nops, int32_t* __restrict__ leafcnt,
                                                        uint8_t* __restrict__ touched, int lgS, int64_t* __restrict__ ins_key,
                                                        double* __restrict__ ins_val, int64_t* __restrict__ ins_pos) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nops) return;
    const uint8_t f = op_flag[i];
    if (f == 0) return;
    const int64_t p = op_pos[i];
    if (f == FL_INSERT) {
        const int32_t j = ins_idx[i];
        ins_key[j] = op_key[i];
        ins_val[j] = op_val[i];
        ins_pos[j] = p;
    } else if (f == FL_DELETE) {
        keys[p] = GAP_KEY;   // the value of a gap cell is never read (exports and SpMV mask by the key)
        atomicSub(&leafcnt[p >> lgS], 1);
        touched[p >> lgS] = 1;
    } else if (OVERWRITES) {
        vals[p] = op_val[i];
    }
}
// A batch of ONE op that turns out to be an insert is applied exactly like the reference's _insert! (writes.jl:26-43), so that
// single writes leave the reference's own layout: the cells between the predecessor and the next gap to its right — wherever
// that gap is, even in another leaf or partition — shift right by one (moves.jl:7-42, semaphore positions follow); if there is
// no gap up to the array end, the cells back to the previous gap shift left (moves.jl:50-85).  The leaf of the new element is
// then walked by the usual density tree (_look_for_rebalance!, pma.jl:105-141): accepted leaf => nothing else moves
// (pma.jl:96-99).  One warp; the op leaves this kernel as "applied" (no pending insert).
__global__ void __launch_bounds__(32) k_single_insert(int64_t* __restrict__ keys, double* __restrict__ vals, int64_t cap,
                                                      const int64_t* __restrict__ op_key, const double* __restrict__ op_val,
                                                      const int64_t* __restrict__ op_pos, uint8_t* __restrict__ op_flag,
                                                      int32_t* __restrict__ ins_flag, int32_t* __restrict__ leafcnt,
                                                      uint8_t* __restrict__ touched, int lgS, int64_t* __restrict__ sem) {
    if (op_flag[0] != FL_INSERT) return;
    const int lane = threadIdx.x;
    const int64_t pp = op_pos[0];   // predecessor cell, -1 = none
    int64_t g = -1;
    for (int64_t b0 = pp + 1; b0 < cap; b0 += 32) {   // _nextemptypos (utils.jl:3-10): scans to the array end
        const int64_t p = b0 + lane;
        const unsigned b = __ballot_sync(0xffffffffu, p < cap && keys[p] == GAP_KEY);
        if (b) {
            g = b0 + __ffs(b) - 1;
            break;
        }
    }
    int64_t newpos;
    if (g >= 0) {   // _movecellstoright!(array, pos + 1, next_empty_pos)
        int64_t hi = g - 1;
        while (hi >= pp + 1) {
            const int64_t lo = hi - 31 > pp + 1 ? hi - 31 : pp + 1;
            const int64_t p = lo + lane;
            const bool valid = p <= hi;
            int64_t k = 0;
            double v = 0.0;
            if (valid) {
                k = keys[p];
                v = vals[p];
            }
            __syncwarp();
            if (valid) {
                keys[p + 1] = k;
                vals[p + 1] = v;
                if (sem && k == 0) sem[(int64_t)v - 1] = p + 1;   // moves.jl:33-37
            }
            __syncwarp();
            hi = lo - 1;
        }
        newpos = pp + 1;
    } else {        // _previousemptypos + _movecellstoleft!(array, pos, previous_empty_pos)
        for (int64_t t0 = pp - 1; t0 >= 0; t0 -= 32) {
            const int64_t p = t0 - lane;
            const unsigned b = __ballot_sync(0xffffffffu, p >= 0 && keys[p] == GAP_KEY);
            if (b) {
                g = t0 - (__ffs(b) - 1);
                break;
            }
        }
        if (g < 0) return;   // "No empty cell to insert a new element": cannot occur below density 1 (writes.jl:39)
        int64_t lo = g + 1;
        while (lo <= pp) {
            const int64_t hi = lo + 31 < pp ? lo + 31 : pp;
            const int64_t p = lo + lane;
            const bool valid = p <= hi;
            int64_t k = 0;
            double v = 0.0;
            if (valid) {
                k = keys[p];
                v = vals[p];
            }
            __syncwarp();
            if (valid) {
                keys[p - 1] = k;
                vals[p - 1] = v;
                if (sem && k == 0) sem[(int64_t)v - 1] = p - 1;   // moves.jl:76-80
            }
            __syncwarp();
            lo = hi + 1;
        }
        newpos = pp;
    }
    if (lane == 0) {
        keys[newpos] = op_key[0];
        vals[newpos] = op_val[0];
        leafcnt[g >> lgS] += 1;          // the cell that was the gap is now occupied; every leaf in between keeps its count
        touched[newpos >> lgS] = 1;      // _look_for_rebalance!(pma, insertion_pos)
        op_flag[0] = 0;
        ins_flag[0] = 0;
    }
}

// per-leaf bookkeeping of the compacted inserts: every new key belongs to the leaf of its predecessor cell; inserts are
// sorted, so the inserts of one leaf are contiguous.  The thread of the FIRST insert of a leaf counts the run and records
// (leaf, first index, count) in the list of leaves that receive inserts (unordered: each entry is independent work).
struct ActiveLeaf {
    int32_t leaf, nins, i0, pad;
};
__global__ void __launch_bounds__(256) k_insert_leaf_info(const int64_t* __restrict__ ins_pos, const int64_t* __restrict__ nins_dev,
                                                           int32_t* __restrict__ inscnt, int32_t* __restrict__ ins_first,
                                                           uint8_t* __restrict__ touched, int lgS, ActiveLeaf* __restrict__ act,
                                                           int64_t* __restrict__ nact_dev) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = *nins_dev;
    if (j >= n) return;
    const int64_t pos = ins_pos[j];
    const int64_t leaf = (pos < 0 ? 0 : pos) >> lgS;
    if (j > 0) {
        const int64_t pq = ins_pos[j - 1];
        if (((pq < 0 ? 0 : pq) >> lgS) == leaf) return;
    }
    // the run of this leaf ends at the first insert whose predecessor lies in a later leaf (positions are sorted).  Runs are
    // short (about one insert per touched leaf on uniform batches): look at the next few entries — the same cache line — before
    // falling back to a binary search over the rest (skewed batches: thousands of inserts on one leaf)
    const int64_t leaf_end = (leaf + 1) << lgS;
    int64_t lo = j + 1, hi = n;
    int near = 0;
    while (lo < n && near < 8 && ins_pos[lo] < leaf_end) {
        ++lo;
        ++near;
    }
    if (near < 8 || lo >= n) hi = lo;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (ins_pos[mid] < leaf_end) lo = mid + 1;
        else hi = mid;
    }
    const int cnt = (int)(lo - j);
    inscnt[leaf] = cnt;
    ins_first[leaf] = (int32_t)j;
    touched[leaf] = 1;
    const unsigned long long slot = atomicAdd((unsigned long long*)nact_dev, 1ull);
    act[slot] = ActiveLeaf{(int32_t)leaf, cnt, (int32_t)j, 0};
}


// ---------------------------------------------------------------------------------------------
// K3 density tree + window pick (_look_for_rebalance!, pma.jl:105-141, for every touched leaf at once).
//   k_tree_low      post[0][l] = leafcnt[l] + inscnt[l]; 10 levels per CTA in shared memory; the LAST CTA to finish (ticket)
//                   sums the upper levels.  In the same pass every touched leaf takes the walk's first step: accepted at its own
//                   level (the common case: pma.jl:120-123 with h = 0) -> marked on the spot; otherwise queued.
//   k_select_pending  the queued leaves continue leaf -> root and mark the first window inside its density bounds.
// ---------------------------------------------------------------------------------------------
constexpr int TREE_LEAVES_PER_THREAD = 4, TREE_THREADS = 256, TREE_TILE = TREE_LEAVES_PER_THREAD * TREE_THREADS;   // 1024 leaves per CTA
constexpr int TREE_UP_NODES = 2048;   // upper levels of the tree that the last CTA finishes in shared memory
__global__ void __launch_bounds__(TREE_THREADS) k_tree_low(const int32_t* __restrict__ leafcnt, const int32_t* __restrict__ inscnt,
                                                            int32_t* __restrict__ post, Levels L, const uint8_t* __restrict__ touched,
                                                            uint8_t* __restrict__ mark, int64_t* __restrict__ status,
                                                            int32_t* __restrict__ pending) {
    __shared__ int32_t s[TREE_THREADS];
    __shared__ int is_last;
    // a thread owns 4 consecutive leaves: levels 0..2 in registers, levels 3..10 in shared memory
    const int64_t idx0 = ((int64_t)blockIdx.x * TREE_THREADS + threadIdx.x) * TREE_LEAVES_PER_THREAD;
    int32_t v[TREE_LEAVES_PER_THREAD];
#pragma unroll
    for (int e = 0; e < TREE_LEAVES_PER_THREAD; ++e) {
        const int64_t idx = idx0 + e;
        v[e] = 0;
        if (idx < L.nsegs) {
            v[e] = leafcnt[idx] + (inscnt ? inscnt[idx] : 0);
            post[L.off[0] + idx] = v[e];
            if (touched[idx]) {
                if (L.mn[0] <= v[e] && v[e] <= L.mx[0]) {
                    mark[L.off[0] + idx] = 1;
                } else {
                    const unsigned long long slot = atomicAdd((unsigned long long*)&status[ST_NPEND], 1ull);
                    pending[slot] = (int32_t)idx;
                }
            }
        }
    }
    const int32_t a = v[0] + v[1], b2 = v[2] + v[3];
    if (L.H >= 1) {
        const int64_t n1 = idx0 >> 1;
        if (n1 < (L.nsegs >> 1)) post[L.off[1] + n1] = a;
        if (n1 + 1 < (L.nsegs >> 1)) post[L.off[1] + n1 + 1] = b2;
    }
    int32_t t = a + b2;
    if (L.H >= 2 && (idx0 >> 2) < (L.nsegs >> 2)) post[L.off[2] + (idx0 >> 2)] = t;
    s[threadIdx.x] = t;
    __syncthreads();
    const int top = L.H < 10 ? L.H : 10;
    for (int k = 3; k <= top; ++k) {
        const int nk = TREE_TILE >> k;
        int32_t u = 0;
        if ((int)threadIdx.x < nk) u = s[2 * threadIdx.x] + s[2 * threadIdx.x + 1];
        __syncthreads();
        if ((int)threadIdx.x < nk) {
            s[threadIdx.x] = u;
            const int64_t node = (((int64_t)blockIdx.x * TREE_TILE) >> k) + threadIdx.x;
            if (node < (L.nsegs >> k)) post[L.off[k] + node] = u;
        }
        __syncthreads();
    }
    if (L.H <= 10) return;
    // upper levels: by the last CTA to get here (its predecessors' level-10 sums are visible: fence + ticket)
    __threadfence();
    if (threadIdx.x == 0) is_last = atomicAdd((unsigned long long*)&status[ST_TICKET], 1ull) == (unsigned long long)gridDim.x - 1;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    int k = 11;
    for (; k <= L.H && (L.nsegs >> (k - 1)) > TREE_UP_NODES; ++k) {   // huge arrays: one global round trip per level
        const int64_t nodes = L.nsegs >> k;
        for (int64_t i = threadIdx.x; i < nodes; i += TREE_THREADS)
            post[L.off[k] + i] = __ldcg(&post[L.off[k - 1] + 2 * i]) + __ldcg(&post[L.off[k - 1] + 2 * i + 1]);
        __syncthreads();
    }
    if (k > L.H) return;
    // the remaining levels hold at most TREE_UP_NODES nodes: one load into shared memory, then no more global round trips
    // (10 levels at ~1 us each otherwise)
    __shared__ int32_t up[2][TREE_UP_NODES];
    int cur = 0;
    {
        const int n = (int)(L.nsegs >> (k - 1));
        for (int i = threadIdx.x; i < n; i += TREE_THREADS) up[0][i] = __ldcg(&post[L.off[k - 1] + i]);
    }
    __syncthreads();
    for (; k <= L.H; ++k) {
        const int nodes = (int)(L.nsegs >> k);
        for (int i = threadIdx.x; i < nodes; i += TREE_THREADS) {
            const int32_t u = up[cur][2 * i] + up[cur][2 * i + 1];
            up[cur ^ 1][i] = u;
            post[L.off[k] + i] = u;
        }
        cur ^= 1;
        __syncthreads();
    }
}

// the queued leaves walk on, from level 1 (pma.jl:113-129).  Windows above leaf level are also appended (once) to a work list.
__global__ void __launch_bounds__(256) k_select_pending(const int32_t* __restrict__ pending, const int32_t* __restrict__ post,
                                                         uint8_t* __restrict__ mark, Levels L, int64_t* __restrict__ status,
                                                         int32_t* __restrict__ hi_h, int64_t* __restrict__ hi_w,
                                                         int32_t* __restrict__ big_h, int64_t* __restrict__ big_w) {
    const int64_t npend = status[ST_NPEND];
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < npend; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = pending[q];
        bool done = false;
        for (int h = 1; h <= L.H && !done; ++h) {
            const int64_t c = post[L.off[h] + (l >> h)];
            if (L.mn[h] <= c && c <= L.mx[h]) {
                const int64_t idx = L.off[h] + (l >> h);
                unsigned* word = (unsigned*)(mark + (idx & ~(int64_t)3));
                const unsigned bit = 1u << (8 * (unsigned)(idx & 3));
                const unsigned old = atomicOr(word, bit);
                if (!(old & bit)) {   // first marker of this window
                    const unsigned long long slot = atomicAdd((unsigned long long*)&status[ST_NHIGH], 1ull);
                    hi_h[slot] = h;
                    hi_w[slot] = l >> h;
                    status[ST_ANYHIGH] = 1;
                    // sizes k_window_small's CTAs (the plain read keeps thousands of windows of one height off the atomic unit)
                    if (h <= L.hsmall && (int64_t)h > *(volatile int64_t*)&status[ST_MAXSMALLH])
                        atomicMax((long long*)&status[ST_MAXSMALLH], (long long)h);
                    if (h > L.hsmall) {   // too large for one CTA's shared memory: its own work list
                        status[ST_ANYBIG] = 1;
                        const unsigned long long bs = atomicAdd((unsigned long long*)&status[ST_NBIG], 1ull);
                        big_h[bs] = h;
                        big_w[bs] = l >> h;
                        atomicMax((long long*)&status[ST_MAXBIGH], (long long)h);
                    }
                }
                done = true;
            }
        }
        if (!done) {
            const int64_t c = post[L.off[L.H]];
            if (c > L.mx[L.H]) status[ST_OVER] = 1;   // density > t  -> _extend!  (pma.jl:132-134)
            else status[ST_UNDER] = 1;                // density < p  -> _shrink!  (pma.jl:135-139)
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) status[ST_ROOT] = post[L.off[L.H]];   // element count after the batch
}

// ---------------------------------------------------------------------------------------------
// K2 + K4 merge / redistribute.  Rank of an item inside its window = prefix of post counts over the window's preceding leaves
// (read off the implicit tree, <= h loads) + position inside the leaf's merged run: the survivors before it + the leaf's
// inserts whose predecessor lies before it.  Destination = window start + closed-form spread! offset.  Leaves accepted at
// their own level are rewritten in place (k_leaf_merge), windows of at most SMALL_CELLS cells through shared memory
// (k_window_small); bigger windows are scattered into the shadow array and copied back (k_merge_scatter_big,
// k_scatter_inserts, k_copyback_big).  Root mode (resize): the same scatter over the root window, into the new arrays.
// ---------------------------------------------------------------------------------------------
struct MergeArgs {
    const int64_t* src_k;
    const double* src_v;
    int64_t* cur_k;   // == src (mutable) for in-place leaves
    double* cur_v;
    int64_t* dst_k;   // shadow or new array
    double* dst_v;
    const int32_t* post;
    const uint8_t* mark;
    const int32_t* inscnt;
    const int32_t* ins_first;
    const int64_t* ins_key;
    const double* ins_val;
    const int64_t* ins_pos;
    int32_t* leafcnt;
    int64_t* sem;   // nullable; 0-based positions per partition id
    int root_mode;  // resize: one window of height L.H, root_c cells, root_m elements, scattered into dst
    int64_t root_c, root_m;
    const uint8_t* cover;      // per leaf: 0 = not inside a window above leaf level, else 1 + height of the outermost one
    const uint8_t* destpos;    // [33][32] spread! offset of rank r in a leaf holding m elements
    const ActiveLeaf* act;     // leaves that receive inserts
    const int64_t* nact_dev;
    const int32_t* hi_h;       // work list of windows above leaf level
    const int64_t* hi_w;
    const int32_t* big_h;      // work list of the windows above SMALL_CELLS
    const int64_t* big_w;
};

// post count of the left sibling of leaf l's ancestor at level k.  The elements of a window of height h that lie before leaf l
// are the sum of these over the levels k < h at which that ancestor is a right child (bit k of l set).
__device__ __forceinline__ int32_t left_sibling_post(const int32_t* __restrict__ post, const Levels& L, int64_t l, int k) {
    return post[L.off[k] + ((l >> k) - 1)];
}
// the same sum by one warp: lane k adds level k
__device__ __forceinline__ int64_t window_prefix(const int32_t* __restrict__ post, const Levels& L, int64_t l, int h, int lane) {
    int64_t term = 0;
    if (lane < h && ((l >> lane) & 1)) term = left_sibling_post(post, L, l, lane);
    return warp_sum_i64(term);
}
// one warp over a leaf, lane = cell p (in = the lane holds a cell): the cell's key and value; returns the leaf's survivors
__device__ __forceinline__ unsigned load_leaf_cell(const int64_t* src_k, const double* src_v, int64_t p, bool in, int64_t& key,
                                                   double& val) {
    key = GAP_KEY;
    val = 0.0;
    if (in) {
        key = src_k[p];
        val = src_v[p];
    }
    return __ballot_sync(0xffffffffu, key != GAP_KEY);
}
// inserts of a leaf (predecessor cells ins_pos[0..nins), sorted) whose predecessor lies before cell p
__device__ __forceinline__ int inserts_before(const int64_t* ins_pos, int nins, int64_t p) {
    int lo = 0, hi = nins;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (ins_pos[mid] < p) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
// survivors of a leaf (mask lm) up to its cell qq (-1 = before the first cell): they precede an insert whose predecessor is qq
__device__ __forceinline__ int survivors_le(unsigned lm, int qq) { return qq < 0 ? 0 : __popc(lm & mask_le(qq)); }
// the window of height h that holds leaf l: first cell, cells, elements after the batch (root: the resized array)
struct Window {
    int64_t cell0, c, m;
};
__device__ __forceinline__ Window window_of(const MergeArgs& A, const Levels& L, int64_t l, int h, bool root) {
    if (root) return Window{0, A.root_c, A.root_m};
    return Window{((l >> h) << h) << L.lgS, (int64_t)(1 << L.lgS) << h, A.post[L.off[h] + (l >> h)]};
}

// one leaf of a big window (one warp, lane = cell): survivors ranked and scattered to their spread! positions in dst.  The
// leaf's inserts are placed by k_scatter_inserts (one thread per insert: a hot leaf may receive millions).
__device__ __forceinline__ void merge_scatter_leaf(const MergeArgs& A, const Levels& L, int64_t l, int h, int lane) {
    const int nins = A.inscnt[l];
    const int64_t i0 = nins ? A.ins_first[l] : 0;
    const Window W = window_of(A, L, l, h, A.root_mode);
    const int64_t base = window_prefix(A.post, L, l, h, lane);
    const int64_t p = (l << L.lgS) + lane;
    int64_t key;
    double val;
    const unsigned lm = load_leaf_cell(A.src_k, A.src_v, p, lane < (1 << L.lgS), key, val);
    const bool live = key != GAP_KEY;
    const int srank = __popc(lm & lanemask_lt());
    const int cntb = live ? inserts_before(A.ins_pos + i0, nins, p) : 0;
    const Spread sp = spread_make(W.c, W.m);
    if (live) {
        const int64_t d = W.cell0 + spread_dest(sp, base + srank + cntb);
        A.dst_k[d] = key;
        A.dst_v[d] = val;
        if (A.sem && key == 0) A.sem[(int64_t)val - 1] = d;   // moves.jl:160-166
    }
}

// outermost = no marked ancestor (a window nested in a larger marked one is re-laid by that one)
__device__ __forceinline__ bool window_is_outermost(const uint8_t* __restrict__ mark, const Levels& L, int h, int64_t w) {
    for (int g = h + 1; g <= L.H; ++g)
        if (mark[L.off[g] + (w >> (g - h))]) return false;
    return true;
}

// grid = (chunks, windows): the blocks of window blockIdx.z * gridDim.y + blockIdx.y (grid.y stops at 65535) share out its
// leaves, one warp per leaf calls leaf_fn(leaf, h, lane).  Only the leaves of the listed windows are visited — a skewed batch
// marks a few hundred windows of a few thousand cells in an array of tens of millions.  Root mode: the one window of height
// L.H, which is every leaf.
template <class LeafFn>
__device__ __forceinline__ void for_each_big_window_leaf(const MergeArgs& A, const Levels& L, int64_t nbig, LeafFn leaf_fn) {
    __shared__ int ok;
    const int64_t i = (int64_t)blockIdx.z * gridDim.y + blockIdx.y;
    if (i >= nbig) return;
    const int h = A.root_mode ? L.H : A.big_h[i];
    const int64_t w = A.root_mode ? 0 : A.big_w[i];
    if (!A.root_mode) {   // (the root has no ancestor: a resize's many short blocks skip the barrier)
        if (threadIdx.x == 0) ok = window_is_outermost(A.mark, L, h, w);
        __syncthreads();
        if (!ok) return;
    }
    const int lane = threadIdx.x & 31;
    const int64_t nleaves = (int64_t)1 << h, first = w << h;
    for (int64_t j = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < nleaves; j += (int64_t)gridDim.x * (blockDim.x >> 5))
        leaf_fn(first + j, h, lane);
}

__global__ void __launch_bounds__(256) k_merge_scatter_big(MergeArgs A, Levels L, int64_t nbig) {
    for_each_big_window_leaf(A, L, nbig, [&](int64_t l, int h, int lane) { merge_scatter_leaf(A, L, l, h, lane); });
}

// ---------------------------------------------------------------------------------------------
// K2 leaf merge (the common case: the leaf itself is the accepted window).  S lanes per leaf, 32/S leaves per warp,
// dense over the leaves with a two-load early exit.  The merged run is re-laid in place from registers; destinations
// come from the precomputed spread! occupancy mask of (S cells, m elements) — no floating point on this path.
// ---------------------------------------------------------------------------------------------
// List-driven: one S-lane group per leaf that receives inserts (32/S leaves per warp), two dependent load rounds.
__global__ void __launch_bounds__(256) k_leaf_merge(MergeArgs A, Levels L) {
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int lgS = L.lgS, S = 1 << lgS;
    const int grp = lane >> lgS, q = lane & (S - 1), gshift = grp << lgS;
    const unsigned gmask = low_bits(S);
    const int64_t e = gw * (32 >> lgS) + grp;
    const int64_t nact = *A.nact_dev;
    if (gw * (32 >> lgS) >= nact) return;
    // round 1: the work item
    ActiveLeaf al = ActiveLeaf{0, 0, 0, 0};
    const bool have = e < nact;
    if (have) al = A.act[e];
    const int64_t l = al.leaf;
    const int nins = al.nins;
    const int64_t p0 = l << lgS, p = p0 + q;
    // round 2: everything else, issued together
    uint8_t cov = 1;
    int64_t key = GAP_KEY, ik = 0;
    double val = 0.0, iv = 0.0;
    int qq = -2;
    const bool has_ins = have && q < nins;
    if (have) {
        cov = A.cover[l];
        key = A.src_k[p];
        val = A.src_v[p];
        if (has_ins) {
            qq = (int)(A.ins_pos[al.i0 + q] - p0);   // predecessor cell inside the leaf, -1 = before the first cell
            ik = A.ins_key[al.i0 + q];
            iv = A.ins_val[al.i0 + q];
        }
    }
    const bool active = have && cov == 0;   // not inside a window above leaf level (those are re-laid by k_window_small)
    const bool live = key != GAP_KEY;
    const unsigned lm = (__ballot_sync(0xffffffffu, live) >> gshift) & gmask;
    const int srank = __popc(lm & ((1u << q) - 1u));
    // rank of insert q in the merged run = survivors up to its predecessor + the inserts before it
    int rj = 0;
    unsigned insbit = 0;
    if (has_ins) {
        rj = survivors_le(lm, qq) + q;
        insbit = 1u << rj;
    }
    const unsigned insmask = __reduce_or_sync(gmask << gshift, insbit);   // merged ranks taken by the inserts
    const int m = __popc(lm) + nins;
    const uint8_t* __restrict__ dtab = A.destpos + m * 32;   // spread! offsets for (S cells, m elements)
    const unsigned mask = L.leafmask[m];
    __syncwarp();
    if (active) {
        if (!((mask >> q) & 1u)) {
            A.cur_k[p] = GAP_KEY;
            A.cur_v[p] = 0.0;
        }
        if (live) {
            // the srank-th rank not taken by an insert: least fixed point of R = srank + #inserts at ranks <= R
            int R = srank;
            while (true) {
                const int Rn = srank + __popc(insmask & mask_le(R));
                if (Rn == R) break;
                R = Rn;
            }
            const int64_t d = p0 + dtab[R];
            A.cur_k[d] = key;
            A.cur_v[d] = val;
            if (A.sem && key == 0) A.sem[(int64_t)val - 1] = d;   // moves.jl:160-166
        }
        if (has_ins) {
            const int64_t d = p0 + dtab[rj];
            A.cur_k[d] = ik;
            A.cur_v[d] = iv;
            if (A.sem && ik == 0) A.sem[(int64_t)iv - 1] = d;
        }
        if (q == 0) A.leafcnt[l] = m;
    }
}

// ---------------------------------------------------------------------------------------------
// K4 windows above leaf level: one CTA per listed window.  Outermost windows mark their leaves as covered; those of at most
// SMALL_CELLS cells are re-laid here: the merged, ranked items are scattered to their spread! offsets in shared memory, then the
// window is written back coalesced (pack! + spread!, moves.jl:94-172, in one pass), with leaf counts and semaphore positions.
// ---------------------------------------------------------------------------------------------
// Shared memory (dynamic) and block size follow the LARGEST small window of the batch (`cells`): a batch whose windows are a few
// leaves each runs 32 CTAs of 64 threads per SM instead of 7 of 256.
__global__ void __launch_bounds__(256) k_window_small(MergeArgs A, Levels L, uint8_t* __restrict__ cover, int cells) {
    extern __shared__ __align__(16) unsigned char window_smem[];
    int64_t* sk = reinterpret_cast<int64_t*>(window_smem);
    double* sv = reinterpret_cast<double*>(sk + cells);
    __shared__ int is_max;
    const int64_t i = blockIdx.x;
    const int h = A.hi_h[i];
    const int64_t w = A.hi_w[i];
    // outermost (no marked ancestor)?  then its leaves are covered by it: k_leaf_merge (launched after this kernel) skips them.
    // One lane per ancestor level (the loads of a serial walk up the tree were most of this kernel's duration).
    if (threadIdx.x < 32) {
        const int g = h + 1 + (int)threadIdx.x;
        const bool mk = g <= L.H && A.mark[L.off[g] + (w >> (g - h))] != 0;
        const unsigned b = __ballot_sync(0xffffffffu, mk);
        if (threadIdx.x == 0) is_max = b == 0;
    }
    __syncthreads();
    if (!is_max) return;
    {
        const int64_t first = w << h, n = (int64_t)1 << h;
        for (int64_t j = threadIdx.x; j < n; j += blockDim.x) cover[first + j] = (uint8_t)(h + 1);
    }
    if (h > L.hsmall) return;   // re-laid by the list-driven big path
    const int lgS = L.lgS, S = 1 << lgS;
    const int c = S << h;
    const int64_t m = A.post[L.off[h] + w];
    const int64_t first_leaf = w << h;
    const int64_t ws_cell = first_leaf << lgS;
    for (int t = threadIdx.x; t < c; t += blockDim.x) {
        sk[t] = GAP_KEY;
        sv[t] = 0.0;
    }
    __syncthreads();
    const Spread sp = spread_make(c, m);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int64_t j = wid; j < ((int64_t)1 << h); j += nw) {
        const int64_t l = first_leaf + j;
        const int64_t base = window_prefix(A.post, L, l, h, lane);
        const int nins = A.inscnt[l];
        const int64_t i0 = nins ? A.ins_first[l] : 0;
        const int64_t p0 = l << lgS, p = p0 + lane;
        int64_t key;
        double val;
        const unsigned lm = load_leaf_cell(A.src_k, A.src_v, p, lane < S, key, val);
        const bool live = key != GAP_KEY;
        const int srank = __popc(lm & lanemask_lt());
        const int cntb = live ? inserts_before(A.ins_pos + i0, nins, p) : 0;
        if (live) {
            const int64_t d = spread_dest(sp, base + srank + cntb);
            sk[d] = key;
            sv[d] = val;
        }
        for (int jj = lane; jj < nins; jj += 32) {
            const int64_t d = spread_dest(sp, base + survivors_le(lm, (int)(A.ins_pos[i0 + jj] - p0)) + jj);
            sk[d] = A.ins_key[i0 + jj];
            sv[d] = A.ins_val[i0 + jj];
        }
    }
    __syncthreads();
    for (int t0 = 0; t0 < c; t0 += blockDim.x) {
        const int t = t0 + threadIdx.x;
        const bool in = t < c;
        int64_t k = GAP_KEY;
        if (in) {
            k = sk[t];
            const double v = sv[t];
            const int64_t p = ws_cell + t;
            A.cur_k[p] = k;
            A.cur_v[p] = v;
            if (A.sem && k == 0) A.sem[(int64_t)v - 1] = p;
        }
        const unsigned b = __ballot_sync(0xffffffffu, in && k != GAP_KEY);
        if (in && (t & (S - 1)) == 0) A.leafcnt[(ws_cell + t) >> lgS] = __popc((b >> lane) & low_bits(S));
    }
}

// Inserts of the big windows / of a resize: one thread per insert (appends and skewed batches pile up to millions of inserts
// on one leaf, so they cannot be left to the leaf's warp).  rank = prefix of post over the window's preceding leaves
// + survivors of the leaf up to the predecessor cell + index among the leaf's inserts.
__global__ void __launch_bounds__(256) k_scatter_inserts(MergeArgs A, Levels L, const int64_t* __restrict__ nins_dev) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *nins_dev) return;
    const int64_t ipos = A.ins_pos[j];
    const int64_t l = (ipos < 0 ? 0 : ipos) >> L.lgS;
    int h;
    if (A.root_mode) h = L.H;
    else {
        h = (int)A.cover[l] - 1;          // height of the outermost window covering the leaf (k_window_small)
        if (h <= L.hsmall) return;        // leaf-level or small window: placed by k_leaf_merge / k_window_small
    }
    const Window W = window_of(A, L, l, h, A.root_mode);
    int64_t base = 0;
    for (int k = 0; k < h; ++k)
        if ((l >> k) & 1) base += left_sibling_post(A.post, L, l, k);
    int surv_le = 0;
    for (int64_t p = l << L.lgS; p <= ipos; ++p) surv_le += A.src_k[p] != GAP_KEY;
    const int64_t r = base + surv_le + (j - A.ins_first[l]);
    const int64_t d = W.cell0 + spread_dest(spread_make(W.c, W.m), r);
    const int64_t ik = A.ins_key[j];
    const double iv = A.ins_val[j];
    A.dst_k[d] = ik;
    A.dst_v[d] = iv;
    if (A.sem && ik == 0) A.sem[(int64_t)iv - 1] = d;
}

// big windows: copy the shadow back, writing the analytic gaps and the new leaf counts
__global__ void __launch_bounds__(256) k_copyback_big(MergeArgs A, Levels L, int64_t nbig) {
    for_each_big_window_leaf(A, L, nbig, [&](int64_t l, int h, int lane) {
        const Window W = window_of(A, L, l, h, false);   // a resize scatters straight into the new arrays: no copy back
        const Spread sp = spread_make(W.c, W.m);
        const int64_t p = (l << L.lgS) + lane;
        bool live = false;
        if (lane < (1 << L.lgS)) {
            live = spread_rank_at(sp, p - W.cell0) >= 0;
            int64_t k = GAP_KEY;
            double v = 0.0;
            if (live) {
                k = A.dst_k[p];
                v = A.dst_v[p];
            }
            A.cur_k[p] = k;
            A.cur_v[p] = v;
        }
        const unsigned b = __ballot_sync(0xffffffffu, live);
        if (lane == 0) A.leafcnt[l] = __popc(b);
    });
}

__global__ void __launch_bounds__(256) k_export_cells(const int64_t* __restrict__ keys, const double* __restrict__ vals, int64_t cap,
                                                       uint8_t* __restrict__ occ, int64_t* __restrict__ ok, double* __restrict__ ov) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < cap) {
        const int64_t k = keys[p];
        const bool live = k != GAP_KEY;
        occ[p] = live ? 1 : 0;
        ok[p] = live ? k : 0;
        ov[p] = live ? vals[p] : 0.0;
    }
}

// =============================================================================================
// Host-side PMA core
// =============================================================================================
struct BatchWorkspace {   // per-handle scratch reused by every batch
    DBuf<int64_t> op_pos;
    DBuf<uint8_t> op_flag;
    DBuf<int32_t> ins_idx, flag32;
    DBuf<int64_t> ins_key, ins_pos;
    DBuf<double> ins_val;
    DBuf<int32_t> ins_first, post, pending;
    // everything that must start a batch as zero lives in ONE block cleared by one memset:
    DBuf<uint8_t> zero_blk;
    int64_t* status = nullptr;   // ST_WORDS
    int32_t* inscnt = nullptr;   // per leaf
    uint8_t* mark = nullptr;     // implicit tree
    uint8_t* touched = nullptr;  // per leaf
    uint8_t* cover = nullptr;    // per leaf
    DBuf<int32_t> hi_h, big_h;
    DBuf<int64_t> hi_w, big_w;
    DBuf<ActiveLeaf> act;
    DBuf<int64_t> shadow_k;
    DBuf<double> shadow_v;
    HPinned<int64_t> h_status;
    ScanWorkspace scan;
    bool single_op = false;      // the running batch is one op: reference-exact single write (k_single_insert, one resize step)
};

struct PmaCore {
    Geometry g{};
    int64_t nnz = 0;   // nb_elements (pma.jl:12)
    DBuf<int64_t> keys;
    DBuf<double> vals;
    DBuf<int32_t> leafcnt;
    DBuf<uint8_t> destpos;     // leaf-level spread! table, rebuilt when the segment capacity is (re)set
    int64_t destpos_S = -1;

    void ensure_destpos(cudaStream_t st) {
        const int S = (int)g.segment_capacity;
        if (destpos_S == S) return;
        std::vector<uint8_t> h(33 * 32, 0);
        for (int m = 0; m <= S; ++m) {
            const Spread sp = spread_make(S, m);
            for (int r = 0; r < m; ++r) h[(size_t)m * 32 + r] = (uint8_t)spread_dest(sp, r);
        }
        destpos.ensure(h.size());
        DSA_CUDA(cudaMemcpyAsync(destpos.p, h.data(), h.size(), cudaMemcpyHostToDevice, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        destpos_S = S;
    }

    Levels levels() const {
        Levels L;
        memset(&L, 0, sizeof(L));
        L.nsegs = g.nb_segments;
        L.H = (int)g.height;
        L.lgS = ilog2_i64(g.segment_capacity);
        int64_t o = 0;
        for (int h = 0; h <= L.H; ++h) {
            L.off[h] = o;
            o += g.nb_segments >> h;
        }
        level_bounds(g.segment_capacity, g.height, g.t_d, g.p_d, L.mn, L.mx);
        const int S = (int)g.segment_capacity;
        L.hsmall = 0;
        while (L.hsmall < L.H && ((int64_t)S << (L.hsmall + 1)) <= SMALL_CELLS) ++L.hsmall;
        for (int m = 0; m <= S; ++m) {
            const Spread sp = spread_make(S, m);
            uint32_t mask = 0;
            for (int r = 0; r < m; ++r) mask |= 1u << (unsigned)spread_dest(sp, r);
            L.leafmask[m] = mask;
        }
        return L;
    }
    int64_t tree_size() const { return 2 * g.nb_segments + 8; }

    void alloc(const Geometry& ng) {
        g = ng;
        keys.ensure((size_t)g.capacity);
        vals.ensure((size_t)g.capacity);
        leafcnt.ensure((size_t)g.nb_segments);
    }

    // PackedMemoryArray(keys, values; sort = false) (pma.jl:69-84) / empty constructor (pma.jl:86-91)
    void build_from_sorted(const int64_t* d_k, const double* d_v, int64_t n, int64_t* d_sem, cudaStream_t st) {
        alloc(geometry_for_build(n));
        nnz = n;
        const int lgS = ilog2_i64(g.segment_capacity);
        if (n == 0) {   // all gaps: any non-null source will do, it is never dereferenced
            d_k = keys.p;
            d_v = vals.p;
        }
        DSA_LAUNCH("layout_build", k_layout, grid_for(g.capacity, 256), 256, 0, st, keys.p, vals.p, g.capacity, n, d_k, d_v,
                   leafcnt.p, d_sem, lgS);
        ensure_destpos(st);   // the segment capacity is fixed from here on (pma.jl:143-161 keep it): no upload inside a batch
    }
    // a copy inherits the table (device to device, no synchronisation)
    void copy_destpos_from(const PmaCore& o, cudaStream_t st) {
        if (o.destpos_S < 0) return;
        destpos.ensure(33 * 32);
        DSA_CUDA(cudaMemcpyAsync(destpos.p, o.destpos.p, 33 * 32, cudaMemcpyDeviceToDevice, st));
        destpos_S = o.destpos_S;
    }

    // The batch tail shared by every mutation: ops are located (op_pos/op_flag), deletes/purges already counted in leafcnt
    // + touched.  Builds the density tree, selects windows, merges/redistributes, resizes when the root fails.
    // d_sem (nullable) = semaphore positions to refresh.  Returns through nnz.
    void rebalance_after(BatchWorkspace& ws, int64_t* d_sem, cudaStream_t st) {
        rebalance_launch(ws, st);
        DSA_CUDA(cudaStreamSynchronize(st));
        rebalance_finish(ws, d_sem, st);
    }

    // first half: density tree + window selection + status read-back (enqueued; the caller synchronises the stream)
    void rebalance_launch(BatchWorkspace& ws, cudaStream_t st) {
        Levels L = levels();
        const int64_t nsegs = g.nb_segments;
        int32_t* post = ws.post.ensure((size_t)tree_size());
        uint8_t* mark = ws.mark;
        int64_t* status = ws.status;
        int32_t* hi_h = ws.hi_h.ensure((size_t)nsegs + 1);
        int64_t* hi_w = ws.hi_w.ensure((size_t)nsegs + 1);
        int32_t* pending = ws.pending.ensure((size_t)nsegs + 1);
        DSA_LAUNCH("tree_low", k_tree_low, grid_for(nsegs, TREE_TILE), TREE_THREADS, 0, st, leafcnt.p, ws.inscnt, post, L, ws.touched, mark, status, pending);
        int32_t* big_h = ws.big_h.ensure((size_t)(nsegs >> (L.hsmall + 1)) + 2);
        int64_t* big_w = ws.big_w.ensure((size_t)(nsegs >> (L.hsmall + 1)) + 2);
        DSA_LAUNCH("select_pending", k_select_pending, 148, 256, 0, st, pending, post, mark, L, status, hi_h, hi_w, big_h, big_w);
        int64_t* hs = ws.h_status.ensure(ST_WORDS);
        DSA_CUDA(cudaMemcpyAsync(hs, status, ST_WORDS * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    }

    // second half (after the stream was synchronised): merges / redistributes, resizes when the root failed
    void rebalance_finish(BatchWorkspace& ws, int64_t* d_sem, cudaStream_t st) {
        Levels L = levels();
        const int64_t nsegs = g.nb_segments;
        int32_t* post = ws.post.p;
        uint8_t* mark = ws.mark;
        uint8_t* cover = ws.cover;
        int32_t* hi_h = ws.hi_h.p;
        int64_t* hi_w = ws.hi_w.p;
        int64_t* hs = ws.h_status.p;
        const int64_t N = (int64_t)(int32_t)(hs[ST_ROOT] & 0xffffffff);
        MergeArgs A;
        memset(&A, 0, sizeof(A));
        A.src_k = keys.p; A.src_v = vals.p; A.cur_k = keys.p; A.cur_v = vals.p;
        A.post = post; A.mark = mark; A.inscnt = ws.inscnt; A.ins_first = ws.ins_first.p;
        A.ins_key = ws.ins_key.p; A.ins_val = ws.ins_val.p; A.ins_pos = ws.ins_pos.p;
        A.leafcnt = leafcnt.p; A.sem = d_sem;
        A.cover = cover; A.hi_h = hi_h; A.hi_w = hi_w;
        ensure_destpos(st);
        A.destpos = destpos.p;
        A.act = ws.act.p;
        A.nact_dev = ws.status + ST_NACT;
        if (hs[ST_OVER] || hs[ST_UNDER]) {
            // root failed: _extend!/_shrink! (pma.jl:132-139) until the root accepts, then one full spread into the new array
            Geometry ng = geometry_after_root_failure(g, N, ws.single_op);
            DBuf<int64_t> nk;
            DBuf<double> nv;
            nk.ensure((size_t)ng.capacity);
            nv.ensure((size_t)ng.capacity);
            A.dst_k = nk.p; A.dst_v = nv.p; A.root_mode = 1; A.root_c = ng.capacity; A.root_m = N;
            // the root window is every leaf (geometries are built with 2^height segments, and resizes keep that)
            if (nsegs != (int64_t)1 << L.H) throw DsaError{DSA_ERR_INTERNAL, "nb_segments is not 2^height"};
            DSA_LAUNCH("merge_scatter_root", k_merge_scatter_big, dim3(grid_for(nsegs * 32, 256), 1), 256, 0, st, A, L, (int64_t)1);
            if (hs[ST_NINS] > 0)
                DSA_LAUNCH("scatter_inserts_root", k_scatter_inserts, grid_for(hs[ST_NINS], 256), 256, 0, st, A, L, ws.status + ST_NINS);
            g = ng;
            leafcnt.ensure((size_t)g.nb_segments);
            DSA_LAUNCH("layout_gaps", k_layout, grid_for(g.capacity, 256), 256, 0, st, nk.p, nv.p, g.capacity, N,
                       (const int64_t*)nullptr, (const double*)nullptr, leafcnt.p, (int64_t*)nullptr, ilog2_i64(g.segment_capacity));
            DSA_CUDA(cudaStreamSynchronize(st));
            keys.swap(nk);
            vals.swap(nv);
        } else {
            const int64_t nhigh = hs[ST_NHIGH];
            // windows above leaf level: cover marks + the small ones re-laid through shared memory, one CTA each (before the leaf
            // merge, which skips covered leaves)
            if (nhigh > 0) {
                const int hmax = (int)std::min<int64_t>(std::max<int64_t>(hs[ST_MAXSMALLH], 1), L.hsmall);
                const int cells = (int)(g.segment_capacity << hmax);
                const int threads = std::min(256, std::max(64, cells / 2));
                DSA_LAUNCH("window_small", k_window_small, (unsigned)nhigh, threads, (size_t)cells * 16, st, A, L, cover, cells);
            }
            // leaves accepted at their own level (the common case), in place
            const int leaves_per_warp = 32 >> L.lgS;
            const int64_t nact = hs[ST_NACT];
            if (nact > 0) {
                const int64_t lm_warps = (nact + leaves_per_warp - 1) / leaves_per_warp;
                DSA_LAUNCH("leaf_merge", k_leaf_merge, grid_for(lm_warps * 32, 256), 256, 0, st, A, L);
            }
            // bigger windows (rare: cascades): warp-per-leaf scatter into the shadow array + copy back
            if (hs[ST_ANYBIG]) {
                A.dst_k = ws.shadow_k.ensure((size_t)g.capacity);
                A.dst_v = ws.shadow_v.ensure((size_t)g.capacity);
                A.big_h = ws.big_h.p;
                A.big_w = ws.big_w.p;
                const int64_t nbig = hs[ST_NBIG];
                // chunks per window: ~2 leaves per warp for the largest window of the batch
                // (and at most ~128k CTAs in all: many listed windows share the chunks of the largest one)
                const int64_t want_chunks = std::min<int64_t>(2048, std::max<int64_t>(1, (int64_t(1) << hs[ST_MAXBIGH]) / 16));
                const unsigned ychunks = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want_chunks, (int64_t(1) << 17) / nbig));
                const int64_t wy = std::min<int64_t>(nbig, 65535);   // grid.y limit: the windows go on in grid.z
                const dim3 grid(ychunks, (unsigned)wy, (unsigned)((nbig + wy - 1) / wy));
                DSA_LAUNCH("merge_scatter_big", k_merge_scatter_big, grid, 256, 0, st, A, L, nbig);
                if (hs[ST_NINS] > 0)
                    DSA_LAUNCH("scatter_inserts_big", k_scatter_inserts, grid_for(hs[ST_NINS], 256), 256, 0, st, A, L, ws.status + ST_NINS);
                DSA_LAUNCH("copyback_big", k_copyback_big, grid, 256, 0, st, A, L, nbig);
            }
        }
        nnz = N;
    }

    void prepare_batch_scratch(BatchWorkspace& ws, int64_t nops, cudaStream_t st) {
        const int64_t nsegs = g.nb_segments;
        ws.single_op = false;
        ws.op_pos.ensure((size_t)nops + 1);
        ws.op_flag.ensure((size_t)nops + 1);
        ws.ins_idx.ensure((size_t)nops + 1);
        ws.ins_key.ensure((size_t)nops + 1);
        ws.ins_val.ensure((size_t)nops + 1);
        ws.ins_pos.ensure((size_t)nops + 1);
        ws.ins_first.ensure((size_t)nsegs);
        const size_t tsz = ((size_t)tree_size() + 15) & ~(size_t)15;
        const size_t lsz = ((size_t)nsegs + 15) & ~(size_t)15;
        const size_t total = ST_WORDS * 8 + (size_t)nsegs * 4 + 16 + tsz + 2 * lsz;
        uint8_t* z = ws.zero_blk.ensure(total);
        ws.status = (int64_t*)z;
        ws.inscnt = (int32_t*)(z + ST_WORDS * 8);
        ws.mark = z + ST_WORDS * 8 + (((size_t)nsegs * 4 + 15) & ~(size_t)15);
        ws.touched = ws.mark + tsz;
        ws.cover = ws.touched + lsz;
        DSA_CUDA(cudaMemsetAsync(z, 0, total, st));
    }

    // sorted unique ops -> located, applied, merged.  op_pid/sem/next_sem nullable (plain PMA).
    void apply_sorted_ops(BatchWorkspace& ws, const int32_t* op_pid, const int64_t* op_key, const double* op_val, int64_t nops,
                          int64_t* d_sem, const int32_t* d_next_slot, cudaStream_t st, const int64_t* n_dev = nullptr,
                          bool launch_only = false) {
        prepare_batch_scratch(ws, nops, st);
        if (nops > 0) {
            const unsigned gr = grid_for(nops, 256);
            int32_t* f32 = ws.flag32.ensure((size_t)nops);
            DSA_LAUNCH("locate", k_locate, gr, 256, 0, st, keys.p, g.capacity, op_pid, op_key, op_val, nops, d_sem, d_next_slot,
                       ws.op_pos.p, ws.op_flag.p, n_dev, f32);
            apply_located_ops<true>(ws, op_key, op_val, nops, d_sem, st);
        }
        rebalance_launch(ws, st);
        if (!launch_only) {
            DSA_CUDA(cudaStreamSynchronize(st));
            rebalance_finish(ws, d_sem, st);
        }
    }

    // located ops (ws.op_pos / op_flag / flag32 = insert flags) -> hits applied, inserts compacted, per-leaf insert runs
    template <bool OVERWRITES>
    void apply_located_ops(BatchWorkspace& ws, const int64_t* op_key, const double* op_val, int64_t nops, int64_t* d_sem, cudaStream_t st) {
        const int lgS = ilog2_i64(g.segment_capacity);
        const unsigned gr = grid_for(nops, 256);
        ws.single_op = nops == 1;
        if (nops == 1)   // a single write keeps the reference's own layout (writes.jl:26-43)
            DSA_LAUNCH("single_insert", k_single_insert, 1, 32, 0, st, keys.p, vals.p, g.capacity, op_key, op_val, (const int64_t*)ws.op_pos.p,
                       ws.op_flag.p, ws.flag32.p, leafcnt.p, ws.touched, lgS, d_sem);
        {
            exclusive_scan_i32<int32_t>(ws.scan, ws.flag32.p, ws.ins_idx.p, nops, ws.status + ST_NINS, st);
            DSA_LAUNCH("apply_compact", k_apply_compact<OVERWRITES>, gr, 256, 0, st, keys.p, vals.p, op_key, op_val, ws.op_pos.p, ws.op_flag.p,
                       ws.ins_idx.p, nops, leafcnt.p, ws.touched, lgS, ws.ins_key.p, ws.ins_val.p, ws.ins_pos.p);
            ActiveLeaf* act = ws.act.ensure((size_t)std::min<int64_t>(nops, g.nb_segments) + 1);
            DSA_LAUNCH("insert_leaf_info", k_insert_leaf_info, gr, 256, 0, st, ws.ins_pos.p, ws.status + ST_NINS, ws.inscnt,
                       ws.ins_first.p, ws.touched, lgS, act, ws.status + ST_NACT);
        }
    }
};

}  // namespace dsa
