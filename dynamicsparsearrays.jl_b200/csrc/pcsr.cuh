// libdsa — partitioned PMA (PackedCSC + MappedPackedCSC, pcsr.jl) on the device: column map, batched set (K1..K5),
// bulk deletecolumn! (K5), column gather and the flat SpMV (K7).
#pragma once
#include <algorithm>
#include <type_traits>
#include <unordered_set>
#include "pma.cuh"
#include "sort.cuh"

namespace dsa {

// ---------------------------------------------------------------------------------------------
// column lookup: partition key -> slot (= partition id - 1) by binary search over the sorted live keys
// (find(mpcsc.col_keys, col), pcsr.jl:342 — tombstones are kept out of the searched list instead of being skipped)
// also reduces: #ops whose column is absent, min/max in-array key, max partition key / in-array key of non-zero writes
// ---------------------------------------------------------------------------------------------
enum { CS_MISSING = 0, CS_MINKEY = 1, CS_MAXKEY = 2, CS_MAXPART_NZ = 3, CS_MAXKEY_NZ = 4, CS_MINPART = 5, CS_MAXBUCKET = 6, CS_N = 7, CS_WORDS = 8 };

// The statistics block starts a batch as ZEROS (it shares the memset of the bucket counters): maxima are kept as
// order-preserving unsigned codes (0 = "none yet" = INT64_MIN), minima as the complement of the code (0 = INT64_MAX).
__host__ __device__ __forceinline__ unsigned long long cs_code(int64_t v) { return (unsigned long long)v ^ 0x8000000000000000ull; }
__host__ __device__ __forceinline__ int64_t cs_max_decode(int64_t stored) { return (int64_t)((unsigned long long)stored ^ 0x8000000000000000ull); }
__host__ __device__ __forceinline__ int64_t cs_min_decode(int64_t stored) { return (int64_t)(~(unsigned long long)stored ^ 0x8000000000000000ull); }

// grid of the (grid-stride) column lookup: one op per thread up to 16 CTAs per SM of a 148-SM part, then strided
inline unsigned lookup_grid(int64_t n) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, 148 * 16)); }

// index of the first a[i] >= key in the ascending a[0, n) (n if there is none)
template <typename T>
__device__ __forceinline__ int64_t lower_bound(const T* a, int64_t n, int64_t key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// The column map of an orientation as the kernels read it (Pcsr::colmap): partition key -> slot through the direct-address
// table when there is one (keymap != nullptr), else by binary search over the sorted live keys.  Which of the two a map has is
// decided by Pcsr::rebuild_live_and_upload.
struct ColMap {
    const int64_t* live_keys;   // ascending
    const int32_t* live_slot;
    int64_t nlive;
    const int32_t* keymap;      // nullable: keymap[key - keymap_min] = slot or -1
    int64_t keymap_min, keymap_len;

    // slot of the live partition with this key, -1 if there is none
    __device__ __forceinline__ int32_t slot(int64_t key) const {
        if (keymap) {
            const uint64_t r = (uint64_t)key - (uint64_t)keymap_min;   // any Int64 key: no signed overflow
            return r < (uint64_t)keymap_len ? keymap[r] : -1;
        }
        const int64_t i = lower_rank(key);
        return (i < nlive && live_keys[i] == key) ? live_slot[i] : -1;
    }
    // index of the first live key >= key (nlive if there is none)
    __device__ __forceinline__ int64_t lower_rank(int64_t key) const { return lower_bound(live_keys, nlive, key); }
};

// Grid-stride: the launch is sized from an upper bound when the op count only exists on the device (n_dev, distributed batches:
// the receive counts of the exchange are never read by the host before this kernel runs); cs[CS_N] reports the count used.
__global__ void __launch_bounds__(256, 6) k_col_lookup(const int64_t* __restrict__ partkeys, const int64_t* __restrict__ inkeys,
                                                     const double* __restrict__ vals, int64_t n_host, const int64_t* __restrict__ n_dev,
                                                     const ColMap cm, int32_t* __restrict__ op_slot, int64_t* __restrict__ cs,
                                                     int32_t* __restrict__ bcnt, int32_t* __restrict__ lidx) {
    int64_t n = n_host;
    if (n_dev) n = *n_dev < n_host ? *n_dev : n_host;
    if (blockIdx.x == 0 && threadIdx.x == 0) cs[CS_N] = n;
    int64_t mink = INT64_MAX, maxk = INT64_MIN, maxp = INT64_MIN, maxknz = INT64_MIN, minp = INT64_MAX;
    int miss = 0;
    int bmax = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pk = partkeys[i];
        minp = pk < minp ? pk : minp;
        const int32_t s = cm.slot(pk);
        op_slot[i] = s;
        miss += s < 0;
        if (bcnt && s >= 0) {   // bucket-sort bookkeeping: arrival-independent local index inside the partition's bucket
            const int li = atomicAdd(&bcnt[s], 1);
            lidx[i] = li;
            bmax = li + 1 > bmax ? li + 1 : bmax;
        }
        if (inkeys) {
            const int64_t k = inkeys[i];
            mink = k < mink ? k : mink;
            maxk = k > maxk ? k : maxk;
            if (vals && vals[i] != 0.0) {
                maxp = pk > maxp ? pk : maxp;
                maxknz = k > maxknz ? k : maxknz;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t a = __shfl_xor_sync(0xffffffffu, mink, o); mink = a < mink ? a : mink;
        a = __shfl_xor_sync(0xffffffffu, maxk, o); maxk = a > maxk ? a : maxk;
        a = __shfl_xor_sync(0xffffffffu, maxp, o); maxp = a > maxp ? a : maxp;
        a = __shfl_xor_sync(0xffffffffu, maxknz, o); maxknz = a > maxknz ? a : maxknz;
        a = __shfl_xor_sync(0xffffffffu, minp, o); minp = a < minp ? a : minp;
        miss += __shfl_xor_sync(0xffffffffu, miss, o);
        const int b2 = __shfl_xor_sync(0xffffffffu, bmax, o);
        bmax = b2 > bmax ? b2 : bmax;
    }
    // block-level combine, then one set of atomics per CTA
    __shared__ int64_t sh[5][8];
    __shared__ int shm[8], shb[8];
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        sh[0][wid] = mink; sh[1][wid] = maxk; sh[2][wid] = maxp; sh[3][wid] = maxknz; sh[4][wid] = minp;
        shm[wid] = miss;
        shb[wid] = bmax;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) {
            mink = sh[0][w] < mink ? sh[0][w] : mink;
            maxk = sh[1][w] > maxk ? sh[1][w] : maxk;
            maxp = sh[2][w] > maxp ? sh[2][w] : maxp;
            maxknz = sh[3][w] > maxknz ? sh[3][w] : maxknz;
            minp = sh[4][w] < minp ? sh[4][w] : minp;
            miss += shm[w];
            bmax = shb[w] > bmax ? shb[w] : bmax;
        }
        unsigned long long* u = (unsigned long long*)cs;
        if (bmax) atomicMax((long long*)&cs[CS_MAXBUCKET], (long long)bmax);
        if (miss) atomicAdd(&u[CS_MISSING], (unsigned long long)miss);
        if (mink != INT64_MAX) atomicMax(&u[CS_MINKEY], ~cs_code(mink));
        if (maxk != INT64_MIN) atomicMax(&u[CS_MAXKEY], cs_code(maxk));
        if (maxp != INT64_MIN) atomicMax(&u[CS_MAXPART_NZ], cs_code(maxp));
        if (maxknz != INT64_MIN) atomicMax(&u[CS_MAXKEY_NZ], cs_code(maxknz));
        if (minp != INT64_MAX) atomicMax(&u[CS_MINPART], ~cs_code(minp));
    }
}

// ops whose column is absent, minus immediate repeats of the same key (columns usually arrive as runs of entries): the
// host only needs every distinct absent key once, in first-arrival order
__device__ __forceinline__ bool missing_head(const int32_t* __restrict__ op_slot, const int64_t* __restrict__ partkeys, int64_t i) {
    return op_slot[i] < 0 && (i == 0 || partkeys[i - 1] != partkeys[i]);
}
__global__ void __launch_bounds__(256) k_flag_missing(const int32_t* __restrict__ op_slot, const int64_t* __restrict__ partkeys, int64_t n,
                                                       int32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = missing_head(op_slot, partkeys, i) ? 1 : 0;
}
__global__ void __launch_bounds__(256) k_compact_missing(const int32_t* __restrict__ op_slot, const int64_t* __restrict__ partkeys,
                                                          const int32_t* __restrict__ idx, int64_t n, int64_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && missing_head(op_slot, partkeys, i)) out[idx[i]] = partkeys[i];
}

// renumbering after new columns: partition ids are slot indices; moved semaphore cells get their new id (pcsr.jl:128-134)
__global__ void __launch_bounds__(256) k_renumber(const int64_t* __restrict__ old_sem, const int32_t* __restrict__ old2new, int64_t nold,
                                                   int64_t* __restrict__ new_sem, double* __restrict__ vals) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nold) return;
    const int64_t pos = old_sem[s];
    const int32_t t = old2new[s];
    if (pos < 0 || t < 0) return;
    new_sem[t] = pos;
    if (t != s) vals[pos] = (double)(t + 1);
}
__global__ void __launch_bounds__(256) k_fill_i64(int64_t* a, int64_t n, int64_t v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}

// ---------------------------------------------------------------------------------------------
// batch assembly: ops + one semaphore insert per new partition; 64-bit sort key = (slot << kb) | (in-array key - kmin + 1), so
// that kb follows the batch's key range, not its largest key
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_make_sortkeys(const int32_t* __restrict__ op_slot, const int64_t* __restrict__ inkeys, int64_t n,
                                                        const int32_t* __restrict__ new_slots, int64_t nnew, int64_t kmin, int kb,
                                                        uint64_t* __restrict__ sk, uint32_t* __restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        sk[i] = ((uint64_t)(uint32_t)op_slot[i] << kb) | ((uint64_t)inkeys[i] - (uint64_t)kmin + 1);
        idx[i] = (uint32_t)i;
    } else if (i < n + nnew) {
        sk[i] = ((uint64_t)(uint32_t)new_slots[i - n] << kb);   // key 0 = semaphore key: sorts first in its partition
        idx[i] = (uint32_t)i;
    }
}
// ---------------------------------------------------------------------------------------------
// Bucket path of K1 (batches whose partitions each receive few ops): ops are dropped into their partition's bucket
// (offsets = exclusive scan of the per-partition counts taken during the column lookup), then every op ranks itself
// inside its bucket by (key, arrival).  Same output as the radix sort — ops ordered by (partition, key), equal keys in
// arrival order — in 3 small kernels instead of 5 passes over 64-bit keys.
// ---------------------------------------------------------------------------------------------
struct __align__(16) BucketRec {
    int64_t key;
    uint32_t arr;
    int32_t slot;
};
__global__ void __launch_bounds__(256) k_bucket_scatter(const int32_t* __restrict__ op_slot, const int32_t* __restrict__ lidx,
                                                         const int64_t* __restrict__ inkeys, int64_t n, const int32_t* __restrict__ boff,
                                                         BucketRec* __restrict__ rec) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t s = op_slot[i];
    const int64_t pos = (int64_t)boff[s] + lidx[i];
    rec[pos] = BucketRec{inkeys[i], (uint32_t)i, s};   // one 16 B store per op
}
// Every op ranks itself inside its bucket by (key, arrival) — its index in the batch's (partition, key, arrival) order — and is
// LOCATED right there (K6, finds.jl:29-57 inside the partition span): the sorted op, its position, its flag and its insert flag
// land at the sorted index.  An op followed by a later write to the same (partition, key) is dead (last writer wins).
// Overwrites store their value at once (a search reads keys only); deletes are applied by k_apply_compact, after every op
// of the batch has been located.
__global__ void __launch_bounds__(256, 8) k_bucket_rank_locate(const BucketRec* __restrict__ rec, const int32_t* __restrict__ boff,
                                                             const int32_t* __restrict__ bcnt, int64_t n, const double* __restrict__ vals,
                                                             const int64_t* __restrict__ keys, double* __restrict__ cell_vals, int64_t cap,
                                                             const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot,
                                                             int64_t* __restrict__ u_key, double* __restrict__ u_val,
                                                             int64_t* __restrict__ op_pos, uint8_t* __restrict__ op_flag,
                                                             int32_t* __restrict__ ins_flag) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const BucketRec me = rec[p];
    const double val = vals[me.arr];
    const int64_t lo = boff[me.slot], hi = lo + bcnt[me.slot];
    int64_t r = lo;
    bool dead = false;
    for (int64_t q = lo; q < hi; ++q) {
        const BucketRec o = rec[q];
        r += (o.key < me.key) || (o.key == me.key && o.arr < me.arr);
        dead |= (o.key == me.key && o.arr > me.arr);
    }
    uint8_t f = 0;
    if (!dead) {
        int64_t pos;
        f = locate_one(keys, cap, true, me.slot, me.key, val != 0.0, sem, next_slot, &pos);
        op_pos[r] = pos;
        if (f == FL_OVERWRITE) cell_vals[pos] = val;   // writes.jl:16-19
        u_key[r] = me.key;
        u_val[r] = val;
    }
    op_flag[r] = f;
    ins_flag[r] = f == FL_INSERT ? 1 : 0;
}

// plain PMA: sort key = key - min
__global__ void __launch_bounds__(256) k_make_sortkeys_vec(const int64_t* __restrict__ keys, int64_t n, int64_t mink,
                                                            uint64_t* __restrict__ sk, uint32_t* __restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        sk[i] = (uint64_t)(keys[i] - mink);
        idx[i] = (uint32_t)i;
    }
}
// last writer wins: keep the last element of every run of equal sort keys (stable sort => last in arrival order)
__global__ void __launch_bounds__(256) k_flag_run_last(const uint64_t* __restrict__ sk, int64_t n, int32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = (i == n - 1 || sk[i] != sk[i + 1]) ? 1 : 0;
}
__global__ void __launch_bounds__(256) k_gather_unique_ops(const uint64_t* __restrict__ sk, const uint32_t* __restrict__ perm,
                                                            const int32_t* __restrict__ flag, const int32_t* __restrict__ uidx, int64_t ntot,
                                                            int64_t n, int kb, const int64_t* __restrict__ inkeys,
                                                            const double* __restrict__ vals, int32_t* __restrict__ u_pid,
                                                            int64_t* __restrict__ u_key, double* __restrict__ u_val) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ntot || !flag[i]) return;
    const int32_t j = uidx[i];
    const uint32_t src = perm[i];
    const int32_t slot = (int32_t)(sk[i] >> kb);
    if (u_pid) u_pid[j] = slot;
    if ((int64_t)src < n) {
        u_key[j] = inkeys[src];
        u_val[j] = vals[src];
    } else {   // semaphore of a new partition: (key 0, T(partition id))   pcsr.jl:39-40
        u_key[j] = 0;
        u_val[j] = (double)(slot + 1);
    }
}

// ---------------------------------------------------------------------------------------------
// builders: duplicate-combine as a left fold in input order (vector.jl:21-31, pcsr.jl:373-398): the head of every run of
// equal sort keys folds its run sequentially (stable sort => input order)
// ---------------------------------------------------------------------------------------------
// min / max are Base.min / Base.max on IEEE floats: NaN if either argument is NaN (the NaN argument itself, as x86 returns it
// from the `x - y` Base computes), -0.0 orders below 0.0, otherwise the smaller / larger argument
__device__ __forceinline__ double julia_min(double a, double b) {
    if (isnan(a)) return a;
    if (isnan(b)) return b;
    if (a == b) return signbit(a) ? a : b;
    return b < a ? b : a;
}
__device__ __forceinline__ double julia_max(double a, double b) {
    if (isnan(a)) return a;
    if (isnan(b)) return b;
    if (a == b) return signbit(a) ? b : a;
    return b > a ? b : a;
}
__device__ __forceinline__ double combine_apply(int c, double a, double b) {
    switch (c) {
        case DSA_COMBINE_ADD: return __dadd_rn(a, b);
        case DSA_COMBINE_MUL: return __dmul_rn(a, b);
        case DSA_COMBINE_LAST: return b;
        case DSA_COMBINE_FIRST: return a;
        case DSA_COMBINE_MIN: return julia_min(a, b);
        case DSA_COMBINE_MAX: return julia_max(a, b);
    }
    return __dadd_rn(a, b);
}
__global__ void __launch_bounds__(256) k_flag_run_first(const uint64_t* __restrict__ sk, int64_t n, int32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = (i == 0 || sk[i] != sk[i - 1]) ? 1 : 0;
}
// second-level run heads for the matrix builder: first element of every partition (column) in the sorted unique stream
__global__ void __launch_bounds__(256) k_flag_part_first(const uint64_t* __restrict__ sk_hi, int64_t n, const int32_t* __restrict__ runflag,
                                                          int32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = (runflag[i] && (i == 0 || sk_hi[i] != sk_hi[i - 1])) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// K5 bulk deletecolumn!: spans of the deleted partitions
// ---------------------------------------------------------------------------------------------
// count the stored cells of (sem, next_sem) per listed slot — one warp per slot
__global__ void __launch_bounds__(256) k_span_count(const int64_t* __restrict__ keys, const int32_t* __restrict__ slots, int64_t nslots,
                                                     const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot, int64_t cap,
                                                     int32_t* __restrict__ counts) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= nslots) return;
    const int32_t s = slots[w];
    const int64_t from = sem[s] + 1, to = span_end(sem, next_slot, s, cap);
    int c = 0;
    for (int64_t p = from + lane; p < to; p += 32) c += keys[p] != GAP_KEY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) counts[w] = c;
}
// emit the stored cells of the span in order (views.jl:15-35 / pcsr.jl:248-258): (key, val) and the owning list index
__global__ void __launch_bounds__(256) k_span_emit(const int64_t* __restrict__ keys, const double* __restrict__ vals,
                                                    const int32_t* __restrict__ slots, int64_t nslots, const int64_t* __restrict__ sem,
                                                    const int32_t* __restrict__ next_slot, int64_t cap, const int32_t* __restrict__ offsets,
                                                    int64_t* __restrict__ out_key, double* __restrict__ out_val,
                                                    int64_t* __restrict__ out_owner, const int64_t* __restrict__ owner_keys) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= nslots) return;
    const int32_t s = slots[w];
    const int64_t from = sem[s] + 1, to = span_end(sem, next_slot, s, cap);
    int64_t o = offsets[w];
    for (int64_t base = from; base < to; base += 32) {
        const int64_t p = base + lane;
        const bool live = p < to && keys[p] != GAP_KEY;
        const unsigned b = __ballot_sync(0xffffffffu, live);
        if (live) {
            const int64_t d = o + __popc(b & lanemask_lt());
            out_key[d] = keys[p];
            if (out_val) out_val[d] = vals[p];
            if (out_owner) out_owner[d] = owner_keys[w];
        }
        o += __popc(b);
    }
}
// purge! (writes.jl:80-92) of [sem, next_sem) for every listed slot + leaf bookkeeping
__global__ void __launch_bounds__(256) k_span_purge(int64_t* __restrict__ keys, double* __restrict__ vals, const int32_t* __restrict__ slots,
                                                     int64_t nslots, const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot, int64_t cap,
                                                     int32_t* __restrict__ leafcnt, uint8_t* __restrict__ touched, int lgS) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= nslots) return;
    const int32_t s = slots[w];
    const int64_t from = sem[s], to = span_end(sem, next_slot, s, cap);
    for (int64_t p = from + lane; p < to; p += 32) {
        if (keys[p] != GAP_KEY) {
            keys[p] = GAP_KEY;
            vals[p] = 0.0;
            atomicSub(&leafcnt[p >> lgS], 1);
            touched[p >> lgS] = 1;
        }
    }
}
__global__ void __launch_bounds__(256) k_clear_sems(int64_t* __restrict__ sem, const int32_t* __restrict__ slots, int64_t nslots) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nslots) sem[slots[i]] = -1;
}

// ---------------------------------------------------------------------------------------------
// K7 SpMV over the gapped array — cell-parallel, deterministic.
// y[key(partition)] = sum over the partition's cells of x[cell key] * cell value, cells in ascending key order, i.e. the
// per-output summation order of _mul_dyn_mat_col_loop! (operations.jl:97-103) when the twin orientation is scanned.
// A warp streams a chunk of consecutive cells, does a segmented reduction with the semaphore cells as in-band segment heads,
// writes every partition that ends inside the chunk, and leaves (a) the partial of the cells before its first head in
// carry[chunk] and (b) the open partial of its last partition in y.  k_spmv_fixup then adds, per chunk with a head, the
// carries of the following head-less chunks in chunk order.  No atomics: the result is bit-reproducible.  mul and add are
// separate roundings (no FMA), as in the reference.
// ---------------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------
// Every lane owns C CONTIGUOUS cells (one 256-bit load of keys, one of values, both L1::no_allocate so that x keeps the L1),
// reduces them sequentially — heads inside the lane close their partition in registers — and the warp then needs ONE
// segmented scan over the 32 lane aggregates per chunk, whatever the number of heads (13 shuffles per 32*C cells; round 1's
// strided kernel paid ~40 per 32-cell step with a head and ran at 83 us on the same data, profiles/gather_probe.cu).
// The C gathers of x are UNCONDITIONAL loads (gap / head lanes read x[0]): a gather under a data-dependent branch is followed
// by a reconvergence point, which serialised the four L2 round trips of a lane (73 us -> see profiles/).
// Per-partition order = ascending cells; association: sequential inside a lane, tree across lanes (within the 1e-12 bar,
// exact for integer-valued data).
// ---------------------------------------------------------------------------------------------
// The big streams (the gapped arrays: 2 x 268 MB per matrix against 126 MB of L2) are loaded with an evict-first L2 policy so that
// the small random-access tables (semaphore positions, column map, x, tile counters and buckets) stay resident between kernels.
#ifndef DSA_L2_EVICT_FIRST
#define DSA_L2_EVICT_FIRST 1
#endif
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void ldg_stream4(const int64_t* p, int64_t& a, int64_t& b, int64_t& c, int64_t& d, uint64_t pol) {
#if DSA_L2_EVICT_FIRST
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s64 {%0,%1,%2,%3}, [%4], %5;" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p), "l"(pol));
#else
    asm volatile("ld.global.nc.L1::no_allocate.v4.s64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
#endif
}
__device__ __forceinline__ void ldg_stream4(const double* p, double& a, double& b, double& c, double& d, uint64_t pol) {
#if DSA_L2_EVICT_FIRST
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p), "l"(pol));
#else
    asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
#endif
}
__device__ __forceinline__ longlong2 ldg_stream2(const longlong2* p, uint64_t pol) {
    longlong2 r;
#if DSA_L2_EVICT_FIRST
    asm volatile("ld.global.L2::cache_hint.v2.s64 {%0,%1}, [%2], %3;" : "=l"(r.x), "=l"(r.y) : "l"(p), "l"(pol));
#else
    r = *p;
#endif
    return r;
}

// A lane's C contiguous cells [p0, p0 + C) of the gapped arrays: 256-bit evict-first loads of keys and of values, cells at or
// past cap read as gaps.  vals = nullptr: keys only (t is not written).
template <int C, typename V>
__device__ __forceinline__ void load_cells(const int64_t* keys, V vals, int64_t cap, int64_t p0, int64_t (&k)[C], double (&t)[C],
                                           uint64_t pol) {
    static_assert(C % 4 == 0, "a lane loads its cells in groups of 4 (256 bits)");
    constexpr bool VALS = !std::is_same<V, std::nullptr_t>::value;
#pragma unroll
    for (int c = 0; c < C; c += 4) {
        if (p0 + c + 4 <= cap) {
            ldg_stream4(keys + p0 + c, k[c], k[c + 1], k[c + 2], k[c + 3], pol);
            if constexpr (VALS) ldg_stream4(vals + p0 + c, t[c], t[c + 1], t[c + 2], t[c + 3], pol);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t p = p0 + c + e;
                k[c + e] = p < cap ? keys[p] : GAP_KEY;
                if constexpr (VALS) t[c + e] = p < cap ? vals[p] : 0.0;
            }
        }
    }
}

// XMODE: 0 = dense x (x[key - 1], every entry stored); 1 = dense x + presence mask (a sparse x scattered into a dense buffer);
// 2 = sparse x looked up by binary search in its ascending key list (xkeys[nx], x = the matching values): for key spaces far
// larger than the number of entries (ids around 1e10 through a key codec), where a dense buffer would not fit.
template <int XMODE, int C>
__global__ void __launch_bounds__(256) k_spmv_blocked(const int64_t* __restrict__ keys, const double* __restrict__ vals, int64_t cap,
                                                       const double* __restrict__ x, const uint8_t* __restrict__ xmask,
                                                       const int64_t* __restrict__ xkeys, int64_t nx,
                                                       double* __restrict__ yslot, int32_t* __restrict__ ycnt,
                                                       double* __restrict__ carry, int32_t* __restrict__ carry_cnt,
                                                       int32_t* __restrict__ chunk_last_slot, int64_t nchunks) {
    const int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (chunk >= nchunks) return;
    const unsigned lt = lanemask_lt();
    const uint64_t l2pol = l2_evict_first_policy();
    const int64_t p0 = chunk * (32 * C) + (int64_t)lane * C;
    int64_t k[C];
    double t[C];
    load_cells(keys, vals, cap, p0, k, t, l2pol);
    // the C gathers of x: independent, branch-free, all in flight together.  t = x[key] * value (separate rounding,
    // operations.jl:101); heads keep their value (the partition id) in t
    double xv[C];
    uint8_t xm[C];
    int tcn[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        xv[c] = 0.0;
        xm[c] = 1;
    }
    constexpr bool SPARSE_X = XMODE != 0;
    if (nx > 0 && XMODE != 2) {   // warp-uniform
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int64_t kk = k[c];
            const int64_t idx = (kk > 0 && kk <= nx) ? kk - 1 : 0;
            xv[c] = __ldg(x + idx);
            if (XMODE == 1) xm[c] = __ldg(xmask + idx);
        }
    }
    if (XMODE == 2) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int64_t kk = k[c];
            xm[c] = 0;
            if (kk > 0) {
                const int64_t lo = lower_bound(xkeys, nx, kk);
                if (lo < nx && __ldg(xkeys + lo) == kk) {
                    xm[c] = 1;
                    xv[c] = __ldg(x + lo);
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int64_t kk = k[c];
        const bool present = kk > 0 && (XMODE == 2 || kk <= nx) && xm[c] != 0;
        tcn[c] = present ? 1 : 0;
        if (kk > 0) t[c] = present ? __dmul_rn(xv[c], t[c]) : 0.0;
    }
    // sequential reduction of the lane's cells
    double run = 0.0, pre = 0.0;   // run: sum since the lane's last head (or lane start); pre: cells before its first head
    int runc = 0, prec = 0;
    bool has_head = false;
    int32_t lastslot = -1;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        if (k[c] == 0) {
            if (!has_head) {
                pre = run;
                prec = runc;
            } else {   // a whole partition inside this lane
                yslot[lastslot] = run;
                if (SPARSE_X) ycnt[lastslot] = runc;
            }
            has_head = true;
            lastslot = (int32_t)t[c] - 1;
            run = 0.0;
            runc = 0;
        } else if (k[c] > 0) {
            run = __dadd_rn(run, t[c]);
            runc += tcn[c];
        }
    }
    // segmented inclusive scan over the lanes: a lane with a head starts a new segment with its tail (run)
    const unsigned hb = __ballot_sync(0xffffffffu, has_head);
    const unsigned hle = hb & (lt | (1u << lane));
    const int seg_lo = hle ? 31 - __clz(hle) : 0;
    double inc = run;
    int incc = runc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(0xffffffffu, inc, o);
        int uc = 0;
        if (SPARSE_X) uc = __shfl_up_sync(0xffffffffu, incc, o);
        if (lane >= o && lane - o >= seg_lo) {
            inc = __dadd_rn(u, inc);
            incc += uc;
        }
    }
    double cin = __shfl_up_sync(0xffffffffu, inc, 1);   // open partition's partial over the lanes before this one
    int cinc = 0;
    if (SPARSE_X) cinc = __shfl_up_sync(0xffffffffu, incc, 1);
    if (lane == 0) {
        cin = 0.0;
        cinc = 0;
    }
    const unsigned hlt = hb & lt;
    const int32_t prev_slot = __shfl_sync(0xffffffffu, lastslot, hlt ? 31 - __clz(hlt) : 0);
    if (has_head) {   // this lane's first head closes the partition that was open before it
        const double tot = __dadd_rn(cin, pre);
        const int totc = cinc + prec;
        if (hlt) {
            yslot[prev_slot] = tot;
            if (SPARSE_X) ycnt[prev_slot] = totc;
        } else {   // it started in an earlier chunk: the fix-up adds this prefix to that chunk's open partition
            carry[chunk] = tot;
            if (SPARSE_X) carry_cnt[chunk] = totc;
        }
    }
    const int32_t end_slot = __shfl_sync(0xffffffffu, lastslot, hb ? 31 - __clz(hb) : 0);
    if (lane == 31) {
        if (hb) {   // open partition at the end of the chunk: partial, completed by the fix-up
            yslot[end_slot] = inc;
            if (SPARSE_X) ycnt[end_slot] = incc;
            chunk_last_slot[chunk] = end_slot;
        } else {    // no head in the whole chunk
            carry[chunk] = inc;
            if (SPARSE_X) carry_cnt[chunk] = incc;
            chunk_last_slot[chunk] = -1;
        }
    }
}

// The carry walk that completes the partition open at the end of chunk c: a + carry[c + 1] + carry[c + 2] + ..., in chunk order,
// up to and including the first chunk that has a head.  Column col's carries lie at carry[chunk * W + col].  cnt (nullable): the
// product counts carry_cnt of the same chunks are added to *cnt.
__device__ __forceinline__ double add_following_carries(double a, const double* __restrict__ carry, const int32_t* __restrict__ chunk_last_slot,
                                                        int64_t c, int64_t nchunks, int64_t W, int64_t col,
                                                        const int32_t* __restrict__ carry_cnt = nullptr, int32_t* cnt = nullptr) {
    for (int64_t d = c + 1; d < nchunks; ++d) {
        a = __dadd_rn(a, carry[d * W + col]);
        if (cnt) *cnt += carry_cnt[d];
        if (chunk_last_slot[d] >= 0) break;
    }
    return a;
}

// sparse output: per chunk c with a head, the last partition of c is completed by the carry walk, product counts included
__global__ void __launch_bounds__(256) k_spmv_fixup(double* __restrict__ yslot, int32_t* __restrict__ ycnt, const double* __restrict__ carry,
                                                     const int32_t* __restrict__ carry_cnt, const int32_t* __restrict__ chunk_last_slot,
                                                     int64_t nchunks) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchunks) return;
    const int32_t slot = chunk_last_slot[c];
    if (slot < 0) return;
    if (c + 1 >= nchunks) return;
    double a = yslot[slot];
    int32_t n = ycnt[slot];
    a = add_following_carries(a, carry, chunk_last_slot, c, nchunks, 1, 0, carry_cnt, &n);
    yslot[slot] = a;
    ycnt[slot] = n;
}

// ---------------------------------------------------------------------------------------------
// K7b multi-vector product Y = A * X over the gapped array, for one pass of 4 * ngroups columns of a row-major X (row stride
// ldx % 4 == 0, 32-byte aligned base).  Bit for bit, column c is k_spmv_blocked<0, C> + the epilogue (W = 1) on column c alone:
// the same 32 * C-cell chunk per warp, the same C contiguous cells per lane summed sequentially, the same segmented scan over
// the lane aggregates (same shuffle order), the same carries added in chunk order by the epilogue, mul and add rounded
// separately.  What is shared: the keys / values are streamed once for all columns, and a cell's x becomes one 256-bit load of
// 4 consecutive entries of its row of X per column group instead of one 8-byte gather per vector.  Column groups run one after
// the other inside the warp, so the registers a group needs do not grow with the pass width.
// Partials: yslot[slot * W + col], carry[chunk * W + col] with W = 4 * ngroups; chunk_last_slot as in k_spmv_blocked.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldg_x4(const double* p, double& a, double& b, double& c, double& d) {
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}

template <int C>
__global__ void __launch_bounds__(256) k_spmm_blocked(const int64_t* __restrict__ keys, const double* __restrict__ vals, int64_t cap,
                                                       const double* __restrict__ X, int64_t nx, int64_t ldx, int ngroups,
                                                       double* __restrict__ yslot, double* __restrict__ carry,
                                                       int32_t* __restrict__ chunk_last_slot, int64_t nchunks) {
    const int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (chunk >= nchunks) return;
    const unsigned lt = lanemask_lt();
    const uint64_t l2pol = l2_evict_first_policy();
    const int64_t p0 = chunk * (32 * C) + (int64_t)lane * C;
    int64_t k[C];
    double t[C];
    load_cells(keys, vals, cap, p0, k, t, l2pol);
    // the segment structure of the chunk is the same for every column
    bool has_head = false;
    int32_t lastslot = -1;
#pragma unroll
    for (int c = 0; c < C; ++c)
        if (k[c] == 0) {
            has_head = true;
            lastslot = (int32_t)t[c] - 1;
        }
    const unsigned hb = __ballot_sync(0xffffffffu, has_head);
    const unsigned hle = hb & (lt | (1u << lane));
    const int seg_lo = hle ? 31 - __clz(hle) : 0;
    const unsigned hlt = hb & lt;
    const int32_t prev_slot = __shfl_sync(0xffffffffu, lastslot, hlt ? 31 - __clz(hlt) : 0);
    const int32_t end_slot = __shfl_sync(0xffffffffu, lastslot, hb ? 31 - __clz(hb) : 0);
    if (lane == 31) chunk_last_slot[chunk] = hb ? end_slot : -1;
    const int64_t W = 4 * (int64_t)ngroups;
#pragma unroll 1
    for (int g = 0; g < ngroups; ++g) {
        // the C row loads of x: independent, branch-free, all in flight together (gap / head lanes read row 0)
        double xv[C][4];
#pragma unroll
        for (int c = 0; c < C; ++c)
#pragma unroll
            for (int j = 0; j < 4; ++j) xv[c][j] = 0.0;
        if (nx > 0) {   // warp-uniform
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const int64_t kk = k[c];
                const int64_t idx = (kk > 0 && kk <= nx) ? kk - 1 : 0;
                ldg_x4(X + idx * ldx + 4 * g, xv[c][0], xv[c][1], xv[c][2], xv[c][3]);
            }
        }
        // sequential reduction of the lane's cells, per column
        double run[4] = {0.0, 0.0, 0.0, 0.0}, pre[4] = {0.0, 0.0, 0.0, 0.0};
        bool seen = false;
        int32_t open = -1;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int64_t kk = k[c];
            if (kk == 0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (!seen) pre[j] = run[j];
                    else yslot[open * W + 4 * g + j] = run[j];   // a whole partition inside this lane
                    run[j] = 0.0;
                }
                seen = true;
                open = (int32_t)t[c] - 1;
            } else if (kk > 0) {
                const bool present = kk <= nx;
#pragma unroll
                for (int j = 0; j < 4; ++j) run[j] = __dadd_rn(run[j], present ? __dmul_rn(xv[c][j], t[c]) : 0.0);
            }
        }
        // segmented inclusive scan over the lanes, per column
        double inc[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) inc[j] = run[j];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double u = __shfl_up_sync(0xffffffffu, inc[j], o);
                if (lane >= o && lane - o >= seg_lo) inc[j] = __dadd_rn(u, inc[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double cin = __shfl_up_sync(0xffffffffu, inc[j], 1);
            if (lane == 0) cin = 0.0;
            const int64_t col = 4 * g + j;
            if (has_head) {   // this lane's first head closes the partition that was open before it
                const double tot = __dadd_rn(cin, pre[j]);
                if (hlt) yslot[prev_slot * W + col] = tot;
                else carry[chunk * W + col] = tot;   // it started in an earlier chunk: the epilogue adds this prefix
            }
            if (lane == 31) {
                if (hb) yslot[end_slot * W + col] = inc[j];   // open partition at the end of the chunk: completed by the epilogue
                else carry[chunk * W + col] = inc[j];         // no head in the whole chunk
            }
        }
    }
}

// Dense-output epilogue of the products in ONE kernel, driven by slot: thread (slot, col) of a pass of W columns completes the
// slot's partial with the carry walk (the additions of k_spmv_fixup, in the same order) and scatters it by partition key to
// Y[(key - key_lo) * ldy + col] for col < ncols.  A slot is the last head of its chunk iff its span reaches the chunk's end.
// ONE: the single-vector product, W = ncols = ldy = 1 as constants (no division, no column arithmetic).
template <bool ONE>
__global__ void __launch_bounds__(256) k_spmm_fix_to_dense(const double* __restrict__ yslot, const double* __restrict__ carry,
                                                            const int32_t* __restrict__ chunk_last_slot, const int64_t* __restrict__ sem,
                                                            const int32_t* __restrict__ next_slot, const int64_t* __restrict__ slot_key,
                                                            int64_t nslots, int64_t cap, int64_t nchunks, int lg_chunk, int W, int ncols,
                                                            double* __restrict__ Y, int64_t ldy, int64_t key_lo, int64_t key_hi) {
    if (ONE) {
        W = ncols = 1;
        ldy = 1;
    }
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t s = i / W;
    const int col = (int)(i - s * W);
    if (s >= nslots || col >= ncols) return;
    const int64_t ps = sem[s];
    if (ps < 0) return;
    const int64_t k = slot_key[s];
    if (k < key_lo || k >= key_hi) return;   // Y holds the partition keys [key_lo, key_hi)
    double a = yslot[s * W + col];
    const int64_t c0 = ps >> lg_chunk;
    if (span_end(sem, next_slot, (int32_t)s, cap) >= ((c0 + 1) << lg_chunk))
        a = add_following_carries(a, carry, chunk_last_slot, c0, nchunks, W, col);
    Y[(k - key_lo) * ldy + col] = a;
}

// touched partitions (at least one product) for the sparse output (operations.jl:11-12, sparsevec(::Dict, n))
__global__ void __launch_bounds__(256) k_flag_touched(const int32_t* __restrict__ ycnt, const int64_t* __restrict__ sem, int64_t nslots,
                                                       int32_t* __restrict__ flag) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < nslots) flag[s] = (sem[s] >= 0 && ycnt[s] > 0) ? 1 : 0;
}
__global__ void __launch_bounds__(256) k_compact_y(const double* __restrict__ yslot, const int64_t* __restrict__ slot_key,
                                                    const int32_t* __restrict__ flag, const int32_t* __restrict__ idx, int64_t nslots,
                                                    int64_t* __restrict__ yk, double* __restrict__ yv) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < nslots && flag[s]) {
        yk[idx[s]] = slot_key[s];
        yv[idx[s]] = yslot[s];
    }
}
__global__ void __launch_bounds__(256) k_scatter_x(const int64_t* __restrict__ xk, const double* __restrict__ xv, int64_t n,
                                                    double* __restrict__ x, uint8_t* __restrict__ xmask, int64_t nx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int64_t k = xk[i];
        if (k >= 1 && k <= nx) {
            x[k - 1] = xv[i];
            xmask[k - 1] = 1;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K8 compressed snapshot: order-preserving compaction of the element cells of an orientation (gaps and semaphore cells
// dropped) = canonical CSC of the column-major twin / CSR of the row-major one, because partitions lie in the array in
// ascending key order and cells in ascending in-array key inside a partition (iterate, pma.jl:165-180; the column / row
// gathers of pcsr.jl:234-291 for every partition at once).  A vector keeps every non-gap cell (nonzeros, vector.jl:93-109).
// Stream compaction with in-band segment heads, bound by HBM, in two passes over the keys:
//   count  one warp per 256-cell chunk, 8 contiguous cells per lane (256-bit loads): element count per CTA tile of 2048 cells,
//          and (dense form, when the host cannot rule it out) the bounds flag
//   scan   int64 offsets of the tiles: exclusive scan inside blocks of 8192 tiles + the block totals (an emitting CTA adds the
//          totals of the blocks before its own): no 32-bit count anywhere, a 2^31-cell orientation can hold > 2^31 entries
//   emit   same chunks: a lane ranks its elements with a warp scan on top of the tile offset and the counts of the warps before
//          it, stages them in shared memory at their rank, and the warp writes its contiguous output range coalesced.  A lane
//          that meets a semaphore cell (value = partition id = slot + 1) writes ptr[live_rank[slot]] = rank of the next element.
// ---------------------------------------------------------------------------------------------
constexpr int CMP_C = 8;                                  // cells per lane
constexpr int CMP_WARPS = 8;                              // warps per CTA
constexpr int CMP_TILE = 32 * CMP_C * CMP_WARPS;          // cells per CTA tile
constexpr int CMP_STAGE = 32 * CMP_C + 32 * CMP_C / 8;    // staging slots per warp: rank r at r + r / 8 (no 16-way bank conflicts)
constexpr int CMP_SCAN_THREADS = 1024, CMP_SCAN_ITEMS = 8, CMP_LG_SCAN_BLOCK = 13;   // tiles per scan block = 1024 x 8
static_assert(CMP_SCAN_THREADS * CMP_SCAN_ITEMS == 1 << CMP_LG_SCAN_BLOCK, "scan block");

// matrices: in-array keys are >= 1 (0 = semaphore); vectors: any key but the gap sentinel
template <bool SEMS>
__device__ __forceinline__ bool cmp_elem(int64_t k) { return SEMS ? k > 0 : k != GAP_KEY; }

// Warp-collective, every lane gets it: the sum of the scan-block totals blk_sum[0 .. q >> CMP_LG_SCAN_BLOCK), which turns item
// q's offset inside its scan block (k_compress_scan) into its global offset.  lane: the caller's threadIdx.x & 31.
__device__ __forceinline__ int64_t scan_block_base(const int64_t* __restrict__ blk_sum, int64_t q, int lane) {
    int64_t a = 0;
    for (int64_t b = lane; b < (q >> CMP_LG_SCAN_BLOCK); b += 32) a += blk_sum[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    return a;
}

// bound_flag (nullable): set when an element lies at or after position sem[bound_slot] (bound_slot = the first live partition
// whose key exceeds the dense dimension: every partition after it in the array has a larger key; -1 = none) or has an
// in-array key > idim
template <bool SEMS>
__global__ void __launch_bounds__(256) k_compress_count(const int64_t* __restrict__ keys, int64_t cap, int32_t* __restrict__ tile_cnt,
                                                         const int64_t* __restrict__ sem, int32_t bound_slot, int64_t idim,
                                                         int32_t* __restrict__ bound_flag) {
    __shared__ int32_t wc[CMP_WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t p0 = (int64_t)blockIdx.x * CMP_TILE + (int64_t)wid * (32 * CMP_C) + (int64_t)lane * CMP_C;
    int64_t k[CMP_C];
    double unused[CMP_C];   // keys only
    load_cells(keys, nullptr, cap, p0, k, unused, l2_evict_first_policy());
    int cnt = 0;
#pragma unroll
    for (int c = 0; c < CMP_C; ++c) cnt += cmp_elem<SEMS>(k[c]) ? 1 : 0;
    if (bound_flag) {   // uniform
        const int64_t pdim = bound_slot >= 0 ? sem[bound_slot] : INT64_MAX;
        bool over = false;
#pragma unroll
        for (int c = 0; c < CMP_C; ++c) over |= cmp_elem<SEMS>(k[c]) && (p0 + c >= pdim || k[c] > idim);
        if (__any_sync(0xffffffffu, over) && lane == 0) atomicOr(bound_flag, 1);
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) wc[wid] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
#pragma unroll
        for (int w = 0; w < CMP_WARPS; ++w) s += wc[w];
        tile_cnt[blockIdx.x] = s;
    }
}

// tile_off[t] = sum of the counts of the tiles before t in its scan block; blk_sum[b] = total of scan block b
__global__ void __launch_bounds__(CMP_SCAN_THREADS) k_compress_scan(const int32_t* __restrict__ tile_cnt, int64_t ntiles,
                                                                     int64_t* __restrict__ tile_off, int64_t* __restrict__ blk_sum) {
    __shared__ int64_t wt[CMP_SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t base = ((int64_t)blockIdx.x << CMP_LG_SCAN_BLOCK) + (int64_t)threadIdx.x * CMP_SCAN_ITEMS;
    int64_t v[CMP_SCAN_ITEMS];
    int64_t s = 0;
#pragma unroll
    for (int i = 0; i < CMP_SCAN_ITEMS; ++i) {
        v[i] = base + i < ntiles ? tile_cnt[base + i] : 0;
        s += v[i];
    }
    int64_t incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wt[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int64_t w = wt[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        wt[lane] = w;
    }
    __syncthreads();
    int64_t run = (wid ? wt[wid - 1] : 0) + incl - s;
#pragma unroll
    for (int i = 0; i < CMP_SCAN_ITEMS; ++i) {
        if (base + i < ntiles) tile_off[base + i] = run;
        run += v[i];
    }
    if (threadIdx.x == CMP_SCAN_THREADS - 1) blk_sum[blockIdx.x] = wt[CMP_SCAN_THREADS / 32 - 1];
}

// out_k = element key + key_shift (dense form: in-array key - 1 + base).  SEMS: ptr[live_rank[slot]] at every semaphore cell,
// ptr[np] = total (by the last tile).  Outputs at ranks >= limit are not written (the caller's capacity).
template <bool SEMS>
__global__ void __launch_bounds__(256) k_compress_emit(const int64_t* __restrict__ keys, const double* __restrict__ vals, int64_t cap,
                                                        const int64_t* __restrict__ tile_off, const int64_t* __restrict__ blk_sum,
                                                        int64_t key_shift, const int32_t* __restrict__ live_rank, int64_t* __restrict__ ptr,
                                                        int64_t np, int64_t limit, int64_t* __restrict__ out_k, double* __restrict__ out_v) {
    __shared__ int64_t sk[CMP_WARPS][CMP_STAGE];
    __shared__ double sv[CMP_WARPS][CMP_STAGE];
    __shared__ int32_t wc[CMP_WARPS];
    __shared__ int64_t s_toff;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t tile = blockIdx.x;
    const int64_t p0 = tile * CMP_TILE + (int64_t)wid * (32 * CMP_C) + (int64_t)lane * CMP_C;
    const uint64_t pol = l2_evict_first_policy();
    int64_t k[CMP_C];
    double t[CMP_C];
    load_cells(keys, vals, cap, p0, k, t, pol);
    int cnt = 0;
#pragma unroll
    for (int c = 0; c < CMP_C; ++c) cnt += cmp_elem<SEMS>(k[c]) ? 1 : 0;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    const int wtot = __shfl_sync(0xffffffffu, incl, 31);
    if (lane == 0) wc[wid] = wtot;
    if (wid == 0) {   // tile offset = offset inside its scan block + totals of the scan blocks before it
        const int64_t a = scan_block_base(blk_sum, tile, lane);
        if (lane == 0) s_toff = tile_off[tile] + a;
    }
    __syncthreads();
    int64_t wbase = s_toff;
    int ttot = 0;
#pragma unroll
    for (int w = 0; w < CMP_WARPS; ++w) {
        if (w < wid) wbase += wc[w];
        ttot += wc[w];
    }
    int r = incl - cnt;   // warp-local rank of the lane's first element
#pragma unroll
    for (int c = 0; c < CMP_C; ++c) {
        if (cmp_elem<SEMS>(k[c])) {
            const int q = r + (r >> 3);
            sk[wid][q] = k[c] + key_shift;
            sv[wid][q] = t[c];
            ++r;
        } else if (SEMS && k[c] == 0) {
            ptr[live_rank[(int32_t)t[c] - 1]] = wbase + r;
        }
    }
    __syncwarp();
    for (int i = lane; i < wtot; i += 32) {
        const int64_t d = wbase + i;
        if (d < limit) {
            out_k[d] = sk[wid][i + (i >> 3)];
            out_v[d] = sv[wid][i + (i >> 3)];
        }
    }
    if (SEMS && threadIdx.x == 0 && tile == (int64_t)gridDim.x - 1) ptr[np] = s_toff + ttot;
}

__global__ void __launch_bounds__(256) k_compress_live_rank(const int32_t* __restrict__ live_slot, int64_t nlive, int32_t* __restrict__ live_rank) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nlive) live_rank[live_slot[i]] = (int32_t)i;
}

// dense pointer over partition keys 1..dim: out[k] = base + ptr[first live partition with key >= k + 1] for k = 0..dim (the
// entries of key k end where the next present key starts); a present key is one load of the direct-address map, others (and
// maps without the table, whose slot lookup is the same binary search) the binary search over the sorted live keys
__global__ void __launch_bounds__(256) k_compress_dense_ptr(const int64_t* __restrict__ ptr, const ColMap cm, const int32_t* __restrict__ live_rank,
                                                             int64_t dim, int64_t base, int64_t* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k > dim) return;
    const int64_t key = k + 1;
    const int32_t s = cm.keymap ? cm.slot(key) : -1;
    out[k] = base + ptr[s >= 0 ? live_rank[s] : cm.lower_rank(key)];
}

struct CompressWorkspace {
    DBuf<int32_t> tile_cnt, live_rank, flag;
    DBuf<int64_t> tile_off, blk_sum, ptr;
    HPinned<int32_t> h_flag;
};

// The dense form's bounds check (see k_compress_count).  check = false: the host has ruled a violation out.
struct CompressBounds {
    bool check = false;
    const int64_t* sem = nullptr;
    int32_t slot = -1;
    int64_t idim = INT64_MAX;
};

// Count, [bounds read-back], scan, emit of the element cells of keys/vals[cap] on st.  A bounds violation throws DSA_ERR_BOUNDS
// before the emit pass: nothing has been written then.
template <bool SEMS>
inline void compress_cells(CompressWorkspace& w, const int64_t* keys, const double* vals, int64_t cap, const CompressBounds& b,
                           int64_t key_shift, const int32_t* live_rank, int64_t* ptr, int64_t np, int64_t limit, int64_t* out_k,
                           double* out_v, cudaStream_t st) {
    const int64_t ntiles = std::max<int64_t>(1, (cap + CMP_TILE - 1) / CMP_TILE);
    const int64_t nblk = (ntiles + (1 << CMP_LG_SCAN_BLOCK) - 1) >> CMP_LG_SCAN_BLOCK;
    int32_t* tile_cnt = w.tile_cnt.ensure((size_t)ntiles);
    int64_t* tile_off = w.tile_off.ensure((size_t)ntiles);
    int64_t* blk_sum = w.blk_sum.ensure((size_t)nblk);
    int32_t* flag = nullptr;
    if (b.check) {
        flag = w.flag.ensure(1);
        DSA_CUDA(cudaMemsetAsync(flag, 0, 4, st));
    }
    DSA_LAUNCH("compress_count", k_compress_count<SEMS>, (unsigned)ntiles, 256, 0, st, keys, cap, tile_cnt, b.sem, b.slot, b.idim, flag);
    if (b.check) {
        int32_t* h = w.h_flag.ensure(1);
        DSA_CUDA(cudaMemcpyAsync(h, flag, 4, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        if (*h)
            throw DsaError{DSA_ERR_BOUNDS, "compress_dense: an entry lies outside dim x idim (a partition key > dim or an in-array key > idim)"};
    }
    DSA_LAUNCH("compress_scan", k_compress_scan, (unsigned)nblk, CMP_SCAN_THREADS, 0, st, tile_cnt, ntiles, tile_off, blk_sum);
    DSA_LAUNCH("compress_emit", k_compress_emit<SEMS>, (unsigned)ntiles, 256, 0, st, keys, vals, cap, tile_off, blk_sum, key_shift, live_rank,
               ptr, np, limit, out_k, out_v);
}

// ---------------------------------------------------------------------------------------------
// K9 sparse-x product driven by x's entries: mat * x over the column-major orientation, transpose(mat) * x over the row-major
// one, exactly as _mul_dyn_mat_col_loop! does it (operations.jl:62-105): for every x entry in ascending key, the cells of that
// partition's span, result[key] = fl(result[key] + fl(x_j * a)).  The cost is the cells of the selected partitions, not the
// size of the matrix.  k right-hand sides (X in CSC over keys: x_ptr[k + 1], keys ascending in each column) go through the same
// kernels in one call: every product is tagged with its column, and column c of the result is the one-vector product with
// X[:, c].  The one-vector product is the case k = 1 with no x_ptr.
//   locate  one thread per x entry: its column (binary search in x_ptr), slot (direct-address map or binary search), span
//           [sem + 1, span_end), the span cut into pieces of at most SPX_PIECE cells (one warp per piece: a 60 000-cell
//           partition does not serialise one warp), and the check that x is strictly ascending inside its column
//   count   one warp per piece: stored cells; int64 exclusive scan of the piece counts (k_compress_scan)
//   cols    one warp per column boundary c: the check of x_ptr, its first piece and its first product (product offsets of
//           the columns, read back with the error flag)
//   rounds  the host cuts the columns into consecutive rounds of at most SPX_ROUND_PRODUCTS products (one column may exceed
//           it alone) and at most 2^(64 - keybits) columns, so that the sort key (column - round start) << keybits | key - 1
//           fits 64 bits.  Per round, with no host synchronisation between rounds:
//     emit  one warp per piece of the round, cells in order: (sort key, product, product index), the index order being x order
//     group stable LSD radix sort over colbits + keybits bits with the product index as payload: a (column, key)'s products
//           stay in ascending x order
//     fold  run heads flagged and ranked; one thread per run folds it left to right from 0.0 and writes (key, value) at the
//           device-resident running output offset, and the first run of a column writes the column pointers
// ---------------------------------------------------------------------------------------------
constexpr int SPX_LG_PIECE = 11, SPX_PIECE = 1 << SPX_LG_PIECE;
constexpr int64_t SPX_ROUND_PRODUCTS = int64_t(1) << 27;   // products of one round: 40 B each, 5.4 GB of workspace
// info words; the column product offsets (k + 1) follow them.  NOUT: outputs of the rounds before the last one folded,
// RUNS: outputs of that round (the next round's emit moves them into NOUT)
enum { SPX_ERR = 0, SPX_NPIECES = 1, SPX_NOUT = 2, SPX_RUNS = 3, SPX_WORDS = 4 };
// grid of the piece kernels (warp-per-piece, grid-stride): 8 CTAs of 8 warps per SM of a 148-SM part at most
inline unsigned spx_piece_grid(int64_t npieces) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((npieces + 7) / 8, 148 * 8)); }

// xptr == nullptr: one column holding all nx entries (xcol not written)
__global__ void __launch_bounds__(256) k_spx_locate(const int64_t* __restrict__ xk, int64_t nx, const int64_t* __restrict__ xptr,
                                                     int64_t ncol, const ColMap cm, const int64_t* __restrict__ sem,
                                                     const int32_t* __restrict__ next_slot, int64_t cap, int64_t* __restrict__ span_from,
                                                     int64_t* __restrict__ span_to, int32_t* __restrict__ npieces, int64_t* __restrict__ xcol,
                                                     int64_t* __restrict__ info) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nx) return;
    const int64_t key = xk[i];
    int64_t first = 0;
    if (xptr) {   // the last column c with xptr[c] <= i (a malformed x_ptr gives some c in [0, ncol): k_spx_cols refuses it)
        const int64_t lo = lower_bound(xptr, ncol, i + 1);
        const int64_t c = lo > 0 ? lo - 1 : 0;
        xcol[i] = c;
        first = xptr[c];
    }
    if (i > first && xk[i - 1] >= key) info[SPX_ERR] = 1;
    const int32_t s = cm.slot(key);
    int64_t from = 0, to = 0;
    if (s >= 0) {
        from = sem[s] + 1;
        to = span_end(sem, next_slot, s, cap);
    }
    span_from[i] = from;
    span_to[i] = to;
    npieces[i] = (int32_t)((to - from + SPX_PIECE - 1) >> SPX_LG_PIECE);
}

// piece q -> x entry i and cells [c0, c1); false for a q that names no piece (past the total, or offsets of a rejected x)
__device__ __forceinline__ bool spx_piece(int64_t q, const int32_t* __restrict__ piece_off, const int32_t* __restrict__ npieces, int64_t nx,
                                          const int64_t* __restrict__ span_from, const int64_t* __restrict__ span_to, int64_t& i,
                                          int64_t& c0, int64_t& c1) {
    i = lower_bound(piece_off, nx, q + 1) - 1;   // the last entry whose first piece is <= q
    if (i < 0) return false;
    const int64_t j = q - piece_off[i];
    if (j < 0 || j >= npieces[i]) return false;
    c0 = span_from[i] + (j << SPX_LG_PIECE);
    c1 = min(span_to[i], c0 + SPX_PIECE);
    return true;
}

// pcnt[q] for every q < nq (zeros past the pieces: the scan reads nq counts)
__global__ void __launch_bounds__(256) k_spx_count(const int64_t* __restrict__ keys, const int32_t* __restrict__ piece_off,
                                                    const int32_t* __restrict__ npieces, int64_t nx, const int64_t* __restrict__ span_from,
                                                    const int64_t* __restrict__ span_to, const int64_t* __restrict__ info, int64_t nq,
                                                    int32_t* __restrict__ pcnt) {
    const int lane = threadIdx.x & 31;
    const int64_t ntot = min(info[SPX_NPIECES], nq);
    const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < nq; q += nw) {
        int64_t i, c0, c1;
        int c = 0;
        if (q < ntot && spx_piece(q, piece_off, npieces, nx, span_from, span_to, i, c0, c1))
            for (int64_t p = c0 + lane; p < c1; p += 32) c += keys[p] != GAP_KEY;
        c = __reduce_add_sync(0xffffffffu, c);
        if (lane == 0) pcnt[q] = c;
    }
}

// one warp per column boundary c in [0, ncol]: x_ptr checked (starts at 0, never decreases, ends at nx), col_piece[c] = first
// piece of column c, info[SPX_WORDS + c] = first product of column c (info[SPX_WORDS + ncol] = the product count).
// xptr == nullptr: one column [0, nx).  Indices are clamped, so a malformed x (refused at the read-back) reads in bounds.
__global__ void __launch_bounds__(256) k_spx_cols(const int64_t* __restrict__ xptr, int64_t ncol, int64_t nx,
                                                   const int32_t* __restrict__ piece_off, const int64_t* __restrict__ poff,
                                                   const int64_t* __restrict__ blk_sum, int64_t nq, int64_t* __restrict__ info,
                                                   int64_t* __restrict__ col_piece) {
    const int lane = threadIdx.x & 31;
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (c > ncol) return;
    int64_t e = c == 0 ? 0 : nx;
    if (xptr) {
        e = xptr[c];
        if (lane == 0 && ((c == 0 ? e != 0 : e < xptr[c - 1]) || (c == ncol && e != nx))) info[SPX_ERR] = 1;
        e = min(max(e, (int64_t)0), nx);
    }
    const int64_t q = min(max(e < nx ? (int64_t)piece_off[e] : info[SPX_NPIECES], (int64_t)0), nq - 1);
    const int64_t a = scan_block_base(blk_sum, q, lane);
    if (lane == 0) {
        col_piece[c] = q;
        info[SPX_WORDS + c] = poff[q] + a;
    }
}

// one round: the pieces of columns [c0, c0 + nc), their products at (global product index - p0).  The sort key of a product is
// (column - c0) << kb | key - 1 (xcol == nullptr: column 0).  Block 0 first folds the previous round's outputs into NOUT.
__global__ void __launch_bounds__(256) k_spx_emit(const int64_t* __restrict__ keys, const double* __restrict__ vals,
                                                   const int32_t* __restrict__ piece_off, const int32_t* __restrict__ npieces,
                                                   const int64_t* __restrict__ span_from, const int64_t* __restrict__ span_to,
                                                   const double* __restrict__ xv, int64_t nx, const int64_t* __restrict__ xcol,
                                                   const int64_t* __restrict__ poff, const int64_t* __restrict__ blk_sum,
                                                   const int64_t* __restrict__ col_piece, int64_t c0, int64_t nc, int kb, int64_t p0,
                                                   int64_t* __restrict__ info, uint64_t* __restrict__ sk, uint32_t* __restrict__ perm,
                                                   double* __restrict__ prod) {
    const int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        info[SPX_NOUT] += info[SPX_RUNS];
        info[SPX_RUNS] = 0;
    }
    const int64_t q1 = col_piece[c0 + nc];
    const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
    const unsigned lt = lanemask_lt();
    for (int64_t q = col_piece[c0] + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); q < q1; q += nw) {
        int64_t i, cf, cl;
        if (!spx_piece(q, piece_off, npieces, nx, span_from, span_to, i, cf, cl)) continue;
        const int64_t a = scan_block_base(blk_sum, q, lane);
        int64_t o = poff[q] + a - p0;
        const double x = xv[i];
        const uint64_t tag = xcol ? (uint64_t)(xcol[i] - c0) << kb : 0;
        for (int64_t base = cf; base < cl; base += 32) {
            const int64_t p = base + lane;
            const int64_t k = p < cl ? keys[p] : GAP_KEY;
            const unsigned b = __ballot_sync(0xffffffffu, k != GAP_KEY);
            if (k != GAP_KEY) {
                const int64_t d = o + __popc(b & lt);
                sk[d] = tag | (uint64_t)(k - 1);
                perm[d] = (uint32_t)d;
                prod[d] = __dmul_rn(x, vals[p]);
            }
            o += __popc(b);
        }
    }
}

// one thread per run of equal sort keys (sk sorted, perm = product indices in x order within a run): the left fold from 0.0,
// written at NOUT + rank when out_k is set and the outputs through this round (NOUT + RUNS) fit cap.  yptr (nullable): the
// first run of a column sets the pointers of the columns since the previous run's, the last run those up to the round's end.
__global__ void __launch_bounds__(256) k_spx_fold(const uint64_t* __restrict__ sk, const uint32_t* __restrict__ perm,
                                                   const double* __restrict__ prod, const int32_t* __restrict__ head,
                                                   const int32_t* __restrict__ rank, int64_t n, const int64_t* __restrict__ info, int64_t cap,
                                                   int64_t* __restrict__ out_k, double* __restrict__ out_v, int kb, int64_t c0, int64_t nc,
                                                   int64_t* __restrict__ yptr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || !head[t]) return;
    const bool write = out_k && info[SPX_NOUT] + info[SPX_RUNS] <= cap;
    if (!write && !yptr) return;
    const uint64_t key = sk[t];
    const int64_t o = info[SPX_NOUT] + rank[t];
    if (write) {
        double acc = 0.0;
        for (int64_t u = t; u < n && sk[u] == key; ++u) acc = __dadd_rn(acc, prod[perm[u]]);
        out_k[o] = (int64_t)(kb ? key & (~uint64_t(0) >> (64 - kb)) : 0) + 1;   // kb = 0: every key is 1
        out_v[o] = acc;
    }
    if (yptr) {
        const int64_t col = (int64_t)(key >> kb);
        for (int64_t j = t ? (int64_t)(sk[t - 1] >> kb) + 1 : 0; j <= col; ++j) yptr[c0 + j] = o;
        if (sk[n - 1] == key)
            for (int64_t j = col + 1; j <= nc; ++j) yptr[c0 + j] = o + 1;
    }
}

// column pointers of a round without products: every one is the running output offset
__global__ void __launch_bounds__(256) k_spx_ptr_fill(const int64_t* __restrict__ info, int64_t c0, int64_t nc, int64_t* __restrict__ yptr) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j <= nc) yptr[c0 + j] = info[SPX_NOUT] + info[SPX_RUNS];
}

struct SpmspvWorkspace {
    DBuf<int64_t> span_from, span_to, poff, blk_sum, info, xcol, col_piece, yptr;
    DBuf<int32_t> npieces, piece_off, pcnt, head, rank;
    DBuf<uint64_t> sk;
    DBuf<uint32_t> perm;
    DBuf<double> prod;
    HPinned<int64_t> h_info;
    std::vector<int64_t> h_cut;   // column boundaries of the rounds
};

// ---- tile-streamed batches (tile.cuh): geometry of a tile and the record an op is bucketed as ----
#ifndef DSA_TILE_LG
#define DSA_TILE_LG 10
#endif
constexpr int TILE_LG = DSA_TILE_LG, TILE_CELLS = 1 << TILE_LG;   // 1024 cells = 16 KB of keys + values
constexpr int TILE_CAP = TILE_CELLS / 4;                  // ops a tile's bucket holds
constexpr int TILE_THREADS = TILE_CELLS / 8;              // a thread moves 4 x 16 bytes of keys and of values each way
constexpr int TILE_CTAS_PER_SM = TILE_LG == 9 ? 20 : TILE_LG == 10 ? 11 : 5;
constexpr int TILE_PREFETCH_DIST = 148 * TILE_CTAS_PER_SM;   // tiles in flight on a B200: the L2 prefetch runs one wave ahead
constexpr int TILE_MAX_LEAVES = TILE_CELLS / 8;           // segment capacity >= 8
#ifndef DSA_TILE_CNT_STRIDE
#define DSA_TILE_CNT_STRIDE 8
#endif
constexpr int TILE_CNT_STRIDE = DSA_TILE_CNT_STRIDE;      // a tile's op counter has a 32-byte sector to itself: the L2 serialises atomics per sector

struct __align__(16) TileRec {   // 32 B: one sector per op
    int64_t key;     // in-array key
    double val;
    uint32_t arr;    // arrival index in the batch (last writer wins)
    int32_t slot;
    uint16_t lo, hi; // tile-local search range (inclusive); lo > hi = empty span: the predecessor is the cell at hi
    uint32_t pad;
};

// =============================================================================================
// MappedPackedCSC on the device
// =============================================================================================
struct PcsrWorkspace {
    BatchWorkspace batch;
    SortWorkspace sort;
    DBuf<int32_t> op_slot, flag32, idx32, u_pid, new_slots, old2new, rank32, del_slots, cnt32, bcnt, boff, lidx, bslot;
    DBuf<BucketRec> brec;
    DBuf<TileRec> trec;          // tile buckets of a tile-streamed batch: TILE_CAP records per tile
    DBuf<int64_t> miss_keys, cs, u_key, live_pos, nuniq, tmp_k, tmp_owner, del_keys;
    DBuf<double> u_val, tmp_v, yslot, carry, xdense;
    DBuf<double> yslot_mv, carry_mv, xpad;   // multi-vector product: partials of a pass (W per slot / chunk), X re-laid to ld % 4 == 0
    DBuf<uint64_t> sk;
    DBuf<uint32_t> perm;
    DBuf<uint8_t> xmask;
    DBuf<int32_t> ycnt, carry_cnt, chunk_last;
    CompressWorkspace cmp;
    SpmspvWorkspace spx;
    HPinned<int64_t> h_cs;
    std::vector<int64_t> h_tmp;
};

struct Pcsr {
    PmaCore pma;
    int64_t nb_partitions = 0;   // pcsr.jl:5
    // col_keys with tombstones (pcsr.jl:17): host mirror is the authority for the map, device copies serve the kernels
    std::vector<int64_t> slot_key;
    std::vector<uint8_t> slot_live;
    std::vector<int64_t> live_keys_h;   // sorted live keys
    std::vector<int32_t> live_slot_h;
    DBuf<int64_t> d_sem;        // per slot: 0-based position of the semaphore cell, -1 = deleted / not yet placed (pcsr.jl:6)
    DBuf<int32_t> d_next_slot;  // per slot: next live, already placed slot (-1 = none): the span ends at its semaphore
    DBuf<int64_t> d_slot_key;
    DBuf<int64_t> d_live_keys;
    DBuf<int32_t> d_live_slot;
    DBuf<int32_t> d_keymap;     // optional direct-address table key - keymap_min -> slot (dense key ranges only)
    std::vector<int32_t> keymap_h;
    int64_t keymap_min = 0, keymap_len = 0;
    std::vector<int32_t> next_slot_h;
    int64_t max_inkey = 0;      // upper bound of the in-array keys ever stored (sizes the dense x of SpMV)
    int tile_penalty = 0;       // batches to wait before the next tile-streamed attempt (after a refused one)
    int64_t last_batch_n = 0;   // ops of the previous batch (the host only has an upper bound of a distributed batch's size)

    ColMap colmap() const {
        return ColMap{d_live_keys.p, d_live_slot.p, nlive(), keymap_len > 0 ? d_keymap.p : nullptr, keymap_min, keymap_len};
    }
    int64_t nslots() const { return (int64_t)slot_key.size(); }
    int64_t nlive() const { return (int64_t)live_keys_h.size(); }
    int64_t nnz() const { return pma.nnz - nb_partitions; }   // pcsr.jl:11

    // unplaced (nullable): slots created by the running batch whose semaphore is not in the array yet
    void rebuild_live_and_upload(cudaStream_t st, const std::vector<int32_t>* unplaced = nullptr) {
        live_keys_h.clear();
        live_slot_h.clear();
        {
            const int64_t nsl = nslots();
            std::vector<uint8_t> placed(slot_live.begin(), slot_live.end());
            if (unplaced)
                for (int32_t u : *unplaced) placed[(size_t)u] = 0;
            next_slot_h.assign((size_t)nsl, -1);
            int32_t nxt = -1;
            for (int64_t q = nsl - 1; q >= 0; --q) {
                next_slot_h[(size_t)q] = nxt;
                if (placed[(size_t)q]) nxt = (int32_t)q;
            }
            d_next_slot.ensure((size_t)nsl + 1);
            if (nsl) DSA_CUDA(cudaMemcpyAsync(d_next_slot.p, next_slot_h.data(), (size_t)nsl * 4, cudaMemcpyHostToDevice, st));
        }
        for (int64_t s = 0; s < nslots(); ++s)
            if (slot_live[s]) { live_keys_h.push_back(slot_key[s]); live_slot_h.push_back((int32_t)s); }
        const size_t ns = (size_t)nslots(), nl = live_keys_h.size();
        d_slot_key.ensure(ns + 1);
        d_live_keys.ensure(nl + 1);
        d_live_slot.ensure(nl + 1);
        if (ns) DSA_CUDA(cudaMemcpyAsync(d_slot_key.p, slot_key.data(), ns * 8, cudaMemcpyHostToDevice, st));
        keymap_len = 0;
        if (nl) {
            DSA_CUDA(cudaMemcpyAsync(d_live_keys.p, live_keys_h.data(), nl * 8, cudaMemcpyHostToDevice, st));
            DSA_CUDA(cudaMemcpyAsync(d_live_slot.p, live_slot_h.data(), nl * 4, cudaMemcpyHostToDevice, st));
            const uint64_t range = (uint64_t)live_keys_h.back() - (uint64_t)live_keys_h.front() + 1;
            if (range <= std::max<uint64_t>(8 * (uint64_t)nl, 1u << 16) && range <= (1u << 27)) {
                keymap_min = live_keys_h.front();
                keymap_len = (int64_t)range;
                keymap_h.assign((size_t)range, -1);
                for (size_t i = 0; i < nl; ++i) keymap_h[(size_t)(live_keys_h[i] - keymap_min)] = live_slot_h[i];
                d_keymap.ensure((size_t)range);
                DSA_CUDA(cudaMemcpyAsync(d_keymap.p, keymap_h.data(), (size_t)range * 4, cudaMemcpyHostToDevice, st));
            }
        }
        DSA_CUDA(cudaStreamSynchronize(st));   // host vectors may be modified after return
    }

    int32_t host_lookup(int64_t key) const {
        auto it = std::lower_bound(live_keys_h.begin(), live_keys_h.end(), key);
        if (it == live_keys_h.end() || *it != key) return -1;
        return live_slot_h[(size_t)(it - live_keys_h.begin())];
    }

    // MappedPackedCSC(K, L, T) (pcsr.jl:82-86)
    void init_empty(cudaStream_t st) {
        pma.build_from_sorted(nullptr, nullptr, 0, nullptr, st);
        nb_partitions = 0;
        slot_key.clear();
        slot_live.clear();
        rebuild_live_and_upload(st);
        d_sem.ensure(1);
        max_inkey = 0;
    }

    // _dynamicsparse (pcsr.jl:354-431): stable sort by (partition key, in-array key), left-fold combine, flatten as
    // [sem_1, col_1..., sem_2, col_2...] (pcsr.jl:37-51), bulk layout + semaphore positions (pcsr.jl:52-61).
    void build_coo_d(PcsrWorkspace& ws, const int64_t* d_inkeys, const int64_t* d_partkeys, const double* d_vals, int64_t n, int combine,
                     cudaStream_t st);

    void get_batch_d(PcsrWorkspace& ws, const int64_t* d_inkeys, const int64_t* d_partkeys, int64_t n, double* d_out, cudaStream_t st) {
        if (n <= 0) return;
        int32_t* op_slot = ws.op_slot.ensure((size_t)n);
        int64_t* cs = ws.cs.ensure(CS_WORDS);   // statistics are not used by reads
        DSA_LAUNCH("col_lookup", k_col_lookup, lookup_grid(n), 256, 0, st, d_partkeys, (const int64_t*)nullptr, (const double*)nullptr, n,
                   (const int64_t*)nullptr, colmap(), op_slot, cs, (int32_t*)nullptr, (int32_t*)nullptr);
        DSA_LAUNCH("get", k_get, grid_for(n, 256), 256, 0, st, pma.keys.p, pma.vals.p, pma.g.capacity, op_slot, d_inkeys, n, d_sem.p,
                       d_next_slot.p, d_out);
    }

    // spans of the listed slots, emitted in list order: returns total count; outputs in ws.tmp_k / tmp_v / tmp_owner
    int64_t gather_spans(PcsrWorkspace& ws, const int32_t* d_slots, int64_t nsl, const int64_t* d_owner_keys, bool want_vals, cudaStream_t st) {
        int32_t* cnt = ws.cnt32.ensure((size_t)nsl + 1);
        int32_t* off = ws.idx32.ensure((size_t)nsl + 1);
        int64_t* tot = ws.nuniq.ensure(4);
        DSA_LAUNCH("span_count", k_span_count, grid_for(nsl * 32, 256), 256, 0, st, pma.keys.p, d_slots, nsl, d_sem.p, d_next_slot.p, pma.g.capacity, cnt);
        exclusive_scan_i32<int32_t>(ws.batch.scan, cnt, off, nsl, tot, st);
        int64_t h_tot = 0;
        DSA_CUDA(cudaMemcpyAsync(&h_tot, tot, 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        if (h_tot > 0) {
            ws.tmp_k.ensure((size_t)h_tot);
            if (want_vals) ws.tmp_v.ensure((size_t)h_tot);
            if (d_owner_keys) ws.tmp_owner.ensure((size_t)h_tot);
            DSA_LAUNCH("span_emit", k_span_emit, grid_for(nsl * 32, 256), 256, 0, st, pma.keys.p, pma.vals.p, d_slots, nsl, d_sem.p, d_next_slot.p, pma.g.capacity,
                       off, ws.tmp_k.p, want_vals ? ws.tmp_v.p : (double*)nullptr, d_owner_keys ? ws.tmp_owner.p : (int64_t*)nullptr,
                       d_owner_keys);
        }
        return h_tot;
    }

    // deletepartition! for a list of slots (pcsr.jl:188-204): purge spans, rebalance, tombstone
    void delete_slots(PcsrWorkspace& ws, const std::vector<int32_t>& slots, const int32_t* d_slots, cudaStream_t st) {
        const int64_t nsl = (int64_t)slots.size();
        if (nsl == 0) return;
        pma.prepare_batch_scratch(ws.batch, 0, st);
        DSA_LAUNCH("span_purge", k_span_purge, grid_for(nsl * 32, 256), 256, 0, st, pma.keys.p, pma.vals.p, d_slots, nsl, d_sem.p, d_next_slot.p, pma.g.capacity,
                   pma.leafcnt.p, ws.batch.touched, ilog2_i64(pma.g.segment_capacity));
        DSA_LAUNCH("clear_sems", k_clear_sems, grid_for(nsl, 256), 256, 0, st, d_sem.p, d_slots, nsl);
        pma.rebalance_after(ws.batch, d_sem.p, st);
        for (int32_t s : slots) slot_live[(size_t)s] = 0;   // pcsr.jl:202,209
        nb_partitions -= nsl;                                // pcsr.jl:191
        rebuild_live_and_upload(st);
    }

    // a warp's chunk = 32 lanes x 8 cells (two 256-bit loads of keys, two of values, 8 gathers of x in flight per lane):
    // product call 71.5 -> 66.5 us at config 2 against 4 cells per lane; 16 cells per lane (114 registers): 83 us
    static constexpr int SPMV_CELLS_PER_LANE = 8, SPMV_LG_CHUNK = 8;
    static_assert(32 * SPMV_CELLS_PER_LANE == 1 << SPMV_LG_CHUNK, "a warp's chunk");
    int64_t spmv_nchunks() const { return (pma.g.capacity + (1 << SPMV_LG_CHUNK) - 1) >> SPMV_LG_CHUNK; }

    // The chunked reduction of mat * x (k_spmv_blocked): partials by slot in ws.yslot, carries in ws.carry / ws.chunk_last, and
    // with a sparse x the product counts in ws.ycnt / ws.carry_cnt.  The caller launches the epilogue that adds the carries.
    // x: dense (d_xmask == nullptr), sparse as a dense buffer with a presence mask, or d_xkeys != nullptr: sparse as
    // (d_xkeys, d_x)[nx] with ascending keys, looked up by binary search (no dense buffer).
    void spmv_reduce(PcsrWorkspace& ws, const double* d_x, const uint8_t* d_xmask, int64_t nx, cudaStream_t st, const int64_t* d_xkeys) {
        constexpr int C = SPMV_CELLS_PER_LANE;
        const int64_t cap = pma.g.capacity, nchunks = spmv_nchunks(), ns = nslots();
        double* yslot = ws.yslot.ensure((size_t)ns + 1);
        int32_t* ycnt = ws.ycnt.ensure((size_t)ns + 1);
        double* carry = ws.carry.ensure((size_t)nchunks);
        int32_t* ccnt = ws.carry_cnt.ensure((size_t)nchunks);
        int32_t* clast = ws.chunk_last.ensure((size_t)nchunks);
        const auto kernel = d_xkeys ? k_spmv_blocked<2, C> : d_xmask ? k_spmv_blocked<1, C> : k_spmv_blocked<0, C>;
        DSA_LAUNCH("spmv_blocked", kernel, grid_for(nchunks * 32, 256), 256, 0, st, pma.keys.p, pma.vals.p, cap, d_x, d_xmask, d_xkeys, nx,
                   yslot, ycnt, carry, ccnt, clast, nchunks);
    }
    // mat * sparse x (a presence mask, or d_xkeys: see spmv_reduce); results and product counts by slot in ws.yslot / ws.ycnt
    void spmv_slots(PcsrWorkspace& ws, const double* d_x, const uint8_t* d_xmask, int64_t nx, cudaStream_t st,
                    const int64_t* d_xkeys = nullptr) {
        spmv_reduce(ws, d_x, d_xmask, nx, st, d_xkeys);
        const int64_t nchunks = spmv_nchunks();
        DSA_LAUNCH("spmv_fixup", k_spmv_fixup, grid_for(nchunks, 256), 256, 0, st, ws.yslot.p, ws.ycnt.p, ws.carry.p, ws.carry_cnt.p,
                   ws.chunk_last.p, nchunks);
    }
    // mat * dense x -> dense y over the partition keys [key_lo, key_hi) (y zeroed by the caller): reduction kernel + one
    // epilogue kernel (fix-up and scatter by key)
    void spmv_dense(PcsrWorkspace& ws, const double* d_x, int64_t nx, double* d_y, int64_t key_lo, int64_t key_hi, cudaStream_t st) {
        spmv_reduce(ws, d_x, nullptr, nx, st, nullptr);
        const int64_t ns = nslots();
        if (ns > 0)
            DSA_LAUNCH("spmv_fix_to_dense", k_spmm_fix_to_dense<true>, grid_for(ns, 256), 256, 0, st, ws.yslot.p, ws.carry.p, ws.chunk_last.p, d_sem.p,
                       d_next_slot.p, d_slot_key.p, ns, pma.g.capacity, spmv_nchunks(), SPMV_LG_CHUNK, 1, 1, d_y, (int64_t)1, key_lo, key_hi);
    }

    // mat * X -> Y for one pass of ncols (<= 4 * ngroups) columns, over the partition keys [key_lo, key_hi) (Y zeroed by the
    // caller; columns >= ncols of Y untouched): X row-major, ldx % 4 == 0, 32-byte aligned; columns ncols .. W-1 of X are read
    // and their results dropped
    void spmm_dense_pass(PcsrWorkspace& ws, const double* d_X, int64_t nx, int64_t ldx, int ncols, double* d_Y, int64_t ldy,
                         int64_t key_lo, int64_t key_hi, cudaStream_t st) {
        constexpr int C = SPMV_CELLS_PER_LANE;
        const int ngroups = (ncols + 3) / 4, W = 4 * ngroups;
        const int64_t cap = pma.g.capacity, ns = nslots(), nchunks = spmv_nchunks();
        double* yslot = ws.yslot_mv.ensure((size_t)(ns + 1) * W);
        double* carry = ws.carry_mv.ensure((size_t)nchunks * W);
        int32_t* clast = ws.chunk_last.ensure((size_t)nchunks);
        DSA_LAUNCH("spmm_blocked", k_spmm_blocked<C>, grid_for(nchunks * 32, 256), 256, 0, st, pma.keys.p, pma.vals.p, cap, d_X, nx, ldx,
                   ngroups, yslot, carry, clast, nchunks);
        if (ns > 0)
            DSA_LAUNCH("spmm_fix_to_dense", k_spmm_fix_to_dense<false>, grid_for(ns * W, 256), 256, 0, st, yslot, carry, clast, d_sem.p,
                       d_next_slot.p, d_slot_key.p, ns, cap, nchunks, SPMV_LG_CHUNK, W, ncols, d_Y, ldy, key_lo, key_hi);
    }

    // slot -> index among the live slots (= rank in array order): built per call, the update path keeps no such map
    const int32_t* compress_live_rank(PcsrWorkspace& ws, cudaStream_t st) {
        int32_t* lr = ws.cmp.live_rank.ensure((size_t)nslots() + 1);
        if (nlive() > 0)
            DSA_LAUNCH("compress_live_rank", k_compress_live_rank, grid_for(nlive(), 256), 256, 0, st, d_live_slot.p, nlive(), lr);
        return lr;
    }
    // sparse-pointer form (K8): part_keys[nlive] (nullable: the host copies its mirror), ptr[nlive + 1], keys / vals[nnz]
    void compress_sparse(PcsrWorkspace& ws, int64_t* d_part_keys, int64_t* d_ptr, int64_t* d_keys, double* d_vals, cudaStream_t st) {
        const int64_t np = nlive();
        if (d_part_keys && np > 0) DSA_CUDA(cudaMemcpyAsync(d_part_keys, d_live_keys.p, (size_t)np * 8, cudaMemcpyDeviceToDevice, st));
        compress_cells<true>(ws.cmp, pma.keys.p, pma.vals.p, pma.g.capacity, CompressBounds{}, 0, compress_live_rank(ws, st), d_ptr, np,
                             nnz(), d_keys, d_vals, st);
    }
    // dense-pointer form (K8): ptr[dim + 1] over partition keys 1..dim, ind = in-array key - 1 + base.  DSA_ERR_BOUNDS (nothing
    // written) if an entry lies in a partition with key > dim or has an in-array key > idim; synchronises only when the host
    // cannot rule that out (a live partition with key > dim, or an in-array key above idim may be stored)
    void compress_dense(PcsrWorkspace& ws, int64_t dim, int64_t idim, int64_t base, int64_t* d_ptr, int64_t* d_ind, double* d_vals,
                        cudaStream_t st) {
        const int64_t np = nlive();
        const int64_t i0 = std::upper_bound(live_keys_h.begin(), live_keys_h.end(), dim) - live_keys_h.begin();
        CompressBounds b;
        b.check = i0 < np || max_inkey > idim;
        if (b.check) {
            b.sem = d_sem.p;
            b.slot = i0 < np ? live_slot_h[(size_t)i0] : -1;
            b.idim = idim;
        }
        const int32_t* lr = compress_live_rank(ws, st);
        int64_t* sptr = ws.cmp.ptr.ensure((size_t)np + 1);
        compress_cells<true>(ws.cmp, pma.keys.p, pma.vals.p, pma.g.capacity, b, base - 1, lr, sptr, np, nnz(), d_ind, d_vals, st);
        DSA_LAUNCH("compress_dense_ptr", k_compress_dense_ptr, grid_for(dim + 1, 256), 256, 0, st, sptr, colmap(), lr, dim, base, d_ptr);
    }

    // sparse-x product (K9): x = (d_xk, d_xv)[nx] with strictly ascending keys (DSA_ERR_ARGUMENT otherwise, nothing written);
    // returns the output count.  stage: the output goes to ws.tmp_k / ws.tmp_v; otherwise to d_yk / d_yv, written only when
    // both are set and the count is <= cap.  Two host synchronisations at most (nx > 0 and a product exists).
    int64_t spmspv(PcsrWorkspace& ws, const int64_t* d_xk, const double* d_xv, int64_t nx, bool stage, int64_t* d_yk, double* d_yv,
                   int64_t cap, cudaStream_t st) {
        return spmspm(ws, nullptr, d_xk, d_xv, 1, nx, stage, nullptr, d_yk, d_yv, cap, st);
    }
    // the same product for k = ncol columns of X (CSC: d_xptr[ncol + 1], keys strictly ascending in each column; a malformed
    // x_ptr or key order is DSA_ERR_ARGUMENT, nothing written).  d_xptr == nullptr: one column of nx entries.  d_yptr
    // (nullable, ncol + 1) is written whatever cap; a round writes its keys and values only when the outputs through it fit
    // cap.  stage: the outputs go to ws.tmp_k / ws.tmp_v (min(cap, products) entries) and ws.spx.yptr (when d_xptr is set).
    // Two host synchronisations at most: the column product offsets, and the output count.
    int64_t spmspm(PcsrWorkspace& ws, const int64_t* d_xptr, const int64_t* d_xk, const double* d_xv, int64_t ncol, int64_t nx, bool stage,
                   int64_t* d_yptr, int64_t* d_yk, double* d_yv, int64_t cap, cudaStream_t st);

    void clone_from(const Pcsr& o, cudaStream_t st) {
        pma.g = o.pma.g;
        pma.nnz = o.pma.nnz;
        pma.alloc(o.pma.g);
        DSA_CUDA(cudaMemcpyAsync(pma.keys.p, o.pma.keys.p, (size_t)pma.g.capacity * 8, cudaMemcpyDeviceToDevice, st));
        DSA_CUDA(cudaMemcpyAsync(pma.vals.p, o.pma.vals.p, (size_t)pma.g.capacity * 8, cudaMemcpyDeviceToDevice, st));
        DSA_CUDA(cudaMemcpyAsync(pma.leafcnt.p, o.pma.leafcnt.p, (size_t)pma.g.nb_segments * 4, cudaMemcpyDeviceToDevice, st));
        pma.copy_destpos_from(o.pma, st);
        nb_partitions = o.nb_partitions;
        slot_key = o.slot_key;
        slot_live = o.slot_live;
        max_inkey = o.max_inkey;
        d_sem.ensure((size_t)nslots() + 1);
        if (nslots()) DSA_CUDA(cudaMemcpyAsync(d_sem.p, o.d_sem.p, (size_t)nslots() * 8, cudaMemcpyDeviceToDevice, st));
        rebuild_live_and_upload(st);
    }
};

// ---------------------------------------------------------------------------------------------
inline int bits_for(uint64_t v) {
    int b = 0;
    while (v) { ++b; v >>= 1; }
    return b;
}

__global__ void __launch_bounds__(256) k_pack_build_keys(const int64_t* __restrict__ partkeys, const int64_t* __restrict__ inkeys, int64_t n,
                                                          int64_t pmin, int64_t kmin, int kb, uint64_t* __restrict__ sk,
                                                          uint32_t* __restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        sk[i] = ((uint64_t)(partkeys[i] - pmin) << kb) | (uint64_t)(inkeys[i] - kmin);
        idx[i] = (uint32_t)i;
    }
}
__global__ void __launch_bounds__(256) k_shift_keys(const uint64_t* __restrict__ sk, int64_t n, int kb, uint64_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = sk[i] >> kb;
}
// left-fold combine of every run, emitted in flattened [sem, col...] order:
//   element with unique index u in partition c (1-based) lands at rank u + c; the semaphore of c at (first u of c) + c - 1
__global__ void __launch_bounds__(256) k_build_flatten(const uint64_t* __restrict__ sk, const uint32_t* __restrict__ perm,
                                                        const int32_t* __restrict__ runflag, const int32_t* __restrict__ uidx,
                                                        const int32_t* __restrict__ partflag, const int32_t* __restrict__ pidx, int64_t n,
                                                        const int64_t* __restrict__ inkeys, const int64_t* __restrict__ partkeys,
                                                        const double* __restrict__ vals, int combine, int with_sems,
                                                        int64_t* __restrict__ out_k, double* __restrict__ out_v,
                                                        int64_t* __restrict__ out_partkey) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !runflag[i]) return;
    const uint32_t src = perm[i];
    double acc = vals[src];
    for (int64_t j = i + 1; j < n && sk[j] == sk[i]; ++j) acc = combine_apply(combine, acc, vals[perm[j]]);
    const int64_t u = uidx[i];
    if (with_sems) {
        const int64_t c = (int64_t)pidx[i] + (partflag[i] ? 1 : 0);   // 1-based partition id (pidx = exclusive scan of partflag)
        out_k[u + c] = inkeys[src];
        out_v[u + c] = acc;
        if (partflag[i]) {
            out_k[u + c - 1] = 0;            // semaphore_key (pcsr.jl:23,39)
            out_v[u + c - 1] = (double)c;    // T(semaphore_id) (pcsr.jl:40)
            out_partkey[c - 1] = partkeys[src];
        }
    } else {
        out_k[u] = inkeys[src];
        out_v[u] = acc;
    }
}

inline int64_t Pcsr::spmspm(PcsrWorkspace& ws, const int64_t* d_xptr, const int64_t* d_xk, const double* d_xv, int64_t ncol, int64_t nx,
                            bool stage, int64_t* d_yptr, int64_t* d_yk, double* d_yv, int64_t cap, cudaStream_t st) {
    if (!d_xptr && nx <= 0) return 0;
    SpmspvWorkspace& w = ws.spx;
    // spans of distinct partitions are disjoint: a column ascending in x has at most (its entries) + capacity / SPX_PIECE
    // pieces, and at most min(ncol, nx) columns have entries
    const int64_t cap_pieces = pma.g.capacity >> SPX_LG_PIECE, busy = std::min(ncol, nx);
    if (nx > INT32_MAX || (busy > 0 && cap_pieces > (INT32_MAX - 1 - nx) / busy))   // piece counts and offsets are scanned in int32
        throw DsaError{DSA_ERR_ARGUMENT, "spmspv: x entries + min(columns, x entries) x capacity / " + std::to_string(SPX_PIECE) +
                                             " exceed the 2^31 - 1 pieces the piece scan indexes"};
    const int64_t nq = nx + busy * cap_pieces + 1;
    const int64_t nblk = (nq + (1 << CMP_LG_SCAN_BLOCK) - 1) >> CMP_LG_SCAN_BLOCK;
    int64_t* info = w.info.ensure((size_t)(SPX_WORDS + ncol + 1));
    int64_t* from = w.span_from.ensure((size_t)nx);
    int64_t* to = w.span_to.ensure((size_t)nx);
    int32_t* np = w.npieces.ensure((size_t)nx);
    int32_t* poff32 = w.piece_off.ensure((size_t)nx);
    int64_t* xcol = d_xptr ? w.xcol.ensure((size_t)nx) : nullptr;
    int64_t* col_piece = w.col_piece.ensure((size_t)ncol + 1);
    int32_t* pcnt = w.pcnt.ensure((size_t)nq);
    int64_t* poff = w.poff.ensure((size_t)nq);
    int64_t* blk = w.blk_sum.ensure((size_t)nblk);
    DSA_CUDA(cudaMemsetAsync(info, 0, SPX_WORDS * sizeof(int64_t), st));
    if (nx > 0)
        DSA_LAUNCH("spmspv_locate", k_spx_locate, grid_for(nx, 256), 256, 0, st, d_xk, nx, d_xptr, ncol, colmap(), d_sem.p, d_next_slot.p,
                   pma.g.capacity, from, to, np, xcol, info);
    exclusive_scan_i32<int32_t>(ws.batch.scan, np, poff32, nx, info + SPX_NPIECES, st);
    DSA_LAUNCH("spmspv_count", k_spx_count, spx_piece_grid(nq), 256, 0, st, pma.keys.p, poff32, np, nx, from, to, info, nq, pcnt);
    DSA_LAUNCH("spmspv_scan", k_compress_scan, (unsigned)nblk, CMP_SCAN_THREADS, 0, st, pcnt, nq, poff, blk);
    DSA_LAUNCH("spmspv_cols", k_spx_cols, grid_for((ncol + 1) * 32, 256), 256, 0, st, d_xptr, ncol, nx, poff32, poff, blk, nq, info, col_piece);
    int64_t* h = w.h_info.ensure((size_t)(SPX_WORDS + ncol + 1));
    DSA_CUDA(cudaMemcpyAsync(h, info, (SPX_WORDS + ncol + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));   // host synchronisation 1: the checks of x and the column product offsets, which cut the rounds
    if (h[SPX_ERR])
        throw DsaError{DSA_ERR_ARGUMENT, d_xptr ? "x_ptr must start at 0, never decrease and end at nnz_x, and x keys must be strictly "
                                                  "ascending inside each column"
                                                : "x keys must be strictly ascending"};
    const int64_t* hc = h + SPX_WORDS;   // hc[c]: first product of column c
    for (int64_t c = 0; c < ncol; ++c)
        if (hc[c + 1] - hc[c] > INT32_MAX)
            throw DsaError{DSA_ERR_ARGUMENT, "spmspv: column " + std::to_string(c) + " has " + std::to_string(hc[c + 1] - hc[c]) +
                                                 " products, more than the 2^31 - 1 the grouping sort indexes"};
    const int64_t total = hc[ncol];
    if (stage) {
        cap = std::min(std::max<int64_t>(cap, 0), total);
        d_yk = ws.tmp_k.ensure((size_t)std::max<int64_t>(cap, 1));
        d_yv = ws.tmp_v.ensure((size_t)std::max<int64_t>(cap, 1));
        d_yptr = d_xptr ? w.yptr.ensure((size_t)ncol + 1) : nullptr;
    }
    if (total == 0 && !d_yptr) return 0;
    // rounds: consecutive columns, at most SPX_ROUND_PRODUCTS products (or one column) and 2^(64 - kb) columns each
    const int kb = bits_for((uint64_t)std::max<int64_t>(max_inkey - 1, 0));
    const int64_t maxcols = kb <= 1 ? INT64_MAX : int64_t(1) << (64 - kb);
    std::vector<int64_t>& cut = w.h_cut;
    cut.assign(1, 0);
    int64_t maxn = 0;
    for (int64_t c0 = 0, c1; c0 < ncol; c0 = c1) {
        for (c1 = c0 + 1; c1 < ncol && c1 - c0 < maxcols && hc[c1 + 1] - hc[c0] <= SPX_ROUND_PRODUCTS; ++c1) {}
        maxn = std::max(maxn, hc[c1] - hc[c0]);
        cut.push_back(c1);
    }
    if (ncol == 0) cut.push_back(0);   // one round without columns: it writes y_ptr[0]
    uint64_t* sk = w.sk.ensure((size_t)maxn);
    uint32_t* perm = w.perm.ensure((size_t)maxn);
    double* prod = w.prod.ensure((size_t)maxn);
    int32_t* head = w.head.ensure((size_t)maxn);
    int32_t* rank = w.rank.ensure((size_t)maxn);
    int64_t* out_k = d_yv ? d_yk : nullptr;
    for (size_t r = 0; r + 1 < cut.size(); ++r) {
        const int64_t c0 = cut[r], nc = cut[r + 1] - c0, n = hc[c0 + nc] - hc[c0];
        if (n == 0) {
            if (d_yptr) DSA_LAUNCH("spmspv_ptr_fill", k_spx_ptr_fill, grid_for(nc + 1, 256), 256, 0, st, info, c0, nc, d_yptr);
            continue;
        }
        DSA_LAUNCH("spmspv_emit", k_spx_emit, spx_piece_grid(nq), 256, 0, st, pma.keys.p, pma.vals.p, poff32, np, from, to, d_xv, nx, xcol,
                   poff, blk, col_piece, c0, nc, kb, hc[c0], info, sk, perm, prod);
        radix_sort_pairs(ws.sort, sk, perm, n, bits_for((uint64_t)(nc - 1)) + kb, st);
        DSA_LAUNCH("flag_run_first", k_flag_run_first, grid_for(n, 256), 256, 0, st, sk, n, head);
        exclusive_scan_i32<int32_t>(ws.batch.scan, head, rank, n, info + SPX_RUNS, st);
        DSA_LAUNCH("spmspv_fold", k_spx_fold, grid_for(n, 256), 256, 0, st, sk, perm, prod, head, rank, n, info, cap, out_k, d_yv, kb, c0, nc,
                   d_yptr);
    }
    if (total == 0) return 0;
    DSA_CUDA(cudaMemcpyAsync(h + SPX_NOUT, info + SPX_NOUT, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));   // host synchronisation 2: the output count
    return h[SPX_NOUT] + h[SPX_RUNS];
}

inline void Pcsr::build_coo_d(PcsrWorkspace& ws, const int64_t* d_inkeys, const int64_t* d_partkeys, const double* d_vals, int64_t n,
                              int combine, cudaStream_t st) {
    if (n == 0) {   // pcsr.jl:443
        init_empty(st);
        return;
    }
    // ranges of both keys -> bit widths of the packed sort key
    int64_t* mm = ws.cs.ensure(CS_WORDS);
    int64_t* hmm = ws.h_cs.ensure(CS_WORDS);
    minmax_i64(d_partkeys, n, mm, st);
    minmax_i64(d_inkeys, n, mm + 2, st);
    DSA_CUDA(cudaMemcpyAsync(hmm, mm, 4 * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    const int64_t pmin = hmm[0], pmax = hmm[1], kmin = hmm[2], kmax = hmm[3];
    if (kmin < 1) throw DsaError{DSA_ERR_ARGUMENT, "in-array keys must be >= 1 (key 0 is the semaphore key, pcsr.jl:23)"};
    const int kb = std::max(1, bits_for((uint64_t)(kmax - kmin)));
    const int pb = std::max(1, bits_for((uint64_t)pmax - (uint64_t)pmin));
    if (kb + pb > 64) throw DsaError{DSA_ERR_ARGUMENT, "key ranges too wide: bits(row range) + bits(column range) must be <= 64"};
    uint64_t* sk = ws.sk.ensure((size_t)n);
    uint32_t* perm = ws.perm.ensure((size_t)n);
    const unsigned gr = grid_for(n, 256);
    DSA_LAUNCH("pack_build_keys", k_pack_build_keys, gr, 256, 0, st, d_partkeys, d_inkeys, n, pmin, kmin, kb, sk, perm);
    radix_sort_pairs(ws.sort, sk, perm, n, kb + pb, st);
    int32_t* runflag = ws.flag32.ensure((size_t)n);
    int32_t* uidx = ws.idx32.ensure((size_t)n);
    int32_t* partflag = ws.rank32.ensure((size_t)n);
    int32_t* pidx = ws.cnt32.ensure((size_t)n);
    int64_t* tot = ws.nuniq.ensure(4);
    DSA_LAUNCH("flag_run_first", k_flag_run_first, gr, 256, 0, st, sk, n, runflag);
    exclusive_scan_i32<int32_t>(ws.batch.scan, runflag, uidx, n, tot, st);
    // partition heads: compare the partition part of the sort key
    uint64_t* skhi = ws.sort.keys_alt.ensure((size_t)n);   // free after the sort
    DSA_LAUNCH("shift_keys", k_shift_keys, gr, 256, 0, st, sk, n, kb, skhi);
    DSA_LAUNCH("flag_part_first", k_flag_part_first, gr, 256, 0, st, skhi, n, runflag, partflag);
    exclusive_scan_i32<int32_t>(ws.batch.scan, partflag, pidx, n, tot + 1, st);
    int64_t h_tot[2];
    DSA_CUDA(cudaMemcpyAsync(h_tot, tot, 16, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    const int64_t nuniq = h_tot[0], nparts = h_tot[1];
    int64_t* fk = ws.u_key.ensure((size_t)(nuniq + nparts));
    double* fv = ws.u_val.ensure((size_t)(nuniq + nparts));
    int64_t* pk = ws.miss_keys.ensure((size_t)nparts);
    DSA_LAUNCH("build_flatten", k_build_flatten, gr, 256, 0, st, sk, perm, runflag, uidx, partflag, pidx, n, d_inkeys, d_partkeys, d_vals,
               combine, 1, fk, fv, pk);
    d_sem.ensure((size_t)nparts + 1);
    pma.build_from_sorted(fk, fv, nuniq + nparts, d_sem.p, st);
    slot_key.resize((size_t)nparts);
    slot_live.assign((size_t)nparts, 1);
    DSA_CUDA(cudaMemcpyAsync(slot_key.data(), pk, (size_t)nparts * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    nb_partitions = nparts;
    max_inkey = kmax;
    rebuild_live_and_upload(st);
}

}  // namespace dsa
