// libdsa — tile-streamed batched setindex! of one PCSR orientation (dense batches: a batch that touches most leaves).
//
// The random-access pipeline (per-partition buckets -> rank + locate in HBM -> apply -> leaf bookkeeping -> leaf merge) moves
// more bytes than one pass over the array once a batch touches about half of the leaves, and moves them as 32-byte sectors.
// Here the array is cut into tiles of TILE_CELLS cells and a batch is applied in two kernels:
//
//   k_tile_assign   one thread per op: column lookup (find(col_keys), pcsr.jl:342) + batch statistics, then the TILE that holds
//                   the op's predecessor cell.  A partition span that lies inside one tile names the tile by itself (two loads of
//                   the semaphore table); a span that straddles tile borders is resolved by probing the first stored cell after
//                   a border (binary search over the borders), not by the gapped search (finds.jl:29-57) over the span in HBM.
//                   The op is dropped into its tile's bucket (fixed capacity: a batch that overflows one falls back).
//   k_tile_merge    one CTA per tile with ops: the tile's KEYS are streamed into shared memory once; every op is located there
//                   (the result of find — hit or predecessor — by a leaf-first search), hits overwrite their value in place or
//                   set their leaf's delete bit (last writer wins by arrival), misses with a value are the leaf's inserts, and
//                   every leaf whose post-batch count stays inside its own density bounds (pma.jl:119-123 with h = 0) is re-laid
//                   at its spread! positions on the spot (pack! + spread!, moves.jl:94-172): these leaves are shared out
//                   over all warps, one lane per cell, and each lane fetches and stores what lands in its own cell.  Leaves
//                   that fail their bounds hand their inserts, in order, to the density tree / window kernels of pma.cuh,
//                   exactly as the random-access pipeline does.  Only modified leaves are written back.
//
// The result is the batch policy's layout (DESIGN.md §4), bit for bit: a leaf accepted at its own level and later covered by a
// larger window is simply re-laid twice (the window kernel reads the merged leaf with no pending inserts).
#pragma once
#include "pcsr.cuh"

namespace dsa {

// ---------------------------------------------------------------------------------------------
// phase 1 of a tile-streamed batch: lookup + statistics (as k_col_lookup) + tile bucket
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 6) k_tile_assign(const int64_t* __restrict__ partkeys, const int64_t* __restrict__ inkeys,
                                                        const double* __restrict__ vals, int64_t n_host, const int64_t* __restrict__ n_dev,
                                                        const ColMap cm, const int64_t* __restrict__ keys, int64_t cap,
                                                        const int64_t* __restrict__ sem, const int32_t* __restrict__ next_slot,
                                                        int64_t nslots, int64_t* __restrict__ cs, int32_t* __restrict__ tcnt,
                                                        TileRec* __restrict__ rec) {
    int64_t n = n_host;
    if (n_dev) n = *n_dev < n_host ? *n_dev : n_host;
    if (blockIdx.x == 0 && threadIdx.x == 0) cs[CS_N] = n;
    int64_t mink = INT64_MAX, maxk = INT64_MIN, maxp = INT64_MIN, maxknz = INT64_MIN, minp = INT64_MAX;
    int miss = 0;
    int bmax = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pk = partkeys[i];
        const int64_t k = inkeys[i];
        const double v = vals[i];
        minp = pk < minp ? pk : minp;
        const int32_t s = cm.slot(pk);
        mink = k < mink ? k : mink;
        maxk = k > maxk ? k : maxk;
        const bool is_set = v != 0.0;   // pcsr.jl:301
        if (is_set) {
            maxp = pk > maxp ? pk : maxp;
            maxknz = k > maxknz ? k : maxknz;
        }
        int64_t ps = -1;
        if (s >= 0) ps = sem[s];
        if (ps < 0) {   // absent column (or a slot without a placed semaphore): the host falls back to the general path
            miss += 1;
            continue;
        }
        if (k < 1) continue;   // refused by the host's validation (statistics) before anything is applied
        const int32_t ns = next_slot ? next_slot[s] : (s + 1 < nslots ? s + 1 : -1);
        const int64_t pe = ns >= 0 ? sem[ns] : cap;   // exclusive end of the span (pcsr.jl:177-186)
        const int64_t from = is_set ? ps + 1 : ps;    // inserts search (sem, end], deletes [sem, end]  (pcsr.jl:305-307)
        const int64_t to = pe - 1;
        int64_t t = ps >> TILE_LG, lo = from, hi = to;
        const int64_t t_last = to >> TILE_LG;
        if (t != t_last) {
            // The span straddles tile borders.  f(b) = key of the first stored cell in [b, end) is non-decreasing over the borders
            // b, and the predecessor of k lies in the tile of the LAST border with f(b) <= k (or in the span's first tile): one
            // probe — a short walk to the right of the border — per step of a binary search over the borders (one border for a
            // span shorter than a tile), instead of the gapped search over the whole span in HBM.
            int64_t blo = t + 1, bhi = t_last;   // border of tile u = u << TILE_LG
            while (blo <= bhi) {
                const int64_t u = (blo + bhi) >> 1;
                int64_t p = u << TILE_LG;
                int64_t kk = keys[p];
                while (kk == GAP_KEY && p < to) kk = keys[++p];
                if (kk != GAP_KEY && kk <= k) {
                    t = u;
                    blo = u + 1;
                } else {
                    bhi = u - 1;
                }
            }
            const int64_t tb0 = t << TILE_LG;
            lo = from > tb0 ? from : tb0;
            hi = to < tb0 + TILE_CELLS - 1 ? to : tb0 + TILE_CELLS - 1;
        }
        const int64_t tb = t << TILE_LG;
        const int li = atomicAdd(&tcnt[t * TILE_CNT_STRIDE], 1);
        bmax = li + 1 > bmax ? li + 1 : bmax;
        if (li < TILE_CAP) {
            int4* out = reinterpret_cast<int4*>(rec + t * TILE_CAP + li);
            const uint64_t ku = (uint64_t)k, vu = (uint64_t)__double_as_longlong(v);
            out[0] = make_int4((int)(uint32_t)ku, (int)(uint32_t)(ku >> 32), (int)(uint32_t)vu, (int)(uint32_t)(vu >> 32));
            out[1] = make_int4((int)(uint32_t)i, s, (int)((uint32_t)(lo - tb) | ((uint32_t)(hi - tb) << 16)), 0);
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

// find (finds.jl:29-57) on the tile in shared memory: position of the hit or of the predecessor of `key` among the stored cells
// of [lo, hi] (all of one partition), else the nearest stored cell to the left of lo (an insert's partition semaphore).
// The reference's gapped binary search probes cells and walks over gaps; here the search first picks the LEAF — fpos[l] is the
// first stored cell at or after the start of leaf l, and "that cell lies in the range and its key is <= key" is monotone in l —
// then scans the leaf's stored cells (its live mask) from the right.  Same result (the answer is a property of the contents),
// a third of the instructions, and no data-dependent walk inside the binary search.
template <int LGS>
__device__ __forceinline__ int tile_find(const int64_t* sk, const uint32_t* live, const uint16_t* fpos, int64_t key, int lo, int hi,
                                         bool* hit) {
    constexpr int S = 1 << LGS;
    *hit = false;
    if (lo <= hi) {
        int a = lo >> LGS, b = hi >> LGS;   // last leaf in (a, b] whose first stored cell is in range with a key <= key; else a
        int best = a;
        ++a;
        while (a <= b) {
            const int mid = (a + b) >> 1;
            const int p = fpos[mid];
            if (p <= hi && sk[p] <= key) {
                best = mid;
                a = mid + 1;
            } else {
                b = mid - 1;
            }
        }
        const int c0 = best << LGS;
        unsigned m = live[best];
        if (lo > c0) m &= ~((1u << (lo - c0)) - 1u);
        if (hi < c0 + S - 1) m &= mask_le(hi - c0);
        while (m) {
            const int q = 31 - __clz(m);
            const int64_t k = sk[c0 + q];
            if (k <= key) {
                *hit = k == key;
                return c0 + q;
            }
            m ^= 1u << q;
        }
        hi = lo - 1;
    }
    int i = hi;
    while (i > 0 && sk[i] == GAP_KEY) --i;   // finds.jl:49-56 (the predecessor lies in this tile by construction)
    return i < 0 ? 0 : i;
}

static_assert(TILE_CAP <= 256 && TILE_CELLS <= 2048, "op indices are stored in 8 bits, tile-local positions in 15");
struct TileSmem {
    int64_t sk[TILE_CELLS];           // the tile's keys (read-only after the load)
    int64_t rkey[TILE_CAP];
    double rval[TILE_CAP];
    union {
        struct {                      // phases B, C: arrival index and slot of every op (last writer wins)
            uint32_t rarr[TILE_CAP];
            int32_t rslot[TILE_CAP];
        } op;
        struct {                      // phases D, R: the leaves re-laid here, and the survivors of each by number
            uint2 leaf[TILE_MAX_LEAVES];   // {survivor mask, spread! mask}, nrelay entries
            uint8_t lid[TILE_MAX_LEAVES];  // ... and the leaf
            uint8_t sidx[TILE_CELLS];      // sidx[leaf cell 0 + i] = the leaf cell of survivor number i
        } lay;
    } u;
    // per leaf
    uint32_t live[TILE_MAX_LEAVES];   // cells stored before the batch
    uint32_t del[TILE_MAX_LEAVES];    // cells blanked by the batch
    uint32_t insm[TILE_MAX_LEAVES];   // merged ranks taken by the inserts (leaves re-laid here)
    int nins[TILE_MAX_LEAVES];        // inserts of the leaf
    int lhead[TILE_MAX_LEAVES];       // first op of the leaf's list (-1 = none)
    uint16_t fpos[TILE_MAX_LEAVES];   // first stored cell at or after the start of the leaf (TILE_CELLS = none)
    // per op
    uint16_t rpos[TILE_CAP];          // tile-local position of the hit / predecessor; bit 15 = hit
    int16_t rnext[TILE_CAP];          // next op of the same leaf (-1 = end)
    uint8_t rstat[TILE_CAP];          // 1 = live insert
    uint8_t rop[TILE_CELLS];          // per re-laid leaf: rop[leaf cell 0 + R] = the op that takes merged rank R
    int nrelay;                       // leaves re-laid here (entries of u.lay.leaf)
};

struct TileArgs {
    int64_t* keys;
    double* vals;
    const TileRec* rec;
    const int32_t* tcnt;
    int64_t* sem;
    const uint8_t* destpos;   // [33][32]: spread! offset of rank r when a leaf holds m elements
    int32_t* leafcnt;
    uint8_t* touched;
    int32_t* inscnt;
    int32_t* ins_first;
    int64_t* ins_key;
    double* ins_val;
    int64_t* ins_pos;
    int64_t* status;
};

// number of the leaf's live inserts ordered before (pp, key): inserts go by (predecessor cell, key)
__device__ __forceinline__ int tile_insert_rank(const TileSmem& s, int head, int pp, int64_t key) {
    int rk = 0;
    for (int o = head; o >= 0; o = s.rnext[o]) {
        if (s.rstat[o]) {
            const int po = s.rpos[o] & 0x7fff;
            rk += (po < pp) || (po == pp && s.rkey[o] < key);
        }
    }
    return rk;
}

// Control flow is data-parallel and kept short (the kernel is bound by instruction issue, not by HBM): op phases run one thread
// per op and only ever walk the list of the ops of the op's own leaf (one or two entries on a uniform batch); the re-laid
// leaves are then shared out over all warps with one lane per cell, and each lane works out what lands in its own cell.
// Only the keys are staged (the searches read them); values are touched where something changes: an overwrite stores its value
// in place, a re-laid leaf is written destination-driven (the r-th survivor, an insert, or a gap per cell), so every cell has
// exactly one writer and a re-laid leaf goes back as full lines.
template <int LGS>
__global__ void __launch_bounds__(TILE_THREADS, TILE_CTAS_PER_SM) k_tile_merge(TileArgs A, Levels L) {
    extern __shared__ __align__(16) unsigned char tile_smem_raw[];
    TileSmem& s = *reinterpret_cast<TileSmem*>(tile_smem_raw);
    const int t = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t tbase = (int64_t)t << TILE_LG;
    constexpr int lgS = LGS, S = 1 << lgS, NL = TILE_CELLS >> lgS;
    const int mn0 = (int)L.mn[0], mx0 = (int)L.mx[0];
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int ROWS = TILE_CELLS / 32, WARPS = TILE_THREADS / 32, RPW = ROWS / WARPS, OPT = TILE_CAP / TILE_THREADS;
    constexpr int VPT = TILE_CELLS / 2 / TILE_THREADS;   // 16-byte key loads per thread

    // ---- A: the tile's keys and the tile's ops, all loads in flight together; live mask per leaf -----------------------
    int nrec = A.tcnt[(int64_t)t * TILE_CNT_STRIDE];
    int4 ra[OPT], rb[OPT];
    {
        // the tile that the CTA taking this one's place will work on: its keys and the head of its bucket are pulled into L2 now
        const int tp = t + TILE_PREFETCH_DIST;
        if (tp < (int)gridDim.x) {
            const char* pk = reinterpret_cast<const char*>(A.keys + ((int64_t)tp << TILE_LG));
            const char* pr = reinterpret_cast<const char*>(A.rec + (int64_t)tp * TILE_CAP);
            if (tid < TILE_CELLS * 8 / 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pk + tid * 128));
            else if (tid < TILE_CELLS * 8 / 128 + 24) asm volatile("prefetch.global.L2 [%0];" ::"l"(pr + (tid - TILE_CELLS * 8 / 128) * 128));
        }
        const uint64_t l2pol = l2_evict_first_policy();
        longlong2 kk[VPT];
        const longlong2* gk = reinterpret_cast<const longlong2*>(A.keys + tbase);
#pragma unroll
        for (int i = 0; i < VPT; ++i) kk[i] = ldg_stream2(gk + tid + i * TILE_THREADS, l2pol);
        if (nrec > TILE_CAP) nrec = TILE_CAP;
#pragma unroll
        for (int i = 0; i < OPT; ++i) {
            const int j = tid + i * TILE_THREADS;
            if (j < nrec) {
                const int4* rp = reinterpret_cast<const int4*>(A.rec + (int64_t)t * TILE_CAP + j);
                ra[i] = rp[0];
                rb[i] = rp[1];
            }
        }
        if (nrec <= 0) return;
#pragma unroll
        for (int i = 0; i < VPT; ++i) reinterpret_cast<longlong2*>(s.sk)[tid + i * TILE_THREADS] = kk[i];
        for (int l = tid; l < NL; l += TILE_THREADS) {
            s.del[l] = 0;
            s.insm[l] = 0;
            s.nins[l] = 0;
            s.lhead[l] = -1;
        }
        if (tid == 0) s.nrelay = 0;
    }
    __syncthreads();
    {   // live masks: a warp reads a row of 32 cells, the first 32/S lanes store the masks of its leaves
        constexpr int G = 32 >> lgS;
        constexpr unsigned gmask = low_bits(S);
#pragma unroll
        for (int i = 0; i < RPW; ++i) {
            const int row = i * WARPS + warp;
            const unsigned b = __ballot_sync(FULL, s.sk[(row << 5) + lane] != GAP_KEY);
            if (lane < G) s.live[row * G + lane] = (b >> (lane << lgS)) & gmask;
        }
    }
    __syncthreads();
    for (int l = tid; l < NL; l += TILE_THREADS) {   // first stored cell at or after the leaf's start (an empty leaf: rare)
        const unsigned m = s.live[l];
        int p = (l << lgS) + __ffs(m) - 1;
        if (m == 0) {
            p = (l + 1) << lgS;
            while (p < TILE_CELLS && s.sk[p] == GAP_KEY) ++p;
        }
        s.fpos[l] = (uint16_t)p;
    }
    __syncthreads();

    // ---- B: every op located in shared memory and pushed on the list of its leaf ---------------------------------------
#pragma unroll
    for (int i = 0; i < OPT; ++i) {
        const int j = tid + i * TILE_THREADS;
        if (j < nrec) {
            const int4 a = ra[i], b = rb[i];
            const int64_t key = (int64_t)((uint64_t)(uint32_t)a.x | ((uint64_t)(uint32_t)a.y << 32));
            const int lo = (int)((uint32_t)b.z & 0xffffu), hi = (int)((uint32_t)b.z >> 16);
            bool hit = false;
            const int pos = tile_find<LGS>(s.sk, s.live, s.fpos, key, lo, hi, &hit);
            s.rkey[j] = key;
            s.rval[j] = __longlong_as_double((long long)((uint64_t)(uint32_t)a.z | ((uint64_t)(uint32_t)a.w << 32)));
            s.u.op.rarr[j] = (uint32_t)b.x;
            s.u.op.rslot[j] = b.y;
            s.rpos[j] = (uint16_t)(pos | (hit ? 0x8000 : 0));
            s.rnext[j] = (int16_t)atomicExch(&s.lhead[pos >> lgS], j);
        }
    }
    __syncthreads();

    // ---- C: last writer wins per key (arrival order); hits overwrite (writes.jl:16-19) or blank (writes.jl:65-68) -------
    for (int j = tid; j < nrec; j += TILE_THREADS) {
        const int64_t key = s.rkey[j];
        const int32_t slot = s.u.op.rslot[j];
        const uint32_t arr = s.u.op.rarr[j];
        const int pp = s.rpos[j];
        const int pos = pp & 0x7fff, l = pos >> lgS;
        bool dead = false;
        for (int o = s.lhead[l]; o >= 0; o = s.rnext[o]) dead |= (s.rkey[o] == key && s.u.op.rslot[o] == slot && s.u.op.rarr[o] > arr);
        const double v = s.rval[j];
        uint8_t st = 0;
        if (!dead) {
            if (pp & 0x8000) {
                if (v != 0.0) A.vals[tbase + pos] = v;   // in place; a re-laid leaf reads it back from there in phase R
                else atomicOr(&s.del[l], 1u << (pos & (S - 1)));
            } else if (v != 0.0) {
                st = 1;
                atomicAdd(&s.nins[l], 1);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(A.vals + tbase + (l << lgS)));   // phase R reads the leaf's values
            }
        }
        s.rstat[j] = st;
    }
    __syncthreads();

    // ---- D: one thread per leaf.  A modified leaf (inserts or deletes) is re-laid here if it has inserts and its post-batch
    //         count m stays inside its own bounds (pma.jl:119-123 with h = 0): it goes on the list of phase R with its
    //         survivors and its spread! mask.  Any other modified leaf is finished here: its deleted cells are blanked, and if
    //         it has inserts they are handed, in order, to the density tree / window kernels. --------------------------------
    for (int l = tid; l < NL; l += TILE_THREADS) {   // NL is a multiple of 32: whole warps
        const int ni = s.nins[l];
        const unsigned dl = s.del[l], surv = s.live[l] & ~dl;
        const int cnt = __popc(surv), m = cnt + ni;
        const bool relay = ni > 0 && m >= mn0 && m <= mx0;
        const unsigned b = __ballot_sync(FULL, relay);
        int base = 0;
        if (lane == 0 && b) base = atomicAdd(&s.nrelay, __popc(b));
        base = __shfl_sync(FULL, base, 0);
        if (ni == 0 && dl == 0) continue;
        const int64_t lg = (int64_t)t * NL + l;
        A.touched[lg] = 1;
        if (relay) {
            A.leafcnt[lg] = m;
            const int i = base + __popc(b & ((1u << lane) - 1u));
            s.u.lay.leaf[i] = make_uint2(surv, L.leafmask[m]);
            s.u.lay.lid[i] = (uint8_t)l;
            continue;
        }
        const int lcell = l << lgS;
        if (dl) {
            A.leafcnt[lg] = cnt;
            for (unsigned d = dl; d; d &= d - 1) A.keys[tbase + lcell + (__ffs(d) - 1)] = GAP_KEY;
        }
        if (ni) {
            const int head = s.lhead[l];
            const int64_t gb = (int64_t)atomicAdd((unsigned long long*)&A.status[ST_NINS], (unsigned long long)ni);
            for (int j = head; j >= 0; j = s.rnext[j]) {
                if (!s.rstat[j]) continue;
                const int pp = s.rpos[j] & 0x7fff;
                const int rk = tile_insert_rank(s, head, pp, s.rkey[j]);
                A.ins_key[gb + rk] = s.rkey[j];
                A.ins_val[gb + rk] = s.rval[j];
                A.ins_pos[gb + rk] = tbase + pp;
            }
            A.inscnt[lg] = ni;
            A.ins_first[lg] = (int32_t)gb;
        }
    }
    //      and the inserts of the leaves re-laid here: merged rank = survivors up to the predecessor cell + inserts ordered before
    for (int j = tid; j < nrec; j += TILE_THREADS) {
        if (!s.rstat[j]) continue;
        const int pp = s.rpos[j] & 0x7fff, l = pp >> lgS;
        const unsigned surv = s.live[l] & ~s.del[l];
        const int m = __popc(surv) + s.nins[l];
        if (m < mn0 || m > mx0) continue;
        const int R = __popc(surv & mask_le(pp & (S - 1))) + tile_insert_rank(s, s.lhead[l], pp, s.rkey[j]);
        s.rop[(l << lgS) + R] = (uint8_t)j;
        atomicOr(&s.insm[l], 1u << R);
    }
    __syncthreads();

    // ---- R: the re-laid leaves (pack! + spread!, moves.jl:94-172), shared out over all warps, 32/S leaves per warp step and
    //         one lane per cell.  Cell q is occupied iff bit q of the spread! mask M is set; it then takes merged rank
    //         r = popc(M below q), which is an insert's (bit r of insm) or else survivor number r - popc(insm below r).  Every
    //         lane loads and stores only its own cell: a survivor's value comes by shuffle from the lane of its old cell (phase
    //         C's in-place overwrites are in global memory), its key from the staged keys. ---------------------------------
    {
        constexpr int G = 32 >> lgS;                       // leaves per warp step
        const int nrelay = s.nrelay;
        const int q = lane & (S - 1), g0 = lane & ~(S - 1);   // this lane's cell in its leaf; the group's first lane
        const unsigned below = (1u << q) - 1u;
        int64_t* const kq = A.keys + tbase + q;
        double* const vq = A.vals + tbase + q;
        for (int i0 = warp * G; i0 < nrelay; i0 += WARPS * G) {   // whole warps: the shuffle and __syncwarp see every lane
            const int i = i0 + (lane >> lgS);
            const bool on = i < nrelay;
            uint2 e = make_uint2(0u, 0u);   // {survivors, spread! mask}
            int lcell = 0;
            double vold = 0.0;              // the cell's value before the re-lay
            if (on) {
                e = s.u.lay.leaf[i];
                lcell = (int)s.u.lay.lid[i] << lgS;
                vold = vq[lcell];
                if ((e.x >> q) & 1u) s.u.lay.sidx[lcell + __popc(e.x & below)] = (uint8_t)q;
            }
            __syncwarp();   // the leaf's survivor numbers are written
            int64_t k = GAP_KEY;
            double v = 0.0;
            int src = -1;   // lane of the survivor that lands here
            if ((e.y >> q) & 1u) {
                const int r = __popc(e.y & below);
                const unsigned insm = s.insm[lcell >> lgS];
                if ((insm >> r) & 1u) {
                    const int o = s.rop[lcell + r];
                    k = s.rkey[o];
                    v = s.rval[o];
                } else {
                    const int c = s.u.lay.sidx[lcell + r - __popc(insm & ((1u << r) - 1u))];
                    k = s.sk[lcell + c];
                    src = g0 + c;
                }
            }
            const double vs = __shfl_sync(FULL, vold, src & 31);   // src < 0: no survivor lands here, vs is not used
            if (on) {
                if (src >= 0) v = vs;
                kq[lcell] = k;
                vq[lcell] = v;
                if (k == 0) A.sem[(int64_t)v - 1] = tbase + lcell + q;   // moves.jl:160-166
            }
        }
    }
}

}  // namespace dsa
