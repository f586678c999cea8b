// libdsa — C ABI (include/dsa.h) over the device structures of pma.cuh / pcsr.cuh.
// Host orchestration only: every data-parallel step is a kernel launched on the handle's stream.
#include <cstdlib>
#include <functional>
#include <memory>
#include <mutex>
#include "pcsr.cuh"
#include "tile.cuh"

namespace dsa {

Prof& prof() {
    static Prof p;
    return p;
}
DevicePool& device_pool(int device) {
    // never destroyed: handles may be released during interpreter shutdown
    static std::mutex mu;
    static std::map<int, DevicePool*>* pools = new std::map<int, DevicePool*>();
    std::lock_guard<std::mutex> lock(mu);
    DevicePool*& p = (*pools)[device];
    if (!p) p = new DevicePool();
    return *p;
}

static thread_local std::string g_last_error;

// ---------------------------------------------------------------------------------------------
// batched setindex! of one orientation (pcsr.jl:341-347 per op), DESIGN.md §4; sequenced by matrix_set_batch_two
// ---------------------------------------------------------------------------------------------
struct BatchStats {
    int64_t missing, minkey, maxkey, maxpart_nz, maxkey_nz, minpart, maxbucket;
};
constexpr int64_t BUCKET_MAX = 256;   // largest per-partition bucket the quadratic in-bucket ranking is used for

// One batched setindex! of one orientation, cut at its two host decisions so that the two orientations of a matrix can
// share each stream synchronisation:
//   phase1_launch  column lookup + batch statistics                     | sync |
//   phase1_finish  validation (nothing mutated yet), new columns        (own syncs, only when columns are created)
//   phase2_launch  sort, last-writer-wins, locate, apply hits, insert bookkeeping, density tree, window selection | sync |
//   phase3         merges / redistribute / resize
struct BatchCtx {
    const int64_t* inkeys = nullptr;
    const int64_t* partkeys = nullptr;
    const double* vals = nullptr;
    int64_t n = 0;                     // number of ops; an UPPER BOUND while n_dev is set and phase 1 has not been read back
    const int64_t* n_dev = nullptr;    // device-side op count (distributed batches: the exchange's receive counts never visit the host)
    BatchStats bs{};
    std::vector<int32_t> new_slots_h;
    bool tile = false;                 // tile-streamed batch (tile.cuh)
    bool no_tile = false;              // the tile-streamed attempt was refused: general path
};

// Tile-streamed batches (tile.cuh): 0 = never, 1 = when the batch is dense enough to touch most leaves (default),
// 2 = whenever the structure allows it (tests).  DSA_TILE overrides the default; dsa_set_tile_mode() changes it at run time.
static int g_tile_mode = [] {
    const char* e = getenv("DSA_TILE");
    return e ? atoi(e) : 1;
}();

static bool tile_eligible(Pcsr& P, const BatchCtx& c) {
    if (g_tile_mode == 0 || c.no_tile || c.n < 2) return false;
    const Geometry& g = P.pma.g;
    if (g.capacity < TILE_CELLS || g.segment_capacity < 8 || g.segment_capacity > 32 || P.nslots() == 0) return false;
    const int64_t ntiles = g.capacity >> TILE_LG;
    // a distributed batch only has an upper bound of its size on the host (W x the largest share): the size of the previous
    // batch of this orientation is the better estimate
    const int64_t n = (c.n_dev && P.last_batch_n > 0) ? std::min(c.n, P.last_batch_n) : c.n;
    if (g_tile_mode >= 2) return n <= ntiles * TILE_CAP;
    if (P.tile_penalty > 0) {   // a recent batch overflowed a tile bucket or created columns: do not pay for the attempt again at once
        P.tile_penalty -= 1;
        return false;
    }
    // measured crossover at config 2's shape (profiles/tile_crossover_r02.log): the random-access pipeline wins below
    // ~capacity/45 ops, one pass over the array above; beyond TILE_CAP/2 ops per tile on average a bucket is likely to overflow
    return n >= g.capacity / 40 && n <= ntiles * (TILE_CAP / 2);
}

static void phase1_launch(Pcsr& P, PcsrWorkspace& ws, BatchCtx& c, cudaStream_t st) {
    int64_t* hcs = ws.h_cs.ensure(CS_WORDS);
    c.tile = tile_eligible(P, c);
    if (c.tile) {   // the buckets are workspace (capacity x 8 bytes): without room for them the batch takes the general path
        try {
            ws.trec.ensure((size_t)(P.pma.g.capacity >> TILE_LG) * TILE_CAP);
        } catch (const DsaError& e) {
            if (e.code != DSA_ERR_OOM) throw;
            c.tile = false;
            c.no_tile = true;
            P.tile_penalty = 64;
        }
    }
    if (c.tile) {
        // one block, one memset: [batch statistics][per-tile op counters]
        const int64_t ntiles = P.pma.g.capacity >> TILE_LG;
        int32_t* blk = ws.bcnt.ensure((size_t)ntiles * TILE_CNT_STRIDE + 1 + 2 * CS_WORDS);
        int64_t* cs = (int64_t*)blk;
        TileRec* rec = ws.trec.ensure((size_t)ntiles * TILE_CAP);
        DSA_CUDA(cudaMemsetAsync(blk, 0, ((size_t)ntiles * TILE_CNT_STRIDE + 1 + 2 * CS_WORDS) * 4, st));
        const int32_t* next_slot = P.nslots() == P.nlive() ? nullptr : P.d_next_slot.p;   // no tombstones: the next slot is s + 1
        // grid-stride over two waves of resident CTAs (6 per SM): 0.449 ms per config-2 step against 0.453 with 16 per SM, 0.464 with 32
        const unsigned assign_grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((c.n + 255) / 256, 148 * 12));
        DSA_LAUNCH("tile_assign", k_tile_assign, assign_grid, 256, 0, st, c.partkeys, c.inkeys, c.vals, c.n, c.n_dev, P.d_live_keys.p,
                   P.d_live_slot.p, P.nlive(), P.keymap(), P.keymap_min, P.keymap_len, P.pma.keys.p, P.pma.g.capacity, P.d_sem.p, next_slot,
                   P.nslots(), cs, blk + 2 * CS_WORDS, rec);
        DSA_CUDA(cudaMemcpyAsync(hcs, cs, CS_WORDS * 8, cudaMemcpyDeviceToHost, st));
        return;
    }
    int32_t* op_slot = ws.op_slot.ensure((size_t)c.n);
    const int64_t ns = P.nslots();
    // one block, one memset: [batch statistics (zero = neutral, pcsr.cuh cs_code)][per-partition bucket counters]
    int32_t* blk = ws.bcnt.ensure((size_t)ns + 1 + 2 * CS_WORDS);
    int64_t* cs = (int64_t*)blk;
    int32_t* bcnt = blk + 2 * CS_WORDS;
    int32_t* lidx = ws.lidx.ensure((size_t)c.n);
    DSA_CUDA(cudaMemsetAsync(blk, 0, ((size_t)ns + 1 + 2 * CS_WORDS) * 4, st));
    DSA_LAUNCH("col_lookup", k_col_lookup, lookup_grid(c.n), 256, 0, st, c.partkeys, c.inkeys, c.vals, c.n, c.n_dev, P.d_live_keys.p,
               P.d_live_slot.p, P.nlive(), P.keymap(), P.keymap_min, P.keymap_len, op_slot, cs, bcnt, lidx);
    DSA_CUDA(cudaMemcpyAsync(hcs, cs, CS_WORDS * 8, cudaMemcpyDeviceToHost, st));
}

static void phase1_read(PcsrWorkspace& ws, BatchCtx& c) {
    const int64_t* hcs = ws.h_cs.p;
    c.bs = BatchStats{hcs[CS_MISSING], cs_min_decode(hcs[CS_MINKEY]), cs_max_decode(hcs[CS_MAXKEY]), cs_max_decode(hcs[CS_MAXPART_NZ]),
                      cs_max_decode(hcs[CS_MAXKEY_NZ]), cs_min_decode(hcs[CS_MINPART]), hcs[CS_MAXBUCKET]};
    if (c.n_dev) {   // the count the kernels used is now known to the host: the remaining phases run on the exact size
        c.n = hcs[CS_N];
        c.n_dev = nullptr;
    }
}

// A tile-streamed attempt is refused when the batch creates columns or overflows a tile's bucket: nothing has been modified
// (k_tile_assign only reads the structure), the batch starts over on the general path.  Returns true if it must be relaunched.
static bool tile_refused(Pcsr& P, BatchCtx& c) {
    P.last_batch_n = c.n;   // exact by now (phase1_read)
    if (!c.tile) return false;
    if (c.bs.missing == 0 && c.bs.maxbucket <= TILE_CAP) return false;
    c.tile = false;
    c.no_tile = true;
    P.tile_penalty = 8;
    return true;
}

// Everything a batch can be refused for, checked on the statistics of phase 1 BEFORE phase1_finish creates columns: a failed
// call leaves the structure unchanged (include/dsa.h).  The bounds are conservative: `missing` counts ops, not distinct keys.
static void phase1_validate(const Pcsr& P, const BatchCtx& c, const char* what) {
    if (c.n <= 0) return;
    if (c.bs.minkey < 1)
        throw DsaError{DSA_ERR_ARGUMENT, std::string(what) + " must be >= 1 (each is an in-array key of one orientation; key 0 is the semaphore key, pcsr.jl:23)"};
    const int64_t slots_after = P.nslots() + std::max<int64_t>(c.bs.missing, 0);
    if (slots_after >= (int64_t(1) << 31)) throw DsaError{DSA_ERR_ARGUMENT, "too many partitions"};
    const int kb = std::max(1, bits_for((uint64_t)c.bs.maxkey - (uint64_t)c.bs.minkey + 1));
    const int pb = std::max(1, bits_for((uint64_t)std::max<int64_t>(slots_after - 1, 1)));
    if (!c.tile && (c.bs.missing > 0 || c.bs.maxbucket > BUCKET_MAX) && kb + pb > 64)   // the radix path packs (slot, key) into one 64-bit sort key
        throw DsaError{DSA_ERR_ARGUMENT, "key range too wide: bits(in-array key range + 1) + bits(#partitions) must be <= 64"};
}

static void phase1_finish(Pcsr& P, PcsrWorkspace& ws, BatchCtx& c, cudaStream_t st) {
    const BatchStats& bs = c.bs;
    const int64_t n = c.n;
    const unsigned gr = grid_for(n, 256);
    c.new_slots_h.clear();
    if (bs.missing > 0) {
        // absent columns: distinct keys in first-arrival order -> addcolumn! plan (pcsr.jl:148-169) on the host mirror
        int32_t* flag = ws.flag32.ensure((size_t)n);
        int32_t* idx = ws.idx32.ensure((size_t)n);
        int64_t* mk = ws.miss_keys.ensure((size_t)bs.missing);
        int64_t* nheads_dev = ws.nuniq.ensure(4) + 3;
        int64_t nheads = 0;
        DSA_LAUNCH("flag_missing", k_flag_missing, gr, 256, 0, st, ws.op_slot.p, c.partkeys, n, flag);
        exclusive_scan_i32<int32_t>(ws.batch.scan, flag, idx, n, nheads_dev, st);
        DSA_LAUNCH("compact_missing", k_compact_missing, gr, 256, 0, st, ws.op_slot.p, c.partkeys, idx, n, mk);
        DSA_CUDA(cudaMemcpyAsync(&nheads, nheads_dev, 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        ws.h_tmp.resize((size_t)nheads);
        DSA_CUDA(cudaMemcpyAsync(ws.h_tmp.data(), mk, (size_t)nheads * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        std::vector<int64_t> distinct;
        {
            std::unordered_set<int64_t> seen;
            seen.reserve(ws.h_tmp.size() * 2);
            for (int64_t k : ws.h_tmp)
                if (seen.insert(k).second) distinct.push_back(k);
        }
        std::vector<int64_t> out_key, out_old;
        std::vector<uint8_t> out_live;
        const int64_t nold = P.nslots();
        const int64_t nnew_slots = colmap_plan(P.slot_key.data(), P.slot_live.data(), nold, distinct.data(), (int64_t)distinct.size(),
                                               out_key, out_live, out_old);
        if (nnew_slots >= (int64_t(1) << 31)) throw DsaError{DSA_ERR_ARGUMENT, "too many partitions"};
        std::vector<int32_t> old2new((size_t)std::max<int64_t>(nold, 1), -1);
        for (int64_t t = 0; t < nnew_slots; ++t) {
            if (out_old[(size_t)t] > 0) old2new[(size_t)out_old[(size_t)t] - 1] = (int32_t)t;
            else if (out_live[(size_t)t]) c.new_slots_h.push_back((int32_t)t);
        }
        DBuf<int64_t> new_sem;
        new_sem.ensure((size_t)nnew_slots + 1);
        DSA_LAUNCH("fill_sem", k_fill_i64, grid_for(nnew_slots, 256), 256, 0, st, new_sem.p, nnew_slots, (int64_t)-1);
        if (nold > 0) {
            int32_t* d_o2n = ws.old2new.ensure((size_t)nold);
            DSA_CUDA(cudaMemcpyAsync(d_o2n, old2new.data(), (size_t)nold * 4, cudaMemcpyHostToDevice, st));
            DSA_LAUNCH("renumber", k_renumber, grid_for(nold, 256), 256, 0, st, P.d_sem.p, d_o2n, nold, new_sem.p, P.pma.vals.p);
        }
        DSA_CUDA(cudaStreamSynchronize(st));
        P.d_sem.swap(new_sem);
        P.slot_key.swap(out_key);
        P.slot_live.swap(out_live);
        P.nb_partitions += (int64_t)distinct.size();
        P.rebuild_live_and_upload(st, &c.new_slots_h);
        // slots changed: look every op up again
        int64_t* cs = ws.cs.ensure(CS_WORDS);   // statistics were already taken
        DSA_LAUNCH("col_lookup", k_col_lookup, lookup_grid(n), 256, 0, st, c.partkeys, (const int64_t*)nullptr, (const double*)nullptr, n,
                   (const int64_t*)nullptr, P.d_live_keys.p, P.d_live_slot.p, P.nlive(), P.keymap(), P.keymap_min, P.keymap_len, ws.op_slot.p, cs,
                   (int32_t*)nullptr, (int32_t*)nullptr);
    }
}

static void phase2_launch(Pcsr& P, PcsrWorkspace& ws, BatchCtx& c, cudaStream_t st) {
    const int64_t n = c.n;
    const int64_t nnew = (int64_t)c.new_slots_h.size();
    const int64_t ntot = n + nnew;
    int32_t* d_new = ws.new_slots.ensure((size_t)nnew + 1);
    if (nnew) DSA_CUDA(cudaMemcpyAsync(d_new, c.new_slots_h.data(), (size_t)nnew * 4, cudaMemcpyHostToDevice, st));
    const int kb = std::max(1, bits_for((uint64_t)c.bs.maxkey - (uint64_t)c.bs.minkey + 1));   // k_make_sortkeys packs key - minkey + 1
    const int pb = std::max(1, bits_for((uint64_t)std::max<int64_t>(P.nslots() - 1, 1)));
    if (c.tile) {
        // one CTA per tile: locate, apply, re-lay the accepted leaves; then the shared tail (density tree, window selection)
        P.pma.prepare_batch_scratch(ws.batch, 0, st);
        ws.batch.ins_key.ensure((size_t)n + 1);
        ws.batch.ins_val.ensure((size_t)n + 1);
        ws.batch.ins_pos.ensure((size_t)n + 1);
        P.pma.ensure_destpos(st);
        const int lgS = ilog2_i64(P.pma.g.segment_capacity);
        void (*kern)(TileArgs, Levels) = lgS == 3 ? k_tile_merge<3> : lgS == 4 ? k_tile_merge<4> : k_tile_merge<5>;
        static std::mutex attr_mu;
        static std::map<std::pair<int, int>, bool> attr_set;
        {
            std::lock_guard<std::mutex> lock(attr_mu);
            bool& done = attr_set[std::make_pair(current_device(), lgS)];
            if (!done) {
                DSA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TileSmem)));
                done = true;
            }
        }
        TileArgs T;
        T.keys = P.pma.keys.p; T.vals = P.pma.vals.p; T.rec = ws.trec.p; T.tcnt = ws.bcnt.p + 2 * CS_WORDS; T.sem = P.d_sem.p;
        T.destpos = P.pma.destpos.p; T.leafcnt = P.pma.leafcnt.p; T.touched = ws.batch.touched; T.inscnt = ws.batch.inscnt;
        T.ins_first = ws.batch.ins_first.p; T.ins_key = ws.batch.ins_key.p; T.ins_val = ws.batch.ins_val.p; T.ins_pos = ws.batch.ins_pos.p;
        T.status = ws.batch.status;
        const int64_t ntiles = P.pma.g.capacity >> TILE_LG;
        DSA_LAUNCH("tile_merge", kern, (unsigned)ntiles, TILE_THREADS, sizeof(TileSmem), st, T, P.pma.levels());
        P.pma.rebalance_launch(ws.batch, st);
        return;
    }
    const unsigned grt = grid_for(ntot, 256);
    int32_t* u_pid = ws.u_pid.ensure((size_t)ntot);
    int64_t* u_key = ws.u_key.ensure((size_t)ntot);
    double* u_val = ws.u_val.ensure((size_t)ntot);
    if (nnew == 0 && c.bs.missing == 0 && c.bs.maxbucket <= BUCKET_MAX) {
        // every partition receives few ops: bucket by partition, rank inside the bucket; superseded writes are flagged dead
        const int64_t ns = P.nslots();
        int32_t* boff = ws.boff.ensure((size_t)ns + 1);
        BucketRec* rec = ws.brec.ensure((size_t)n);
        int32_t* bcnt = ws.bcnt.p + 2 * CS_WORDS;
        exclusive_scan_i32<int32_t>(ws.batch.scan, bcnt, boff, ns, nullptr, st);
        DSA_LAUNCH("bucket_scatter", k_bucket_scatter, grt, 256, 0, st, ws.op_slot.p, ws.lidx.p, c.inkeys, n, boff, rec);
        // rank inside the bucket + locate + overwrite in one kernel, then the shared tail (deletes, insert compaction, density tree)
        P.pma.prepare_batch_scratch(ws.batch, n, st);
        int32_t* f32 = ws.batch.flag32.ensure((size_t)n);
        DSA_LAUNCH("bucket_rank_locate", k_bucket_rank_locate, grt, 256, 0, st, rec, boff, bcnt, n, c.vals, P.pma.keys.p, P.pma.vals.p,
                   P.pma.g.capacity, P.d_sem.p, P.d_next_slot.p, u_key, u_val, ws.batch.op_pos.p, ws.batch.op_flag.p, f32);
        P.pma.apply_located_ops<false>(ws.batch, u_key, u_val, n, P.d_sem.p, st);
        P.pma.rebalance_launch(ws.batch, st);
        return;
    }
    // only the radix path packs (slot, key) into one 64-bit sort key.  A guard, not the refusal: phase1_validate refuses such a
    // batch first, with a partition count at least as large (it counts absent ops, not distinct keys), before any column is
    // created; were this throw ever reached, phase1_finish would already have changed the column map.
    if (kb + pb > 64) throw DsaError{DSA_ERR_ARGUMENT, "key range too wide: bits(in-array key range + 1) + bits(#partitions) must be <= 64"};
    uint64_t* sk = ws.sk.ensure((size_t)ntot);
    uint32_t* perm = ws.perm.ensure((size_t)ntot);
    DSA_LAUNCH("make_sortkeys", k_make_sortkeys, grt, 256, 0, st, ws.op_slot.p, c.inkeys, n, d_new, nnew, c.bs.minkey, kb, sk, perm);
    radix_sort_pairs(ws.sort, sk, perm, ntot, kb + pb, st);
    int32_t* flag = ws.flag32.ensure((size_t)ntot);
    int32_t* uidx = ws.idx32.ensure((size_t)ntot);
    int64_t* nuniq_dev = ws.nuniq.ensure(4) + 2;
    DSA_LAUNCH("flag_run_last", k_flag_run_last, grt, 256, 0, st, sk, ntot, flag);
    exclusive_scan_i32<int32_t>(ws.batch.scan, flag, uidx, ntot, nuniq_dev, st);
    DSA_LAUNCH("gather_unique_ops", k_gather_unique_ops, grt, 256, 0, st, sk, perm, flag, uidx, ntot, n, kb, c.inkeys, c.vals, u_pid,
               u_key, u_val);
    P.pma.apply_sorted_ops(ws.batch, u_pid, u_key, u_val, ntot, P.d_sem.p, P.d_next_slot.p, st, nuniq_dev, /*launch_only=*/true);
}

static void phase3(Pcsr& P, PcsrWorkspace& ws, BatchCtx& c, cudaStream_t st) {
    P.pma.rebalance_finish(ws.batch, P.d_sem.p, st);
    if (c.bs.maxkey > P.max_inkey) P.max_inkey = c.bs.maxkey;
    if (!c.new_slots_h.empty()) P.rebuild_live_and_upload(st);   // the new partitions are placed now: they end the spans before them
}

// ---------------------------------------------------------------------------------------------
// handles
// ---------------------------------------------------------------------------------------------
struct StreamHolder {
    cudaStream_t st = nullptr;
    bool owned = false;
    void create() {   // highest priority: the work a caller waits for (row-major phases, SpMV) goes ahead of the twin stream's
        int least = 0, greatest = 0;
        DSA_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        DSA_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, greatest));
        owned = true;
    }
    void set(cudaStream_t s) {
        if (owned && st) cudaStreamDestroy(st);
        st = s;
        owned = false;
    }
    ~StreamHolder() {
        if (owned && st) cudaStreamDestroy(st);
    }
};

// staging of host batches
struct Staging {
    DBuf<int64_t> a, b;
    DBuf<double> v, out;
};

}  // namespace dsa

using namespace dsa;

struct dsa_vec {
    PmaCore pma;
    int64_t n = 0;   // vector.jl:2
    PcsrWorkspace ws;
    Staging stg;
    StreamHolder sh;
};

struct dsa_matrix {
    Pcsr colmajor, rowmajor;   // matrix.jl:6-7
    int64_t m = 0, n = 0;      // matrix.jl:2-3
    PcsrWorkspace ws, ws2;     // ws2: batch scratch of the row-major twin (both orientations are in flight together)
    Staging stg;
    StreamHolder sh;
    // double-buffered staging of host batches (dsa_matrix_stage_batch / dsa_matrix_apply_staged)
    struct Slot {
        DBuf<int64_t> r, c;
        DBuf<double> v;
        cudaEvent_t ev = nullptr;
        int64_t n = 0;
    } slot[2];
    cudaStream_t copy_st = nullptr;
    int staged_head = 0, staged_count = 0;
    // the column-major orientation's batch phases run on their own stream, forked from / joined to sh.st, when both orientations have ops
    cudaStream_t twin_st = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    ~dsa_matrix() {
        for (auto& s : slot)
            if (s.ev) cudaEventDestroy(s.ev);
        if (copy_st) cudaStreamDestroy(copy_st);
        if (twin_st) cudaStreamDestroy(twin_st);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
    }
    DBuf<int32_t> d_slots;
    DBuf<int64_t> d_ids;
};

#define DSA_TRY try { ::dsa::NvtxRange _nvtx_range(__func__);
#define DSA_CATCH                                                              \
    }                                                                          \
    catch (const DsaError& e) {                                                \
        g_last_error = e.msg;                                                  \
        return e.code;                                                         \
    }                                                                          \
    catch (const std::bad_alloc&) {                                            \
        g_last_error = "host out of memory";                                   \
        return DSA_ERR_OOM;                                                    \
    }                                                                          \
    catch (const std::exception& e) {                                          \
        g_last_error = e.what();                                               \
        return DSA_ERR_INTERNAL;                                               \
    }

static void require_device() {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess || c == 0) {
        cudaGetLastError();
        throw DsaError{DSA_ERR_CUDA, "no CUDA device available: libdsa has no CPU fallback"};
    }
}

template <typename T>
static T* h2d(DBuf<T>& buf, const T* h, int64_t n, cudaStream_t st) {
    T* d = buf.ensure((size_t)std::max<int64_t>(n, 1));
    if (n > 0) DSA_CUDA(cudaMemcpyAsync(d, h, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, st));
    return d;
}

// ---- vector batch (plain PMA): sort by key, last writer wins, merge -----------------------------------------------
static void vec_sorted_unique(dsa_vec* v, const int64_t* d_keys, const double* d_vals, int64_t n, bool build, int combine,
                              int64_t** out_k, double** out_v, int64_t* nuniq_host, int64_t** nuniq_dev, int64_t* maxkey) {
    cudaStream_t st = v->sh.st;
    PcsrWorkspace& ws = v->ws;
    int64_t* mm = ws.cs.ensure(CS_WORDS);
    int64_t* hmm = ws.h_cs.ensure(CS_WORDS);
    minmax_i64(d_keys, n, mm, st);
    DSA_CUDA(cudaMemcpyAsync(hmm, mm, 16, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    const int64_t kmin = hmm[0], kmax = hmm[1];
    if (kmin == GAP_KEY) throw DsaError{DSA_ERR_ARGUMENT, "key typemin(Int64) is reserved"};
    *maxkey = kmax;
    const int nbits = std::max(1, bits_for((uint64_t)kmax - (uint64_t)kmin));
    uint64_t* sk = ws.sk.ensure((size_t)n);
    uint32_t* perm = ws.perm.ensure((size_t)n);
    const unsigned gr = grid_for(n, 256);
    DSA_LAUNCH("make_sortkeys_vec", k_make_sortkeys_vec, gr, 256, 0, st, d_keys, n, kmin, sk, perm);
    radix_sort_pairs(ws.sort, sk, perm, n, nbits, st);
    int32_t* flag = ws.flag32.ensure((size_t)n);
    int32_t* uidx = ws.idx32.ensure((size_t)n);
    int64_t* tot = ws.nuniq.ensure(4) + 2;
    int64_t* uk = ws.u_key.ensure((size_t)n);
    double* uv = ws.u_val.ensure((size_t)n);
    if (build) {
        DSA_LAUNCH("flag_run_first", k_flag_run_first, gr, 256, 0, st, sk, n, flag);
        exclusive_scan_i32<int32_t>(ws.batch.scan, flag, uidx, n, tot, st);
        DSA_LAUNCH("build_flatten", k_build_flatten, gr, 256, 0, st, sk, perm, flag, uidx, (const int32_t*)nullptr, (const int32_t*)nullptr, n,
                   d_keys, (const int64_t*)nullptr, d_vals, combine, 0, uk, uv, (int64_t*)nullptr);
    } else {
        DSA_LAUNCH("flag_run_last", k_flag_run_last, gr, 256, 0, st, sk, n, flag);
        exclusive_scan_i32<int32_t>(ws.batch.scan, flag, uidx, n, tot, st);
        DSA_LAUNCH("gather_unique_ops", k_gather_unique_ops, gr, 256, 0, st, sk, perm, flag, uidx, n, n, 0, d_keys, d_vals, (int32_t*)nullptr, uk,
                   uv);
    }
    *out_k = uk;
    *out_v = uv;
    *nuniq_dev = tot;
    if (nuniq_host) {
        DSA_CUDA(cudaMemcpyAsync(nuniq_host, tot, 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
    }
}

__global__ void __launch_bounds__(256) k_max_key_nonzero(const int64_t* __restrict__ keys, const double* __restrict__ vals, int64_t n,
                                                          int64_t* __restrict__ out) {
    int64_t hi = INT64_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (vals[i] != 0.0 && keys[i] > hi) hi = keys[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t h2 = __shfl_down_sync(0xffffffffu, hi, o);
        hi = h2 > hi ? h2 : hi;
    }
    if ((threadIdx.x & 31) == 0 && hi != INT64_MIN) atomicMax((long long*)out, (long long)hi);
}
__global__ void __launch_bounds__(256) k_max_live_key(const int64_t* __restrict__ keys, int64_t n, int64_t* __restrict__ out) {
    int64_t hi = INT64_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (keys[i] != GAP_KEY && keys[i] > hi) hi = keys[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t h2 = __shfl_down_sync(0xffffffffu, hi, o);
        hi = h2 > hi ? h2 : hi;
    }
    if ((threadIdx.x & 31) == 0 && hi != INT64_MIN) atomicMax((long long*)out, (long long)hi);
}
__global__ void k_set_i64(int64_t* p, int64_t v) { *p = v; }

static void vec_set_batch_dev(dsa_vec* v, const int64_t* d_keys, const double* d_vals, int64_t n) {
    if (n <= 0) return;
    cudaStream_t st = v->sh.st;
    // n = max(n, key) for non-zero writes (vector.jl:77-79)
    int64_t* mx = v->ws.cs.ensure(CS_WORDS) + 6;
    DSA_LAUNCH("set_i64", k_set_i64, 1, 1, 0, st, mx, (int64_t)INT64_MIN);
    DSA_LAUNCH("max_key_nonzero", k_max_key_nonzero, (unsigned)std::min<int64_t>((n + 255) / 256, 1184), 256, 0, st, d_keys, d_vals, n, mx);
    int64_t h_mx = INT64_MIN;
    DSA_CUDA(cudaMemcpyAsync(&h_mx, mx, 8, cudaMemcpyDeviceToHost, st));
    int64_t *uk, *nu_dev, maxkey;
    double* uv;
    vec_sorted_unique(v, d_keys, d_vals, n, false, 0, &uk, &uv, nullptr, &nu_dev, &maxkey);   // syncs (h_mx valid after)
    v->pma.apply_sorted_ops(v->ws.batch, nullptr, uk, uv, n, nullptr, nullptr, st, nu_dev);
    if (h_mx != INT64_MIN && h_mx > v->n) v->n = h_mx;
}

// ---- matrix helpers -----------------------------------------------------------------------------------------------
// One orientation's part of a matrix batch: its structure, its scratch, its ops, the stream its phases run on and the two
// dimensions its keys grow.
struct OrientationBatch {
    Pcsr& P;
    PcsrWorkspace& ws;
    BatchCtx c;
    cudaStream_t st;
    int64_t& part_dim;   // grown by the partition keys of non-zero writes
    int64_t& key_dim;    // grown by the in-array keys of non-zero writes
};

// The orientations that have ops go through the batch phases together so that they share the host decisions.  A plain matrix
// batch feeds both with the same triples; a shard of a distributed matrix feeds them different ones; the delete list of
// deletecolumn! / deleterow! feeds only the twin of the purged orientation.
// nc_dev / nr_dev (nullable): device-side op counts; nc / nr are then upper bounds (distributed batches).
static void matrix_set_batch_two(dsa_matrix* A, const int64_t* rows_c, const int64_t* cols_c, const double* vals_c, int64_t nc,
                                 const int64_t* rows_r, const int64_t* cols_r, const double* vals_r, int64_t nr,
                                 const int64_t* nc_dev = nullptr, const int64_t* nr_dev = nullptr,
                                 const std::function<void()>* pre_mutate = nullptr) {
    cudaStream_t st = A->sh.st;
    // The two orientations are independent (own structure, own workspace), so when both have ops the column-major one runs on a
    // second, low-priority stream that forks from st here; the row-major one stays on st and, being ahead, finishes first.
    const bool two = nc > 0 && nr > 0;
    if (two) {
        if (!A->twin_st) {
            int least = 0, greatest = 0;
            DSA_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
            DSA_CUDA(cudaStreamCreateWithPriority(&A->twin_st, cudaStreamNonBlocking, least));
            DSA_CUDA(cudaEventCreateWithFlags(&A->ev_fork, cudaEventDisableTiming));
            DSA_CUDA(cudaEventCreateWithFlags(&A->ev_join, cudaEventDisableTiming));
        }
        DSA_CUDA(cudaEventRecord(A->ev_fork, st));        // everything queued on st so far (input copies) precedes the twin's work
        DSA_CUDA(cudaStreamWaitEvent(A->twin_st, A->ev_fork, 0));
    }
    // row-major first: rowmajor[col, row] = v (matrix.jl:57-59), then colmajor[row, col] = v (matrix.jl:53-55)
    std::vector<OrientationBatch> obs;
    obs.reserve(2);
    if (nr > 0) obs.push_back({A->rowmajor, A->ws2, {cols_r, rows_r, vals_r, nr, nr_dev}, st, A->m, A->n});
    if (nc > 0) obs.push_back({A->colmajor, A->ws, {rows_c, cols_c, vals_c, nc, nc_dev}, two ? A->twin_st : st, A->n, A->m});
    try {
        for (OrientationBatch& o : obs) phase1_launch(o.P, o.ws, o.c, o.st);
        for (OrientationBatch& o : obs) DSA_CUDA(cudaStreamSynchronize(o.st));
        for (OrientationBatch& o : obs) phase1_read(o.ws, o.c);   // c.n is exact from here on: a distributed batch may bring 0 ops
        // a refused tile-streamed attempt starts over on the general path (nothing was modified)
        std::vector<OrientationBatch*> redo;
        for (OrientationBatch& o : obs)
            if (o.c.n > 0 && tile_refused(o.P, o.c)) redo.push_back(&o);
        for (OrientationBatch* o : redo) phase1_launch(o->P, o->ws, o->c, o->st);
        for (OrientationBatch* o : redo) DSA_CUDA(cudaStreamSynchronize(o->st));
        for (OrientationBatch* o : redo) phase1_read(o->ws, o->c);
        if (pre_mutate) (*pre_mutate)();   // caller-side validation that needs the first host synchronisation (may throw: nothing is mutated yet)
        // validate before mutate: rows are the in-array keys of the col-major structure, columns those of the row-major one
        // (both orientations are checked before either one creates a column; the col-major one first, so that a batch both
        // refuse reports the col-major one's reason)
        for (auto o = obs.rbegin(); o != obs.rend(); ++o)
            if (o->c.n > 0) phase1_validate(o->P, o->c, "row and column keys");
        for (OrientationBatch& o : obs)
            if (o.c.n > 0) phase1_finish(o.P, o.ws, o.c, o.st);
        for (OrientationBatch& o : obs)
            if (o.c.n > 0) phase2_launch(o.P, o.ws, o.c, o.st);
        for (OrientationBatch& o : obs) {   // the row-major orientation's phase 3 is not held back by the other one
            DSA_CUDA(cudaStreamSynchronize(o.st));
            if (o.c.n > 0) phase3(o.P, o.ws, o.c, o.st);
        }
        if (two) {   // later work on st that needs the column-major orientation sees its merges
            DSA_CUDA(cudaEventRecord(A->ev_join, A->twin_st));
            DSA_CUDA(cudaStreamWaitEvent(st, A->ev_join, 0));
        }
    } catch (...) {
        if (two) cudaStreamSynchronize(A->twin_st);
        throw;
    }
    // matrix.jl:44-47: dimensions grow on non-zero writes (the statistics are INT64_MIN when there is none)
    for (OrientationBatch& o : obs)
        if (o.c.n > 0) {
            o.part_dim = std::max(o.part_dim, o.c.bs.maxpart_nz);
            o.key_dim = std::max(o.key_dim, o.c.bs.maxkey_nz);
        }
}
static void matrix_set_batch_dev(dsa_matrix* A, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n) {
    if (n <= 0) return;
    matrix_set_batch_two(A, d_rows, d_cols, d_vals, n, d_rows, d_cols, d_vals, n);
}

static void matrix_delete(dsa_matrix* A, bool rows, const int64_t* ids, int64_t n) {
    if (n <= 0) return;
    cudaStream_t st = A->sh.st;
    Pcsr& primary = rows ? A->rowmajor : A->colmajor;
    // validate before mutate (pcsr.jl:208)
    std::vector<int32_t> slots;
    {
        std::unordered_set<int32_t> seen;
        for (int64_t i = 0; i < n; ++i) {
            int32_t s = primary.host_lookup(ids[i]);
            if (s < 0) throw DsaError{DSA_ERR_ARGUMENT, (rows ? "row " : "column ") + std::to_string(ids[i]) + " does not exist."};
            if (!seen.insert(s).second) throw DsaError{DSA_ERR_ARGUMENT, "column listed twice."};
            slots.push_back(s);
        }
    }
    int32_t* d_slots = A->d_slots.ensure((size_t)n);
    int64_t* d_ids = A->d_ids.ensure((size_t)n);
    DSA_CUDA(cudaMemcpyAsync(d_slots, slots.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    DSA_CUDA(cudaMemcpyAsync(d_ids, ids, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    // entries to delete from the twin: for (row, val) in view(matrix, :, col): rowmajor[col, row] = 0  (matrix.jl:97-99)
    // gathered into the primary orientation's own workspace: the twin's batch runs on the other one and reads the list in place
    PcsrWorkspace& pws = rows ? A->ws2 : A->ws;
    const int64_t tot = primary.gather_spans(pws, d_slots, n, d_ids, false, st);
    if (tot > 0) {
        // twin partition key = in-array key of the primary cell (tmp_k), twin in-array key = deleted id (tmp_owner), value 0.0
        DBuf<double> zeros;
        zeros.ensure((size_t)tot);
        DSA_CUDA(cudaMemsetAsync(zeros.p, 0, (size_t)tot * 8, st));
        if (rows) matrix_set_batch_two(A, pws.tmp_owner.p, pws.tmp_k.p, zeros.p, tot, nullptr, nullptr, nullptr, 0);
        else matrix_set_batch_two(A, nullptr, nullptr, nullptr, 0, pws.tmp_k.p, pws.tmp_owner.p, zeros.p, tot);
        DSA_CUDA(cudaStreamSynchronize(st));
    }
    primary.delete_slots(A->ws, slots, d_slots, st);   // deletecolumn!(colmajor, col)  (matrix.jl:100)
}

static void matrix_spmv_slots(dsa_matrix* A, int trans, const double* d_x, const uint8_t* d_mask, int64_t nx) {
    // mat * x sums, per row, over ascending columns (operations.jl:97-103): that is a segmented reduction over the
    // ROW-major twin; transpose(mat) * x is the same over the column-major structure.
    Pcsr& P = trans ? A->colmajor : A->rowmajor;
    P.spmv_slots(A->ws, d_x, d_mask, nx, A->sh.st);
}

extern "C" {

int dsa_version(void) { return 100; }
const char* dsa_last_error(void) { return g_last_error.c_str(); }
int dsa_device_count(int* count_out) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        cudaGetLastError();
        c = 0;
    }
    *count_out = c;
    return DSA_OK;
}
int dsa_set_device(int device) {
    DSA_TRY
    DSA_CUDA(cudaSetDevice(device));
    return DSA_OK;
    DSA_CATCH
}

// ---- host logic ----------------------------------------------------------------------------------------------------
int dsa_pma_geometry(int64_t nb_elements, int64_t* out4) {
    Geometry g = geometry_for_build(nb_elements);
    out4[0] = g.capacity; out4[1] = g.segment_capacity; out4[2] = g.nb_segments; out4[3] = g.height;
    return DSA_OK;
}
int dsa_level_bounds(int64_t segment_capacity, int64_t height, int64_t* mn, int64_t* mx) {
    if (height < 1 || height >= MAX_LEVELS) { g_last_error = "height out of range"; return DSA_ERR_ARGUMENT; }
    level_bounds(segment_capacity, height, (T_H - T_0) / (double)height, (P_H - P_0) / (double)height, mn, mx);
    return DSA_OK;
}
int64_t dsa_spread_dest(int64_t c, int64_t m, int64_t r) { return spread_dest(spread_make(c, m), r); }
int64_t dsa_spread_rank(int64_t c, int64_t m, int64_t p) { return spread_rank_at(spread_make(c, m), p); }
int64_t dsa_colmap_plan(const int64_t* slot_key, const uint8_t* slot_live, int64_t nslots, const int64_t* new_keys, int64_t nnew,
                        int64_t* out_key, uint8_t* out_live, int64_t* out_old) {
    std::vector<int64_t> k, o;
    std::vector<uint8_t> l;
    int64_t n = colmap_plan(slot_key, slot_live, nslots, new_keys, nnew, k, l, o);
    for (int64_t i = 0; i < n; ++i) { out_key[i] = k[(size_t)i]; out_live[i] = l[(size_t)i]; out_old[i] = o[(size_t)i]; }
    return n;
}

// ---- vector -----------------------------------------------------------------------------------------------------------
int dsa_vec_create(int64_t expected_nb_elems, dsa_vec_t** out) {
    DSA_TRY
    require_device();
    std::unique_ptr<dsa_vec> v(new dsa_vec());
    v->sh.create();
    v->pma.alloc(geometry_for_build(0, expected_nb_elems > 0 ? expected_nb_elems : 100));
    v->pma.nnz = 0;
    DSA_LAUNCH("layout_build", k_layout, grid_for(v->pma.g.capacity, 256), 256, 0, v->sh.st, v->pma.keys.p, v->pma.vals.p, v->pma.g.capacity,
               (int64_t)0, (const int64_t*)v->pma.keys.p, (const double*)v->pma.vals.p, v->pma.leafcnt.p, (int64_t*)nullptr,
               ilog2_i64(v->pma.g.segment_capacity));
    DSA_CUDA(cudaStreamSynchronize(v->sh.st));
    *out = v.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_build(const int64_t* keys, const double* vals, int64_t n, int combine, int64_t len, int len_given, dsa_vec_t** out) {
    DSA_TRY
    require_device();
    if (n < 0) throw DsaError{DSA_ERR_ARGUMENT, "negative length"};
    std::unique_ptr<dsa_vec> v(new dsa_vec());
    v->sh.create();
    cudaStream_t st = v->sh.st;
    if (n == 0) {
        v->pma.build_from_sorted(nullptr, nullptr, 0, nullptr, st);
        v->n = len_given ? len : 0;
    } else {
        int64_t* dk = h2d(v->stg.a, keys, n, st);
        double* dv = h2d(v->stg.v, vals, n, st);
        int64_t *uk, *nu_dev, nu = 0, maxkey = 0;
        double* uv;
        vec_sorted_unique(v.get(), dk, dv, n, true, combine, &uk, &uv, &nu, &nu_dev, &maxkey);
        v->pma.build_from_sorted(uk, uv, nu, nullptr, st);
        v->n = len_given ? len : std::max<int64_t>(maxkey, 0);   // _guess_length (vector.jl:6) = maximum(keys; init = 0)
    }
    DSA_CUDA(cudaStreamSynchronize(st));
    *out = v.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_destroy(dsa_vec_t* v) {
    delete v;
    return DSA_OK;
}
int dsa_vec_clone(const dsa_vec_t* v, dsa_vec_t** out) {
    DSA_TRY
    std::unique_ptr<dsa_vec> c(new dsa_vec());
    c->sh.create();
    cudaStream_t st = c->sh.st;
    DSA_CUDA(cudaStreamSynchronize(v->sh.st));
    c->pma.alloc(v->pma.g);
    c->pma.nnz = v->pma.nnz;
    c->n = v->n;
    DSA_CUDA(cudaMemcpyAsync(c->pma.keys.p, v->pma.keys.p, (size_t)v->pma.g.capacity * 8, cudaMemcpyDeviceToDevice, st));
    DSA_CUDA(cudaMemcpyAsync(c->pma.vals.p, v->pma.vals.p, (size_t)v->pma.g.capacity * 8, cudaMemcpyDeviceToDevice, st));
    DSA_CUDA(cudaMemcpyAsync(c->pma.leafcnt.p, v->pma.leafcnt.p, (size_t)v->pma.g.nb_segments * 4, cudaMemcpyDeviceToDevice, st));
    c->pma.copy_destpos_from(v->pma, st);
    DSA_CUDA(cudaStreamSynchronize(st));
    *out = c.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_set_stream(dsa_vec_t* v, void* cuda_stream) {
    v->sh.set((cudaStream_t)cuda_stream);
    return DSA_OK;
}
int dsa_vec_set_batch(dsa_vec_t* v, const int64_t* keys, const double* vals, int64_t n) {
    DSA_TRY
    if (n <= 0) return DSA_OK;
    cudaStream_t st = v->sh.st;
    int64_t* dk = h2d(v->stg.a, keys, n, st);
    double* dv = h2d(v->stg.v, vals, n, st);
    vec_set_batch_dev(v, dk, dv, n);
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_set_batch_d(dsa_vec_t* v, const int64_t* d_keys, const double* d_vals, int64_t n) {
    DSA_TRY
    vec_set_batch_dev(v, d_keys, d_vals, n);
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_get_batch(dsa_vec_t* v, const int64_t* keys, int64_t n, double* out) {
    DSA_TRY
    if (n <= 0) return DSA_OK;
    cudaStream_t st = v->sh.st;
    int64_t* dk = h2d(v->stg.a, keys, n, st);
    double* dout = v->stg.out.ensure((size_t)n);
    DSA_LAUNCH("get", k_get, grid_for(n, 256), 256, 0, st, v->pma.keys.p, v->pma.vals.p, v->pma.g.capacity, (const int32_t*)nullptr, dk, n,
                   (const int64_t*)nullptr, (const int32_t*)nullptr, dout);
    DSA_CUDA(cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_info(const dsa_vec_t* v, int64_t* out6) {
    out6[0] = v->pma.g.capacity; out6[1] = v->pma.g.segment_capacity; out6[2] = v->pma.g.nb_segments;
    out6[3] = v->pma.nnz; out6[4] = v->pma.g.height; out6[5] = v->n;
    return DSA_OK;
}
int dsa_vec_nonzeros(dsa_vec_t* v, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out) {
    DSA_TRY
    // the compaction of the matrices' compressed snapshot without semaphores: a vector keeps every non-gap cell
    const int64_t n = v->pma.nnz;
    *count_out = n;
    if (n > 0 && keys_out && n <= cap) {
        cudaStream_t st = v->sh.st;
        int64_t* ck = v->ws.tmp_k.ensure((size_t)n);
        double* cv = v->ws.tmp_v.ensure((size_t)n);
        compress_cells<false>(v->ws.cmp, v->pma.keys.p, v->pma.vals.p, v->pma.g.capacity, CompressBounds{}, 0, nullptr, nullptr, 0, n, ck,
                              cv, st);
        DSA_CUDA(cudaMemcpyAsync(keys_out, ck, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaMemcpyAsync(vals_out, cv, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
    }
    return DSA_OK;
    DSA_CATCH
}
int dsa_vec_shrink_size(dsa_vec_t* v, int64_t* n_out) {
    DSA_TRY
    cudaStream_t st = v->sh.st;
    int64_t* mx = v->ws.cs.ensure(CS_WORDS);
    DSA_LAUNCH("set_i64", k_set_i64, 1, 1, 0, st, mx, (int64_t)INT64_MIN);
    DSA_LAUNCH("max_live_key", k_max_live_key, (unsigned)std::min<int64_t>((v->pma.g.capacity + 255) / 256, 1184), 256, 0, st, v->pma.keys.p,
               v->pma.g.capacity, mx);
    int64_t h = 0;
    DSA_CUDA(cudaMemcpyAsync(&h, mx, 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    v->n = h == INT64_MIN ? 0 : std::max<int64_t>(h, 0);   // mapreduce(max; init = zero(K))  (vector.jl:7-8)
    *n_out = v->n;
    return DSA_OK;
    DSA_CATCH
}
static void export_cells(Staging& stg, const PmaCore& p, uint8_t* occ, int64_t* keys, double* vals, cudaStream_t st) {
    const int64_t cap = p.g.capacity;
    DBuf<uint8_t> d_occ;
    d_occ.ensure((size_t)cap);
    int64_t* dk = stg.a.ensure((size_t)cap);
    double* dv = stg.v.ensure((size_t)cap);
    DSA_LAUNCH("export_cells", k_export_cells, grid_for(cap, 256), 256, 0, st, p.keys.p, p.vals.p, cap, d_occ.p, dk, dv);
    DSA_CUDA(cudaMemcpyAsync(occ, d_occ.p, (size_t)cap, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaMemcpyAsync(keys, dk, (size_t)cap * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaMemcpyAsync(vals, dv, (size_t)cap * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
}
int dsa_vec_export(dsa_vec_t* v, uint8_t* occupied, int64_t* keys, double* vals) {
    DSA_TRY
    export_cells(v->stg, v->pma, occupied, keys, vals, v->sh.st);
    return DSA_OK;
    DSA_CATCH
}

// ---- matrix -----------------------------------------------------------------------------------------------------------
int dsa_matrix_create(dsa_matrix_t** out) {
    DSA_TRY
    require_device();
    std::unique_ptr<dsa_matrix> A(new dsa_matrix());
    A->sh.create();
    A->colmajor.init_empty(A->sh.st);
    A->rowmajor.init_empty(A->sh.st);
    DSA_CUDA(cudaStreamSynchronize(A->sh.st));
    *out = A.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_build_coo(const int64_t* rows, const int64_t* cols, const double* vals, int64_t n, int64_t m, int64_t ncols, int dims_given,
                         int combine, dsa_matrix_t** out) {
    DSA_TRY
    require_device();
    if (n < 0) throw DsaError{DSA_ERR_ARGUMENT, "negative length"};
    std::unique_ptr<dsa_matrix> A(new dsa_matrix());
    A->sh.create();
    cudaStream_t st = A->sh.st;
    int64_t* dr = h2d(A->stg.a, rows, n, st);
    int64_t* dc = h2d(A->stg.b, cols, n, st);
    double* dv = h2d(A->stg.v, vals, n, st);
    if (n > 0) {
        int64_t* mm = A->ws.cs.ensure(CS_WORDS);
        int64_t* hmm = A->ws.h_cs.ensure(CS_WORDS);
        minmax_i64(dr, n, mm, st);
        minmax_i64(dc, n, mm + 2, st);
        DSA_CUDA(cudaMemcpyAsync(hmm, mm, 32, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        if (hmm[0] < 1 || hmm[2] < 1)
            throw DsaError{DSA_ERR_ARGUMENT, "row and column keys must be >= 1 (each is an in-array key of one orientation; key 0 is the semaphore key, pcsr.jl:23)"};
        A->m = dims_given ? m : hmm[1];        // _guess_length (vector.jl:6)
        A->n = dims_given ? ncols : hmm[3];
    } else {
        A->m = dims_given ? m : 0;
        A->n = dims_given ? ncols : 0;
    }
    A->colmajor.build_coo_d(A->ws, dr, dc, dv, n, combine, st);   // dynamicsparsecolmajor(I, J, V)  (matrix.jl:17)
    A->rowmajor.build_coo_d(A->ws, dc, dr, dv, n, combine, st);   // dynamicsparsecolmajor(J, I, V)
    DSA_CUDA(cudaStreamSynchronize(st));
    *out = A.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_destroy(dsa_matrix_t* A) {
    delete A;
    return DSA_OK;
}
int dsa_matrix_clone(const dsa_matrix_t* A, dsa_matrix_t** out) {
    DSA_TRY
    std::unique_ptr<dsa_matrix> C(new dsa_matrix());
    C->sh.create();
    DSA_CUDA(cudaStreamSynchronize(A->sh.st));
    C->colmajor.clone_from(A->colmajor, C->sh.st);
    C->rowmajor.clone_from(A->rowmajor, C->sh.st);
    C->m = A->m;
    C->n = A->n;
    DSA_CUDA(cudaStreamSynchronize(C->sh.st));
    *out = C.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_set_stream(dsa_matrix_t* A, void* cuda_stream) {
    A->sh.set((cudaStream_t)cuda_stream);
    return DSA_OK;
}
int dsa_matrix_set_batch(dsa_matrix_t* A, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n) {
    DSA_TRY
    if (n <= 0) return DSA_OK;
    cudaStream_t st = A->sh.st;
    int64_t* dr = h2d(A->stg.a, rows, n, st);
    int64_t* dc = h2d(A->stg.b, cols, n, st);
    double* dv = h2d(A->stg.v, vals, n, st);
    matrix_set_batch_dev(A, dr, dc, dv, n);
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_stage_batch(dsa_matrix_t* A, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n) {
    DSA_TRY
    if (A->staged_count >= 2) throw DsaError{DSA_ERR_ERROR, "two batches are already staged: call dsa_matrix_apply_staged first"};
    if (n < 0) throw DsaError{DSA_ERR_ARGUMENT, "negative length"};
    if (!A->copy_st) DSA_CUDA(cudaStreamCreateWithFlags(&A->copy_st, cudaStreamNonBlocking));
    dsa_matrix::Slot& s = A->slot[(A->staged_head + A->staged_count) & 1];
    if (!s.ev) DSA_CUDA(cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming));
    s.n = n;
    int64_t* dr = s.r.ensure((size_t)std::max<int64_t>(n, 1));
    int64_t* dc = s.c.ensure((size_t)std::max<int64_t>(n, 1));
    double* dv = s.v.ensure((size_t)std::max<int64_t>(n, 1));
    if (n > 0) {
        DSA_CUDA(cudaMemcpyAsync(dr, rows, (size_t)n * 8, cudaMemcpyHostToDevice, A->copy_st));
        DSA_CUDA(cudaMemcpyAsync(dc, cols, (size_t)n * 8, cudaMemcpyHostToDevice, A->copy_st));
        DSA_CUDA(cudaMemcpyAsync(dv, vals, (size_t)n * 8, cudaMemcpyHostToDevice, A->copy_st));
    }
    DSA_CUDA(cudaEventRecord(s.ev, A->copy_st));
    A->staged_count += 1;
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_apply_staged(dsa_matrix_t* A) {
    DSA_TRY
    if (A->staged_count <= 0) throw DsaError{DSA_ERR_ERROR, "no staged batch"};
    dsa_matrix::Slot& s = A->slot[A->staged_head & 1];
    A->staged_head ^= 1;
    A->staged_count -= 1;
    DSA_CUDA(cudaStreamWaitEvent(A->sh.st, s.ev, 0));
    matrix_set_batch_dev(A, s.r.p, s.c.p, s.v.p, s.n);
    DSA_CUDA(cudaStreamSynchronize(A->sh.st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_set_batch_d(dsa_matrix_t* A, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n) {
    DSA_TRY
    matrix_set_batch_dev(A, d_rows, d_cols, d_vals, n);
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_get_batch(dsa_matrix_t* A, int which, const int64_t* rows, const int64_t* cols, int64_t n, double* out) {
    DSA_TRY
    if (n <= 0) return DSA_OK;
    cudaStream_t st = A->sh.st;
    int64_t* dr = h2d(A->stg.a, rows, n, st);
    int64_t* dc = h2d(A->stg.b, cols, n, st);
    double* dout = A->stg.out.ensure((size_t)n);
    if (which == DSA_COLMAJOR) A->colmajor.get_batch_d(A->ws, dr, dc, n, dout, st);
    else A->rowmajor.get_batch_d(A->ws, dc, dr, n, dout, st);
    DSA_CUDA(cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_delete_columns(dsa_matrix_t* A, const int64_t* cols, int64_t n) {
    DSA_TRY
    matrix_delete(A, false, cols, n);
    DSA_CUDA(cudaStreamSynchronize(A->sh.st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_delete_rows(dsa_matrix_t* A, const int64_t* rows, int64_t n) {
    DSA_TRY
    matrix_delete(A, true, rows, n);
    DSA_CUDA(cudaStreamSynchronize(A->sh.st));
    return DSA_OK;
    DSA_CATCH
}
static int matrix_span(dsa_matrix_t* A, Pcsr& P, int64_t id, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out) {
    DSA_TRY
    cudaStream_t st = A->sh.st;
    *count_out = 0;
    const int32_t s = P.host_lookup(id);
    if (s < 0) return DSA_OK;   // empty view (views.jl:11-12)
    int32_t* d_s = A->d_slots.ensure(1);
    DSA_CUDA(cudaMemcpyAsync(d_s, &s, 4, cudaMemcpyHostToDevice, st));
    const int64_t tot = P.gather_spans(A->ws, d_s, 1, nullptr, true, st);
    *count_out = tot;
    if (tot > 0 && keys_out && tot <= cap) {
        DSA_CUDA(cudaMemcpyAsync(keys_out, A->ws.tmp_k.p, (size_t)tot * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaMemcpyAsync(vals_out, A->ws.tmp_v.p, (size_t)tot * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
    }
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_column(dsa_matrix_t* A, int64_t col, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out) {
    return matrix_span(A, A->colmajor, col, keys_out, vals_out, cap, count_out);
}
int dsa_matrix_row(dsa_matrix_t* A, int64_t row, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out) {
    return matrix_span(A, A->rowmajor, row, keys_out, vals_out, cap, count_out);
}
int dsa_matrix_spmv(dsa_matrix_t* A, int trans, const int64_t* x_keys, const double* x_vals, int64_t nx, int64_t* y_keys, double* y_vals,
                    int64_t cap, int64_t* count_out) {
    DSA_TRY
    cudaStream_t st = A->sh.st;
    Pcsr& P = trans ? A->colmajor : A->rowmajor;
    *count_out = 0;
    const int64_t dim = std::max<int64_t>(P.max_inkey, 1);
    // x as a dense buffer indexed by key (one load per cell) as long as the key space is not far larger than the data; beyond
    // that (ids around 1e10 through a key codec: a dense x would not fit, the reference's Dict does) x stays a sorted list
    // and every cell looks its key up by binary search
    const bool lookup = dim > (int64_t(1) << 26) && dim > 16 * (nx + P.pma.nnz + 1);
    if (lookup) {
        for (int64_t i = 1; i < nx; ++i)
            if (x_keys[i] <= x_keys[i - 1]) throw DsaError{DSA_ERR_ARGUMENT, "x keys must be strictly ascending"};
        int64_t* dk = h2d(A->stg.a, x_keys, nx, st);
        double* dv = h2d(A->stg.v, x_vals, nx, st);
        P.spmv_slots(A->ws, dv, nullptr, nx, st, dk);
    } else {
        double* xd = A->ws.xdense.ensure((size_t)dim);
        uint8_t* xm = A->ws.xmask.ensure((size_t)dim);
        DSA_CUDA(cudaMemsetAsync(xd, 0, (size_t)dim * 8, st));
        DSA_CUDA(cudaMemsetAsync(xm, 0, (size_t)dim, st));
        if (nx > 0) {
            int64_t* dk = h2d(A->stg.a, x_keys, nx, st);
            double* dv = h2d(A->stg.v, x_vals, nx, st);
            DSA_LAUNCH("scatter_x", k_scatter_x, grid_for(nx, 256), 256, 0, st, dk, dv, nx, xd, xm, dim);
        }
        matrix_spmv_slots(A, trans, xd, xm, dim);
    }
    const int64_t ns = P.nslots();
    if (ns == 0) return DSA_OK;
    int32_t* flag = A->ws.flag32.ensure((size_t)ns);
    int32_t* idx = A->ws.idx32.ensure((size_t)ns);
    int64_t* tot = A->ws.nuniq.ensure(4);
    DSA_LAUNCH("flag_touched", k_flag_touched, grid_for(ns, 256), 256, 0, st, A->ws.ycnt.p, P.d_sem.p, ns, flag);
    exclusive_scan_i32<int32_t>(A->ws.batch.scan, flag, idx, ns, tot, st);
    int64_t h_tot = 0;
    DSA_CUDA(cudaMemcpyAsync(&h_tot, tot, 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    *count_out = h_tot;
    if (h_tot > 0 && y_keys && h_tot <= cap) {
        int64_t* yk = A->ws.tmp_k.ensure((size_t)h_tot);
        double* yv = A->ws.tmp_v.ensure((size_t)h_tot);
        DSA_LAUNCH("compact_y", k_compact_y, grid_for(ns, 256), 256, 0, st, A->ws.yslot.p, P.d_slot_key.p, flag, idx, ns, yk, yv);
        DSA_CUDA(cudaMemcpyAsync(y_keys, yk, (size_t)h_tot * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaMemcpyAsync(y_vals, yv, (size_t)h_tot * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
    }
    return DSA_OK;
    DSA_CATCH
}
static void spmv_dense_dev(dsa_matrix_t* A, int trans, const double* d_x, int64_t nx, double* d_y, int64_t ny) {
    cudaStream_t st = A->sh.st;
    Pcsr& P = trans ? A->colmajor : A->rowmajor;
    DSA_CUDA(cudaMemsetAsync(d_y, 0, (size_t)ny * 8, st));
    P.spmv_dense(A->ws, d_x, nx, d_y, 1, ny + 1, st);
}
int dsa_matrix_spmv_dense(dsa_matrix_t* A, int trans, const double* x, int64_t nx, double* y, int64_t ny) {
    DSA_TRY
    cudaStream_t st = A->sh.st;
    double* dx = h2d(A->stg.v, x, nx, st);
    double* dy = A->stg.out.ensure((size_t)std::max<int64_t>(ny, 1));
    spmv_dense_dev(A, trans, dx, nx, dy, ny);
    if (ny > 0) DSA_CUDA(cudaMemcpyAsync(y, dy, (size_t)ny * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_spmv_dense_d(dsa_matrix_t* A, int trans, const double* d_x, int64_t nx, double* d_y, int64_t ny) {
    DSA_TRY
    spmv_dense_dev(A, trans, d_x, nx, d_y, ny);
    return DSA_OK;
    DSA_CATCH
}
// Columns per pass over the matrix: the pass's partials take (slots + chunks) x 8 B per column of workspace
static constexpr int64_t SPMM_COLS_PER_PASS = 32;
static void check_spmm_args(int64_t nx, int64_t k, int64_t ldx, int64_t ny, int64_t ldy) {
    if (nx < 0 || ny < 0 || k < 0 || ldx < k || ldy < k)
        throw DsaError{DSA_ERR_ARGUMENT, "spmm_dense: need nx >= 0, ny >= 0, k >= 0, ldx >= k and ldy >= k"};
}
// X row-major with ld % 4 == 0, 32-byte aligned, every row readable up to column k rounded up to 4
static void spmm_dense_run(dsa_matrix_t* A, int trans, const double* X, int64_t nx, int64_t k, int64_t ld, double* d_Y, int64_t ny,
                           int64_t ldy) {
    cudaStream_t st = A->sh.st;
    Pcsr& P = trans ? A->colmajor : A->rowmajor;
    if (ny > 0) DSA_CUDA(cudaMemset2DAsync(d_Y, (size_t)ldy * 8, 0, (size_t)k * 8, (size_t)ny, st));
    for (int64_t c0 = 0; c0 < k; c0 += SPMM_COLS_PER_PASS)
        P.spmm_dense_pass(A->ws, nx > 0 ? X + c0 : X, nx, ld, (int)std::min(SPMM_COLS_PER_PASS, k - c0), d_Y + c0, ldy, 1, ny + 1, st);
}
static void spmm_dense_dev(dsa_matrix_t* A, int trans, const double* d_X, int64_t nx, int64_t k, int64_t ldx, double* d_Y, int64_t ny,
                           int64_t ldy) {
    if (k == 1 && ldx == 1 && ldy == 1) {   // one contiguous vector: the single-vector product itself
        spmv_dense_dev(A, trans, d_X, nx, d_Y, ny);
        return;
    }
    // a cell reads 4 consecutive entries of its row of X with one 256-bit load: other layouts are re-laid with ld = k rounded up
    // to 4 (the padding columns are read, their results dropped)
    if (nx > 0 && (k % 4 != 0 || ldx % 4 != 0 || (uintptr_t)d_X % 32 != 0)) {
        const int64_t ld = (k + 3) / 4 * 4;
        double* xp = A->ws.xpad.ensure((size_t)(nx * ld));
        DSA_CUDA(cudaMemcpy2DAsync(xp, (size_t)ld * 8, d_X, (size_t)ldx * 8, (size_t)k * 8, (size_t)nx, cudaMemcpyDeviceToDevice,
                                   A->sh.st));
        spmm_dense_run(A, trans, xp, nx, k, ld, d_Y, ny, ldy);
    } else {
        spmm_dense_run(A, trans, d_X, nx, k, ldx, d_Y, ny, ldy);
    }
}
int dsa_matrix_spmm_dense(dsa_matrix_t* A, int trans, const double* X, int64_t nx, int64_t k, int64_t ldx, double* Y, int64_t ny,
                          int64_t ldy) {
    DSA_TRY
    check_spmm_args(nx, k, ldx, ny, ldy);
    if (k == 0) return DSA_OK;
    cudaStream_t st = A->sh.st;
    // staged in the layout the kernel reads in place: ld = k rounded up to 4 (a single column stays a contiguous vector)
    const int64_t lds = k == 1 ? 1 : (k + 3) / 4 * 4;
    double* dx = A->stg.v.ensure((size_t)std::max<int64_t>(nx * lds, 1));
    if (nx > 0)
        DSA_CUDA(cudaMemcpy2DAsync(dx, (size_t)lds * 8, X, (size_t)ldx * 8, (size_t)k * 8, (size_t)nx, cudaMemcpyHostToDevice, st));
    double* dy = A->stg.out.ensure((size_t)std::max<int64_t>(ny * k, 1));
    if (k == 1) spmv_dense_dev(A, trans, dx, nx, dy, ny);
    else spmm_dense_run(A, trans, dx, nx, k, lds, dy, ny, k);
    if (ny > 0)
        DSA_CUDA(cudaMemcpy2DAsync(Y, (size_t)ldy * 8, dy, (size_t)k * 8, (size_t)k * 8, (size_t)ny, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_spmm_dense_d(dsa_matrix_t* A, int trans, const double* d_X, int64_t nx, int64_t k, int64_t ldx, double* d_Y, int64_t ny,
                            int64_t ldy) {
    DSA_TRY
    check_spmm_args(nx, k, ldx, ny, ldy);
    if (k > 0) spmm_dense_dev(A, trans, d_X, nx, k, ldx, d_Y, ny, ldy);
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_get_stream(const dsa_matrix_t* A, void** cuda_stream_out) {
    *cuda_stream_out = (void*)A->sh.st;
    return DSA_OK;
}
int dsa_matrix_info(const dsa_matrix_t* A, int which, int64_t* out10) {
    const Pcsr& P = which == DSA_COLMAJOR ? A->colmajor : A->rowmajor;
    out10[0] = P.pma.g.capacity; out10[1] = P.pma.g.segment_capacity; out10[2] = P.pma.g.nb_segments; out10[3] = P.pma.nnz;
    out10[4] = P.pma.g.height; out10[5] = P.nb_partitions; out10[6] = P.nslots(); out10[7] = A->m; out10[8] = A->n; out10[9] = P.nnz();
    return DSA_OK;
}
int dsa_matrix_export(dsa_matrix_t* A, int which, uint8_t* occupied, int64_t* keys, double* vals, int64_t* semaphores, int64_t* col_keys,
                      uint8_t* col_live) {
    DSA_TRY
    Pcsr& P = which == DSA_COLMAJOR ? A->colmajor : A->rowmajor;
    cudaStream_t st = A->sh.st;
    export_cells(A->stg, P.pma, occupied, keys, vals, st);
    const int64_t ns = P.nslots();
    if (ns > 0) {
        DSA_CUDA(cudaMemcpyAsync(semaphores, P.d_sem.p, (size_t)ns * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        for (int64_t s = 0; s < ns; ++s) {
            semaphores[s] = (P.slot_live[(size_t)s] && semaphores[s] >= 0) ? semaphores[s] + 1 : 0;   // 1-based, 0 = nothing
            col_keys[s] = P.slot_live[(size_t)s] ? P.slot_key[(size_t)s] : 0;
            col_live[s] = P.slot_live[(size_t)s];
        }
    }
    return DSA_OK;
    DSA_CATCH
}

// ---- compressed snapshot (K8, pcsr.cuh) -------------------------------------------------------------------------------
static Pcsr& orientation(dsa_matrix_t* A, int which) {
    if (which != DSA_COLMAJOR && which != DSA_ROWMAJOR) throw DsaError{DSA_ERR_ARGUMENT, "which must be DSA_COLMAJOR or DSA_ROWMAJOR"};
    return which == DSA_COLMAJOR ? A->colmajor : A->rowmajor;
}
// both counts are known on the host; a buffer whose required length is 0 may be NULL
static bool compress_fits(Pcsr& P, const int64_t* part_keys, const int64_t* ptr, const int64_t* keys, const double* vals, int64_t cap_parts,
                          int64_t cap_nnz, int64_t* counts_out2) {
    const int64_t np = P.nlive(), nnz = P.nnz();
    counts_out2[0] = np;
    counts_out2[1] = nnz;
    return ptr && cap_parts >= np && cap_nnz >= nnz && (np == 0 || part_keys) && (nnz == 0 || (keys && vals));
}
static bool compress_dense_fits(Pcsr& P, int64_t dim, int64_t idim, int base, const int64_t* ptr, const int64_t* ind, const double* vals,
                                int64_t cap_nnz, int64_t* nnz_out) {
    if (base != 0 && base != 1) throw DsaError{DSA_ERR_ARGUMENT, "compress_dense: base must be 0 or 1"};
    if (dim < 0 || idim < 0) throw DsaError{DSA_ERR_ARGUMENT, "compress_dense: dim and idim must be >= 0"};
    const int64_t nnz = P.nnz();
    *nnz_out = nnz;
    return ptr && cap_nnz >= nnz && (nnz == 0 || (ind && vals));
}
int dsa_matrix_compress(dsa_matrix_t* A, int which, int64_t* part_keys, int64_t* ptr, int64_t* keys, double* vals, int64_t cap_parts,
                        int64_t cap_nnz, int64_t* counts_out2) {
    DSA_TRY
    Pcsr& P = orientation(A, which);
    if (!compress_fits(P, part_keys, ptr, keys, vals, cap_parts, cap_nnz, counts_out2)) return DSA_OK;
    cudaStream_t st = A->sh.st;
    const int64_t np = counts_out2[0], nnz = counts_out2[1];
    int64_t* dptr = A->stg.b.ensure((size_t)np + 1);
    int64_t* dk = A->stg.a.ensure((size_t)std::max<int64_t>(nnz, 1));
    double* dv = A->stg.v.ensure((size_t)std::max<int64_t>(nnz, 1));
    P.compress_sparse(A->ws, nullptr, dptr, dk, dv, st);
    if (np > 0) memcpy(part_keys, P.live_keys_h.data(), (size_t)np * 8);
    DSA_CUDA(cudaMemcpyAsync(ptr, dptr, (size_t)(np + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (nnz > 0) {
        DSA_CUDA(cudaMemcpyAsync(keys, dk, (size_t)nnz * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaMemcpyAsync(vals, dv, (size_t)nnz * 8, cudaMemcpyDeviceToHost, st));
    }
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_compress_d(dsa_matrix_t* A, int which, int64_t* d_part_keys, int64_t* d_ptr, int64_t* d_keys, double* d_vals, int64_t cap_parts,
                          int64_t cap_nnz, int64_t* counts_out2) {
    DSA_TRY
    Pcsr& P = orientation(A, which);
    if (compress_fits(P, d_part_keys, d_ptr, d_keys, d_vals, cap_parts, cap_nnz, counts_out2))
        P.compress_sparse(A->ws, d_part_keys, d_ptr, d_keys, d_vals, A->sh.st);
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_compress_dense(dsa_matrix_t* A, int which, int64_t dim, int64_t idim, int base, int64_t* ptr, int64_t* ind, double* vals,
                              int64_t cap_nnz, int64_t* nnz_out) {
    DSA_TRY
    Pcsr& P = orientation(A, which);
    if (!compress_dense_fits(P, dim, idim, base, ptr, ind, vals, cap_nnz, nnz_out)) return DSA_OK;
    cudaStream_t st = A->sh.st;
    const int64_t nnz = *nnz_out;
    int64_t* dptr = A->stg.b.ensure((size_t)dim + 1);
    int64_t* di = A->stg.a.ensure((size_t)std::max<int64_t>(nnz, 1));
    double* dv = A->stg.v.ensure((size_t)std::max<int64_t>(nnz, 1));
    P.compress_dense(A->ws, dim, idim, base, dptr, di, dv, st);
    DSA_CUDA(cudaMemcpyAsync(ptr, dptr, (size_t)(dim + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (nnz > 0) {
        DSA_CUDA(cudaMemcpyAsync(ind, di, (size_t)nnz * 8, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaMemcpyAsync(vals, dv, (size_t)nnz * 8, cudaMemcpyDeviceToHost, st));
    }
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_matrix_compress_dense_d(dsa_matrix_t* A, int which, int64_t dim, int64_t idim, int base, int64_t* d_ptr, int64_t* d_ind, double* d_vals,
                                int64_t cap_nnz, int64_t* nnz_out) {
    DSA_TRY
    Pcsr& P = orientation(A, which);
    if (compress_dense_fits(P, dim, idim, base, d_ptr, d_ind, d_vals, cap_nnz, nnz_out))
        P.compress_dense(A->ws, dim, idim, base, d_ptr, d_ind, d_vals, A->sh.st);
    return DSA_OK;
    DSA_CATCH
}

// ---- measurement ------------------------------------------------------------------------------------------------------
int dsa_trim_memory(void) {
    DSA_TRY
    cudaDeviceSynchronize();
    device_pool(current_device()).trim();
    return DSA_OK;
    DSA_CATCH
}
int64_t dsa_cached_bytes(void) { return (int64_t)device_pool(current_device()).cached_bytes; }
int64_t dsa_launch_count(void) { return prof().launches; }
int dsa_set_tile_mode(int mode) {
    const int prev = g_tile_mode;
    g_tile_mode = mode;
    return prev;
}
int dsa_prof_enable(int on) {
    if (!on) prof().resolve();
    prof().enabled = on != 0;
    return DSA_OK;
}
int dsa_prof_reset(void) {
    prof().resolve();
    prof().entries.clear();
    return DSA_OK;
}
int64_t dsa_prof_dump(char* buf, int64_t cap) {
    prof().resolve();
    std::string s;
    for (auto& kv : prof().entries) {
        char line[256];
        snprintf(line, sizeof(line), "%s,%lld,%.6f\n", kv.first.c_str(), (long long)kv.second.count, kv.second.ms);
        s += line;
    }
    if (buf && cap > 0) {
        size_t n = std::min<size_t>(s.size(), (size_t)cap - 1);
        memcpy(buf, s.data(), n);
        buf[n] = 0;
    }
    return (int64_t)s.size() + 1;
}

}  // extern "C"

#include "dist_api.cuh"
