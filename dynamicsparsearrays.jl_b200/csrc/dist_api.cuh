// libdsa — host side of the multi-GPU entry points (include/dsa.h, "multi-GPU"): handles, peer-memory exchange set-up,
// the routed batch, the gathered SpMV, routed deletes / reads / bulk build.  Included by libdsa.cu (needs dsa_matrix).
#pragma once
#include <functional>
#include "dist.cuh"

struct dsa_dist {
    ncclComm_t comm = nullptr;
    bool own_comm = false;
    int rank = 0, world = 1;
    int transport = 0;   // 0 = peer-memory stores (CUDA IPC), 1 = ncclSend/ncclRecv
    ~dsa_dist() {
        if (own_comm && comm) dsa::nccl().CommDestroy(comm);
    }
};

struct dsa_dmatrix {
    dsa_dist* ctx = nullptr;
    dsa_matrix* A = nullptr;   // this rank's shards (owned)
    int64_t m = 0, n = 0;
    std::vector<int64_t> split[2];   // [0] col_split, [1] row_split: world + 1 first-owned keys
    bool even[2] = {true, true};
    int64_t per[2] = {0, 0};         // widest shard (slice length of the SpMV gather buffer)
    dsa::RouteTables T{};
    int64_t region_cap = 0;          // = max_share
    int64_t words_per_parity = 0;    // words of one slot of the receive regions
    int64_t* xbuf = nullptr;         // receive regions, DIST_SLOTS slots (plain cudaMalloc: exported through CUDA IPC)
    int64_t* peer[dsa::DIST_MAX_RANKS] = {nullptr};   // every rank's xbuf as mapped here (own = xbuf)
    int64_t seq = 0;                 // batches routed so far: batch s uses slot s % DIST_SLOTS
    int row_stride = 0;              // words per rank in the count matrix: 2 * world counts + flags
    struct Routed { int slot; int64_t n; int omask; };
    std::vector<Routed> staged;      // routed (pushed) but not applied yet, oldest first: at most 2
    cudaStream_t xst = nullptr;      // routing + peer stores run here, so that they overlap the previous batch's pipeline
    cudaEvent_t ev_main = nullptr, ev_routed[3] = {nullptr, nullptr, nullptr};
    dsa::DBuf<int32_t> tile_cnt, tile_off;
    dsa::DBuf<int64_t> counts, rx_n, misc;
    dsa::HPinned<int64_t> h_counts, h_misc;
    dsa::DBuf<int64_t> rx_rows[2], rx_cols[2];
    dsa::DBuf<double> rx_vals[2];
    dsa::DBuf<int64_t> sendbuf;      // nccl transport: local staging in the receive-region layout
    dsa::DBuf<int64_t> stg_r[3], stg_c[3];   // device copies of staged HOST shares, one set per slot
    dsa::DBuf<double> stg_v[3];
    dsa::DBuf<double> ybuf, dtmp;
    dsa::DBuf<int64_t> itmp, itmp2;
    dsa::DBuf<double> ztmp;
    ~dsa_dmatrix() {
        cudaDeviceSynchronize();
        if (ctx)
            for (int r = 0; r < ctx->world; ++r)
                if (r != ctx->rank && peer[r]) cudaIpcCloseMemHandle(peer[r]);
        if (xbuf) cudaFree(xbuf);
        if (xst) cudaStreamDestroy(xst);
        if (ev_main) cudaEventDestroy(ev_main);
        for (auto& e : ev_routed)
            if (e) cudaEventDestroy(e);
        delete A;
    }
};

namespace dsa {

// Receive regions, count matrices and send staging exist in 3 slots (batch s uses slot s % 3).  A rank may route batch s+1
// while batch s is still being applied anywhere: its stores go to slot (s+1) % 3, whose last reader on any peer was the unpack
// of batch s-2, and that unpack precedes the peer's contribution to the count all-gather of batch s-1, which this rank has
// seen complete (it has returned from applying batch s-1) before it can route batch s+1.
constexpr int DIST_SLOTS = 3;

static void dist_all_gather(dsa_dist* d, const void* send, void* recv, size_t count, ncclDataType_t t, cudaStream_t st) {
    if (d->world == 1) {
        const size_t bytes = count * (t == ncclInt8 || t == ncclUint8 ? 1 : 8);
        if (send != recv) DSA_CUDA(cudaMemcpyAsync(recv, send, bytes, cudaMemcpyDeviceToDevice, st));
        return;
    }
    DSA_NCCL(nccl().AllGather(send, recv, count, t, d->comm, st));
}
static void dist_all_reduce(dsa_dist* d, void* buf, size_t count, ncclDataType_t t, ncclRedOp_t op, cudaStream_t st) {
    if (d->world == 1) return;
    DSA_NCCL(nccl().AllReduce(buf, buf, count, t, op, d->comm, st));
}

// collective: max over ranks of a host integer (host-synchronous; set-up and cold paths only)
static int64_t dist_host_max(dsa_dmatrix* D, int64_t v, cudaStream_t st) {
    if (D->ctx->world == 1) return v;
    int64_t* d = D->misc.ensure(8);
    int64_t* h = D->h_misc.ensure(8);
    h[0] = v;
    DSA_CUDA(cudaMemcpyAsync(d, h, 8, cudaMemcpyHostToDevice, st));
    dist_all_reduce(D->ctx, d, 1, ncclInt64, ncclMax, st);
    DSA_CUDA(cudaMemcpyAsync(h, d, 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return h[0];
}

// receive regions + peer mappings (collective)
static void dist_setup_exchange(dsa_dmatrix* D, int64_t max_share, cudaStream_t st) {
    dsa_dist* d = D->ctx;
    const int W = d->world;
    D->region_cap = std::max<int64_t>(max_share, 1);
    D->words_per_parity = (int64_t)2 * W * 3 * D->region_cap;
    D->row_stride = 2 * W + 4;   // 2 W send counts, bad-key flag, wide-key flag, packed flag (what the sender actually used), pad
    DSA_CUDA(cudaMalloc(&D->xbuf, (size_t)D->words_per_parity * DIST_SLOTS * 8));
    D->peer[d->rank] = D->xbuf;
    D->counts.ensure((size_t)DIST_SLOTS * W * D->row_stride);
    D->h_counts.ensure((size_t)DIST_SLOTS * W * D->row_stride);
    D->rx_n.ensure(4);
    DSA_CUDA(cudaMemsetAsync(D->counts.p, 0, (size_t)DIST_SLOTS * W * D->row_stride * 8, st));
    DSA_CUDA(cudaStreamCreateWithFlags(&D->xst, cudaStreamNonBlocking));
    DSA_CUDA(cudaEventCreateWithFlags(&D->ev_main, cudaEventDisableTiming));
    for (auto& e : D->ev_routed) DSA_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    const char* tr = getenv("DSA_DIST_TRANSPORT");
    int want_p2p = !(tr && std::string(tr) == "nccl");
    if (W > 1) {
        // CUDA IPC: every rank publishes the handle of its receive buffer; peers map it and store into it directly
        cudaIpcMemHandle_t mine;
        memset(&mine, 0, sizeof(mine));
        int ok = want_p2p;
        if (want_p2p && cudaIpcGetMemHandle(&mine, D->xbuf) != cudaSuccess) {
            cudaGetLastError();
            ok = 0;
        }
        const size_t hb = sizeof(cudaIpcMemHandle_t);   // 64 bytes
        DBuf<uint8_t> dh;
        dh.ensure(hb * W);
        std::vector<uint8_t> all(hb * W);
        DSA_CUDA(cudaMemcpyAsync(dh.p + hb * d->rank, &mine, hb, cudaMemcpyHostToDevice, st));
        dist_all_gather(d, dh.p + hb * d->rank, dh.p, hb, ncclUint8, st);
        DSA_CUDA(cudaMemcpyAsync(all.data(), dh.p, hb * W, cudaMemcpyDeviceToHost, st));
        DSA_CUDA(cudaStreamSynchronize(st));
        if (ok) {
            for (int r = 0; r < W && ok; ++r) {
                if (r == d->rank) continue;
                cudaIpcMemHandle_t h;
                memcpy(&h, all.data() + hb * r, hb);
                void* p = nullptr;
                if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                    cudaGetLastError();
                    ok = 0;
                } else {
                    D->peer[r] = (int64_t*)p;
                }
            }
        }
        // every rank must use the same transport: peer stores only if everybody mapped everybody
        const int64_t all_ok = -dist_host_max(D, ok ? 0 : 1, st) + 1;
        if (!all_ok) {
            for (int r = 0; r < W; ++r)
                if (r != d->rank && D->peer[r]) {
                    cudaIpcCloseMemHandle(D->peer[r]);
                    D->peer[r] = nullptr;
                }
            d->transport = 1;
        } else {
            d->transport = 0;
        }
    }
    const int64_t bound = (int64_t)W * D->region_cap;
    for (int o = 0; o < 2; ++o) {
        D->rx_rows[o].ensure((size_t)bound);
        D->rx_cols[o].ensure((size_t)bound);
        D->rx_vals[o].ensure((size_t)bound);
    }
    if (d->transport == 1) D->sendbuf.ensure((size_t)D->words_per_parity * DIST_SLOTS);
}

// First half of the exchange, on the routing stream: count, scan, and push this rank's (rows, cols, vals)[n] into the owners'
// receive regions (orientations in omask).  Nothing here waits for the host or for a collective.
static void dist_route(dsa_dmatrix* D, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n, int omask) {
    dsa_dist* d = D->ctx;
    const int W = d->world;
    if (D->staged.size() >= 2) throw DsaError{DSA_ERR_ERROR, "two batches are already staged: call dsa_dmatrix_apply_staged first"};
    // A share larger than the receive regions cannot be pushed.  The refusal must be COLLECTIVE (a rank that threw here alone
    // would leave its peers waiting in the count all-gather): the rank routes nothing and raises its flag in the count row;
    // every rank sees it after the all-gather and refuses the batch.
    const bool oversize = n > D->region_cap;
    if (oversize) n = 0;
    cudaStream_t st = D->A->sh.st, xs = D->xst;
    const int slot = (int)(D->seq % DIST_SLOTS);
    D->seq += 1;
    DSA_CUDA(cudaEventRecord(D->ev_main, st));   // the share is ready in the handle's stream order
    DSA_CUDA(cudaStreamWaitEvent(xs, D->ev_main, 0));
    RouteTables T = D->T;
    T.omask = omask;
    int64_t* row = D->counts.p + ((size_t)slot * W + d->rank) * D->row_stride;
    DSA_CUDA(cudaMemsetAsync(row, 0, (size_t)D->row_stride * 8, xs));
    const int64_t ntiles = (n + RT_TILE - 1) / RT_TILE;
    PushTargets P;
    memset(&P, 0, sizeof(P));
    for (int r = 0; r < W; ++r) {
        if (d->transport == 0) {
            P.base[r] = D->peer[r] + (size_t)slot * D->words_per_parity;
            P.region[r] = d->rank;
        } else {
            P.base[r] = D->sendbuf.p + (size_t)slot * D->words_per_parity;
            P.region[r] = r;
        }
    }
    if (n > 0) {
        int32_t* tc = D->tile_cnt.ensure((size_t)ntiles * 2 * W);
        int32_t* to = D->tile_off.ensure((size_t)ntiles * 2 * W);
        DSA_LAUNCH("route_count", k_route_count, (unsigned)ntiles, RT_THREADS, 0, xs, d_rows, d_cols, n, T, tc, row + 2 * W);
        DSA_LAUNCH("route_scan", k_route_scan, (unsigned)(2 * W), 1024, 0, xs, (const int32_t*)tc, ntiles, W, to, row);
        // peer-memory transport: 16-byte ops when every key of the share fits 32 bits (decided on the device by k_route_count)
        int64_t* wide = d->transport == 0 ? row + 2 * W + 1 : nullptr;
        DSA_LAUNCH("route_push", k_route_push, (unsigned)ntiles, RT_THREADS, 0, xs, d_rows, d_cols, d_vals, n, T, (const int32_t*)to, P,
                   D->region_cap, wide);
    }
    if (oversize) {
        static const int64_t two = 2;
        DSA_CUDA(cudaMemcpyAsync(row + 2 * W, &two, 8, cudaMemcpyHostToDevice, xs));
    }
    DSA_CUDA(cudaEventRecord(D->ev_routed[slot], xs));
    D->staged.push_back(dsa_dmatrix::Routed{slot, n, omask});
}

static int64_t* dist_host_counts(dsa_dmatrix* D, int slot) { return D->h_counts.p + (size_t)slot * D->ctx->world * D->row_stride; }

// Second half, on the handle's stream: the count all-gather (the only collective of the exchange, and the barrier behind which
// every peer's stores are complete) and the unpack of what this rank received into rx_{rows,cols,vals}[o] (rank-major, arrival
// order) with the counts in rx_n[o] (device).  Returns true when the host already knows the receive counts (nccl transport).
static bool dist_complete(dsa_dmatrix* D, const dsa_dmatrix::Routed& R, int64_t* hn0, int64_t* hn1) {
    dsa_dist* d = D->ctx;
    const int W = d->world;
    cudaStream_t st = D->A->sh.st;
    const int slot = R.slot;
    DSA_CUDA(cudaStreamWaitEvent(st, D->ev_routed[slot], 0));
    int64_t* cmat = D->counts.p + (size_t)slot * W * D->row_stride;
    int64_t* row = cmat + (size_t)d->rank * D->row_stride;
    dist_all_gather(d, row, cmat, (size_t)D->row_stride, ncclInt64, st);
    int64_t* hc = dist_host_counts(D, slot);
    DSA_CUDA(cudaMemcpyAsync(hc, cmat, (size_t)W * D->row_stride * 8, cudaMemcpyDeviceToHost, st));   // read at the next host sync
    if (d->transport == 0) {
        DSA_LAUNCH("dist_unpack", k_dist_unpack, dim3(148 * 2, 2), 256, 0, st, (const int64_t*)cmat, D->row_stride, W, d->rank,
                   (const int64_t*)(D->xbuf + (size_t)slot * D->words_per_parity), D->region_cap, D->rx_rows[0].p, D->rx_cols[0].p,
                   D->rx_vals[0].p, D->rx_rows[1].p, D->rx_cols[1].p, D->rx_vals[1].p, D->rx_n.p);
        return false;
    }
    // nccl transport: exact sizes need the counts on the host
    DSA_CUDA(cudaStreamSynchronize(st));
    const int64_t* sendbuf = D->sendbuf.p + (size_t)slot * D->words_per_parity;
    int64_t tot[2] = {0, 0};
    if (W > 1) DSA_NCCL(nccl().GroupStart());
    for (int o = 0; o < 2; ++o) {
        int64_t off = 0;
        for (int s = 0; s < W; ++s) {
            const int64_t rc = hc[(size_t)s * D->row_stride + o * W + d->rank];   // what s sends me
            const int64_t sc = hc[(size_t)d->rank * D->row_stride + o * W + s];   // what I send s
            for (int a = 0; a < 3; ++a) {
                int64_t* dst = (a == 0 ? D->rx_rows[o].p : a == 1 ? D->rx_cols[o].p : (int64_t*)D->rx_vals[o].p) + off;
                const int64_t* src = sendbuf + region_word(o, s, a, W, D->region_cap);
                if (s == d->rank) {
                    if (rc > 0) DSA_CUDA(cudaMemcpyAsync(dst, src, (size_t)rc * 8, cudaMemcpyDeviceToDevice, st));
                } else {
                    if (sc > 0) DSA_NCCL(nccl().Send(src, (size_t)sc, ncclInt64, s, d->comm, st));
                    if (rc > 0) DSA_NCCL(nccl().Recv(dst, (size_t)rc, ncclInt64, s, d->comm, st));
                }
            }
            off += rc;
        }
        tot[o] = off;
    }
    if (W > 1) DSA_NCCL(nccl().GroupEnd());
    *hn0 = tot[0];
    *hn1 = tot[1];
    return true;
}

// 0 = fine, 1 = some rank passed a key < 1, 2 = some rank passed a share larger than max_share (identical on every rank)
static int dist_refusal(dsa_dmatrix* D, int slot) {
    const int W = D->ctx->world;
    const int64_t* hc = dist_host_counts(D, slot);
    int worst = 0;
    for (int s = 0; s < W; ++s) worst = std::max(worst, (int)hc[(size_t)s * D->row_stride + 2 * W]);
    return worst;
}
static void dist_throw_if_refused(dsa_dmatrix* D, int slot) {
    const int r = dist_refusal(D, slot);
    if (r == 2) throw DsaError{DSA_ERR_ARGUMENT, "a rank's share of the batch exceeds max_share = " + std::to_string(D->region_cap)};
    if (r == 1)
        throw DsaError{DSA_ERR_ARGUMENT, "row and column keys must be >= 1 (each is an in-array key of one orientation; key 0 is the semaphore key, pcsr.jl:23)"};
}

// the oldest routed batch: exchange completed + the per-GPU pipeline on what arrived
static void dist_apply_staged(dsa_dmatrix* D) {
    if (D->staged.empty()) throw DsaError{DSA_ERR_ERROR, "no staged batch"};
    const dsa_dmatrix::Routed R = D->staged.front();
    D->staged.erase(D->staged.begin());
    dsa_matrix* A = D->A;
    const int omask = R.omask;
    int64_t hn0 = 0, hn1 = 0;
    const bool host_counts = dist_complete(D, R, &hn0, &hn1);
    if (host_counts) {
        dist_throw_if_refused(D, R.slot);   // every rank sees every flag: all of them throw
        if (hn0 > 0 || hn1 > 0)
            matrix_set_batch_two(A, D->rx_rows[0].p, D->rx_cols[0].p, D->rx_vals[0].p, (omask & 1) ? hn0 : 0, D->rx_rows[1].p, D->rx_cols[1].p,
                                 D->rx_vals[1].p, (omask & 2) ? hn1 : 0);
        return;
    }
    // counts live on the device: the pipeline runs on upper bounds until its own first host synchronisation
    const int64_t bound = (int64_t)D->ctx->world * D->region_cap;
    const int slot = R.slot;
    std::function<void()> pre_mutate = [&] { dist_throw_if_refused(D, slot); };
    matrix_set_batch_two(A, D->rx_rows[0].p, D->rx_cols[0].p, D->rx_vals[0].p, (omask & 1) ? bound : 0, D->rx_rows[1].p, D->rx_cols[1].p,
                         D->rx_vals[1].p, (omask & 2) ? bound : 0, D->rx_n.p, D->rx_n.p + 1, &pre_mutate);
}

// routed batch in one call
static void dist_set_batch(dsa_dmatrix* D, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n, int omask) {
    if (!D->staged.empty()) throw DsaError{DSA_ERR_ERROR, "a staged batch is pending: call dsa_dmatrix_apply_staged first"};
    dist_route(D, d_rows, d_cols, d_vals, n, omask);
    dist_apply_staged(D);
}

static void dist_spmv(dsa_dmatrix* D, int trans, const double* d_x, int64_t nx, double* d_y, int64_t ny) {
    dsa_matrix* A = D->A;
    dsa_dist* d = D->ctx;
    cudaStream_t st = A->sh.st;
    const int which = trans ? 0 : 1;   // A * x gathers over the row-major shards (rows split), transpose(A) * x over the col-major ones
    const int W = d->world;
    const int64_t per = D->per[which];
    double* yb = D->ybuf.ensure((size_t)per * W);
    const int64_t lo = D->split[which][(size_t)d->rank], hi = D->split[which][(size_t)d->rank + 1];
    double* slice = yb + (size_t)d->rank * per;
    DSA_CUDA(cudaMemsetAsync(slice, 0, (size_t)per * 8, st));
    Pcsr& Pm = trans ? A->colmajor : A->rowmajor;
    // the epilogue (carry fix-up + scatter by key) writes this rank's slice straight into the gather buffer (nothing when the
    // rank holds no keys: hi <= lo)
    Pm.spmv_dense(A->ws, d_x, nx, slice, lo, hi, st);
    dist_all_gather(d, slice, yb, (size_t)per, ncclFloat64, st);
    if (ny <= 0) return;
    if (D->even[which]) {
        DSA_CUDA(cudaMemcpyAsync(d_y, yb, (size_t)std::min<int64_t>(ny, per * W) * 8, cudaMemcpyDeviceToDevice, st));
        if (ny > per * W) DSA_CUDA(cudaMemsetAsync(d_y + per * W, 0, (size_t)(ny - per * W) * 8, st));
    } else {
        DSA_LAUNCH("dist_assemble_y", k_dist_assemble_y, grid_for(ny, 256), 256, 0, st, (const double*)yb, per, W, D->T, which, (int64_t)0, d_y, ny);
    }
}

static int dist_owner_host(const dsa_dmatrix* D, int which, int64_t key) {
    int o = 0;
    for (int i = 1; i < D->ctx->world; ++i) o += D->split[which][(size_t)i] <= key;
    return o;
}

// deletecolumn! / deleterow! over the group (matrix.jl:95-111): validation is agreed on before anything changes
static void dist_delete(dsa_dmatrix* D, bool rows, const int64_t* ids, int64_t n) {
    if (n <= 0) return;
    dsa_matrix* A = D->A;
    dsa_dist* d = D->ctx;
    cudaStream_t st = A->sh.st;
    Pcsr& primary = rows ? A->rowmajor : A->colmajor;
    const int which = rows ? 1 : 0;
    std::vector<int32_t> slots;
    std::vector<int64_t> mine;
    int64_t bad = 0;
    {
        std::unordered_set<int64_t> seen;
        for (int64_t i = 0; i < n; ++i) {
            if (!seen.insert(ids[i]).second) { bad = 2; continue; }
            if (dist_owner_host(D, which, ids[i]) != d->rank) continue;
            const int32_t s = primary.host_lookup(ids[i]);
            if (s < 0) { bad = std::max<int64_t>(bad, 1); continue; }
            slots.push_back(s);
            mine.push_back(ids[i]);
        }
    }
    bad = dist_host_max(D, bad, st);
    if (bad == 2) throw DsaError{DSA_ERR_ARGUMENT, "column listed twice."};
    if (bad == 1) throw DsaError{DSA_ERR_ARGUMENT, std::string(rows ? "row" : "column") + " does not exist."};   // pcsr.jl:208
    const int64_t nm = (int64_t)mine.size();
    // entries of the purged spans -> delete list for the twin orientation (matrix.jl:97-99), routed to the twin's owners
    int64_t tot = 0;
    int32_t* d_slots = nullptr;
    if (nm > 0) {
        d_slots = A->d_slots.ensure((size_t)nm);
        int64_t* d_ids = A->d_ids.ensure((size_t)nm);
        DSA_CUDA(cudaMemcpyAsync(d_slots, slots.data(), (size_t)nm * 4, cudaMemcpyHostToDevice, st));
        DSA_CUDA(cudaMemcpyAsync(d_ids, mine.data(), (size_t)nm * 8, cudaMemcpyHostToDevice, st));
        tot = primary.gather_spans(A->ws, d_slots, nm, d_ids, false, st);   // ws.tmp_k = in-array keys, ws.tmp_owner = deleted id
    }
    const int64_t tot_max = dist_host_max(D, tot, st);
    const int64_t rounds = (tot_max + D->region_cap - 1) / D->region_cap;
    if (rounds > 0) {
        // copy out of the shared workspace (the twin's batch reuses it)
        int64_t* ik = D->itmp.ensure((size_t)std::max<int64_t>(tot, 1));
        int64_t* pk = D->itmp2.ensure((size_t)std::max<int64_t>(tot, 1));
        double* z = D->ztmp.ensure((size_t)std::max<int64_t>(std::min(tot, D->region_cap), 1));
        if (tot > 0) {
            DSA_CUDA(cudaMemcpyAsync(ik, A->ws.tmp_k.p, (size_t)tot * 8, cudaMemcpyDeviceToDevice, st));
            DSA_CUDA(cudaMemcpyAsync(pk, A->ws.tmp_owner.p, (size_t)tot * 8, cudaMemcpyDeviceToDevice, st));
            DSA_CUDA(cudaMemsetAsync(z, 0, (size_t)std::min(tot, D->region_cap) * 8, st));
        }
        for (int64_t r = 0; r < rounds; ++r) {
            const int64_t a = std::min(tot, r * D->region_cap), b = std::min(tot, (r + 1) * D->region_cap);
            // deleting columns: twin = row-major, op (row = in-array key, col = deleted id) routed by row; rows: the mirror image
            if (rows) dist_set_batch(D, pk + a, ik + a, z, b - a, /*omask=*/1);
            else dist_set_batch(D, ik + a, pk + a, z, b - a, /*omask=*/2);
            DSA_CUDA(cudaStreamSynchronize(st));
        }
    }
    if (nm > 0) primary.delete_slots(A->ws, slots, d_slots, st);   // deletecolumn!(colmajor, col)  (matrix.jl:100)
    DSA_CUDA(cudaStreamSynchronize(st));
}

}  // namespace dsa

using namespace dsa;

static void dist_make_tables(dsa_dmatrix* D) {
    const int W = D->ctx->world;
    memset(&D->T, 0, sizeof(D->T));
    D->T.world = W;
    D->T.me = D->ctx->rank;
    D->T.nsplit = W - 1;
    D->T.omask = 3;
    for (int o = 0; o < 2; ++o) {
        for (int i = 1; i < W; ++i) D->T.split[o][i - 1] = D->split[o][(size_t)i];
        int64_t per = 0;
        bool even = true;
        for (int r = 0; r < W; ++r) per = std::max(per, D->split[o][(size_t)r + 1] - D->split[o][(size_t)r]);
        for (int r = 0; r < W; ++r) even = even && D->split[o][(size_t)r] == 1 + r * per;
        D->per[o] = std::max<int64_t>(per, 1);
        D->even[o] = even;
    }
}

extern "C" {

int dsa_dist_unique_id(void* id_out128) {
    DSA_TRY
    static_assert(sizeof(ncclUniqueId) == DSA_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    DSA_NCCL(nccl().GetUniqueId(&id));
    memcpy(id_out128, &id, sizeof(id));
    return DSA_OK;
    DSA_CATCH
}
int dsa_dist_init(const void* id128, int rank, int world, dsa_dist_t** out) {
    DSA_TRY
    require_device();
    if (world < 1 || world > DIST_MAX_RANKS || rank < 0 || rank >= world)
        throw DsaError{DSA_ERR_ARGUMENT, "rank / world out of range (at most " + std::to_string(DIST_MAX_RANKS) + " ranks)"};
    std::unique_ptr<dsa_dist> d(new dsa_dist());
    d->rank = rank;
    d->world = world;
    if (world > 1) {
        ncclUniqueId id;
        memcpy(&id, id128, sizeof(id));
        DSA_NCCL(nccl().CommInitRank(&d->comm, world, id, rank));
        d->own_comm = true;
    }
    *out = d.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_dist_init_comm(void* nccl_comm, int rank, int world, dsa_dist_t** out) {
    DSA_TRY
    require_device();
    if (world < 1 || world > DIST_MAX_RANKS || rank < 0 || rank >= world) throw DsaError{DSA_ERR_ARGUMENT, "rank / world out of range"};
    if (world > 1) nccl();   // bind the library now: a missing NCCL fails here, not inside the first collective
    std::unique_ptr<dsa_dist> d(new dsa_dist());
    d->rank = rank;
    d->world = world;
    d->comm = (ncclComm_t)nccl_comm;
    d->own_comm = false;
    *out = d.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_dist_destroy(dsa_dist_t* d) {
    delete d;
    return DSA_OK;
}
int dsa_dist_info(const dsa_dist_t* d, int64_t* out4) {
    DSA_TRY
    out4[0] = d->rank; out4[1] = d->world; out4[2] = d->transport;
    int v = 0;
    if (d->world > 1 && nccl().GetVersion) nccl().GetVersion(&v);
    out4[3] = v;
    return DSA_OK;
    DSA_CATCH
}

int dsa_dmatrix_create(dsa_dist_t* d, int64_t m, int64_t n, const int64_t* row_split, const int64_t* col_split, int64_t max_share,
                       dsa_dmatrix_t** out) {
    DSA_TRY
    require_device();
    if (m < 0 || n < 0 || max_share < 1) throw DsaError{DSA_ERR_ARGUMENT, "dimensions must be >= 0 and max_share >= 1"};
    std::unique_ptr<dsa_dmatrix> D(new dsa_dmatrix());
    D->ctx = d;
    D->m = m;
    D->n = n;
    const int W = d->world;
    const int64_t dims[2] = {n, m};   // split[0] cuts the columns, split[1] the rows
    const int64_t* given[2] = {col_split, row_split};
    for (int o = 0; o < 2; ++o) {
        D->split[o].resize((size_t)W + 1);
        if (given[o]) {
            for (int r = 0; r <= W; ++r) D->split[o][(size_t)r] = given[o][r];
            if (D->split[o][0] != 1) throw DsaError{DSA_ERR_ARGUMENT, "split[0] must be 1"};
            for (int r = 0; r < W; ++r)
                if (D->split[o][(size_t)r + 1] < D->split[o][(size_t)r]) throw DsaError{DSA_ERR_ARGUMENT, "splitters must be ascending"};
        } else {   // equal key ranges
            const int64_t per = std::max<int64_t>((dims[o] + W - 1) / W, 1);
            for (int r = 0; r < W; ++r) D->split[o][(size_t)r] = 1 + r * per;
            D->split[o][(size_t)W] = std::max(dims[o], per * W) + 1;
        }
    }
    dist_make_tables(D.get());
    D->A = new dsa_matrix();
    D->A->sh.create();
    D->A->colmajor.init_empty(D->A->sh.st);
    D->A->rowmajor.init_empty(D->A->sh.st);
    D->A->m = m;
    D->A->n = n;
    dist_setup_exchange(D.get(), max_share, D->A->sh.st);
    DSA_CUDA(cudaStreamSynchronize(D->A->sh.st));
    *out = D.release();
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_destroy(dsa_dmatrix_t* D) {
    delete D;
    return DSA_OK;
}
int dsa_dmatrix_set_stream(dsa_dmatrix_t* D, void* cuda_stream) {
    D->A->sh.set((cudaStream_t)cuda_stream);
    return DSA_OK;
}
dsa_matrix_t* dsa_dmatrix_local(dsa_dmatrix_t* D) { return D->A; }

int dsa_dmatrix_build_local(dsa_dmatrix_t* D, int which, const int64_t* inkeys, const int64_t* partkeys, const double* vals, int64_t n,
                            int combine) {
    DSA_TRY
    dsa_matrix* A = D->A;
    cudaStream_t st = A->sh.st;
    Pcsr& P = which == DSA_COLMAJOR ? A->colmajor : A->rowmajor;
    int64_t* dk = h2d(A->stg.a, inkeys, n, st);
    int64_t* dp = h2d(A->stg.b, partkeys, n, st);
    double* dv = h2d(A->stg.v, vals, n, st);
    P.build_coo_d(A->ws, dk, dp, dv, n, combine, st);
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}

int dsa_dmatrix_build_local_d(dsa_dmatrix_t* D, int which, const int64_t* d_inkeys, const int64_t* d_partkeys, const double* d_vals, int64_t n,
                              int combine) {
    DSA_TRY
    dsa_matrix* A = D->A;
    cudaStream_t st = A->sh.st;
    Pcsr& P = which == DSA_COLMAJOR ? A->colmajor : A->rowmajor;
    P.build_coo_d(A->ws, d_inkeys, d_partkeys, d_vals, n, combine, st);
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}

int dsa_dmatrix_build_coo(dsa_dmatrix_t* D, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n, int combine) {
    DSA_TRY
    dsa_matrix* A = D->A;
    cudaStream_t st = A->sh.st;
    if (n < 0) throw DsaError{DSA_ERR_ARGUMENT, "negative length"};
    const int64_t cap = D->region_cap;
    const int64_t rounds = (dist_host_max(D, n, st) + cap - 1) / cap;
    // what this rank receives, per orientation, appended round after round
    DBuf<int64_t> acc_r[2], acc_c[2];
    DBuf<double> acc_v[2];
    int64_t have[2] = {0, 0}, room[2] = {0, 0};
    bool bad = false;
    for (int64_t r = 0; r < rounds; ++r) {
        const int64_t a = std::min(n, r * cap), b = std::min(n, (r + 1) * cap);
        int64_t* dr = h2d(A->stg.a, rows + a, b - a, st);
        int64_t* dc = h2d(A->stg.b, cols + a, b - a, st);
        double* dv = h2d(A->stg.v, vals + a, b - a, st);
        int64_t hn[2] = {0, 0};
        dist_route(D, dr, dc, dv, b - a, 3);
        const dsa_dmatrix::Routed R = D->staged.front();
        D->staged.erase(D->staged.begin());
        const bool known = dist_complete(D, R, &hn[0], &hn[1]);
        if (!known) {
            int64_t* h = D->h_misc.ensure(8);
            DSA_CUDA(cudaMemcpyAsync(h, D->rx_n.p, 16, cudaMemcpyDeviceToHost, st));
            DSA_CUDA(cudaStreamSynchronize(st));
            hn[0] = h[0];
            hn[1] = h[1];
        } else {
            DSA_CUDA(cudaStreamSynchronize(st));
        }
        bad = bad || dist_refusal(D, R.slot) != 0;
        for (int o = 0; o < 2; ++o) {
            if (have[o] + hn[o] > room[o]) {   // grow geometrically, keeping what was received so far
                const int64_t nr = std::max<int64_t>({2 * room[o], have[o] + hn[o], 1024});
                DBuf<int64_t> nr_, nc_;
                DBuf<double> nv_;
                nr_.ensure((size_t)nr); nc_.ensure((size_t)nr); nv_.ensure((size_t)nr);
                if (have[o] > 0) {
                    DSA_CUDA(cudaMemcpyAsync(nr_.p, acc_r[o].p, (size_t)have[o] * 8, cudaMemcpyDeviceToDevice, st));
                    DSA_CUDA(cudaMemcpyAsync(nc_.p, acc_c[o].p, (size_t)have[o] * 8, cudaMemcpyDeviceToDevice, st));
                    DSA_CUDA(cudaMemcpyAsync(nv_.p, acc_v[o].p, (size_t)have[o] * 8, cudaMemcpyDeviceToDevice, st));
                    DSA_CUDA(cudaStreamSynchronize(st));
                }
                acc_r[o].swap(nr_); acc_c[o].swap(nc_); acc_v[o].swap(nv_);
                room[o] = nr;
            }
            if (hn[o] > 0) {
                DSA_CUDA(cudaMemcpyAsync(acc_r[o].p + have[o], D->rx_rows[o].p, (size_t)hn[o] * 8, cudaMemcpyDeviceToDevice, st));
                DSA_CUDA(cudaMemcpyAsync(acc_c[o].p + have[o], D->rx_cols[o].p, (size_t)hn[o] * 8, cudaMemcpyDeviceToDevice, st));
                DSA_CUDA(cudaMemcpyAsync(acc_v[o].p + have[o], D->rx_vals[o].p, (size_t)hn[o] * 8, cudaMemcpyDeviceToDevice, st));
                have[o] += hn[o];
            }
        }
        DSA_CUDA(cudaStreamSynchronize(st));
    }
    if (bad) throw DsaError{DSA_ERR_ARGUMENT, "row and column keys must be >= 1 (each is an in-array key of one orientation; key 0 is the semaphore key, pcsr.jl:23)"};
    A->colmajor.build_coo_d(A->ws, acc_r[0].p, acc_c[0].p, acc_v[0].p, have[0], combine, st);   // dynamicsparsecolmajor(I, J, V) of the owned columns
    A->rowmajor.build_coo_d(A->ws, acc_c[1].p, acc_r[1].p, acc_v[1].p, have[1], combine, st);   // dynamicsparsecolmajor(J, I, V) of the owned rows
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}

int dsa_dmatrix_stage_batch_d(dsa_dmatrix_t* D, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n) {
    DSA_TRY
    dist_route(D, d_rows, d_cols, d_vals, std::max<int64_t>(n, 0), 3);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_stage_batch(dsa_dmatrix_t* D, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n) {
    DSA_TRY
    n = std::max<int64_t>(n, 0);
    if (D->staged.size() >= 2) throw DsaError{DSA_ERR_ERROR, "two batches are already staged: call dsa_dmatrix_apply_staged first"};
    if (n > D->region_cap) {   // refused collectively by the routing (every rank learns it from the count all-gather)
        dist_route(D, nullptr, nullptr, nullptr, n, 3);
        return DSA_OK;
    }
    const int slot = (int)(D->seq % DIST_SLOTS);
    // the copies run on the routing stream: the previous user of this slot's staging buffers was the routing of batch seq - 3,
    // on the same stream
    int64_t* dr = D->stg_r[slot].ensure((size_t)std::max<int64_t>(n, 1));
    int64_t* dc = D->stg_c[slot].ensure((size_t)std::max<int64_t>(n, 1));
    double* dv = D->stg_v[slot].ensure((size_t)std::max<int64_t>(n, 1));
    if (n > 0) {
        DSA_CUDA(cudaMemcpyAsync(dr, rows, (size_t)n * 8, cudaMemcpyHostToDevice, D->xst));
        DSA_CUDA(cudaMemcpyAsync(dc, cols, (size_t)n * 8, cudaMemcpyHostToDevice, D->xst));
        DSA_CUDA(cudaMemcpyAsync(dv, vals, (size_t)n * 8, cudaMemcpyHostToDevice, D->xst));
    }
    dist_route(D, dr, dc, dv, n, 3);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_apply_staged(dsa_dmatrix_t* D) {
    DSA_TRY
    dist_apply_staged(D);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_set_batch_d(dsa_dmatrix_t* D, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n) {
    DSA_TRY
    dist_set_batch(D, d_rows, d_cols, d_vals, std::max<int64_t>(n, 0), 3);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_set_batch(dsa_dmatrix_t* D, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n) {
    DSA_TRY
    dsa_matrix* A = D->A;
    cudaStream_t st = A->sh.st;
    n = std::max<int64_t>(n, 0);
    int64_t* dr = h2d(A->stg.a, rows, n, st);
    int64_t* dc = h2d(A->stg.b, cols, n, st);
    double* dv = h2d(A->stg.v, vals, n, st);
    dist_set_batch(D, dr, dc, dv, n, 3);
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_spmv_dense_d(dsa_dmatrix_t* D, int trans, const double* d_x, int64_t nx, double* d_y, int64_t ny) {
    DSA_TRY
    dist_spmv(D, trans, d_x, nx, d_y, ny);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_spmv_dense(dsa_dmatrix_t* D, int trans, const double* x, int64_t nx, double* y, int64_t ny) {
    DSA_TRY
    dsa_matrix* A = D->A;
    cudaStream_t st = A->sh.st;
    double* dx = h2d(A->stg.v, x, nx, st);
    double* dy = A->stg.out.ensure((size_t)std::max<int64_t>(ny, 1));
    dist_spmv(D, trans, dx, nx, dy, ny);
    if (ny > 0) DSA_CUDA(cudaMemcpyAsync(y, dy, (size_t)ny * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_get_batch(dsa_dmatrix_t* D, int which, const int64_t* rows, const int64_t* cols, int64_t n, double* out) {
    DSA_TRY
    dsa_matrix* A = D->A;
    dsa_dist* d = D->ctx;
    cudaStream_t st = A->sh.st;
    const int W = d->world;
    n = std::max<int64_t>(n, 0);
    const int64_t nmax = dist_host_max(D, n, st);
    if (nmax == 0) return DSA_OK;
    // all queries to all ranks (padded with key -1: absent everywhere); every rank answers from its shard (a column lives on its
    // owner only, the others read 0.0); the sum over ranks is exact: one non-zero term at most
    int64_t* q = D->itmp.ensure((size_t)W * 2 * nmax);
    std::vector<int64_t> hq((size_t)2 * nmax, -1);
    for (int64_t i = 0; i < n; ++i) { hq[(size_t)i] = rows[i]; hq[(size_t)(nmax + i)] = cols[i]; }
    int64_t* mine = q + (size_t)d->rank * 2 * nmax;
    DSA_CUDA(cudaMemcpyAsync(mine, hq.data(), (size_t)2 * nmax * 8, cudaMemcpyHostToDevice, st));
    dist_all_gather(d, mine, q, (size_t)2 * nmax, ncclInt64, st);
    double* ans = D->dtmp.ensure((size_t)W * nmax);
    for (int s = 0; s < W; ++s) {
        const int64_t* qr = q + (size_t)s * 2 * nmax;
        const int64_t* qc = qr + nmax;
        if (which == DSA_COLMAJOR) A->colmajor.get_batch_d(A->ws, qr, qc, nmax, ans + (size_t)s * nmax, st);
        else A->rowmajor.get_batch_d(A->ws, qc, qr, nmax, ans + (size_t)s * nmax, st);
    }
    dist_all_reduce(d, ans, (size_t)W * nmax, ncclFloat64, ncclSum, st);
    if (n > 0) DSA_CUDA(cudaMemcpyAsync(out, ans + (size_t)d->rank * nmax, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_delete_columns(dsa_dmatrix_t* D, const int64_t* cols, int64_t n) {
    DSA_TRY
    dist_delete(D, false, cols, n);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_delete_rows(dsa_dmatrix_t* D, const int64_t* rows, int64_t n) {
    DSA_TRY
    dist_delete(D, true, rows, n);
    return DSA_OK;
    DSA_CATCH
}
int dsa_dmatrix_info(dsa_dmatrix_t* D, int64_t* out8) {
    DSA_TRY
    dsa_matrix* A = D->A;
    cudaStream_t st = A->sh.st;
    DSA_CUDA(cudaStreamSynchronize(st));
    int64_t* dv = D->misc.ensure(8);
    int64_t* h = D->h_misc.ensure(8);
    h[0] = A->rowmajor.nnz();              // matrix.jl:91: nnz(rowmajor), summed over the row shards
    h[1] = A->colmajor.nb_partitions;
    h[2] = A->rowmajor.nb_partitions;
    h[3] = A->colmajor.nnz();
    DSA_CUDA(cudaMemcpyAsync(dv, h, 32, cudaMemcpyHostToDevice, st));
    dist_all_reduce(D->ctx, dv, 4, ncclInt64, ncclSum, st);
    DSA_CUDA(cudaMemcpyAsync(h, dv, 32, cudaMemcpyDeviceToHost, st));
    DSA_CUDA(cudaStreamSynchronize(st));
    out8[0] = D->m; out8[1] = D->n; out8[2] = h[0]; out8[3] = h[1]; out8[4] = h[2]; out8[5] = D->region_cap; out8[6] = h[3];
    out8[7] = D->ctx->transport;
    return DSA_OK;
    DSA_CATCH
}

}  // extern "C"
