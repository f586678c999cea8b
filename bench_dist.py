"""bench.py's multi-GPU arm (launched by torchrun, one rank per GPU), through libdsa's dsa_dmatrix_* entry points.

value  — WEAK scaling of the single-GPU workload (configs[1] per GPU): a (1e5*N) x (1e5*N) PCSR with 1e7*N nnz sharded by key
         range; one step = a global batch of 1M*N logical updates (every rank contributes 1M: ~50% inserts of new entries, ~50%
         deletes of its previous inserts; routed to the owners of both orientations by the fused route+push kernel over NVLink
         peer memory) + one SpMV A*x with the y slices all-gathered (NCCL).  Per-GPU work is that of the N = 1 line, so the
         driver's efficiency is value_N / (N * value_1).
c4     — BASELINE.json configs[3] at its stated size (N >= 2): PCSR 1e7 x 1e7 with 1e9 nnz generated shard-locally, global batches
         of 100M updates (90% insert/overwrite, 10% delete; 100M/N per rank) + SpMV.  Checked in place through size-independent
         properties (both orientations agree: 1'(A x) == (A'1)'x, nnz of the col-major shards == nnz of the row-major shards,
         routed point reads of a sample of the last batch return the written values).
"""
import ctypes as C
import datetime
import json
import os
import time

import numpy as np


def _block(torch, dev, seed, a, b, lo_r, hi_r, lo_c, hi_c, nnz, parity):
    """entries of global block (row range a, col range b): the same device-side stream on every rank.  (i + j) has the given
    parity, so that later inserts (opposite parity) can never collide with an initial entry."""
    g = torch.Generator(device=dev)
    g.manual_seed(((seed * 1_000_003 + a) * 1_000_003 + b) % (1 << 62))
    I = torch.randint(lo_r, hi_r, (nnz,), generator=g, device=dev, dtype=torch.int64)
    J = torch.randint(lo_c, hi_c, (nnz,), generator=g, device=dev, dtype=torch.int64)
    fix = ((I + J) & 1) != parity
    J = torch.where(fix, torch.where(J + 1 < hi_c, J + 1, J - 1), J)
    V = torch.rand(nnz, generator=g, device=dev, dtype=torch.float64) + 1e-3
    return I, J, V


def _build_blocks(torch, dev, A, seed, rank, world, rows_per, cols_per, nnz_block):
    """column-major shard = blocks (a, rank) for all a ; row-major shard = blocks (rank, b) for all b (one consistent global matrix)"""
    rng = lambda r, per: (1 + r * per, 1 + (r + 1) * per)
    parts = [_block(torch, dev, seed, a, rank, *rng(a, rows_per), *rng(rank, cols_per), nnz_block, 0) for a in range(world)]
    I, J, V = (torch.cat(x) for x in zip(*parts))
    del parts
    A.build_local(0, I, J, V)
    del I, J, V
    parts = [_block(torch, dev, seed, rank, b, *rng(rank, rows_per), *rng(b, cols_per), nnz_block, 0) for b in range(world)]
    I, J, V = (torch.cat(x) for x in zip(*parts))
    del parts
    A.build_local(1, J, I, V)
    del I, J, V
    torch.cuda.empty_cache()


def _fresh(torch, dev, g, m, n, k):
    """k uniform (i, j) with (i + j) odd: disjoint from the initial entries by construction"""
    I = torch.randint(1, m + 1, (k,), generator=g, device=dev, dtype=torch.int64)
    J = torch.randint(1, n + 1, (k,), generator=g, device=dev, dtype=torch.int64)
    fix = ((I + J) & 1) != 1
    J = torch.where(fix, torch.where(J + 1 <= n, J + 1, J - 1), J)
    return I, J


def _properties(torch, dist, A, dev, m, n, tag):
    """size-independent checks that tie the two orientations together after all the routed batches"""
    x = torch.rand(n, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(99))
    y = A.spmv(x)                                                     # row-major shards
    t = A.spmv(torch.ones(m, device=dev, dtype=torch.float64), trans=True)   # col-major shards
    lhs, rhs = float(y.sum().item()), float(torch.dot(t, x).item())
    inf = A.info()
    ok = abs(lhs - rhs) <= 1e-9 * max(abs(lhs), abs(rhs), 1.0) and inf["nnz"] == inf["nnz_colmajor"]
    return {"workload": tag, "ok": bool(ok), "sum_Ax": lhs, "dot_At1_x": rhs, "nnz_rowmajor": inf["nnz"], "nnz_colmajor": inf["nnz_colmajor"]}


def main_dist(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import bench as B
    import dsa_b200 as D
    from dsa_b200.sharded import DistContext, DistMatrix

    # stdout carries exactly ONE JSON line: everything else (NCCL banners, warnings) goes to stderr
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    L = D.lib()
    L.dsa_set_device(C.c_int(local_rank))
    dev = torch.device("cuda", local_rank)
    # a short collective timeout: a hang must abort within minutes instead of holding N GPUs
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    ctx = DistContext()
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    K, W = args.steps, max(args.warmup, 3)
    P = W + K

    # ---------------------------------------------------------------- weak scaling of configs[1] ----------------------
    per = B.M_ROWS
    m = n = per * world
    nnz_block = B.NNZ0 // world          # every (a, b) block holds nnz/world entries -> each shard holds ~1e7 per orientation
    A = DistMatrix(ctx, m, n, B.BATCH, stream=stream.cuda_stream)
    _build_blocks(torch, dev, A, B.SEED, rank, world, per, per, nnz_block)
    # a CYCLE of P shares per rank: share k inserts S_k (new entries) and deletes S_{k-1}; S_{P-1} is inserted before the
    # warm-up, so the chain is periodic and the structure stays at ~1e7 nnz per shard however many repeats are timed
    g = torch.Generator(device=dev)
    g.manual_seed((B.SEED * 7 + rank) % (1 << 62))
    half = B.BATCH // 2
    S = [_fresh(torch, dev, g, m, n, half) for _ in range(P)]
    shares = []
    for k in range(P):
        ii, jj = torch.cat([S[k][0], S[k - 1][0]]), torch.cat([S[k][1], S[k - 1][1]])
        vv = torch.cat([torch.rand(half, generator=g, device=dev, dtype=torch.float64) + 1e-3, torch.zeros(half, device=dev, dtype=torch.float64)])
        p = torch.randperm(B.BATCH, generator=g, device=dev)
        shares.append((ii[p].contiguous(), jj[p].contiguous(), vv[p].contiguous()))
    A.set_batch(S[-1][0], S[-1][1], torch.rand(half, generator=g, device=dev, dtype=torch.float64) + 1e-3)
    d_x = torch.rand(n, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(B.SEED + 9))
    d_y = torch.empty(m, device=dev, dtype=torch.float64)

    # The step in two halves (dsa_dmatrix_stage_batch_d / dsa_dmatrix_apply_staged): the routing + NVLink push of batch s+1 run
    # on the library's side stream while the kernels of batch s run.  Every batch of a timed region is staged inside it.
    def run_dev(first, nsteps):
        A.stage_batch(*shares[first % P])
        for s in range(first, first + nsteps):
            if s + 1 < first + nsteps:
                A.stage_batch(*shares[(s + 1) % P])
            A.apply_staged()
            A.spmv(d_x, out=d_y)

    def step_dev(s):
        A.set_batch(*shares[s % P])
        return A.spmv(d_x, out=d_y)

    sampler = B.ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    windows = []
    for s in range(W):
        step_dev(s)
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(first, nsteps):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        run_dev(first, nsteps)
        e1.record(stream)
        torch.cuda.synchronize()
        dist.barrier()
        windows.append((t0, time.perf_counter()))
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)      # the slowest rank's device time
        return float(ms.item())

    launches0 = L.dsa_launch_count()
    ms_total = timed(W, K)                             # exactly K timed steps
    launches = L.dsa_launch_count() - launches0
    s_next = W + K
    ms_step = ms_total / K
    value = B.BATCH * world / (ms_step * 1e-3) / 1e6
    checksum = float(d_y.sum().item())
    parity = [_properties(torch, dist, A, dev, m, n, "weak C2-per-GPU")]

    # e2e: pinned host shares through the host-pointer entry points: H2D + step + D2H of y inside the timed region
    e2e = None
    if not args.no_e2e:
        h_sh = [tuple(t.cpu().pin_memory() for t in shares[k]) for k in range(P)]
        h_x = d_x.cpu().pin_memory()
        h_y = torch.empty(m, dtype=torch.float64).pin_memory()

        def run_host(first, nsteps):   # pinned host shares, staged: the PCIe copy and the exchange of batch s+1 overlap batch s
            A.stage_batch(*h_sh[first % P])
            for s in range(first, first + nsteps):
                if s + 1 < first + nsteps:
                    A.stage_batch(*h_sh[(s + 1) % P])
                A.apply_staged()
                D._lib.check(L.dsa_dmatrix_spmv_dense(A._h, C.c_int(0), C.c_void_p(h_x.data_ptr()), C.c_int64(n), C.c_void_p(h_y.data_ptr()), C.c_int64(m)))

        run_host(s_next, W)
        s_next += W
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        run_host(s_next, K)
        torch.cuda.synchronize()
        dist.barrier()
        windows.append((t0, time.perf_counter()))
        s_next += K
        wall = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        ms_e2e = 1e3 * float(wall.item()) / K
        e2e = {"value": B.BATCH * world / (ms_e2e * 1e-3) / 1e6, "unit": "Mupdates/s", "h2d_bytes_per_step": (24 * B.BATCH + 8 * n) * world,
               "d2h_bytes_per_step": 8 * m * world, "ms_per_step": ms_e2e, "steps": K, "checksum": float(h_y.sum().item()),
               "api": "dsa_dmatrix_stage_batch + dsa_dmatrix_apply_staged + dsa_dmatrix_spmv_dense (host pinned buffers)"}
        del h_sh

    # per-kernel durations on rank 0 (CUDA events around every launch, outside the timed region; collectives keep the ranks in step)
    L.dsa_prof_reset()
    L.dsa_prof_enable(C.c_int(1))
    for s in range(s_next, s_next + 3):
        step_dev(s)
    s_next += 3
    torch.cuda.synchronize()
    L.dsa_prof_enable(C.c_int(0))
    need = L.dsa_prof_dump(None, C.c_int64(0))
    buf = C.create_string_buffer(int(need) + 16)
    L.dsa_prof_dump(buf, C.c_int64(len(buf)))
    kernels = {}
    for ln in buf.value.decode().strip().splitlines():
        name, cnt, tms = ln.split(",")
        kernels[name] = {"launches_per_step": int(cnt) / 3, "ms_per_step": float(tms) / 3, "avg_us": 1e3 * float(tms) / int(cnt)}
    inf_local = A.local.info(1)
    spmv = None
    spmv_name = next((k for k in ("spmv_blocked", "spmv_flat") if k in kernels), None)
    if spmv_name:
        us = kernels[spmv_name]["avg_us"]
        peak, src = B.measured_peak_gbs()
        alg = 16 * (inf_local["nnz"] + inf_local["nb_partitions"]) + 8 * (n + per)
        a = alg / (us * 1e-6) / 1e9
        spmv = {"kernel": spmv_name, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak, "avg_us": us,
                "algorithmic_bytes": alg, "traffic": None, "peak_source": src, "scope": "rank 0 shard"}
    dist_info = A.info()
    A.close()
    del shares, S
    torch.cuda.empty_cache()
    L.dsa_trim_memory()

    # ---------------------------------------------------------------- configs[3] at its stated size --------------------
    c4 = None
    if world >= 2 and not args.no_c4:
        c4 = run_c4(torch, dist, B, D, ctx, dev, stream, rank, world, parity)

    clocks = sampler.stop(windows) if sampler else None
    if rank == 0:
        cfg = B.workload_config(world)
        cfg["workload"] = (f"value = weak scaling of C2 per GPU: PCSR {m} x {n}, {nnz_block * world * world} nnz sharded by key range over {world} GPUs; "
                           f"step = {B.BATCH * world} updates routed to both orientations (fused route+push over NVLink peer memory) + SpMV with "
                           f"all-gather.  c4 = C4 at its stated size: PCSR 1e7 x 1e7, 1e9 nnz, 100M-update global batches + SpMV")
        cfg.update(rows=m, cols=n, nnz=nnz_block * world * world, batch=B.BATCH * world, transport=dist_info["transport"],
                   nccl_version=ctx.info()["nccl_version"])
        os.dup2(saved_stdout, 1)
        print(json.dumps({
            "metric": "batched PCSR insert/delete Mupdates/s", "value": value, "unit": "Mupdates/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_step, "timed_steps": K, "timed_region_s": ms_total * 1e-3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64 keys / f64 values", "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "gpu_launches_per_step": launches / K, "parity": parity, "c4": c4,
            "roofline": spmv, "spmv": spmv, "cpu_baseline": None, "kernels": kernels, "checksum": checksum,
            "shard_nnz_rank0": inf_local["nnz"], "nnz_global": dist_info["nnz"]}), flush=True)
        os.dup2(2, 1)
    ctx.close()
    dist.destroy_process_group()


def run_c4(torch, dist, B, D, ctx, dev, stream, rank, world, parity):
    """PCSR 1e7 x 1e7, 1e9 nnz over `world` GPUs; global batches of 100M updates (90% insert/overwrite, 10% delete)."""
    from dsa_b200.sharded import DistMatrix
    L = D.lib()
    m = n = 10_000_000
    nnz_total, batch_total = 1_000_000_000, 100_000_000
    rows_per = cols_per = m // world
    nnz_block = nnz_total // (world * world)
    share = batch_total // world
    warm, steps = 2, 3   # every step adds ~0.8 * share entries per shard: 5 steps stay below the root's upper density bound
    t_build = time.perf_counter()
    A = DistMatrix(ctx, m, n, share, stream=stream.cuda_stream)
    _build_blocks(torch, dev, A, B.SEED + 4, rank, world, rows_per, cols_per, nnz_block)
    torch.cuda.synchronize()
    dist.barrier()
    t_build = time.perf_counter() - t_build
    inf0 = A.local.info(1)
    g = torch.Generator(device=dev)
    g.manual_seed(((B.SEED + 4) * 7 + rank) % (1 << 62))
    n_del = share // 10
    n_ins = share - n_del
    x = torch.rand(n, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(B.SEED + 13))
    y = torch.empty(m, device=dev, dtype=torch.float64)
    prev = None
    batches = []
    for s in range(warm + steps):
        I, J = _fresh(torch, dev, g, m, n, n_ins)
        V = torch.rand(n_ins, generator=g, device=dev, dtype=torch.float64) + 1e-3
        if prev is None:   # first batch: its delete slots are deletes of absent keys (silent no-ops, writes.jl:62)
            dI, dJ = _fresh(torch, dev, g, m, n, n_del)
        else:
            dI, dJ = prev[0][:n_del], prev[1][:n_del]
        p = torch.randperm(share, generator=g, device=dev)
        batches.append((torch.cat([I, dI])[p].contiguous(), torch.cat([J, dJ])[p].contiguous(),
                        torch.cat([V, torch.zeros(n_del, device=dev, dtype=torch.float64)])[p].contiguous()))
        prev = (I, J)
    del prev
    for s in range(warm):
        A.set_batch(*batches[s])
        A.spmv(x, out=y)
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = L.dsa_launch_count()
    e0.record(stream)
    for s in range(warm, warm + steps):
        A.set_batch(*batches[s])
        A.spmv(x, out=y)
    e1.record(stream)
    torch.cuda.synchronize()
    dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = L.dsa_launch_count() - launches0
    ms_step = float(ms.item()) / steps
    # SpMV alone (all ranks in step)
    torch.cuda.synchronize()
    dist.barrier()
    e0.record(stream)
    for _ in range(5):
        A.spmv(x, out=y)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_spmv = torch.tensor([e0.elapsed_time(e1) / 5], dtype=torch.float64, device=dev)
    dist.all_reduce(ms_spmv, op=dist.ReduceOp.MAX)
    inf = A.info()
    # routed point reads of a sample of the last batch: the written values (keys written twice in the share are left out)
    bi, bj, bv = batches[-1]
    lin = bi * (n + 1) + bj
    srt, _ = torch.sort(lin)
    dup = srt[1:][srt[1:] == srt[:-1]]
    pick = torch.randperm(share, generator=g, device=dev)[:20_000]
    keep = ~torch.isin(lin[pick], dup)
    qi, qj, qv = bi[pick][keep].cpu().numpy(), bj[pick][keep].cpu().numpy(), bv[pick][keep].cpu().numpy()
    got = A.get_batch(qi, qj)
    got_r = A.get_batch(qi, qj, which=1)
    reads_ok = bool(np.array_equal(got, qv) and np.array_equal(got_r, qv))
    prop = _properties(torch, dist, A, dev, m, n, "C4")
    prop["routed_reads_ok"] = reads_ok
    prop["ok"] = bool(prop["ok"] and reads_ok)
    parity.append(prop)
    peak, src = B.measured_peak_gbs()
    inf_local = A.local.info(1)
    alg = 16 * (inf_local["nnz"] + inf_local["nb_partitions"]) + 8 * (n + rows_per)
    out = {"workload": "C4: PCSR 1e7 x 1e7, 1e9 nnz sharded by key range, 100M-update global batches (90% insert/overwrite, 10% delete) + SpMV",
           "value": batch_total / (ms_step * 1e-3) / 1e6, "unit": "Mupdates/s", "ms_per_step": ms_step, "steps": steps, "warmup": warm,
           "nnz_initial": nnz_block * world * world, "nnz_after": inf["nnz"], "batch": batch_total, "share_per_rank": share,
           "shard_capacity_cells": inf_local["capacity"], "shard_capacity_initial": inf0["capacity"], "build_s": t_build,
           "gpu_launches": int(launches), "spmv_ms": float(ms_spmv.item()),
           "spmv_effective_gbs_per_gpu": alg / (float(ms_spmv.item()) * 1e-3) / 1e9, "spmv_frac_of_measured_peak": alg / (float(ms_spmv.item()) * 1e-3) / 1e9 / peak,
           "peak_source": src}
    A.close()
    return out
