#!/usr/bin/env python
"""bench.py — BASELINE.json configs[1]: PCSR 1e5 x 1e5 with 1e7 nnz resident in HBM; one step = one batched update of
1M logical entries (both orientations) followed by one SpMV (A * x, dense x).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line.
  value              whole-job Mupdates/s with inputs resident in HBM on the stationary chain (each 1M-update batch inserts
                     ~0.5M new entries, overwrites a few, deletes the previous batch's inserts): exactly K timed steps after
                     max(W, 3) warm-up steps
  value_insert_only  configs[1] as written: fresh 1e7-nnz matrix -> ONE batched insert of 1M new entries -> SpMV (the matrix is
                     restored from a pristine device clone outside the timed bracket of every repetition)
  e2e                the stationary step through the host-pointer C-ABI calls (pinned host buffers; every H2D copy of the batch
                     and of x and the D2H read of y happen inside the timed region)
  parity             y of the GPU arm after the first W+K steps and after the insert-only step, against the CPU oracle fed the
                     SAME batches (<= 1e-12 relative), plus nnz — the number the driver times is tied to a correctness check
  roofline / spmv    dominant kernel of the step / the SpMV kernel against the measured HBM peak
  cpu_baseline       the CPU oracle (C++ restatement of the reference, 1 core) on the same W+K steps
`--impl reference` times the oracle on the same W+K batches (same generator, same x) and prints the same checksum.
`--dump-outputs DIR` writes what the timed path returned after its last step (outputs_of_last_step) and y of the insert-only
step as float64 .npy files, ~34 MB; the inputs depend on W and K only, so two builds run with the same arguments can be
compared file by file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

M_ROWS = N_COLS = 100_000
NNZ0 = 10_000_000
BATCH = 1_000_000
N_OVER = 1_000                 # overwrites of resident entries per batch (100 of them written twice: last writer wins)
SEED = 0xD5A00002
BYTES_PER_UPDATE = 80          # SURVEY.md §8d: 2 orientations x (24 B triple read + 16 B cell write)
BYTES_PER_UPDATE_ONE = 40      # one orientation (what a single kernel launch of the update pipeline processes)
SPMV_RTOL = 1e-12              # north_star: Float64 SpMV within 1e-12 relative
DUMP_SAMPLE = 1 << 20          # stored entries in the seeded sample of --dump-outputs (3 arrays x 8 MB)


def make_workload(ncycle, m=M_ROWS, n=N_COLS, nnz0=NNZ0, nb=BATCH, seed=SEED):
    """x, the initial COO, a CYCLE of `ncycle` batches and one insert-only batch — all over distinct (i, j).

    Batch k = (nb/2 - N_OVER) inserts of new entries S_k + N_OVER overwrites of resident entries (100 keys written twice)
    + (nb/2 - N_OVER) deletes (v = 0.0) of S_{k-1} + N_OVER deletes of absent keys (silent no-ops, writes.jl:62), shuffled.
    The initial matrix holds S_{ncycle-1}, so the chain is periodic: after every full cycle the contents are those of the
    start and nnz stays at nnz0 - N_OVER during the whole run, however long."""
    rng = np.random.default_rng(seed)
    x = rng.random(n)                                   # drawn FIRST: identical for every arm and every step count
    half = nb // 2
    fresh = half - N_OVER
    nbase = nnz0 - half
    need = nbase + ncycle * (fresh + N_OVER) + nb
    lin = np.sort(rng.integers(0, m * n, int(need * 1.02) + 1000))       # sort + adjacent difference (np.unique is 80x slower)
    lin = lin[np.concatenate([[True], lin[1:] != lin[:-1]])]
    assert len(lin) >= need, "not enough distinct keys"
    lin = rng.permutation(lin)[:need]

    def ij(l):
        return l // n + 1, l % n + 1

    base = lin[:nbase]
    off = nbase
    S, noop = [], []
    for _ in range(ncycle):
        S.append(lin[off:off + fresh]); off += fresh
        noop.append(lin[off:off + N_OVER]); off += N_OVER
    ins_only = lin[off:off + nb]
    init = np.concatenate([base, S[-1]])
    I, J = ij(init)
    V = rng.random(len(init)) + 1e-3
    batches = []
    for k in range(ncycle):
        ov = base[rng.integers(0, nbase, N_OVER - 100)]
        ov = np.concatenate([ov, ov[:100]])             # 100 keys appear twice in the batch: the later write wins
        keys = np.concatenate([S[k], ov, S[k - 1], noop[k]])
        vals = np.concatenate([rng.random(fresh + N_OVER) + 1e-3, np.zeros(fresh + N_OVER)])
        p = rng.permutation(nb)
        bi, bj = ij(keys[p])
        batches.append((np.ascontiguousarray(bi), np.ascontiguousarray(bj), np.ascontiguousarray(vals[p])))
    oi, oj = ij(ins_only)
    insert_only = (np.ascontiguousarray(oi), np.ascontiguousarray(oj), rng.random(nb) + 1e-3)
    return x, (I, J, V), batches, insert_only


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, windows=()):
        """windows: (t0, t1) perf_counter intervals of the timed regions; samples inside them are the ones 'under load'."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, sm_load, reasons = [], [], [], set()
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                s_, m_ = float(f[1]), float(f[2])
            except ValueError:
                continue
            sm.append(s_)
            mx.append(m_)
            inside = any(a <= ts <= b for a, b in windows)
            if inside:
                sm_load.append(s_)
            if inside or not windows:
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        use = sm_load if sm_load else sm
        return {"sm_mhz": float(np.median(use)) if use else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_in_timed_regions": len(sm_load)}


def ncu_traffic(kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu --set full capture."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["kernels"][kernel]["dram_bytes"]
    except Exception:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def rel_err(y, yo):
    d = np.abs(y - yo)
    s = np.maximum(np.abs(y), np.abs(yo))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(s > 0, d / s, 0.0)
    return float(r.max()) if len(r) else 0.0


def outputs_of_last_step(A, y, last_batch):
    """What a caller of the timed step holds after its last step: y = A * x, the values stored at the last batch's (i, j)
    (getindex), and a seeded sample of DUMP_SAMPLE stored entries (rows, cols, vals in column-major order, to_coo).  ~33 MB."""
    import dsa_b200 as D
    rows, cols, vals = D.to_coo(A)
    pick = np.sort(np.random.default_rng(SEED).choice(len(rows), min(DUMP_SAMPLE, len(rows)), replace=False))
    return {"y": y, "batch_vals": A.get_batch(last_batch[0], last_batch[1]),
            "entries_rows": rows[pick], "entries_cols": cols[pick], "entries_vals": vals[pick]}


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def oracle_chain(coo, batches, x, insert_only=None):
    """The reference's CPU path on the same inputs: build, then per step a loop of setindex! over the batch (the reference has
    no batched update, matrix.jl:119-121) + mat * x.  One host core (C++ oracle; Julia is not installed).  Returns the
    per-step times, y after the last step, nnz, and (optionally) y / nnz of the insert-only step on the pristine matrix."""
    from oracle import oracle as O
    t0 = time.perf_counter()
    M = O.Matrix(coo[0], coo[1], coo[2], m=M_ROWS, n=N_COLS)
    t_build = time.perf_counter() - t0
    io = None
    if insert_only is not None:
        P = M.clone()
        P.set_many(*insert_only)
        io = (P.mul_dense(x, M_ROWS), P.nnz())
        del P
    upd, spmv = [], []
    y = None
    for bi, bj, bv in batches:
        t0 = time.perf_counter()
        M.set_many(bi, bj, bv)
        t1 = time.perf_counter()
        y = M.mul_dense(x, M_ROWS)
        t2 = time.perf_counter()
        upd.append(t1 - t0)
        spmv.append(t2 - t1)
    return dict(t_build=t_build, upd=upd, spmv=spmv, y=y, nnz=M.nnz(), insert_only=io)


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (C++ oracle port), rank 0 only."""
    if rank != 0:
        return
    K, W = args.steps, max(args.warmup, 3)
    x, coo, batches, _ = make_workload(W + K)
    r = oracle_chain(coo, batches, x)
    times = [a + b for a, b in zip(r["upd"], r["spmv"])][W:]
    total = sum(times)
    val = BATCH * len(times) / total / 1e6
    line = {
        "impl": "reference", "metric": "batched PCSR insert/delete Mupdates/s", "value": val, "unit": "Mupdates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64 keys / f64 values", "data": "synthetic",
        "config": workload_config(1),
        "cpu_baseline": {"value": val, "unit": "Mupdates/s", "cores": 1, "kind": "port",
                         "sample": f"{len(times)} full steps (1M-update batch as a loop of setindex! + SpMV) on 1 host core; "
                                   "C++ restatement of the reference (Julia not installed)"},
        "e2e": {"value": val, "unit": "Mupdates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "checksum": float(np.sum(r["y"])), "checksum_after_steps": W + K, "nnz_after": r["nnz"],
    }
    print(json.dumps(line))


def workload_config(n_gpus):
    return {"workload": "C2: dynamicsparse PCSR 1e5 x 1e5, 1e7 nnz resident; step = 1M-update batch (~50% inserts of new entries, 0.1% "
                        "overwrites, ~50% deletes; both orientations) + SpMV A*x (dense x); value_insert_only = configs[1] as written "
                        "(one batched insert of 1M new entries into the fresh matrix + SpMV)",
            "rows": M_ROWS, "cols": N_COLS, "nnz": NNZ0, "batch": BATCH,
            "l2_policy": "inputs larger than L2 (2 x 268 MB gapped arrays per matrix vs 126 MB L2)", "seed": hex(SEED),
            "parallelism": f"column-range shards x{n_gpus}" if n_gpus > 1 else "single GPU",
            # batches of >= capacity/40 ops are tile-streamed (one pass over each orientation's keys, DESIGN.md 4b): config 2's are
            "batch_pipeline": "tile-streamed (k_tile_assign + k_tile_merge) above capacity/40 ops per batch, random-access below",
            # kernel switches in effect (empty = the validated defaults)
            "switches": {k: os.environ[k] for k in sorted(os.environ) if k.startswith("DSA_")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle legs (cpu_baseline AND the parity check)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="multi-GPU arm: skip the full-size configs[3] run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or world > 1 or os.environ.get("DSA_BENCH_FORCE_DIST") == "1"):
        ap.error("--dump-outputs is implemented for the single-GPU arm of --impl ours")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1 or os.environ.get("DSA_BENCH_FORCE_DIST") == "1":   # the latter: the sharded code path on one rank (no NVLink traffic)
        from bench_dist import main_dist   # sharded path (dsa_dist_*: peer-memory routing + NCCL all-gather)
        main_dist(args, rank, world, local_rank)
        return

    import torch

    import dsa_b200 as D
    D.require_gpu()
    L = D.lib()
    torch.cuda.set_device(local_rank)
    L.dsa_set_device(C.c_int(local_rank))
    K, W = args.steps, max(args.warmup, 3)
    P = W + K                                           # cycle length: the chain is periodic with this period
    x, coo, batches, insert_only = make_workload(P)
    A = D.dynamicsparse(coo[0], coo[1], coo[2], m=M_ROWS, n=N_COLS)
    stream = torch.cuda.current_stream()
    D._lib.check(L.dsa_matrix_set_stream(A._h, C.c_void_p(stream.cuda_stream)))
    dev = torch.device("cuda", local_rank)

    def vp(t):
        return C.c_void_p(t.data_ptr())

    def clone_handle(h):
        out = C.c_void_p()
        D._lib.check(L.dsa_matrix_clone(h, C.byref(out)))
        D._lib.check(L.dsa_matrix_set_stream(out, C.c_void_p(stream.cuda_stream)))
        return out

    pristine = clone_handle(A._h)                       # the fresh 1e7-nnz matrix, for the insert-only repetitions

    # ---- value: inputs resident in HBM --------------------------------------------------------------------
    d_batches = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in batches]
    d_x = torch.from_numpy(x).to(dev)
    d_y = torch.zeros(M_ROWS, dtype=torch.float64, device=dev)

    def step_dev(s, h=None):
        bi, bj, bv = d_batches[s % P]
        D._lib.check(L.dsa_matrix_set_batch_d(h or A._h, vp(bi), vp(bj), vp(bv), C.c_int64(BATCH)))
        D._lib.check(L.dsa_matrix_spmv_dense_d(h or A._h, C.c_int(0), vp(d_x), C.c_int64(N_COLS), vp(d_y), C.c_int64(M_ROWS)))

    sampler = ClockSampler(local_rank)
    sampler.start()
    windows = []
    for s in range(W):
        step_dev(s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the timed region: exactly K steps; afterwards the structure has seen batches 0 .. W+K-1 = one full cycle -> parity snapshot
    launches0 = L.dsa_launch_count()
    t_w0 = time.perf_counter()
    e0.record(stream)
    for s in range(W, W + K):
        step_dev(s)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    launches = L.dsa_launch_count() - launches0
    windows.append((t_w0, time.perf_counter()))
    y_gpu = d_y.cpu().numpy().copy()
    nnz_gpu = A.info(1)["nnz"]
    dumped = outputs_of_last_step(A, y_gpu, batches[(W + K - 1) % P]) if args.dump_outputs else None
    s_next = W + K
    ms_step = ms_total / K
    value = BATCH / (ms_step * 1e-3) / 1e6
    checksum = float(y_gpu.sum())

    # ---- configs[1] as written: fresh matrix -> one batched insert of 1M new entries -> SpMV ------------------------------
    d_io = tuple(torch.from_numpy(a).to(dev) for a in insert_only)
    io_ms, y_io, nnz_io = [], None, None
    for rep in range(8):
        Cc = clone_handle(pristine)                     # untimed: restore the fresh matrix
        torch.cuda.synchronize()
        e0.record(stream)
        D._lib.check(L.dsa_matrix_set_batch_d(Cc, vp(d_io[0]), vp(d_io[1]), vp(d_io[2]), C.c_int64(BATCH)))
        D._lib.check(L.dsa_matrix_spmv_dense_d(Cc, C.c_int(0), vp(d_x), C.c_int64(N_COLS), vp(d_y), C.c_int64(M_ROWS)))
        e1.record(stream)
        torch.cuda.synchronize()
        if rep >= 2:                                    # two warm-up repetitions (buffer growth of the clone's workspace)
            io_ms.append(e0.elapsed_time(e1))
        if rep == 7:
            y_io = d_y.cpu().numpy().copy()
            out10 = np.zeros(10, np.int64)
            L.dsa_matrix_info(Cc, C.c_int(1), C.c_void_p(out10.ctypes.data))
            nnz_io = int(out10[9])
        L.dsa_matrix_destroy(Cc)
    io_ms_step = float(np.mean(io_ms))

    # ---- per-kernel durations (CUDA events around every launch, outside the timed region) -------------------
    prof_steps = 3
    L.dsa_prof_reset()
    L.dsa_prof_enable(C.c_int(1))
    for s in range(s_next, s_next + prof_steps):
        step_dev(s)
    s_next += prof_steps
    torch.cuda.synchronize()
    L.dsa_prof_enable(C.c_int(0))
    need = L.dsa_prof_dump(None, C.c_int64(0))
    buf = C.create_string_buffer(int(need) + 16)
    L.dsa_prof_dump(buf, C.c_int64(len(buf)))
    kernels = {}
    for ln in buf.value.decode().strip().splitlines():
        name, cnt, ms = ln.split(",")
        kernels[name] = {"launches_per_step": int(cnt) / prof_steps, "ms_per_step": float(ms) / prof_steps,
                         "avg_us": 1e3 * float(ms) / int(cnt)}
    inf = A.info(1)
    peak, peak_src = measured_peak_gbs()
    spmv_alg_bytes = 16 * (inf["nnz"] + inf["nb_partitions"]) + 8 * (N_COLS + M_ROWS)
    spmv_phys_bytes = 16 * inf["capacity"] + 8 * (N_COLS + M_ROWS)
    spmv_name = next((k for k in ("spmv_blocked", "spmv_flat") if k in kernels), "spmv_flat")
    # The SpMV's own duration: CUDA events around 30 back-to-back products on the library's stream (a kernel timed alone right
    # after a synchronisation starts on an idle GPU and reads ~15 us longer).  One product = the reduction kernel + the carry
    # fix-up + the scatter of y by row key (+ the memset of y): the whole call is charged to the kernel.
    n_sp = 30
    for _ in range(3):
        D._lib.check(L.dsa_matrix_spmv_dense_d(A._h, C.c_int(0), vp(d_x), C.c_int64(N_COLS), vp(d_y), C.c_int64(M_ROWS)))
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(n_sp):
        D._lib.check(L.dsa_matrix_spmv_dense_d(A._h, C.c_int(0), vp(d_x), C.c_int64(N_COLS), vp(d_y), C.c_int64(M_ROWS)))
    e1.record(stream)
    torch.cuda.synchronize()
    spmv_us = 1e3 * e0.elapsed_time(e1) / n_sp
    a = spmv_alg_bytes / (spmv_us * 1e-6) / 1e9
    spmv = {"kernel": spmv_name, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
            "frac_of_8TBs": a / 8000.0, "avg_us": spmv_us, "algorithmic_bytes": spmv_alg_bytes, "physical_bytes": spmv_phys_bytes,
            "traffic": ncu_traffic(spmv_name), "peak_source": peak_src,
            "how": f"{n_sp} back-to-back dsa_matrix_spmv_dense_d calls between two CUDA events (kernel + fix-up + epilogue per call)",
            "avg_us_single_launch_after_sync": kernels.get(spmv_name, {}).get("avg_us")}
    dom = max(kernels.items(), key=lambda kv: kv[1]["ms_per_step"]) if kernels else (None, None)
    roofline = None
    if dom[0]:
        name, k = dom
        if name == spmv_name:
            alg = spmv_alg_bytes
        else:   # a kernel of the update pipeline processes one orientation's share of the batch per launch
            alg = BYTES_PER_UPDATE_ONE * BATCH
        a = alg / (k["avg_us"] * 1e-6) / 1e9
        roofline = {"kernel": name, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak, "traffic": ncu_traffic(name),
                    "avg_us": k["avg_us"], "algorithmic_bytes": alg, "share_of_step": k["ms_per_step"] / sum(v["ms_per_step"] for v in kernels.values()),
                    "peak_source": peak_src}
        if roofline["traffic"]:   # what the kernel physically moves (ncu DRAM bytes of the committed capture) over the live duration
            roofline["physical_gbs"] = roofline["traffic"] / (k["avg_us"] * 1e-6) / 1e9
            roofline["physical_frac"] = roofline["physical_gbs"] / peak
        if name == "tile_merge":
            roofline["note"] = ("one pass over the orientation's keys (8 B per cell, changed or not) replaces the random-access locate / "
                                "apply / merge kernels for dense batches; the kernel is bound by instruction issue (DESIGN.md 6, 7)")

    # ---- e2e: host buffers through the host-pointer C-ABI calls ---------------------------------------------
    e2e = None
    if not args.no_e2e:
        hb = [tuple(torch.from_numpy(a).pin_memory() for a in b) for b in batches]
        h_x = torch.from_numpy(x).pin_memory()
        h_y = torch.zeros(M_ROWS, dtype=torch.float64).pin_memory()

        # The flush is double-buffered (dsa_matrix_stage_batch / dsa_matrix_apply_staged): the PCIe transfer of batch s+1 overlaps
        # the kernels of batch s.  Every copy (all K batches, x in, y out) happens inside the timed region: nothing is staged
        # before it starts.
        def run_host(first, last):
            bi, bj, bv = hb[first % P]
            D._lib.check(L.dsa_matrix_stage_batch(A._h, vp(bi), vp(bj), vp(bv), C.c_int64(BATCH)))
            for s in range(first, last):
                if s + 1 < last:
                    bi, bj, bv = hb[(s + 1) % P]
                    D._lib.check(L.dsa_matrix_stage_batch(A._h, vp(bi), vp(bj), vp(bv), C.c_int64(BATCH)))
                D._lib.check(L.dsa_matrix_apply_staged(A._h))
                D._lib.check(L.dsa_matrix_spmv_dense(A._h, C.c_int(0), vp(h_x), C.c_int64(N_COLS), vp(h_y), C.c_int64(M_ROWS)))

        run_host(s_next, s_next + W)
        s_next += W
        torch.cuda.synchronize()
        t_w0 = time.perf_counter()
        e0.record(stream)
        run_host(s_next, s_next + K)
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t_w0
        windows.append((t_w0, t_w0 + wall))
        s_next += K
        ms_e2e = max(e0.elapsed_time(e1), wall * 1e3) / K
        e2e = {"value": BATCH / (ms_e2e * 1e-3) / 1e6, "unit": "Mupdates/s", "h2d_bytes_per_step": 24 * BATCH + 8 * N_COLS,
               "d2h_bytes_per_step": 8 * M_ROWS, "ms_per_step": ms_e2e, "steps": K, "checksum": float(h_y.sum().item()),
               "api": "dsa_matrix_stage_batch + dsa_matrix_apply_staged + dsa_matrix_spmv_dense (host pinned buffers)"}
        # the same step through the plain synchronous call (no overlap of the copy), for reference
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(s_next, s_next + K):
            bi, bj, bv = hb[s % P]
            D._lib.check(L.dsa_matrix_set_batch(A._h, vp(bi), vp(bj), vp(bv), C.c_int64(BATCH)))
            D._lib.check(L.dsa_matrix_spmv_dense(A._h, C.c_int(0), vp(h_x), C.c_int64(N_COLS), vp(h_y), C.c_int64(M_ROWS)))
        torch.cuda.synchronize()
        s_next += K
        ms_sync = 1e3 * (time.perf_counter() - t0) / K
        e2e["synchronous_call"] = {"value": BATCH / (ms_sync * 1e-3) / 1e6, "ms_per_step": ms_sync, "steps": K,
                                   "api": "dsa_matrix_set_batch + dsa_matrix_spmv_dense"}

    clocks = sampler.stop(windows)

    # ---- CPU oracle on the SAME batches: parity of what was timed + cpu_baseline --------------------------------------------
    cpu, parity = None, {"checked": False, "reason": "--no-cpu-baseline"}
    if not args.no_cpu_baseline:
        r = oracle_chain(coo, batches, x, insert_only)
        err = rel_err(y_gpu, r["y"])
        err_io = rel_err(y_io, r["insert_only"][0])
        ok = err <= SPMV_RTOL and err_io <= SPMV_RTOL and nnz_gpu == r["nnz"] and nnz_io == r["insert_only"][1]
        parity = {"checked": True, "ok": bool(ok), "steps_compared": W + K, "y_max_rel_err": err, "y_insert_only_max_rel_err": err_io,
                  "rtol": SPMV_RTOL, "nnz": [int(nnz_gpu), int(r["nnz"])], "nnz_insert_only": [int(nnz_io), int(r["insert_only"][1])],
                  "oracle_checksum": float(np.sum(r["y"]))}
        t_upd, t_spmv = float(np.sum(r["upd"])), float(np.sum(r["spmv"]))
        cpu = {"value": BATCH * P / (t_upd + t_spmv) / 1e6, "unit": "Mupdates/s", "cores": 1, "kind": "port",
               "sample": f"{P} full steps (1M-update batch as a loop of setindex! + SpMV) on 1 host core; C++ restatement of the "
                         "reference (Julia not installed)",
               "update_s_per_step": t_upd / P, "spmv_s_per_step": t_spmv / P, "build_s": r["t_build"],
               "spmv_effective_gbs": spmv_alg_bytes / (t_spmv / P) / 1e9, "host_cores_available": os.cpu_count()}

    line = {
        "metric": "batched PCSR insert/delete Mupdates/s", "value": value, "unit": "Mupdates/s", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "timed_steps": K, "timed_region_s": ms_total * 1e-3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "value_insert_only": BATCH / (io_ms_step * 1e-3) / 1e6, "ms_per_step_insert_only": io_ms_step, "insert_only_repetitions": len(io_ms),
        "dtype": "int64 keys / f64 values", "data": "synthetic", "config": workload_config(1), "clocks": clocks, "e2e": e2e,
        "gpu_launches": int(launches), "gpu_launches_per_step": launches / K, "parity": parity,
        "roofline": roofline, "spmv": spmv, "cpu_baseline": cpu,
        "update_effective_gbs": BYTES_PER_UPDATE * BATCH / (ms_step * 1e-3) / 1e9, "kernels": kernels, "checksum": checksum,
        "checksum_after_steps": W + K, "nnz_after": int(nnz_gpu),
    }
    if dumped is not None:
        dumped["y_insert_only"] = y_io
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line))
    if parity.get("checked") and not parity["ok"]:
        sys.exit(3)


if __name__ == "__main__":
    main()
