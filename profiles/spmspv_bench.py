"""Sparse-x product driven by x's entries (dsa_matrix_spmspv[_d]) against the streaming product (dsa_matrix_spmv) on config 2
(bench.py's matrix: 1e5 x 1e5, 1e7 nnz, after two bench batches so that the layout is the one the bench step leaves).

    python profiles/spmspv_bench.py [--window-s 1.0] [--reps 3] [--out FILE]     one JSON line (stdout, and FILE if given)

For nx random present columns (A·x, trans 0) or rows (Aᵀ·x, trans 1), nx in 1, 16, 256, 4096, 32768, 100000, three arms on the
same x: dsa_matrix_spmspv_d (x and y on the device), dsa_matrix_spmspv (host buffers) and dsa_matrix_spmv (host buffers, the
streaming product).  Every arm is timed with CUDA events over as many back-to-back calls as fill --window-s, after a warm-up;
the arms alternate inside each of --reps repetitions, and the median and spread (min, max) are reported.
Algorithmic bytes of the new call: 16 B per cell of the selected spans (keys and values read once; gaps included) + 8 B per x
entry + 16 B per output entry.  The crossover is the first nx of the list at which the new call is no faster than the
streaming one.  The outputs of the new call are checked bit for bit against the oracle's mul (the reference's loop) at
nx = 256 and 4096 in both orientations.  Per-kernel times of the new call (dsa_prof_*: every launch waited for, so a small
kernel's time includes its launch latency) at nx = 1, 256, 32768 and 100000, after the timed windows."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402
import dsa_b200 as D  # noqa: E402
from oracle import oracle as O  # noqa: E402

NXS = (1, 16, 256, 4096, 32768, 100_000)
CHECK_NX = (256, 4096)
PROF_NX = (1, 256, 32768, 100_000)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"card": name, "power_limit": power}


def span_cells(A, which):
    """partition key -> cells of its span (semaphore excluded, gaps included), from the raw layout"""
    e = A.export(which)
    live = e["col_live"].astype(bool)
    keys, sem = e["col_keys"][live], e["semaphores"][live] - 1      # 0-based semaphore positions
    o = np.argsort(sem)
    keys, sem = keys[o], sem[o]
    end = np.append(sem[1:], e["capacity"])
    return dict(zip(keys.tolist(), (end - sem - 1).tolist())), np.sort(keys)


def prof(L, fn, calls=20):
    """per-kernel (and per-copy) times of one call, us, from the library's per-launch events"""
    fn()
    torch.cuda.synchronize()
    L.dsa_prof_reset()
    L.dsa_prof_enable(C.c_int(1))
    for _ in range(calls):
        fn()
    L.dsa_prof_enable(C.c_int(0))
    L.dsa_prof_dump.restype = C.c_int64
    buf = C.create_string_buffer(int(L.dsa_prof_dump(None, C.c_int64(0))) + 16)
    L.dsa_prof_dump(buf, C.c_int64(len(buf)))
    L.dsa_prof_reset()
    return {ln.split(",")[0]: 1e3 * float(ln.split(",")[2]) / calls for ln in buf.value.decode().strip().splitlines() if ln}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    D.require_gpu()
    L = D.lib()
    _, coo, batches, _ = B.make_workload(3)
    A = D.dynamicsparse(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    om = O.Matrix(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    for b in batches[:2]:
        A.set_batch(*b)
        om.set_batch_policy(*b)
    st = torch.cuda.current_stream()
    D._lib.check(L.dsa_matrix_set_stream(A._h, C.c_void_p(st.cuda_stream)))
    rng = np.random.default_rng(6)
    p = lambda a: C.c_void_p(a.data_ptr() if isinstance(a, torch.Tensor) else a.ctypes.data)  # noqa: E731

    def timed(fn, calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(calls):
            fn()
        e1.record(st)
        e1.synchronize()
        return 1e3 * e0.elapsed_time(e1) / calls   # us per call

    line = {"arms": {}, "crossover": {}}
    for trans in (0, 1):
        cells, live = span_cells(A, 1 if trans else 0)     # x selects partitions of the row-major (trans) / column-major twin
        cap = A.info(0 if trans else 1)["nb_semaphores"]
        yk, yv = np.zeros(cap, np.int64), np.zeros(cap)
        dyk, dyv = torch.empty(cap, dtype=torch.int64, device="cuda"), torch.empty(cap, dtype=torch.float64, device="cuda")
        cnt = C.c_int64()
        ori = "Atx" if trans else "Ax"
        rows = {}
        for nx in NXS:
            xk = np.sort(rng.choice(live, min(nx, len(live)), replace=False)).astype(np.int64)
            xv = rng.random(len(xk)) * 2.0 - 1.0
            dxk, dxv = torch.from_numpy(xk).cuda(), torch.from_numpy(xv).cuda()
            torch.cuda.synchronize()

            def new_d(xk=xk, dxk=dxk, dxv=dxv):
                D._lib.check(L.dsa_matrix_spmspv_d(A._h, C.c_int(trans), p(dxk), p(dxv), C.c_int64(len(xk)), p(dyk), p(dyv), C.c_int64(cap),
                                                   C.byref(cnt)))

            def new_h(xk=xk, xv=xv):
                D._lib.check(L.dsa_matrix_spmspv(A._h, C.c_int(trans), p(xk), p(xv), C.c_int64(len(xk)), p(yk), p(yv), C.c_int64(cap),
                                                 C.byref(cnt)))

            def old_h(xk=xk, xv=xv):
                D._lib.check(L.dsa_matrix_spmv(A._h, C.c_int(trans), p(xk), p(xv), C.c_int64(len(xk)), p(yk), p(yv), C.c_int64(cap),
                                               C.byref(cnt)))

            fns = {"spmspv_d": new_d, "spmspv_host": new_h, "spmv_host": old_h}
            new_d()
            torch.cuda.synchronize()
            count = cnt.value
            row = {"nx": len(xk), "count": count, "span_cells": int(sum(cells[k] for k in xk.tolist()))}
            row["bytes_new"] = 16 * row["span_cells"] + 8 * len(xk) + 16 * count
            if nx in CHECK_NX:
                ok, ov = om.mul(xk, xv, trans=bool(trans))
                gk, gv = dyk[:count].cpu().numpy(), dyv[:count].cpu().numpy()
                new_h()
                row["bit_identical_to_oracle"] = bool(np.array_equal(gk, ok) and np.array_equal(gv.view(np.int64), ov.view(np.int64))
                                                      and np.array_equal(yk[:count], ok) and np.array_equal(yv[:count].view(np.int64), ov.view(np.int64)))
                old_h()
                row["same_keys_as_streaming"] = bool(cnt.value == count and np.array_equal(yk[:count], ok))
            calls = {}
            for name, fn in fns.items():
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                calls[name] = max(3, int(args.window_s * 1e6 / timed(fn, 5)))
            t = {name: [] for name in fns}
            for _ in range(args.reps):   # the arms alternate inside every repetition
                for name, fn in fns.items():
                    t[name].append(timed(fn, calls[name]))
            for name in fns:
                med = float(np.median(t[name]))
                row[name] = {"us_per_call": med, "spread_us": [min(t[name]), max(t[name])], "calls_per_window": calls[name]}
            row["spmspv_d_gbs"] = row["bytes_new"] / row["spmspv_d"]["us_per_call"] / 1e3
            if nx in PROF_NX:
                row["spmspv_d_us_by_kernel"] = prof(L, new_d)
            rows[str(nx)] = row
            print(json.dumps({ori: {str(nx): row}}), file=sys.stderr, flush=True)
        line["arms"][ori] = rows
        for arm in ("spmspv_d", "spmspv_host"):
            slower = [nx for nx in NXS if rows[str(nx)][arm]["us_per_call"] >= rows[str(nx)]["spmv_host"]["us_per_call"]]
            line["crossover"][f"{ori}_{arm}_vs_spmv_host"] = slower[0] if slower else None
    line.update(card())
    line["matrix"] = {"m": B.M_ROWS, "n": B.N_COLS, "nnz": A.info(1)["nnz"], "capacity_colmajor": A.info(0)["capacity"],
                      "capacity_rowmajor": A.info(1)["capacity"], "state": "bulk build + 2 bench batches"}
    out = json.dumps(line)
    print(out, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
