"""Multi-vector product against k single-vector products, config 2 (bench.py's matrix: 1e5 x 1e5, 1e7 nnz, after two bench
batches so that the layout is the one the bench step leaves).

    python profiles/spmm_bench.py [--window-s 1.0] [--reps 3]     one JSON line per k in {1, 2, 4, 8, 16, 32}
    python profiles/spmm_bench.py --prof                         per-kernel times (dsa_prof_*) of both arms, k = 8

Arms, both on device-resident data and both orientations: ONE dsa_matrix_spmm_dense_d call on X (nx x k, row-major), against k
back-to-back dsa_matrix_spmv_dense_d calls on the k columns (prepared as contiguous vectors outside the timed region).  Each
arm is timed with CUDA events over as many calls as fill --window-s, after a warm-up; the arms alternate, --reps times, and
the median and the spread (min, max) of the repetitions are reported.  The gapped arrays (2 x 268 MB) are larger than the
126 MB L2, so every pass over the matrix streams them from HBM.
Algorithmic bytes of a call: 16 B per cell (key + value) of the partitions' elements and semaphores per pass over the matrix,
plus 8 B per entry of X and of Y: 16 (nnz + partitions) passes + 8 k (nx + ny), passes = ceil(k / 32) for the multi-vector
call and k for the single products.  The result of the multi-vector arm is checked in the same run against the stacked
single products, bit for bit."""
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

KS = (1, 2, 4, 8, 16, 32)
COLS_PER_PASS = 32   # dsa_matrix_spmm_dense: columns carried by one pass over the matrix


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"card": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prof", action="store_true")
    args = ap.parse_args()
    D.require_gpu()
    L = D.lib()
    _, coo, batches, _ = B.make_workload(3)
    A = D.dynamicsparse(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    for b in batches[:2]:
        A.set_batch(*b)
    st = torch.cuda.current_stream()
    D._lib.check(L.dsa_matrix_set_stream(A._h, C.c_void_p(st.cuda_stream)))
    m, n = A.size
    cells = {t: A.info(D._lib.COLMAJOR if t else D._lib.ROWMAJOR)["nb_elements"] for t in (0, 1)}   # nnz + partitions
    gen = torch.Generator(device="cuda").manual_seed(0x5EED)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def arms(k, trans):
        nx, ny = (m, n) if trans else (n, m)
        X = torch.rand((nx, k), dtype=torch.float64, device="cuda", generator=gen)
        Y = torch.empty((ny, k), dtype=torch.float64, device="cuda")
        xs = [X[:, c].contiguous() for c in range(k)]
        ys = [torch.empty(ny, dtype=torch.float64, device="cuda") for _ in range(k)]

        def multi():
            D._lib.check(L.dsa_matrix_spmm_dense_d(A._h, C.c_int(trans), p(X), C.c_int64(nx), C.c_int64(k), C.c_int64(k), p(Y),
                                                   C.c_int64(ny), C.c_int64(k)))

        def single():
            for c in range(k):
                D._lib.check(L.dsa_matrix_spmv_dense_d(A._h, C.c_int(trans), p(xs[c]), C.c_int64(nx), p(ys[c]), C.c_int64(ny)))

        return nx, ny, Y, ys, multi, single

    if args.prof:
        for trans in (0, 1):
            _, _, _, _, multi, single = arms(8, trans)
            for name, fn in (("multi", multi), ("single", single)):
                fn()
                torch.cuda.synchronize()
                L.dsa_prof_reset()
                L.dsa_prof_enable(C.c_int(1))
                for _ in range(20):
                    fn()
                L.dsa_prof_enable(C.c_int(0))
                buf = C.create_string_buffer(int(L.dsa_prof_dump(None, C.c_int64(0))) + 16)
                L.dsa_prof_dump(buf, C.c_int64(len(buf)))
                kern = {}
                for ln in buf.value.decode().strip().splitlines():
                    kname, cnt, ms = ln.split(",")
                    kern[kname] = {"launches_per_call": int(cnt) / 20, "us_per_call": 1e3 * float(ms) / 20}
                print(json.dumps({"k": 8, "trans": trans, "arm": name, "kernels": kern, **card()}))
        return

    def timed(fn, calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(calls):
            fn()
        e1.record(st)
        e1.synchronize()
        return 1e3 * e0.elapsed_time(e1) / calls   # us per call

    prov = card()
    for k in KS:
        line = {"k": k}
        for trans in (0, 1):
            nx, ny, Y, ys, multi, single = arms(k, trans)
            calls = {}
            for name, fn in (("multi", multi), ("single", single)):
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                calls[name] = max(3, int(args.window_s * 1e6 / timed(fn, 5)))
            t = {"multi": [], "single": []}
            for _ in range(args.reps):
                for name, fn in (("multi", multi), ("single", single)):
                    t[name].append(timed(fn, calls[name]))
            torch.cuda.synchronize()
            Yh = Y.cpu().numpy()
            exact = all(np.array_equal(Yh[:, c], ys[c].cpu().numpy()) for c in range(k))
            res = {}
            for name, passes in (("multi", -(-k // COLS_PER_PASS)), ("single", k)):
                med = float(np.median(t[name]))
                nbytes = 16 * cells[trans] * passes + 8 * k * (nx + ny)
                res[name] = {"us_per_call": med, "spread_us": [min(t[name]), max(t[name])], "calls_per_window": calls[name],
                             "passes": passes, "bytes": nbytes, "gbs": nbytes / med / 1e3}
            res["multi_over_single"] = res["multi"]["us_per_call"] / res["single"]["us_per_call"]
            res["bit_identical"] = bool(exact)
            line[f"trans{trans}"] = res
        line.update(prov)
        line["matrix"] = {"m": m, "n": n, "cells_rowmajor": cells[0], "cells_colmajor": cells[1], "state": "bulk build + 2 bench batches"}
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
