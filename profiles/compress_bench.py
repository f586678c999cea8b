"""Compressed snapshot of config 2 (bench.py's matrix: 1e5 x 1e5, 1e7 nnz, after two bench batches so that the layout is the one
the bench step leaves): dsa_matrix_compress_d (sparse pointer) and dsa_matrix_compress_dense_d (dense pointer, base 0), both
orientations.

    python profiles/compress_bench.py [--window-s 1.0] [--reps 3]     one JSON line
    python profiles/compress_bench.py --prof                         per-kernel times (dsa_prof_*), one JSON line

Every call is timed with CUDA events over as many back-to-back calls as fill --window-s, after a warm-up, --reps times: the
median and the spread (min, max) are reported.  The gapped arrays (2 x 134 MB per orientation) and the outputs (160 MB) are
larger than the 126 MB L2, so every call streams from HBM.  Copy-rate reference, in the same process: a device-to-device copy
of a 430 MB buffer (torch copy_, 860 MB moved), timed the same way.
Bytes a call moves (two passes): keys 8 B x capacity read twice, values 8 B x capacity read once, writes 16 B x nnz plus the
pointer, 8 B x (np + 1) (sparse form) or 8 B x (dim + 1) (dense form).  Each output is checked bit for bit against a numpy
compaction of export(which).  The host path it replaces (to_coo: raw export + numpy compaction) is timed once for context."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench as B  # noqa: E402
import dsa_b200 as D  # noqa: E402
from compress_ref import compact, dense  # noqa: E402

COPY_BYTES = 430_000_000


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
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    dev = lambda k, dt=torch.int64: torch.empty(k, dtype=dt, device="cuda")  # noqa: E731

    arms = {}
    for which in (0, 1):
        inf = A.info(which)
        npart, nnz, cap = inf["nb_partitions"], inf["nnz"], inf["capacity"]
        dim, idim = (n, m) if which == 0 else (m, n)
        cnt, cnt1 = np.zeros(2, np.int64), C.c_int64()
        sp = (dev(npart), dev(npart + 1), dev(nnz), dev(nnz, torch.float64))
        dn = (dev(dim + 1), dev(nnz), dev(nnz, torch.float64))

        def sparse(which=which, sp=sp, npart=npart, nnz=nnz, cnt=cnt):
            D._lib.check(L.dsa_matrix_compress_d(A._h, C.c_int(which), *(p(t) for t in sp), C.c_int64(npart), C.c_int64(nnz), cnt.ctypes.data_as(C.c_void_p)))

        def dense0(which=which, dn=dn, dim=dim, idim=idim, nnz=nnz, cnt1=cnt1):
            D._lib.check(L.dsa_matrix_compress_dense_d(A._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(0), *(p(t) for t in dn),
                                                       C.c_int64(nnz), C.byref(cnt1)))

        reads = 8 * cap * 2 + 8 * cap
        arms[f"{'col' if which == 0 else 'row'}major_sparse"] = (sparse, reads + 16 * nnz + 8 * (npart + 1), which, sp, None)
        arms[f"{'col' if which == 0 else 'row'}major_dense"] = (dense0, reads + 16 * nnz + 8 * (dim + 1), which, dn, (dim, idim))

    if args.prof:
        out = {}
        for name, (fn, _, _, _, _) in arms.items():
            fn()
            torch.cuda.synchronize()
            L.dsa_prof_reset()
            L.dsa_prof_enable(C.c_int(1))
            for _ in range(20):
                fn()
            L.dsa_prof_enable(C.c_int(0))
            L.dsa_prof_dump.restype = C.c_int64
            buf = C.create_string_buffer(int(L.dsa_prof_dump(None, C.c_int64(0))) + 16)
            L.dsa_prof_dump(buf, C.c_int64(len(buf)))
            out[name] = {ln.split(",")[0]: 1e3 * float(ln.split(",")[2]) / 20 for ln in buf.value.decode().strip().splitlines()}
        print(json.dumps({"us_per_call_by_kernel": out, **card()}), flush=True)
        return

    # bit-for-bit check of every output against the numpy compaction of the raw export
    exact = {}
    for name, (fn, _, which, outs, dims) in arms.items():
        fn()
        torch.cuda.synchronize()
        pk, ptr, k, v = compact(A.export(which))
        got = [t.cpu().numpy() for t in outs]
        if dims is None:
            want = (pk, ptr, k, v)
        else:
            want = dense(pk, ptr, k, dims[0], 0) + (v,)
        exact[name] = all(np.array_equal(g.view(np.uint64) if g.dtype == np.float64 else g,
                                         w.view(np.uint64) if w.dtype == np.float64 else w) for g, w in zip(got, want))

    src, dst = torch.empty(COPY_BYTES // 8, dtype=torch.float64, device="cuda"), torch.empty(COPY_BYTES // 8, dtype=torch.float64, device="cuda")
    src.fill_(1.0)

    def copy():
        dst.copy_(src)

    def timed(fn, calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(calls):
            fn()
        e1.record(st)
        e1.synchronize()
        return 1e3 * e0.elapsed_time(e1) / calls   # us per call

    fns = {name: a[0] for name, a in arms.items()}
    fns["copy_430MB"] = copy
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
    copy_us = float(np.median(t["copy_430MB"]))
    copy_rate = 2 * COPY_BYTES / copy_us / 1e3   # GB/s, read + write
    line = {"copy_430MB": {"us": copy_us, "spread_us": [min(t["copy_430MB"]), max(t["copy_430MB"])], "gbs": copy_rate}}
    for name, (_, nbytes, _, _, _) in arms.items():
        med = float(np.median(t[name]))
        line[name] = {"us_per_call": med, "spread_us": [min(t[name]), max(t[name])], "calls_per_window": calls[name], "bytes": nbytes,
                      "gbs": nbytes / med / 1e3, "of_copy_rate": nbytes / med / 1e3 / copy_rate,
                      "floor_us_at_copy_rate": nbytes / copy_rate / 1e3, "bit_identical": exact[name]}
    t0 = time.perf_counter()
    api_rows, _, _ = D.to_coo(A)
    line["host_to_coo_ms_once"] = 1e3 * (time.perf_counter() - t0)
    line.update(card())
    line["matrix"] = {"m": m, "n": n, "nnz": int(len(api_rows)), "capacity_colmajor": A.info(0)["capacity"],
                      "capacity_rowmajor": A.info(1)["capacity"], "state": "bulk build + 2 bench batches"}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
