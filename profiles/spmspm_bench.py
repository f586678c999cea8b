"""Sparse multi-vector product (dsa_matrix_spmspm_d) against k back-to-back one-vector calls (dsa_matrix_spmspv_d) and against
cuSPARSE SpGEMM (torch.sparse.mm of A's CSR with X's CSR), on config 2 (bench.py's matrix: 1e5 x 1e5, 1e7 nnz, after two
bench batches so that the layout is the one the bench step leaves).

    python profiles/spmspm_bench.py [--window-s 1.0] [--reps 3] [--out FILE]     one JSON line (stdout, and FILE if given)
    python profiles/spmspm_bench.py --prof [--out FILE]                          per-kernel times (dsa_prof_*), in a run of its own

For (k, nnz per column) in CASES and both orientations (A·X: X's rows are columns of A; Aᵀ·X: rows of A), X has k columns of
distinct random present partition keys with values in [-1, 1).  Arms, all with inputs and outputs on the device and prepared
outside the timing: one spmspm_d call; k spmspv_d calls, one per column; torch.sparse.mm(A_csr, X_csr) (A's compressed snapshot
and X as torch sparse CSR tensors).  Every arm is timed with CUDA events over as many back-to-back calls as fill --window-s,
after a warm-up; the arms alternate inside each of --reps repetitions, and the median and spread (min, max) are reported.
Checks in the same run: spmspm equals the stacked spmspv results bit for bit; cuSPARSE touches the same keys, and each value
is within 2 L u sum |x_j a_ij| of ours (L = terms of that output, u = 2^-53; the bound of any summation order)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import scipy.sparse as sp
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402
import dsa_b200 as D  # noqa: E402

CASES = ((16, 16), (256, 16), (256, 256), (4096, 16), (1024, 1024))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"card": name, "power_limit": power}


def prof(L, fn, calls=10):
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
    out = {}
    for ln in buf.value.decode().strip().splitlines():
        name, cnt, ms = ln.split(",")
        out[name] = {"us": 1e3 * float(ms) / calls, "launches": int(cnt) / calls}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prof", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    D.require_gpu()
    L = D.lib()
    _, coo, batches, _ = B.make_workload(3)
    A = D.dynamicsparse(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    for b in batches[:2]:
        A.set_batch(*b)
    st = torch.cuda.current_stream()
    D._lib.check(L.dsa_matrix_set_stream(A._h, C.c_void_p(st.cuda_stream)))
    rng = np.random.default_rng(8)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    m, n = A.size

    def timed(fn, calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(calls):
            fn()
        e1.record(st)
        e1.synchronize()
        return 1e3 * e0.elapsed_time(e1) / calls   # us per call

    line = {"arms": {}}
    for trans in (0, 1):
        ori = "AtX" if trans else "AX"
        dim = m if trans else n
        Acsr = A.to_torch(torch.sparse_csr)
        if trans:   # Aᵀ as CSR is A's CSC read with the dimensions swapped
            c = A.to_torch(torch.sparse_csc)
            Acsr = torch.sparse_csr_tensor(c.ccol_indices(), c.row_indices(), c.values(), size=(n, m))
        Aabs = torch.sparse_csr_tensor(Acsr.crow_indices(), Acsr.col_indices(), Acsr.values().abs(), size=Acsr.shape)
        live = np.unique((coo[0] if trans else coo[1]))
        rows = {}
        for k, per in CASES:
            cols = [np.sort(rng.choice(live, per, replace=False)) for _ in range(k)]
            ptr = np.concatenate([[0], np.cumsum([per] * k)]).astype(np.int64)
            xk = np.concatenate(cols).astype(np.int64)
            xv = rng.random(len(xk)) * 2.0 - 1.0
            dp, dk, dv = (torch.from_numpy(a).cuda() for a in (ptr, xk, xv))
            cnt = C.c_int64()
            D._lib.check(L.dsa_matrix_spmspm_d(A._h, C.c_int(trans), p(dp), p(dk), p(dv), C.c_int64(k), C.c_int64(len(xk)), None, None,
                                               None, C.c_int64(0), C.byref(cnt)))
            nnz = cnt.value
            yp = torch.empty(k + 1, dtype=torch.int64, device="cuda")
            yk = torch.empty(max(nnz, 1), dtype=torch.int64, device="cuda")
            yv = torch.empty(max(nnz, 1), dtype=torch.float64, device="cuda")
            cap1 = A.info(0 if trans else 1)["nb_semaphores"]
            y1k = torch.empty(cap1, dtype=torch.int64, device="cuda")
            y1v = torch.empty(cap1, dtype=torch.float64, device="cuda")
            S = sp.csr_matrix((xv, (xk - 1, np.repeat(np.arange(k), per))), shape=(dim, k))   # X's row key r at row r - 1
            Xcsr = torch.sparse_csr_tensor(torch.from_numpy(S.indptr.astype(np.int64)).cuda(), torch.from_numpy(S.indices.astype(np.int64)).cuda(),
                                           torch.from_numpy(S.data).cuda(), size=(dim, k))
            Xabs = torch.sparse_csr_tensor(Xcsr.crow_indices(), Xcsr.col_indices(), Xcsr.values().abs(), size=Xcsr.shape)

            def spmspm():
                D._lib.check(L.dsa_matrix_spmspm_d(A._h, C.c_int(trans), p(dp), p(dk), p(dv), C.c_int64(k), C.c_int64(len(xk)), p(yp),
                                                   p(yk), p(yv), C.c_int64(nnz), C.byref(cnt)))

            def loop(collect=None):
                c1 = C.c_int64()
                for c in range(k):
                    o = int(ptr[c])
                    D._lib.check(L.dsa_matrix_spmspv_d(A._h, C.c_int(trans), C.c_void_p(dk.data_ptr() + 8 * o),
                                                       C.c_void_p(dv.data_ptr() + 8 * o), C.c_int64(per), p(y1k), p(y1v), C.c_int64(cap1),
                                                       C.byref(c1)))
                    if collect is not None:
                        collect.append((y1k[:c1.value].cpu().numpy(), y1v[:c1.value].cpu().numpy()))

            def cusparse():
                return torch.sparse.mm(Acsr, Xcsr)

            if args.prof:
                rows[f"{k}x{per}"] = {"k": k, "nnz_per_col": per, "count": nnz, "spmspm_d_us_by_kernel": prof(L, spmspm)}
                print(json.dumps({ori: rows[f"{k}x{per}"]}), file=sys.stderr, flush=True)
                continue
            spmspm()
            torch.cuda.synchronize()
            gp, gk, gv = yp.cpu().numpy(), yk[:nnz].cpu().numpy(), yv[:nnz].cpu().numpy()
            stacked = []
            loop(stacked)
            bit_identical = all(np.array_equal(gk[gp[c]:gp[c + 1]], s[0]) and
                                np.array_equal(gv[gp[c]:gp[c + 1]].view(np.int64), s[1].view(np.int64)) for c, s in enumerate(stacked))
            Y = cusparse().to_sparse_csc()
            Yabs = torch.sparse.mm(Aabs, Xabs).to_sparse_csc()
            cp, ck, cv = Y.ccol_indices().cpu().numpy(), Y.row_indices().cpu().numpy() + 1, Y.values().cpu().numpy()
            same_keys = bool(np.array_equal(cp, gp) and np.array_equal(ck, gk))
            within = False
            if same_keys:
                within = bool(np.all(np.abs(cv - gv) <= 2.0 * per * 2.0 ** -53 * Yabs.values().cpu().numpy()))
            fns = {"spmspm_d": spmspm, "spmspv_d_loop": loop, "cusparse_spgemm": cusparse}
            calls = {}
            for name, fn in fns.items():
                for _ in range(2):
                    fn()
                torch.cuda.synchronize()
                calls[name] = max(2, int(args.window_s * 1e6 / timed(fn, 2)))
            t = {name: [] for name in fns}
            for _ in range(args.reps):   # the arms alternate inside every repetition
                for name, fn in fns.items():
                    t[name].append(timed(fn, calls[name]))
            row = {"k": k, "nnz_per_col": per, "nnz_x": len(xk), "count": nnz, "spmspm_equals_stacked_spmspv": bool(bit_identical),
                   "cusparse_same_keys": same_keys, "cusparse_within_bound": within}
            for name in fns:
                row[name] = {"us_per_call": float(np.median(t[name])), "spread_us": [min(t[name]), max(t[name])], "calls_per_window": calls[name]}
            row["loop_over_spmspm"] = row["spmspv_d_loop"]["us_per_call"] / row["spmspm_d"]["us_per_call"]
            row["cusparse_over_spmspm"] = row["cusparse_spgemm"]["us_per_call"] / row["spmspm_d"]["us_per_call"]
            rows[f"{k}x{per}"] = row
            print(json.dumps({ori: {f"{k}x{per}": row}}), file=sys.stderr, flush=True)
        line["arms"][ori] = rows
    line.update(card())
    line["matrix"] = {"m": B.M_ROWS, "n": B.N_COLS, "nnz": A.info(1)["nnz"], "state": "bulk build + 2 bench batches"}
    out = json.dumps(line)
    print(out, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
