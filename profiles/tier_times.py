"""Per-launch times of the rebalance tiers the bench step never runs: windows above SMALL_CELLS cells (merge_scatter_big,
scatter_inserts_big, copyback_big) and a resize (merge_scatter_root, scatter_inserts_root, layout_gaps).

    python profiles/tier_times.py [--reps N] [--tag NAME]

Each case copies a freshly built structure and applies one batch under the library's per-kernel event profile (prof mode: one
kernel at a time), N times after one warm-up.  One JSON line per case: mean microseconds per launch of each tier kernel, and
a digest of the layout the batch left (so two builds can be compared on the same inputs)."""
import argparse
import copy
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dsa_b200 as D  # noqa: E402

TIERS = ("merge_scatter_big", "scatter_inserts_big", "copyback_big", "merge_scatter_root", "scatter_inserts_root", "layout_gaps")


def profiled(fn):
    L = D.lib()
    L.dsa_prof_reset()
    L.dsa_prof_enable(C.c_int(1))
    try:
        fn()
    finally:
        L.dsa_prof_enable(C.c_int(0))
    buf = C.create_string_buffer(int(L.dsa_prof_dump(None, C.c_int64(0))) + 16)
    L.dsa_prof_dump(buf, C.c_int64(len(buf)))
    L.dsa_prof_reset()
    out = {}
    for ln in buf.value.decode().strip().splitlines():
        name, cnt, ms = ln.split(",")
        out[name] = (int(cnt), float(ms))
    return out


def digest(x):
    h = hashlib.sha256()
    exports = [x.export()] if isinstance(x, D.DynamicSparseVector) else [x.export(0), x.export(1)]
    for e in exports:
        for a in (e if isinstance(e, tuple) else (e["tag"], e["key"], e["val"], e["semaphores"])):
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def cases():
    rng = np.random.default_rng(0xD5A00001)
    keys = np.unique(rng.integers(1, 10_000_000_000, 1_000_000))   # the vector of config 1: 2^21 cells
    vals = rng.integers(10, 100001, len(keys)) / 10.0
    vec = D.dynamicsparsevec(keys, vals)
    wide = np.nonzero(np.diff(keys) > 4000)[0]
    wide = wide[np.linspace(0, len(wide) - 1, 64).astype(int)]      # 64 gaps far apart: 4000 consecutive keys into each
    k = np.concatenate([keys[i] + 1 + np.arange(4000) for i in wide])
    yield "vector_big_windows", vec, lambda x: x.set_batch(k, np.full(len(k), 1.5))
    k2 = rng.integers(1, 10_000_000_000, 1_100_000)                # more elements than cells: 2^21 -> 2^22 cells
    yield "vector_resize", vec, lambda x: x.set_batch(k2, np.full(len(k2), 2.5))

    m = n = 5_000                                                   # config 5's matrix and its monotone batch
    I, J = rng.integers(1, m + 1, 200_000), rng.integers(1, n + 1, 200_000)
    mat = D.dynamicsparse(I, J, rng.random(200_000) + 0.01, m=m, n=n)
    hot = rng.choice(n, 100, replace=False) + 1
    I2, J2 = np.concatenate([np.arange(m + 1, m + 401) for _ in hot]), np.repeat(hot, 400)
    yield "matrix_big_windows", mat, lambda x: x.set_batch(I2, J2, np.full(len(I2), 0.5))
    m = n = 100_000
    I, J = rng.integers(1, m + 1, 2_000_000), rng.integers(1, n + 1, 2_000_000)
    big = D.dynamicsparse(I, J, rng.random(2_000_000) + 0.5, m=m, n=n)
    I3, J3 = rng.integers(1, m + 1, 2_000_000), rng.integers(1, n + 1, 2_000_000)
    yield "matrix_resize", big, lambda x: x.set_batch(I3, J3, np.full(len(I3), 0.25))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    D.require_gpu()
    for name, base, batch in cases():
        tot = {}
        dig = None
        for rep in range(args.reps + 1):
            x = copy.deepcopy(base)
            prof = profiled(lambda: batch(x))
            if rep == 0:
                dig = digest(x)
                continue
            for t in TIERS:
                if t in prof:
                    c, ms = tot.get(t, (0, 0.0))
                    tot[t] = (c + prof[t][0], ms + prof[t][1])
            del x
        us = {t: round(1000.0 * ms / c, 2) for t, (c, ms) in tot.items()}
        launches = {t: c // args.reps for t, (c, _) in tot.items()}
        print(json.dumps({"tag": args.tag, "case": name, "us_per_launch": us, "launches_per_batch": launches, "layout": dig}), flush=True)


if __name__ == "__main__":
    main()
