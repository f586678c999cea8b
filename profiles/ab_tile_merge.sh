#!/bin/bash
# A/B of k_tile_merge against the parent commit, on ONE GPU, everything in one run:
#   git archive <parent> | tar -x -C ab_parent      (an untracked, git-ignored copy of the parent tree)
#   bash profiles/ab_tile_merge.sh OUTDIR [PAIRS] [tests]
# Writes under OUTDIR: the card, both builds, the outputs of bench.py --dump-outputs for both trees and their comparison,
# PAIRS alternating parent/branch bench runs (ab.jsonl), and with "tests" the GPU suite of both trees and smoke() of the branch.
set +e
[ -n "$1" ] || { echo "usage: bash profiles/ab_tile_merge.sh OUTDIR [PAIRS] [tests]"; exit 2; }
mkdir -p "$1"
OUT=$(realpath "$1")
PAIRS=${2:-3}
export PYTHONUNBUFFERED=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
for tree in ab_parent .; do
    (cd "$tree" && python -c "import __graft_entry__ as g; g.build()" > "$OUT/build_$(basename "$(realpath "$tree")").log" 2>&1) || echo "build failed: $tree"
done
if [ "$3" = "tests" ]; then
    python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee "$OUT/smoke.log"
    for tree in ab_parent .; do
        name=$( [ "$tree" = . ] && echo branch || echo parent )
        (cd "$tree" && timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -4) > "$OUT/pytest_gpu_$name.log"
        echo "gpu suite $name: $(tail -1 "$OUT/pytest_gpu_$name.log")"
    done
fi
# same results: the outputs of the last timed step, bit for bit
for tree in ab_parent .; do
    name=$( [ "$tree" = . ] && echo branch || echo parent )
    (cd "$tree" && timeout 600 python bench.py --steps 20 --warmup 5 --dump-outputs "$OUT/dump_$name" > "$OUT/dump_$name.json" 2> "$OUT/dump_$name.err")
    echo "dump $name rc=$?"
done
python - "$OUT" <<'EOF'
import glob, json, os, sys
import numpy as np
out = sys.argv[1]
names = sorted(os.path.basename(f) for f in glob.glob(f"{out}/dump_parent/*.npy"))
same = {n: bool(np.array_equal(np.load(f"{out}/dump_parent/{n}"), np.load(f"{out}/dump_branch/{n}"))) for n in names}
js = [json.loads(open(f"{out}/dump_{w}.json").read().strip().splitlines()[-1]) for w in ("parent", "branch")]
pick = lambda j: (j.get("gpu_launches"), j.get("nnz_after"), (j.get("parity") or {}).get("ok"))
print("arrays identical:", same, "| launches, nnz_after, parity.ok:", [pick(j) for j in js])
EOF
rm -rf "$OUT/dump_parent" "$OUT/dump_branch"   # the arrays are large; the comparison above is what is kept
# timing: alternating pairs
: > "$OUT/ab.jsonl"
for i in $(seq 1 "$PAIRS"); do
    for tree in ab_parent .; do
        name=$( [ "$tree" = . ] && echo branch || echo parent )
        line=$(cd "$tree" && timeout 600 python bench.py --steps 20 --warmup 5 2> "$OUT/ab_${name}_$i.err" | tail -1)
        echo "{\"tree\": \"$name\", \"pair\": $i, \"result\": ${line:-null}}" >> "$OUT/ab.jsonl"
    done
done
python - "$OUT" <<'EOF'
import json, sys
for ln in open(f"{sys.argv[1]}/ab.jsonl"):
    d = json.loads(ln); r = d["result"] or {}
    print(d["tree"], d["pair"], "value %.1f" % r.get("value", 0), "tile_merge %.1f us" % r.get("kernels", {}).get("tile_merge", {}).get("avg_us", 0),
          "insert_only %.1f" % r.get("value_insert_only", 0), "e2e %.1f" % (r.get("e2e") or {}).get("value", 0))
EOF
