#!/bin/bash
# A/B of the inference benchmark between a checkout of the parent commit and this tree, alternating, in one session on
# one GPU: card name / power limit / max SM clock, RUNS x bench.py per tree (no CPU / eager legs), one --breakdown per
# tree (inference and training), and --dump-outputs of both trees compared (max |logits difference|, mask agreement).
#   usage: tools/ab_decoder_split.sh PARENT_TREE OUT_DIR [RUNS]      (OUT_DIR: where the logs and the summary go)
set -u
cd "$(dirname "$0")/.."
PARENT=$(cd "$1" && pwd)
mkdir -p "$2"
OUT=$(cd "$2" && pwd)
RUNS=${3:-5}
BRANCH=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv"
cat "$OUT/gpu.csv"
for t in parent branch; do
  d=$PARENT; [ $t = branch ] && d=$BRANCH
  (cd "$d" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_$t.log" 2>&1 || { echo "build $t failed"; tail -5 "$OUT/build_$t.log"; exit 1; }
done
for i in $(seq 1 "$RUNS"); do
  for t in parent branch; do
    d=$PARENT; [ $t = branch ] && d=$BRANCH
    (cd "$d" && timeout 600 python bench.py --no-cpu-baseline --no-eager-baseline) > "$OUT/bench_${t}_$i.json" 2> "$OUT/bench_${t}_$i.err"
    echo "run $i $t rc=$?"
  done
done
for t in parent branch; do
  d=$PARENT; [ $t = branch ] && d=$BRANCH
  (cd "$d" && timeout 600 python bench.py --no-cpu-baseline --no-eager-baseline --no-train-leg --breakdown \
     --dump-outputs "$OUT/dump_$t") > "$OUT/breakdown_$t.json" 2> "$OUT/breakdown_$t.txt"
  echo "breakdown $t rc=$?"
  (cd "$d" && timeout 600 python bench.py --workload train --steps 20 --warmup 5 --breakdown) \
     > "$OUT/train_breakdown_$t.json" 2> "$OUT/train_breakdown_$t.txt"
  echo "train breakdown $t rc=$?"
done
python - "$OUT" "$RUNS" <<'PY'
import glob, json, os, sys
import numpy as np
out, runs = sys.argv[1], int(sys.argv[2])
keys = [("value", lambda d: d["value"]), ("e2e", lambda d: d["e2e"]["value"]), ("ms_per_step", lambda d: d["ms_per_step"]),
        ("train_img_s", lambda d: d["config"]["train_img_s"]), ("train_ms_per_step", lambda d: d["config"]["train_ms_per_step"]),
        ("sm_mhz", lambda d: d["clocks"]["sm_mhz"])]
res = {}
for t in ("parent", "branch"):
    rows = []
    for i in range(1, runs + 1):
        try:
            rows.append(json.loads(open(f"{out}/bench_{t}_{i}.json").read().strip().splitlines()[-1]))
        except Exception as e:  # noqa: BLE001
            print(t, i, "no result:", e)
    res[t] = {k: [f(d) for d in rows] for k, f in keys}
lines = []
for k, _ in keys:
    p, b = res["parent"][k], res["branch"][k]
    if not p or not b:
        continue
    fmt = lambda v: f"median {np.median(v):.4g} min {min(v):.4g} max {max(v):.4g}"   # noqa: E731
    lines.append(f"{k:18s} parent {fmt(p)} | branch {fmt(b)} | median ratio {np.median(b) / np.median(p):.4f}")
for t in ("parent", "branch"):
    with open(f"{out}/breakdown_{t}.txt") as f:
        for ln in f:
            if ln.split() and (".up " in ln or "conv.conv.0 " in ln):
                lines.append(f"{t:6s} {ln.rstrip()}")
dump = {}
for t in ("parent", "branch"):
    for f in sorted(glob.glob(f"{out}/dump_{t}/*.npy")):
        dump.setdefault(os.path.basename(f), {})[t] = np.load(f)
for name, d in sorted(dump.items()):
    if len(d) != 2:
        continue
    a, b = d["parent"], d["branch"]
    if name.startswith("mask"):
        lines.append(f"{name}: agreement {float((a == b).mean()):.6f} ({int((a != b).sum())} of {a.size} differ)")
    else:
        diff = np.abs(a.astype(np.float64) - b.astype(np.float64))
        lines.append(f"{name}: max |diff| {diff.max():.4g}  mean |diff| {diff.mean():.3g}  max |parent| {np.abs(a).max():.4g}")
print("\n".join(lines))
open(f"{out}/summary.txt", "w").write("\n".join(lines) + "\n")
PY
rm -rf "$OUT"/dump_parent "$OUT"/dump_branch      # 16 MB arrays: compared above, not kept
