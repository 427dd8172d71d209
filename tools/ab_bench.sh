#!/bin/bash
# On a machine with a B200: alternating A/B of bench.py between the in-tree library ("new") and every variant under
# tools/_alt/ (tools/ab_build.sh; e.g. the parent commit's library, named after its file), all in one run:
#   tools/ab_bench.sh [ROUNDS] [WORKLOAD...]
# - for each WORKLOAD (default c3), ROUNDS rounds (default 3) of `bench.py --workload WORKLOAD --no-cpu`, every
#   library once per round, the order reversed from one round to the next;
# - every library once with --dump-outputs on c3, c2 and c4s; each dump is compared with new's array by array
#   (np.array_equal).
# Output under $OUT (default: a new temporary directory, printed at the start): bench.jsonl (every JSON line,
# tagged with library, workload and round), gpu.csv (card name, power limit), the dumps and the stderr of every run.
# Exit status 1 if a run failed or a dump differs.
set -u
cd "$(dirname "$0")/.."
rounds=${1:-3}
shift || true
workloads=${*:-c3}
OUT=${OUT:-$(mktemp -d -t ab_bench.XXXXXX)}
mkdir -p "$OUT"
echo "output: $OUT"
lib=steered-mixture-of-experts_b200/libsmoe_b200.so
python __graft_entry__.py > /dev/null || exit 1
tmp=$(mktemp -d)
cp $lib "$tmp/new.so"
trap 'cp "$tmp/new.so" $lib; rm -rf "$tmp"' EXIT
names="new"
for v in tools/_alt/*.so; do
  [ -e "$v" ] || continue
  n=$(basename "$v" .so)
  cp "$v" "$tmp/$n.so"
  names="$names $n"
done
rev=$(echo $names | tr ' ' '\n' | tac | tr '\n' ' ')
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv"
status=0

run() {  # library workload round [bench args...]
  local n=$1 wl=$2 r=$3
  shift 3
  cp "$tmp/$n.so" $lib              # a fresh mtime: bench.py's build() keeps it
  if ! python bench.py --workload $wl --no-cpu "$@" > "$tmp/line" 2> "$OUT/err_${n}_${wl}_$r.txt"; then
    echo "FAILED: $n $wl round $r"; tail -3 "$OUT/err_${n}_${wl}_$r.txt"; status=1; return
  fi
  python - "$n" "$wl" "$r" "$tmp/line" >> "$OUT/bench.jsonl" <<'PY'
import json, sys
n, wl, r, path = sys.argv[1:]
print(json.dumps({"lib": n, "workload": wl, "round": r, "bench": json.loads(open(path).read().strip().splitlines()[-1])}))
PY
}

for wl in $workloads; do
  for ((r = 0; r < rounds; r++)); do
    order=$names; (( r % 2 )) && order=$rev
    for n in $order; do run $n $wl $r; done
  done
done
for wl in c3 c2 c4s; do
  for n in $names; do
    run $n $wl dump --steps 3 --no-dense --no-aux --pruned-iters 0 --dump-outputs "$OUT/dump_${n}_$wl"
  done
done

python - "$OUT" $names <<'PY' || status=1
import glob, json, os, sys
import numpy as np
out, names = sys.argv[1], sys.argv[2:]
rows = [json.loads(l) for l in open(os.path.join(out, "bench.jsonl"))] if os.path.exists(os.path.join(out, "bench.jsonl")) else []
print(open(os.path.join(out, "gpu.csv")).read().strip())
def get(b, path):
    for k in path.split("."):
        b = b.get(k) if isinstance(b, dict) else None
    return b
fields = ["value", "ms_per_step", "roofline.product_mode.backward_ms", "roofline.dense_backward_ms",
          "states.ms_per_step", "states.backward_ms"]
for wl in sorted({r["workload"] for r in rows if r["round"] != "dump"}):
    for n in names:
        sel = [r["bench"] for r in rows if r["workload"] == wl and r["lib"] == n and r["round"] != "dump"]
        if not sel:
            continue
        stat = {}
        for f in fields:
            v = [get(b, f) for b in sel]
            v = [x for x in v if isinstance(x, (int, float))]
            if v:
                stat[f] = (float(np.mean(v)), float(min(v)), float(max(v)))
        thr = sorted({x for b in sel for x in (get(b, "clocks.reasons") or [])})
        print(f"{wl} {n} runs={len(sel)} throttle={thr or 'none'}")
        for f, (m, lo, hi) in stat.items():
            print(f"    {f:36s} mean {m:.6g}  [{lo:.6g}, {hi:.6g}]")
bad = 0
for wl in ("c3", "c2", "c4s"):
    ref = os.path.join(out, f"dump_new_{wl}")
    files = sorted(os.path.basename(p) for p in glob.glob(os.path.join(ref, "*.npy")))
    for n in names[1:]:
        other = os.path.join(out, f"dump_{n}_{wl}")
        diff = [f for f in files if not os.path.exists(os.path.join(other, f))
                or not np.array_equal(np.load(os.path.join(ref, f)), np.load(os.path.join(other, f)))]
        same = bool(files) and not diff
        bad += not same
        print(f"dump {wl}: new vs {n}: {len(files)} arrays, {'bitwise equal' if same else 'DIFFER: ' + str(diff or 'no dump')}")
sys.exit(1 if bad else 0)
PY
exit $status
