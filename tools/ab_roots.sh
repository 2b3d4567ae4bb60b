#!/bin/bash
# A/B of two source trees on one GPU: builds each, then runs `bench.py --no-train --no-comparator --no-cpu --steps 100`
# RUNS times per tree, alternating A and B, with --dump-outputs on the first run of each; compares the two dumps with
# tools/compare_dumps.py and prints the headline numbers of every run. Logs and bench JSON lines go to <out_dir>.
#   bash tools/ab_roots.sh <root_a> <root_b> <out_dir> [runs]
A=$(realpath "${1:?usage: tools/ab_roots.sh <root_a> <root_b> <out_dir> [runs]}")
B=$(realpath "${2:?usage: tools/ab_roots.sh <root_a> <root_b> <out_dir> [runs]}")
mkdir -p "${3:?usage: tools/ab_roots.sh <root_a> <root_b> <out_dir> [runs]}"
OUT=$(realpath "$3")
RUNS=${4:-3}
HERE=$(dirname "$(realpath "$0")")
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/smi.txt" 2>&1
cat "$OUT/smi.txt"
for arm in a b; do
  root=$A; [ $arm = b ] && root=$B
  (cd "$root" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_$arm.log" 2>&1 || { echo "build $arm failed"; tail -30 "$OUT/build_$arm.log"; exit 1; }
done
DUMPS=$(mktemp -d)
for i in $(seq 1 "$RUNS"); do
  for arm in a b; do
    root=$A; [ $arm = b ] && root=$B
    extra=""
    [ "$i" -eq 1 ] && extra="--dump-outputs $DUMPS/$arm"
    (cd "$root" && timeout 400 python bench.py --no-train --no-comparator --no-cpu --steps 100 $extra) > "$OUT/bench_${arm}_$i.json" 2>> "$OUT/bench.err"
    echo "bench $arm $i exit $?"
  done
done
python "$HERE/compare_dumps.py" "$DUMPS/a" "$DUMPS/b" > "$OUT/compare.json"; echo "compare exit $?"
cut -c1-400 "$OUT/compare.json"
rm -rf "$DUMPS"
python - "$OUT" <<'PY'
import glob, json, sys
out = sys.argv[1]
for f in sorted(glob.glob(out + "/bench_*.json")):
    try:
        b = json.loads(open(f).read().strip().splitlines()[-1])
    except Exception as e:
        print(f, "unreadable", e)
        continue
    L = b["config"]["layers_ms"]
    fp = b.get("fp16_activation_mode") or {}
    gr = b.get("graph_replay") or {}
    print(f.split("/")[-1], f"value {b['value']:.1f} ms {b['ms_per_step']:.3f} heads.fused {L.get('heads.fused', 0):.3f}",
          "fp16", fp.get("ms_per_step"), "graph", gr.get("ms_per_step"))
PY
