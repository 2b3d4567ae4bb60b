#!/bin/bash
# A/B of the output heads on one B200: the fused kernel (default) against the separate conv1 / conv2 launches
# (ABCNET_FUSED_HEADS=0). Build, the fused-heads parity tests, then `bench.py --no-train --no-comparator --no-cpu` RUNS times
# per arm, alternating, with --dump-outputs on the first run of each arm; compares the dumps and prints the headline numbers.
# Logs and bench JSON lines go to <out_dir>.
#   bash tools/ab_fused_heads.sh <out_dir> [runs] [extra pytest files...]
OUT=${1:?usage: tools/ab_fused_heads.sh <out_dir> [runs] [extra pytest files...]}
RUNS=${2:-3}
shift 2 2>/dev/null
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/smi.txt" 2>&1
cat "$OUT/smi.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1 || { echo "build failed"; tail -30 "$OUT/build.log"; exit 1; }
timeout 600 python -m pytest -x -q -p no:cacheprovider tests/test_heads_fused_gpu.py "$@" > "$OUT/pytest.log" 2>&1
rc=$?
echo "pytest exit $rc"; tail -15 "$OUT/pytest.log" | cut -c1-300
[ $rc -eq 0 ] || exit 1
DUMPS=$(mktemp -d)
for i in $(seq 1 "$RUNS"); do
  for arm in base fused; do
    extra=""
    [ "$i" -eq 1 ] && extra="--dump-outputs $DUMPS/$arm"
    if [ $arm = base ]; then
      ABCNET_FUSED_HEADS=0 timeout 400 python bench.py --no-train --no-comparator --no-cpu --steps 100 $extra > "$OUT/bench_${arm}_$i.json" 2>> "$OUT/bench.err"
    else
      timeout 400 python bench.py --no-train --no-comparator --no-cpu --steps 100 $extra > "$OUT/bench_${arm}_$i.json" 2>> "$OUT/bench.err"
    fi
    echo "bench $arm $i exit $?"
  done
done
python tools/compare_dumps.py "$DUMPS/base" "$DUMPS/fused" > "$OUT/compare.json"; echo "compare exit $?"
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
    heads = L.get("heads.fused", L.get("heads.conv1", 0) + L.get("heads.conv2", 0))
    fp = b.get("fp16_activation_mode") or {}
    gr = b.get("graph_replay") or {}
    print(f.split("/")[-1], f"value {b['value']:.1f} ms {b['ms_per_step']:.3f} heads_ms {heads:.3f}",
          {k: round(v, 3) for k, v in L.items() if k.startswith("heads")}, "fp16", fp.get("ms_per_step"), "graph", gr.get("ms_per_step"))
PY
