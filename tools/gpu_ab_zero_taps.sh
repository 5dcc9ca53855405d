#!/bin/bash
# A/B of the exact-2x kernel with the exactly-zero taps skipped (default) against every tap
# (JINCRESIZE_B200_UP2X_ZERO_TAPS=0), in one GPU session:
#   card, power limit and clocks; build; the GPU test suite; for configs 2, 1 and 3 alternated pairs of kernel-only bench
#   lines; the dumped outputs of both settings compared plane for plane; one default bench line.
# Usage: bash tools/gpu_ab_zero_taps.sh OUT_DIR [pairs] [steps]      writes OUT_DIR/r03_*
set -u
OUT=${1:?usage: bash tools/gpu_ab_zero_taps.sh OUT_DIR [pairs] [steps]}
PAIRS=${2:-3}
S=${3:-2000}
mkdir -p $OUT
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r03_smi.txt 2>&1
cat $OUT/r03_smi.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r03_build.log 2>&1 || { tail -30 $OUT/r03_build.log; exit 1; }
python -m pytest -q -m gpu tests/ > $OUT/r03_pytest_gpu.log 2>&1
tail -3 $OUT/r03_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r03_smoke.log 2>&1
tail -1 $OUT/r03_smoke.log

B="--steps $S --warmup 20 --no-cpu --no-all-configs --plugin-threads 0 --bands 0"
DUMP=$(mktemp -d)
for c in 2 1 3; do
    for p in $(seq 1 $PAIRS); do
        for v in 0 1; do
            d=""
            [ $p = 1 ] && d="--dump-outputs $DUMP/c${c}_v$v"
            if [ $v = 0 ]; then
                JINCRESIZE_B200_UP2X_ZERO_TAPS=0 python bench.py --config $c $B $d 2>/dev/null | tail -1 > $OUT/r03_ab_config${c}_taps${v}_$p.json
            else
                python bench.py --config $c $B $d 2>/dev/null | tail -1 > $OUT/r03_ab_config${c}_taps${v}_$p.json
            fi
        done
    done
    python - $c $DUMP <<'EOF'
import glob, os, sys
import numpy as np
c, d = sys.argv[1], sys.argv[2]
names = sorted(os.path.basename(p) for p in glob.glob(f"{d}/c{c}_v0/plane*.npy"))
same = [np.array_equal(np.load(f"{d}/c{c}_v0/{n}"), np.load(f"{d}/c{c}_v1/{n}")) for n in names]
print(f"config {c}: {len(names)} dumped planes, identical between every tap and zero taps skipped: {all(same) and len(names) > 0} {same}")
EOF
done 2>&1 | tee $OUT/r03_ab_outputs_identical.txt
rm -rf $DUMP

python - $OUT <<'EOF' | tee $OUT/r03_ab_summary.txt
import glob, json, statistics, sys
out = sys.argv[1]
for c in (2, 1, 3):
    v = {}
    for t in (0, 1):
        runs = []
        for f in sorted(glob.glob(f"{out}/r03_ab_config{c}_taps{t}_*.json")):
            try:
                d = json.load(open(f))
            except ValueError:
                continue
            runs.append((d["value"], d["roofline"]["launch_ms"], (d.get("verified") or {}).get("ok"), d.get("clocks", {}).get("sm_mhz")))
        v[t] = runs
    m0 = statistics.median(r[0] for r in v[0]) if v[0] else float("nan")
    m1 = statistics.median(r[0] for r in v[1]) if v[1] else float("nan")
    print(f"config {c}: every tap {[round(r[0]) for r in v[0]]} launch ms {[round(r[1], 4) for r in v[0]]}")
    print(f"config {c}: zero taps skipped {[round(r[0]) for r in v[1]]} launch ms {[round(r[1], 4) for r in v[1]]}")
    print(f"config {c}: median ratio {m1 / m0:.3f}; every default above every switch-off: "
          f"{min(r[0] for r in v[1]) > max(r[0] for r in v[0]) if v[0] and v[1] else None}; "
          f"verified {[r[2] for r in v[0] + v[1]]}; sm MHz {[r[3] for r in v[0] + v[1]]}")
EOF
python bench.py 2>/dev/null | tail -1 > $OUT/r03_bench_config2_default.json
python - $OUT/r03_bench_config2_default.json profiles/r02z_bench_config2_default.json <<'EOF'
import json, sys
for f in sys.argv[1:]:
    d = json.load(open(f))
    a = d.get("all_configs", {})
    print(f, "config 2", round(d["value"]), "launch ms", round(d["roofline"]["launch_ms"], 4), "frac", round(d["roofline"]["frac"], 3),
          "verified", (d.get("verified") or {}).get("ok"), "sm MHz", d.get("clocks", {}).get("sm_mhz"),
          "| " + " ".join(f"config {k}: {round(v['value'])} ({v.get('verified')})" for k, v in sorted(a.items())))
EOF
