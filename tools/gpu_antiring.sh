#!/bin/bash
# The anti-ringing pass on one GPU session:
#   card, power limit and max SM clock (queries only); build; the anti-ringing GPU tests and the smoke test;
#   tools/bench_antiring.py (strength 0 against 1: kernel-only, the pass alone, end to end; configs 1-5); one default
#   bench line for config 2 next to the round-4 one.
# Usage: bash tools/gpu_antiring.sh OUT_DIR [pairs] [steps]      writes OUT_DIR/r05_antiring_*
set -u
OUT=${1:?usage: bash tools/gpu_antiring.sh OUT_DIR [pairs] [steps]}
PAIRS=${2:-3}
S=${3:-50}
mkdir -p $OUT
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $OUT/r05_antiring_smi.txt 2>&1
cat $OUT/r05_antiring_smi.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r05_antiring_build.log 2>&1 || { tail -30 $OUT/r05_antiring_build.log; exit 1; }
python -m pytest -q -m gpu tests/test_gpu_antiring.py > $OUT/r05_antiring_pytest_antiring.log 2>&1
tail -3 $OUT/r05_antiring_pytest_antiring.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r05_antiring_smoke.log 2>&1
tail -1 $OUT/r05_antiring_smoke.log

python tools/bench_antiring.py --pairs $PAIRS --steps $S > $OUT/r05_antiring_bench.jsonl 2> $OUT/r05_antiring_bench.err
tail -3 $OUT/r05_antiring_bench.err
python - $OUT/r05_antiring_bench.jsonl <<'PY' | tee $OUT/r05_antiring_summary.txt
import json, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    k, p, e = d["kernel"], d["pass"], d["e2e"]
    dr = k["delta_rate"] or {}
    print(f"config {d['config']} ({', '.join(d['kernel_paths'])}; {d['frames_per_batch']} frames, {d['batch_mb']} MB): kernel-only "
          f"s=0 {k['s0_gpixel_s']} Gpixel/s, s=1 {k['s1_gpixel_s']} Gpixel/s (+{100 * k['delta_frac_of_s0']:.1f} %, launches "
          f"{k['launches_per_batch']}; the added time moves {dr.get('gb_s')} GB/s = {dr.get('frac_of_7p7_tb_s_datasheet')} of 7.7 TB/s); "
          f"pass alone ({p['calls_per_sweep']} calls) {p['gb_s']} GB/s = {p['frac_of_7p7_tb_s_datasheet']} of 7.7 TB/s (data sheet); "
          f"e2e s=0 {e['s0_fps']} fps, s=1 {e['s1_fps']} fps, ratio {e['median_fps_ratio_s1_over_s0']}")
PY

python bench.py 2>/dev/null | tail -1 > $OUT/r05_antiring_bench_config2_default.json
python - $OUT/r05_antiring_bench_config2_default.json profiles/r04_f16_bench_config2_default.json <<'PY' | tee -a $OUT/r05_antiring_summary.txt
import json, sys
for f in sys.argv[1:]:
    d = json.load(open(f))
    print(f, "config 2", round(d["value"]), "launch ms", round(d["roofline"]["launch_ms"], 4), "frac", round(d["roofline"]["frac"], 3),
          "verified", (d.get("verified") or {}).get("ok"), "sm MHz", d.get("clocks", {}).get("sm_mhz"))
PY
