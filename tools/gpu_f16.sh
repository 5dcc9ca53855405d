#!/bin/bash
# Half-precision planes (JINC_SAMPLE_F16) on one GPU session:
#   card, power limit and max SM clock (queries only); build; the half tests, then the whole GPU suite and the smoke
#   test; tools/bench_f16.py (float32 against half, kernel-only and end to end, configs 2, 4, 5); one default bench line
#   for config 2 next to the latest round-3 one.
# Usage: bash tools/gpu_f16.sh OUT_DIR [pairs] [steps]      writes OUT_DIR/r04_f16_*
set -u
OUT=${1:?usage: bash tools/gpu_f16.sh OUT_DIR [pairs] [steps]}
PAIRS=${2:-3}
S=${3:-50}
mkdir -p $OUT
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r04_f16_smi.txt 2>&1
cat $OUT/r04_f16_smi.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r04_f16_build.log 2>&1 || { tail -30 $OUT/r04_f16_build.log; exit 1; }
python -m pytest -q -m gpu tests/test_gpu_f16.py > $OUT/r04_f16_pytest_f16.log 2>&1
tail -3 $OUT/r04_f16_pytest_f16.log
python -m pytest -q -m gpu tests/ > $OUT/r04_f16_pytest_gpu.log 2>&1
tail -3 $OUT/r04_f16_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r04_f16_smoke.log 2>&1
tail -1 $OUT/r04_f16_smoke.log

python tools/bench_f16.py --pairs $PAIRS --steps $S > $OUT/r04_f16_bench.jsonl 2> $OUT/r04_f16_bench.err
python - $OUT/r04_f16_bench.jsonl <<'EOF' | tee $OUT/r04_f16_summary.txt
import json, statistics, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    k, e = d["kernel"], d["e2e"]
    m = lambda v: statistics.median(v)
    print(f"config {d['config']} ({', '.join(d['kernel_paths'])}; {d['frames_per_batch']} frames, {d['batch_mb']['f16']} / "
          f"{d['batch_mb']['f32']} MB half / float32): kernel-only f32 {k['f32']['gpixel_s']} Gpixel/s (FMA frac "
          f"{m(k['f32']['fma_frac'])}), f16 {k['f16']['gpixel_s']} Gpixel/s (FMA frac {m(k['f16']['fma_frac'])}), "
          f"time ratio f16/f32 {k['median_time_ratio_f16_over_f32']}; e2e f32 {e['f32_fps']} fps, f16 {e['f16_fps']} fps, "
          f"ratio {e['median_fps_ratio_f16_over_f32']}; check {d['check']['ok']} ({d['check']['samples']} samples)")
EOF

python bench.py 2>/dev/null | tail -1 > $OUT/r04_f16_bench_config2_default.json
python - $OUT/r04_f16_bench_config2_default.json profiles/r03_bench_config2_default.json <<'EOF' | tee -a $OUT/r04_f16_summary.txt
import json, sys
for f in sys.argv[1:]:
    d = json.load(open(f))
    print(f, "config 2", round(d["value"]), "launch ms", round(d["roofline"]["launch_ms"], 4), "frac", round(d["roofline"]["frac"], 3),
          "verified", (d.get("verified") or {}).get("ok"), "sm MHz", d.get("clocks", {}).get("sm_mhz"))
EOF
