#!/bin/bash
# Differentiable anti-ringing on one GPU session:
#   card, power limit and SM clocks (queries only); build; the new tests, the adjoint / anti-ringing / VapourSynth tests,
#   the whole GPU suite and the smoke test; tools/bench_antiring_adjoint.py (backward at strength 1 against the plain
#   adjoint and the tensor forward with and without anti-ringing, configs 2, 4, 5, float32 and half), its torch.profiler
#   run (time per launch and bytes per second of the two new passes); tools/bench_adjoint.py on configs 2 and 4 (the plain
#   adjoint against the forward); one default bench line for config 2, which shows the forward path is unchanged.
# Usage: bash tools/gpu_antiring_adjoint.sh OUT_DIR [pairs] [seconds]      writes OUT_DIR/r07_antiring_adjoint_*
set -u
OUT=${1:?usage: bash tools/gpu_antiring_adjoint.sh OUT_DIR [pairs] [seconds]}
PAIRS=${2:-3}
SEC=${3:-1.0}
P=$OUT/r07_antiring_adjoint
mkdir -p $OUT
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > ${P}_smi.txt 2>&1
cat ${P}_smi.txt
python -c "import __graft_entry__ as g; g.build()" > ${P}_build.log 2>&1 || { tail -30 ${P}_build.log; exit 1; }
python -m pytest -q tests/test_gpu_tensor_antiring.py > ${P}_pytest_new.log 2>&1
tail -3 ${P}_pytest_new.log
python -m pytest -q -m gpu tests/test_gpu_tensor_adjoint.py tests/test_gpu_antiring.py tests/test_vapoursynth.py > ${P}_pytest_related.log 2>&1
tail -3 ${P}_pytest_related.log
python -m pytest -q -m gpu tests/ > ${P}_pytest_gpu.log 2>&1
tail -3 ${P}_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > ${P}_smoke.log 2>&1
tail -1 ${P}_smoke.log
python tools/bench_antiring_adjoint.py --pairs $PAIRS --seconds $SEC > ${P}_bench.jsonl 2> ${P}_bench.err
cat ${P}_bench.jsonl
python tools/bench_antiring_adjoint.py --profile > ${P}_profile.jsonl 2> ${P}_profile.err
cat ${P}_profile.jsonl
python tools/bench_adjoint.py --configs 2 4 --pairs $PAIRS --seconds $SEC --torch-steps 10 > ${P}_bench_adjoint.jsonl 2> ${P}_bench_adjoint.err
cat ${P}_bench_adjoint.jsonl
python bench.py 2>/dev/null | tail -1 > ${P}_bench_config2_default.json
python - ${P}_bench_config2_default.json profiles/r04_f16_bench_config2_default.json <<'EOF'
import json, sys
for f in sys.argv[1:]:
    d = json.load(open(f))
    print(f, "config 2", round(d["value"]), "frac", round(d["roofline"]["frac"], 3), "verified", (d.get("verified") or {}).get("ok"),
          "sm MHz", d.get("clocks", {}).get("sm_mhz"))
EOF
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv,noheader >> ${P}_smi.txt 2>&1
