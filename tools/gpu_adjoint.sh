#!/bin/bash
# The adjoint and the PyTorch front-end on one GPU session:
#   card, power limit and max SM clock (queries only); build; the tensor / adjoint tests, then the whole GPU suite and the
#   smoke test; tools/bench_adjoint.py (forward against adjoint, kernel-only, configs 1-6; one torch-level training step);
#   a torch.profiler run of its own (which adjoint kernels run on configs 2 and 4); one default bench line for config 2,
#   which shows the forward path is unchanged.
# Usage: bash tools/gpu_adjoint.sh OUT_DIR [pairs] [seconds]      writes OUT_DIR/r06_adjoint_*
set -u
OUT=${1:?usage: bash tools/gpu_adjoint.sh OUT_DIR [pairs] [seconds]}
PAIRS=${2:-3}
SEC=${3:-1.0}
mkdir -p $OUT
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r06_adjoint_smi.txt 2>&1
cat $OUT/r06_adjoint_smi.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/r06_adjoint_build.log 2>&1 || { tail -30 $OUT/r06_adjoint_build.log; exit 1; }
python -m pytest -q -m gpu tests/test_gpu_tensor_adjoint.py > $OUT/r06_adjoint_pytest_adjoint.log 2>&1
tail -3 $OUT/r06_adjoint_pytest_adjoint.log
python -m pytest -q -m gpu tests/ > $OUT/r06_adjoint_pytest_gpu.log 2>&1
tail -3 $OUT/r06_adjoint_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r06_adjoint_smoke.log 2>&1
tail -1 $OUT/r06_adjoint_smoke.log
python tools/bench_adjoint.py --pairs $PAIRS --seconds $SEC > $OUT/r06_adjoint_bench.jsonl 2> $OUT/r06_adjoint_bench.err
cat $OUT/r06_adjoint_bench.jsonl
python tools/bench_adjoint.py --profile $OUT > /dev/null 2> $OUT/r06_adjoint_profile.err
grep -E "^==|adjoint_" $OUT/r06_adjoint_profile.txt | cut -c1-120
python bench.py 2>/dev/null | tail -1 > $OUT/r06_adjoint_bench_config2_default.json
python - $OUT/r06_adjoint_bench_config2_default.json profiles/r04_f16_bench_config2_default.json <<'EOF'
import json, sys
for f in sys.argv[1:]:
    d = json.load(open(f))
    print(f, "config 2", round(d["value"]), "frac", round(d["roofline"]["frac"], 3), "verified", (d.get("verified") or {}).get("ok"),
          "sm MHz", d.get("clocks", {}).get("sm_mhz"))
EOF
