#!/usr/bin/env bash
# Final check of the multi-sweep schedule: per-kernel split of config 2 under both schedules (tools/msdt_nodes.py), the
# config-2 bench dump with CALS_B200_MSDT=0 against the default (factors and lambda within 1e-11), the GPU test suite,
# smoke() and one full bench line.
# Usage: tools/msdt_final.sh OUTPUT_DIR
set -u
O=${1:?usage: tools/msdt_final.sh OUTPUT_DIR}; mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu.csv 2>&1
timeout 300 python tools/msdt_nodes.py 2 $O > $O/nodes.log 2>&1; echo "nodes rc=$?" >> $O/nodes.log
CALS_B200_MSDT=0 timeout 400 python bench.py --config 2 --no-secondary --no-cpu-baseline --dump-outputs $O/dump_m0 \
  > $O/dump_m0.json 2>> $O/err.log
timeout 400 python bench.py --config 2 --no-secondary --no-cpu-baseline --dump-outputs $O/dump_default \
  > $O/dump_default.json 2>> $O/err.log
python - $O > $O/dump_compare.log 2>&1 <<'EOF'
import glob, os, sys
import numpy as np
out = sys.argv[1]
worst = 0.0
for f in sorted(glob.glob(os.path.join(out, "dump_m0", "*.npy"))):
    name = os.path.basename(f)
    a, b = np.load(f), np.load(os.path.join(out, "dump_default", name))
    if name.startswith("factors") or name.startswith("lambda"):
        e = float(np.linalg.norm(a - b) / np.linalg.norm(a))
        worst = max(worst, e)
        print("%-20s rel diff %.3e" % (name, e))
    else:
        print("%-20s max abs diff %.3e" % (name, float(np.abs(a - b).max())))
print("worst factor / lambda rel diff %.3e -> %s" % (worst, "ok" if worst <= 1e-11 else "FAIL"))
EOF
timeout 1500 python -m pytest tests/ -q -m gpu > $O/tests.log 2>&1; echo "tests rc=$?" >> $O/tests.log
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1; echo "smoke rc=$?" >> $O/smoke.log
timeout 900 python bench.py > $O/bench.json 2> $O/bench.err
cat $O/gpu.csv; tail -3 $O/nodes.log; cat $O/dump_compare.log; tail -3 $O/tests.log; tail -2 $O/smoke.log
head -c 400 $O/bench.json
