#!/usr/bin/env bash
# A/B of the multi-sweep dimension tree (CALS_B200_MSDT=1) against the one-sweep pair node (CALS_B200_MSDT=0):
# config 2 and its 8-way shard alternated three times each, configs 1, 3 and 4 once per schedule.  Every bench line
# carries its own per-kernel split (roofline.share_of_step, from the event-timed passes).
# Usage: tools/msdt_ab.sh OUTPUT_DIR
set -u
O=${1:?usage: tools/msdt_ab.sh OUTPUT_DIR}; mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,temperature.gpu --format=csv > $O/gpu.csv 2>&1
run() { local name=$1; shift; timeout 400 python bench.py --no-secondary --no-cpu-baseline --steps 5 --warmup 3 "$@" \
          > $O/$name.json 2>> $O/err.log; }
for rep in 1 2 3; do
  for m in 0 1; do
    CALS_B200_MSDT=$m run c2_m${m}_$rep --config 2
    CALS_B200_MSDT=$m run c2s8_m${m}_$rep --config 2 --shard-of 8
  done
done
for cfg in 1 3 4; do
  for m in 0 1; do
    CALS_B200_MSDT=$m run c${cfg}_m$m --config $cfg
  done
done
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,temperature.gpu --format=csv >> $O/gpu.csv 2>&1
python - $O <<'EOF'
import glob, json, os, sys
out = sys.argv[1]
rows = []
for f in sorted(glob.glob(os.path.join(out, "*.json"))):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except Exception as e:  # a failed run leaves an empty or partial file
        rows.append("%-14s  no result (%s)" % (os.path.basename(f)[:-5], type(e).__name__))
        continue
    r = d.get("roofline") or {}
    sh = r.get("share_of_step") or {}
    rows.append("%-14s  %10.1f %s  contractions/it %.2f  shares %s" % (
        os.path.basename(f)[:-5], d.get("value", float("nan")), d.get("unit", ""),
        r.get("launches_per_als_iteration", float("nan")),
        " ".join("%s=%.3f" % (k, v) for k, v in sh.items())))
open(os.path.join(out, "summary.txt"), "w").write("\n".join(rows) + "\n")
print("\n".join(rows))
EOF
cat $O/gpu.csv
