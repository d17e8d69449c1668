#!/bin/bash
# Session of round 13 (one host chunk pipeline, workspace sizes derived from the carves): a checkout of the parent commit
# (directory in $1) against this tree: smoke, the whole GPU suite, then the parent and this tree timed alternately, twice
# each, on bench.py default / --workload guided / --workload stereo / --workload stereo_chain, tools/bench_stereo_chain.py
# and tools/bench_superpixels_bgr.py, with the default workload's dumped outputs compared byte for byte.
# The GPU's name, power limit and SM clocks are read with nvidia-smi --query-gpu only; no setting is changed.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r13_host_pipeline.sh /path/to/parent/checkout OUT_DIR
# SUITE=0 skips the GPU suite; LEGS and ROUNDS (space-separated) pick the timed legs and the round numbers.
set -u
P=$(realpath "$1")
out=$(realpath -m "${2:?output directory}")
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > $out/gpu.txt 2>&1
cat $out/gpu.txt
t0=$(date +%s)
(cd $P && timeout 900 python -c "import __graft_entry__ as g; g.build()") > $out/build_parent.log 2>&1; echo "parent build rc=$?"
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $out/smoke.log 2>&1; echo "smoke rc=$?" | tee -a $out/smoke.log
tail -2 $out/smoke.log
echo "t=$(( $(date +%s) - t0 ))"
if [ "${SUITE:-1}" = 1 ]; then
  timeout 1800 python -m pytest tests -q -m gpu > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $out/pytest_gpu.log
  tail -8 $out/pytest_gpu.log
  echo "t=$(( $(date +%s) - t0 ))"
fi
legs=(${LEGS:-default guided stereo stereo_chain tool_stereo_chain tool_superpixels_bgr})
run_leg() {  # leg, output file (from the current directory)
  case $1 in
    default) timeout 600 python bench.py --gpus 1 --no-cpu-baseline ;;
    tool_stereo_chain) timeout 600 python tools/bench_stereo_chain.py ;;
    tool_superpixels_bgr) timeout 600 python tools/bench_superpixels_bgr.py ;;
    *) timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $1 ;;
  esac > $2 2>> $out/bench.err
}
for i in ${ROUNDS:-1 2}; do
  for leg in "${legs[@]}"; do
    (cd $P && run_leg $leg $out/bench_${leg}_before_$i.json); echo "$leg before $i rc=$?"
    run_leg $leg $out/bench_${leg}_after_$i.json; echo "$leg after $i rc=$?"
  done
  echo "t=$(( $(date +%s) - t0 ))"
done
tmp=$(mktemp -d)
(cd $P && timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/before) > /dev/null 2>> $out/dump.err; echo "dump before rc=$?"
timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/after > /dev/null 2>> $out/dump.err; echo "dump after rc=$?"
(cd $tmp/before && sha256sum *) > $out/dump_sha256_before.txt
(cd $tmp/after && sha256sum *) > $out/dump_sha256_after.txt
cmp $out/dump_sha256_before.txt $out/dump_sha256_after.txt && echo "dumped outputs identical" | tee $out/dump_cmp.txt
rm -rf $tmp
# every numeric key of the last JSON line of each run: median and range per side
OUT="$out" python - <<'PY' | tee $out/summary.txt
import json, glob, os, statistics as s
out = os.environ["OUT"]
legs = sorted({os.path.basename(f).rsplit("_", 2)[0][len("bench_"):] for f in glob.glob(os.path.join(out, "bench_*_*_*.json"))})
for leg in legs:
    for side in ("before", "after"):
        vals = {}
        for f in sorted(glob.glob(os.path.join(out, f"bench_{leg}_{side}_*.json"))):
            try:
                d = json.loads(open(f).read().strip().splitlines()[-1])
            except Exception as e:
                print(os.path.basename(f), "unreadable", e); continue
            stack = [("", d)]
            while stack:
                k, v = stack.pop()
                if isinstance(v, dict):
                    stack += [(f"{k}.{kk}" if k else kk, vv) for kk, vv in v.items()]
                elif isinstance(v, (int, float)) and not isinstance(v, bool):
                    vals.setdefault(k, []).append(v)
        for k in sorted(vals):
            v = vals[k]
            print(f"{leg:22s} {side:6s} {k:40s} median {s.median(v):.6g} [{min(v):.6g}, {max(v):.6g}]")
PY
echo "t=$(( $(date +%s) - t0 ))"
