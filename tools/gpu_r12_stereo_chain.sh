#!/bin/bash
# Session of round 12 (the stereo program's chain in one call, dcmt_stereo_chain_f32*): a checkout of the parent commit
# (directory in $1) against this tree: smoke, the new GPU tests, tools/bench_stereo_chain.py, the whole GPU suite, and
# bench.py default and --workload stereo_chain alternating twice each, with the default workload's dumped outputs compared.
# The GPU's name, power limit and SM clocks are read with nvidia-smi --query-gpu only; no setting is changed.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r12_stereo_chain.sh /path/to/parent/checkout OUT_DIR
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
timeout 1200 python -m pytest tests/test_stereo_chain_call.py -q -m gpu > $out/pytest_new.log 2>&1; echo "pytest new rc=$?" | tee -a $out/pytest_new.log
tail -8 $out/pytest_new.log
echo "t=$(( $(date +%s) - t0 ))"
timeout 1200 python tools/bench_stereo_chain.py --steps 3 --warmup 1 > $out/bench_stereo_chain.json 2> $out/bench_stereo_chain.err
echo "bench_stereo_chain rc=$?"
cat $out/bench_stereo_chain.json; tail -12 $out/bench_stereo_chain.err
echo "t=$(( $(date +%s) - t0 ))"
timeout 2400 python -m pytest tests -q -m gpu --ignore=tests/test_stereo_chain_call.py > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $out/pytest_gpu.log
tail -8 $out/pytest_gpu.log
echo "t=$(( $(date +%s) - t0 ))"
for w in lidar_only stereo_chain; do
  for i in 1 2; do
    (cd $P && timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w) > $out/bench_${w}_before_$i.json 2>> $out/bench.err; echo "$w before $i rc=$?"
    timeout 600 python bench.py --gpus 1 --no-cpu-baseline --workload $w > $out/bench_${w}_after_$i.json 2>> $out/bench.err; echo "$w after $i rc=$?"
  done
done
tmp=$(mktemp -d)
(cd $P && timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/before) > /dev/null 2>> $out/dump.err; echo "dump before rc=$?"
timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/after > /dev/null 2>> $out/dump.err; echo "dump after rc=$?"
sha256sum $tmp/before/depth.npy $tmp/after/depth.npy | sed "s|$tmp/||" | tee $out/dump_sha256.txt
cmp $tmp/before/depth.npy $tmp/after/depth.npy && echo "depth.npy identical" | tee -a $out/dump_sha256.txt
rm -rf $tmp
OUT="$out" python - <<'PY'
import json, glob, os, statistics as s
for w in ("lidar_only", "stereo_chain"):
    for side in ("before", "after"):
        v = []
        for f in sorted(glob.glob(os.path.join(os.environ["OUT"], f"bench_{w}_{side}_*.json"))):
            try:
                d = json.loads(open(f).read().strip().splitlines()[-1])
            except Exception as e:
                print(f, "unreadable", e); continue
            v.append(d["value"])
            val = d.get("validation", {})
            print(os.path.basename(f), round(d["value"]), "golden", val.get("golden_sha256_match"), "replicas", val.get("replicas_equal"))
        if v:
            print(f"{w} {side}: value median {s.median(v):.0f} [{min(v):.0f}, {max(v):.0f}]")
PY
echo "t=$(( $(date +%s) - t0 ))"
