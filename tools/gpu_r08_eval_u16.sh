#!/bin/bash
# Session of round 8 (evaluation on KITTI uint16 ground truth): a built checkout of the parent commit (directory in $1; its own
# bench.py, binding and libdcmt.so -- this tree's binding requires entry points the parent library lacks) against this tree:
# smoke, tools/bench_eval_u16.py with the parent's dcmt_evaluate_f32 timed in the same alternation and its records compared,
# the GPU suite, and bench.py default alternating twice with its dumped outputs compared.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r08_eval_u16.sh /path/to/parent/checkout OUT_DIR
set -u
P=$(realpath "$1")
out=$(realpath -m "${2:?output directory}")
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $out/gpu.txt 2>&1
cat $out/gpu.txt
t0=$(date +%s)
(cd $P && timeout 900 python -c "import __graft_entry__ as g; g.build()") > $out/build_parent.log 2>&1; echo "parent build rc=$?"
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $out/smoke.log 2>&1; echo "smoke rc=$?" | tee -a $out/smoke.log
tail -2 $out/smoke.log
echo "t=$(( $(date +%s) - t0 ))"
timeout 900 python tools/bench_eval_u16.py --steps 20 --warmup 3 --parent-lib $P/depth_completion_mt_b200/libdcmt.so > $out/eval_u16.json 2> $out/eval_u16.err
echo "bench_eval_u16 rc=$?"
cat $out/eval_u16.json; tail -3 $out/eval_u16.err
echo "t=$(( $(date +%s) - t0 ))"
timeout 1800 python -m pytest tests -q -m gpu > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $out/pytest_gpu.log
tail -8 $out/pytest_gpu.log
echo "t=$(( $(date +%s) - t0 ))"
for i in 1 2; do
  (cd $P && timeout 600 python bench.py --no-cpu-baseline) > $out/bench_before_$i.json 2>> $out/bench.err; echo "before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline > $out/bench_after_$i.json 2>> $out/bench.err; echo "after $i rc=$?"
done
tmp=$(mktemp -d)
(cd $P && timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/before) > /dev/null 2>> $out/dump.err; echo "dump before rc=$?"
timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/after > /dev/null 2>> $out/dump.err; echo "dump after rc=$?"
sha256sum $tmp/before/depth.npy $tmp/after/depth.npy | sed "s|$tmp/||" | tee $out/dump_sha256.txt
cmp $tmp/before/depth.npy $tmp/after/depth.npy && echo "depth.npy identical" | tee -a $out/dump_sha256.txt
rm -rf $tmp
echo "t=$(( $(date +%s) - t0 ))"
OUT="$out" python - <<'PY'
import json, glob, os, statistics as s
for side in ("before", "after"):
    v = []
    for f in sorted(glob.glob(os.path.join(os.environ["OUT"], f"bench_{side}_*.json"))):
        try:
            d = json.loads(open(f).read().strip().splitlines()[-1])
        except Exception as e:
            print(f, "unreadable", e); continue
        v.append(d["value"])
        val = d.get("validation", {})
        print(os.path.basename(f), round(d["value"]), "golden", val.get("golden_sha256_match"), "replicas", val.get("replicas_equal"))
    if v:
        print(f"{side}: value median {s.median(v):.0f} [{min(v):.0f}, {max(v):.0f}]")
PY
echo "t=$(( $(date +%s) - t0 ))"
