#!/bin/bash
# A/B session of round 4: a parent-commit build of libdcmt.so (path in $1, selected through DCMT_LIB) against this tree's
# libdcmt.so, alternating, plus smoke, phase profiles, dumped outputs, the GPU suite and the fuzz run.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r04_ab.sh /path/to/parent/libdcmt.so OUT_DIR
set -u
P=$(realpath "$1")
out=${2:?output directory}
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $out/gpu.txt 2>&1
cat $out/gpu.txt
t0=$(date +%s)
timeout 600 python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $out/smoke.log 2>&1; echo "smoke rc=$?" | tee -a $out/smoke.log
echo "t=$(( $(date +%s) - t0 ))"
for i in 1 2 3; do
  DCMT_LIB=$P timeout 600 python bench.py --no-cpu-baseline > $out/bench_before_$i.json 2> $out/bench_before_$i.err; echo "before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline > $out/bench_after_$i.json 2> $out/bench_after_$i.err; echo "after $i rc=$?"
  echo "t=$(( $(date +%s) - t0 ))"
done
for i in 1 2; do
  DCMT_LIB=$P timeout 600 python bench.py --no-cpu-baseline --input u16 > $out/bench_u16_before_$i.json 2>> $out/bench_u16.err; echo "u16 before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline --input u16 > $out/bench_u16_after_$i.json 2>> $out/bench_u16.err; echo "u16 after $i rc=$?"
  DCMT_LIB=$P timeout 600 python bench.py --no-cpu-baseline --input float --path rank > $out/bench_rank_before_$i.json 2>> $out/bench_rank.err; echo "rank before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline --input float --path rank > $out/bench_rank_after_$i.json 2>> $out/bench_rank.err; echo "rank after $i rc=$?"
done
echo "t=$(( $(date +%s) - t0 ))"
DCMT_LIB=$P timeout 300 python tools/q8_phase_profile.py 158 > $out/phase_before.txt 2>&1; echo "phase before rc=$?"
timeout 300 python tools/q8_phase_profile.py 158 > $out/phase_after.txt 2>&1; echo "phase after rc=$?"
cat $out/phase_before.txt $out/phase_after.txt
tmp=$(mktemp -d)
DCMT_LIB=$P timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/before > /dev/null 2>> $out/dump.err; echo "dump before rc=$?"
timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/after > /dev/null 2>> $out/dump.err; echo "dump after rc=$?"
sha256sum $tmp/before/depth.npy $tmp/after/depth.npy | sed "s|$tmp/||" | tee $out/dump_sha256.txt
cmp $tmp/before/depth.npy $tmp/after/depth.npy && echo "depth.npy identical" | tee -a $out/dump_sha256.txt
rm -rf $tmp
echo "t=$(( $(date +%s) - t0 ))"
timeout 1500 python -m pytest tests -q -m gpu > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $out/pytest_gpu.log
tail -5 $out/pytest_gpu.log
echo "t=$(( $(date +%s) - t0 ))"
timeout 200 python tools/fuzz_gpu.py 90 > $out/fuzz_gpu.txt 2>&1; echo "fuzz rc=$?" | tee -a $out/fuzz_gpu.txt
tail -5 $out/fuzz_gpu.txt
OUT="$out" python - <<'PY'
import json, glob, os, statistics as s
for tag in ("", "u16_", "rank_"):
    for side in ("before", "after"):
        v, k = [], []
        for f in sorted(glob.glob(os.path.join(os.environ["OUT"], f"bench_{tag}{side}_*.json"))):
            try:
                d = json.loads(open(f).read().strip().splitlines()[-1])
            except Exception as e:
                print(f, "unreadable", e); continue
            v.append(d["value"]); k.append(((d["roofline"].get("kernels") or {}).get("k_q8_front") or {}).get("ms_per_step", float("nan")))
            val = d.get("validation", {})
            print(f, round(d["value"]), round(k[-1], 4), "golden", val.get("golden_sha256_match"), "replicas", val.get("replicas_equal"))
        if v:
            print(f"{tag or 'f32_'}{side}: value median {s.median(v):.0f} [{min(v):.0f}, {max(v):.0f}]  front ms median {s.median(k):.4f} [{min(k):.4f}, {max(k):.4f}]")
PY
echo "t=$(( $(date +%s) - t0 ))"
