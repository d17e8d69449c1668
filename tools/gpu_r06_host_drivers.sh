#!/bin/bash
# Session of round 6 (one device driver and one host-pointer driver for every completion entry point): a checkout of the
# parent commit (directory in $1, built here with its own __graft_entry__; its bench.py, binding and libdcmt.so) against this
# tree, alternating: bench.py default, --input u16 and --host-multi, tools/bench_kitti_io.py; plus smoke, dumped outputs and
# the GPU suite.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r06_host_drivers.sh /path/to/parent/checkout OUT_DIR
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
for i in 1 2 3; do
  (cd $P && timeout 600 python bench.py --no-cpu-baseline) > $out/bench_before_$i.json 2> $out/bench_before_$i.err; echo "before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline > $out/bench_after_$i.json 2> $out/bench_after_$i.err; echo "after $i rc=$?"
done
for i in 1 2 3 4; do
  (cd $P && timeout 600 python bench.py --no-cpu-baseline --input u16) > $out/bench_u16_before_$i.json 2>> $out/bench_u16.err; echo "u16 before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline --input u16 > $out/bench_u16_after_$i.json 2>> $out/bench_u16.err; echo "u16 after $i rc=$?"
done
for i in 1 2; do
  (cd $P && timeout 600 python bench.py --no-cpu-baseline --host-multi) > $out/bench_multi_before_$i.json 2>> $out/bench_multi.err; echo "multi before $i rc=$?"
  timeout 600 python bench.py --no-cpu-baseline --host-multi > $out/bench_multi_after_$i.json 2>> $out/bench_multi.err; echo "multi after $i rc=$?"
done
echo "t=$(( $(date +%s) - t0 ))"
for i in 1 2; do
  (cd $P && timeout 900 python tools/bench_kitti_io.py --steps 10 --warmup 2) > $out/kitti_io_before_$i.json 2>> $out/kitti_io.err; echo "kitti_io before $i rc=$?"
  timeout 900 python tools/bench_kitti_io.py --steps 10 --warmup 2 > $out/kitti_io_after_$i.json 2>> $out/kitti_io.err; echo "kitti_io after $i rc=$?"
done
tail -n 3 $out/kitti_io.err
echo "t=$(( $(date +%s) - t0 ))"
tmp=$(mktemp -d)
(cd $P && timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/before) > /dev/null 2>> $out/dump.err; echo "dump before rc=$?"
timeout 600 python bench.py --no-cpu-baseline --steps 1 --warmup 1 --dump-outputs $tmp/after > /dev/null 2>> $out/dump.err; echo "dump after rc=$?"
sha256sum $tmp/before/depth.npy $tmp/after/depth.npy | sed "s|$tmp/||" | tee $out/dump_sha256.txt
cmp $tmp/before/depth.npy $tmp/after/depth.npy && echo "depth.npy identical" | tee -a $out/dump_sha256.txt
rm -rf $tmp
echo "t=$(( $(date +%s) - t0 ))"
timeout 1800 python -m pytest tests -q -m gpu > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $out/pytest_gpu.log
tail -8 $out/pytest_gpu.log
echo "t=$(( $(date +%s) - t0 ))"
OUT="$out" python - <<'PY'
import json, glob, os, statistics as s
for tag in ("", "u16_", "multi_"):
    for side in ("before", "after"):
        v = []
        for f in sorted(glob.glob(os.path.join(os.environ["OUT"], f"bench_{tag}{side}_*.json"))):
            try:
                d = json.loads(open(f).read().strip().splitlines()[-1])
            except Exception as e:
                print(f, "unreadable", e); continue
            v.append(d["value"])
            val = d.get("validation", {})
            print(f, round(d["value"]), "golden", val.get("golden_sha256_match"), "replicas", val.get("replicas_equal"),
                  "e2e", {k: round(x["value"]) for k, x in d.items() if k.startswith("e2e") and isinstance(x, dict) and "value" in x})
        if v:
            print(f"{tag or 'f32_'}{side}: value median {s.median(v):.0f} [{min(v):.0f}, {max(v):.0f}]")
for side in ("before", "after"):
    for f in sorted(glob.glob(os.path.join(os.environ["OUT"], f"kitti_io_{side}_*.json"))):
        d = json.loads(open(f).read().strip().splitlines()[-1])
        print(f, {k: round(d[k]) for k in ("device_u16_f32", "device_u16_u16")},
              {k: round(d[k]["e2e"]) for k in d if k.startswith("host_")}, "rule", all(d["outputs_follow_rule"].values()))
PY
echo "t=$(( $(date +%s) - t0 ))"
