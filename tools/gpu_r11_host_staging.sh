#!/bin/bash
# Session of round 11 (the single-shot host entry points staged through one helper, arguments checked before any copy): a
# built checkout of the parent commit (directory in $1) against this tree: smoke, the whole GPU suite, bench.py default and
# --workload lidar_camera_chain alternating twice each with the default workload's dumped outputs compared,
# tools/bench_eval_u16.py with the parent's library, tools/bench_superpixels_bgr.py (its host leg times
# dcmt_slic_bgr_u8c3_host) alternating twice, and the numpy forms of api.bgr2gray / bgr2lab / lidar_project /
# generate_superpixels at 352 x 1216 timed with perf_counter, alternating twice.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r11_host_staging.sh /path/to/parent/checkout OUT_DIR
set -u
P=$(realpath "$1")
out=$(realpath -m "${2:?output directory}")
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > $out/gpu.txt 2>&1
cat $out/gpu.txt
t0=$(date +%s)
timeout 900 python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $out/smoke.log 2>&1; echo "smoke rc=$?" | tee -a $out/smoke.log
tail -2 $out/smoke.log
echo "t=$(( $(date +%s) - t0 ))"
timeout 2400 python -m pytest tests -q -m gpu > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $out/pytest_gpu.log
tail -8 $out/pytest_gpu.log
echo "t=$(( $(date +%s) - t0 ))"
for w in lidar_only lidar_camera_chain; do
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
echo "t=$(( $(date +%s) - t0 ))"
timeout 900 python tools/bench_eval_u16.py --steps 20 --warmup 3 --parent-lib $P/depth_completion_mt_b200/libdcmt.so > $out/eval_u16.json 2> $out/eval_u16.err
echo "bench_eval_u16 rc=$?"
cat $out/eval_u16.json; tail -3 $out/eval_u16.err
echo "t=$(( $(date +%s) - t0 ))"
for i in 1 2; do
  (cd $P && timeout 900 python tools/bench_superpixels_bgr.py --steps 3 --warmup 1) > $out/bgr_before_$i.json 2>> $out/bgr.err; echo "bench_superpixels_bgr before $i rc=$?"
  timeout 900 python tools/bench_superpixels_bgr.py --steps 3 --warmup 1 > $out/bgr_after_$i.json 2>> $out/bgr.err; echo "bench_superpixels_bgr after $i rc=$?"
done
echo "t=$(( $(date +%s) - t0 ))"
# the numpy forms of the single-shot host calls: median wall time of one synchronous call, 352 x 1216
cat > $out/host_api.py <<'PY'
import json, statistics, sys, time
sys.path.insert(0, sys.argv[1])
import numpy as np
from depth_completion_mt_b200 import api, synth
rng = np.random.default_rng(0)
bgr = rng.integers(0, 256, (352, 1216, 3), dtype=np.uint8)
lab = api.bgr2lab(bgr)
pts = np.c_[rng.uniform(2, 80, 120000), rng.uniform(-40, 40, 120000), rng.uniform(-3, 2, 120000), rng.uniform(0, 1, 120000)].astype(np.float32)
calls = {"bgr2gray": lambda: api.bgr2gray(bgr), "bgr2lab": lambda: api.bgr2lab(bgr),
         "lidar_project": lambda: api.lidar_project(pts, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, 352, 1216),
         "generate_superpixels": lambda: api.generate_superpixels(lab, 18, 50)}
res = {}
for name, f in calls.items():
    for _ in range(5):
        f()
    t = []
    for _ in range(40 if name != "generate_superpixels" else 15):
        a = time.perf_counter(); f(); t.append(time.perf_counter() - a)
    res[name + "_ms"] = round(statistics.median(t) * 1e3, 4)
print(json.dumps(res))
PY
for i in 1 2; do
  timeout 600 python $out/host_api.py $P > $out/host_api_before_$i.json 2>> $out/host_api.err; echo "host api before $i rc=$?"
  timeout 600 python $out/host_api.py $PWD > $out/host_api_after_$i.json 2>> $out/host_api.err; echo "host api after $i rc=$?"
done
cat $out/host_api_*.json
OUT="$out" python - <<'PY'
import json, glob, os, statistics as s
for w in ("lidar_only", "lidar_camera_chain"):
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
