#!/bin/bash
# Session of round 7 (the fused path's dead alternatives removed): a checkout of the parent commit (directory in $1, built
# here with its own __graft_entry__; its bench.py, binding and libdcmt.so) against this tree, alternating three times each:
# bench.py default, --input u16, --workload guided and --input float --path rank (k_q8_tail<true>); plus smoke and the
# dumped outputs of every leg.  The GPU suite runs in a call of its own.
# Usage (on the GPU box, from the repository root): bash tools/gpu_r07_fused_cleanup.sh /path/to/parent/checkout OUT_DIR
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
legs=("default:" "u16:--input u16" "guided:--workload guided" "rank:--input float --path rank")
for leg in "${legs[@]}"; do
  tag=${leg%%:*}; args=${leg#*:}
  for i in 1 2 3; do
    (cd $P && timeout 600 python bench.py --no-cpu-baseline $args) > $out/bench_${tag}_before_$i.json 2>> $out/bench_${tag}.err; echo "$tag before $i rc=$?"
    timeout 600 python bench.py --no-cpu-baseline $args > $out/bench_${tag}_after_$i.json 2>> $out/bench_${tag}.err; echo "$tag after $i rc=$?"
  done
  echo "t=$(( $(date +%s) - t0 ))"
done
tmp=$(mktemp -d)
for leg in "${legs[@]}"; do
  tag=${leg%%:*}; args=${leg#*:}
  (cd $P && timeout 600 python bench.py --no-cpu-baseline $args --steps 1 --warmup 1 --dump-outputs $tmp/before_$tag) > /dev/null 2>> $out/dump.err
  echo "dump $tag before rc=$?"
  timeout 600 python bench.py --no-cpu-baseline $args --steps 1 --warmup 1 --dump-outputs $tmp/after_$tag > /dev/null 2>> $out/dump.err
  echo "dump $tag after rc=$?"
  sha256sum $tmp/before_$tag/depth.npy $tmp/after_$tag/depth.npy | sed "s|$tmp/||" | tee -a $out/dump_sha256.txt
  cmp $tmp/before_$tag/depth.npy $tmp/after_$tag/depth.npy && echo "$tag: depth.npy identical" | tee -a $out/dump_sha256.txt
done
rm -rf $tmp
echo "t=$(( $(date +%s) - t0 ))"
OUT="$out" python - <<'PY'
import json, glob, os, statistics as s
for tag in ("default", "u16", "guided", "rank"):
    for side in ("before", "after"):
        v = []
        for f in sorted(glob.glob(os.path.join(os.environ["OUT"], f"bench_{tag}_{side}_*.json"))):
            try:
                d = json.loads(open(f).read().strip().splitlines()[-1])
            except Exception as e:
                print(f, "unreadable", e); continue
            v.append(d["value"])
            val = d.get("validation", {})
            print(os.path.basename(f), round(d["value"]), "golden", val.get("golden_sha256_match"), "replicas", val.get("replicas_equal"))
        if v:
            print(f"{tag} {side}: value median {s.median(v):.0f} [{min(v):.0f}, {max(v):.0f}]")
PY
echo "t=$(( $(date +%s) - t0 ))"
