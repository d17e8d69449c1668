#!/usr/bin/env python
"""bench.py -- throughput of the img_completion hot path (BASELINE.json metric: frames/s at 1216x352).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload lidar_only|guided|stereo] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A step is one pass of the hot path over one batch of synthetic frames (default: BASELINE configs[1],
DC_lidar_only, 1024 frames of 352x1216 at 5 % valid pixels, 64 unique frames x 16).  Per-GPU work is
fixed as N grows (weak scaling): frames are independent and sharded frame-wise, no collective on the
hot path; NCCL only gathers timings / checksums (depth_completion_mt_b200/sharding.py).

  value     frames/s, device-resident inputs, CUDA events on the launch stream, max over ranks
  e2e       the same through the C ABI host entry point: pinned HOST buffers in and out, H2D + D2H inside
            the timed region
  roofline  algorithmic bytes (SURVEY.md 8d: 8 B/px lidar-only, 12 guided, 10 stereo) / time vs the measured
            HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the reference CPU path, one process per host core: the reference's own sources (oracle/_ref, kind
                "reference") when the prebuilt library is present, else the cv2 oracle port
            timed on a bounded sample of the same workload, rank 0 at N=1 only
`--impl reference` prints the reference-CPU arm alone in the same JSON shape.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# SURVEY.md 8d (stereo_chain: a2 + a4-a9, 14 B/px; lidar_camera_chain: Lab image 3 + sparse 4 + dense 4 B/px, the labels stay on the device)
BYTES_PER_PX = {"lidar_only": 8, "guided": 12, "stereo": 10, "stereo_chain": 14, "lidar_camera_chain": 11}
METRIC = "frames/sec @1216x352 sparse depth"
UNIQUE = 64


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="lidar_only", choices=list(BYTES_PER_PX))
    ap.add_argument("--frames", type=int, default=1024, help="frames per GPU per step")
    ap.add_argument("--rows", type=int, default=352)
    ap.add_argument("--cols", type=int, default=1216)
    ap.add_argument("--density", type=float, default=0.05)
    ap.add_argument("--path", default="auto", choices=["auto", "generic", "fused", "rank"])
    ap.add_argument("--input", default="f32", choices=["f32", "u16", "float"],
                    help="lidar_only / guided: float32 metres on the KITTI q8 grid (the reference's cv::Mat, default), KITTI uint16 = metres * 256 "
                         "(main.cpp:75-82), or `float`: arbitrary float32 depths (what DC_stereo_lidar completes after cv::normalize; use --path rank)")
    ap.add_argument("--labels", default="grid", choices=["grid", "slic"],
                    help="guided workload: jittered grid labels (SURVEY 8d) or real SLIC output of synthetic Lab images (step 18, nc 50)")
    ap.add_argument("--host-input", default="pinned", choices=["pinned", "wc"],
                    help="e2e leg, lidar_only: input in torch pinned memory, or in write-combined page-locked memory (dcmt_host_alloc)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--host-multi", action="store_true", help="single process: also time dcmt_img_completion_u16_host_multi over all visible GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-frames-per-core", type=int, default=16, help="reference arm: frames per host core per step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl ours: after the timed steps, write the output of the last one as DIR/<name>.npy (float32, at most "
                         "64 MB: a fixed, seeded sample of frames when the batch is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":  # the reference arm's workers hand back one pixel per frame, not the frames
        ap.error("--dump-outputs needs --impl ours: the reference arm keeps only out[0, 0] of each frame it times")
    return args


# --------------------------------------------------------------------------- reference (CPU) arm
_W = {}


def _ref_worker_init(workload, rows, cols, density):
    sys.path.insert(0, ROOT)
    from depth_completion_mt_b200 import synth
    try:
        from oracle import cv2_oracle as cvo
        have_cv2 = cvo.HAVE_CV2
    except Exception:
        have_cv2 = False
    ref_ok = False
    if have_cv2:
        # the reference's own sources compiled from /root/reference in the build container (oracle/_ref/libdcmt_ref.so,
        # OpenCV calls forwarded to cv2)
        try:
            from oracle import ref_oracle as ro

            ref_ok = ro.available()
        except Exception:
            ref_ok = False
    if ref_ok:
        ro.lib()  # registers the cv2 callbacks, cv2.setNumThreads(1)
        _W["impl"] = ro
        _W["kind"] = "ref"
    elif have_cv2:
        import cv2

        cv2.setNumThreads(1)
        _W["impl"] = cvo
        _W["kind"] = "cv2"
    else:
        from oracle import c_oracle as co

        _W["impl"] = co
        _W["kind"] = "c"
    _W.update(workload=workload, rows=rows, cols=cols, density=density, synth=synth, cache={})


def _ref_inputs(f):
    c = _W["cache"]
    if f not in c:
        synth, rows, cols = _W["synth"], _W["rows"], _W["cols"]
        if _W["workload"] == "lidar_only":
            c[f] = (synth.sparse_depth(f, rows, cols, _W["density"]),)
        elif _W["workload"] == "guided":
            lab, k = synth.superpixel_labels(f, rows, cols)
            c[f] = (synth.sparse_depth(f, rows, cols, _W["density"]), lab, k)
        elif _W["workload"] == "stereo_chain":
            lab, k = synth.superpixel_labels(f, rows, cols, 65)
            _, left, right = synth.stereo_pair(f, rows, cols)
            c[f] = (synth.velodyne_cloud(f, 120000), lab, k, left, right)
        elif _W["workload"] == "lidar_camera_chain":
            c[f] = (synth.sparse_depth(f, rows, cols, _W["density"]), synth.lab_image(f, rows, cols))
        else:
            c[f] = synth.stereo_pair(f, rows, cols)
    return c[f]


def _ref_task(f):
    impl, args = _W["impl"], _ref_inputs(f % UNIQUE)
    if _W["workload"] == "lidar_only":
        out = impl.img_completion(args[0], "gaussian")
    elif _W["workload"] == "guided":
        if _W["kind"] == "ref":
            out = impl.interpolate_with_superpixels(args[1], args[0], n_clusters=args[2])
        else:
            out = impl.interpolate_with_superpixels(args[0], args[1], args[2])
    elif _W["workload"] == "lidar_camera_chain":
        from oracle import c_oracle as co

        if _W["kind"] == "ref":
            labels, centers = impl.generate_superpixels(args[1], 18, 50)[:2]
            out = impl.interpolate_with_superpixels(labels, args[0], n_clusters=len(centers))
        else:
            labels, centers = co.slic(args[1], 18, 50)
            out = impl.interpolate_with_superpixels(args[0], labels, len(centers))
    elif _W["workload"] == "stereo_chain":
        synth = _W["synth"]
        pts, lab, k, left, right = args
        if _W["kind"] == "ref":
            nrm = impl.lidar_project(pts, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, _W["rows"], _W["cols"])[1]
            dense = impl.interpolate_with_superpixels(lab, nrm, n_clusters=k)
        else:
            from oracle import c_oracle as co

            nrm = co.lidar_project(pts, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, _W["rows"], _W["cols"])[1]
            dense = impl.interpolate_with_superpixels(nrm, lab, k)
        out = impl.stereo_refine(dense, left, right)
    else:
        out = impl.stereo_refine(*args)
    return float(out[0, 0])


def _single_frame_ms(runs):
    """BASELINE configs[0]: one frame, one thread (cv2.setNumThreads(1) in the worker), median of `runs` calls."""
    _ref_task(0)
    ts = []
    for _ in range(runs):
        t0 = time.perf_counter()
        _ref_task(0)
        ts.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(ts)


def run_reference(args, quiet=False):
    """Reference CPU arm: the reference's own CPU implementation (oracle/_ref, else the oracle port) on all host cores.
    `config` is the GPU arm's (same workload, same frames per step); each timed step is a BOUNDED SAMPLE of that step
    (cpu_baseline.sample says how many frames), and the rate is what is compared."""
    import multiprocessing as mp

    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_step = max(1, args.ref_frames_per_core) * cores
    if args.workload in ("guided", "lidar_camera_chain"):
        per_step = cores  # ~2 s per frame per core
    if args.workload == "stereo_chain":
        per_step = 2 * cores  # ~100 superpixels: about 0.25 s per frame per core
    if not quiet:
        # --impl reference: load the reference build in THIS process as well (the work runs in forked workers), so that whoever lists
        # the libraries this process loaded sees which implementation `kind` names.  Not in the GPU arm's cpu_baseline leg: that
        # process is the product's, its list should show libdcmt.so alone.
        try:
            from oracle import cv2_oracle as _cvo, ref_oracle as _ro

            if _cvo.HAVE_CV2 and _ro.available():
                _ro.lib()
        except Exception:
            pass
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_ref_worker_init, initargs=(args.workload, args.rows, args.cols, args.density)) as pool:
        kind = pool.apply(_kind)
        single_ms = pool.apply(_single_frame_ms, (20 if args.workload not in ("guided", "lidar_camera_chain") else 3,))
        frames = list(range(per_step))
        chunk = max(1, per_step // (cores * 2))
        for _ in range(max(1, args.warmup)):
            pool.map(_ref_task, frames, chunksize=chunk)  # also fills the per-worker input caches
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_ref_task, frames, chunksize=chunk)
        dt = time.perf_counter() - t0
    fps = per_step * args.steps / dt
    is_ref = kind.startswith("reference")
    sample = (f"{per_step} frames per timed step (a bounded sample of the {args.frames}-frame step of `config`) x {args.steps} steps of the {args.workload} workload "
              f"({args.rows}x{args.cols}, {args.density:.0%} valid), {kind}{'' if is_ref else ' oracle port'}, "
              "one single-threaded process per core")
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.frames),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "reference" if is_ref else "port", "sample": sample,
                         "sample_frames_per_step": per_step, "single_thread_ms": single_ms,
                         "single_thread_note": "one frame, one thread, median of 20 calls (BASELINE configs[0]); the imgproc calls go "
                                               "through Python / cv2 callbacks (7 per frame), a native OpenCV build would be somewhat faster"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not quiet:
        emit(line)
    return line


def _kind():
    if _W["kind"] == "ref":
        import cv2

        return ("reference sources compiled from /root/reference (oracle/_ref/libdcmt_ref.so), "
                "imgproc calls forwarded to cv2 (OpenCV %s)" % cv2.__version__)
    return "cv2 (OpenCV %s)" % _W["impl"].cv2.__version__ if _W["kind"] == "cv2" else "plain-C"


def workload_config(args, frames_per_step_per_gpu):
    names = {"lidar_only": "DC_lidar_only img_completion, fused dilate/erode/fill/blur (BASELINE configs[1])",
             "guided": "DC_lidar_camera interpolate_with_superpixels (BASELINE configs[2])",
             "stereo": "DC_stereo_lidar disparity refinement (BASELINE configs[3])",
             "lidar_camera_chain": "DC_lidar_camera chain: Slic::generate_superpixels (step 18, nc 50, 10 iterations) on the Lab image -> "
                                   "interpolate_with_superpixels (main_lc.cpp:184-220; BASELINE configs[2])",
             "stereo_chain": "DC_stereo_lidar chain: LiDAR projection + cv::normalize -> interpolate_with_superpixels on the normalised floats -> "
                             "disparity refinement (main_sl.cpp:478-540,1162-1253; BASELINE configs[3])"}
    return {"workload": names[args.workload], "rows": args.rows, "cols": args.cols, "valid_density": args.density,
            "frames_per_gpu_per_step": frames_per_step_per_gpu, "global_batch": frames_per_step_per_gpu * max(1, args.gpus),
            "unique_frames": UNIQUE, "blur": "gaussian", "labels": getattr(args, "labels", "grid") if args.workload == "guided" else None, "input": getattr(args, "input", "f32") if args.workload == "lidar_only" else "f32", "parallelism": f"frame-sharded dp{max(1, args.gpus)}, no collective on the hot path",
            "l2_policy": "inputs larger than L2 (batch >> 126 MB), no flush needed"}


# --------------------------------------------------------------------------- GPU arm
class ClockSampler:
    """nvidia-smi sampling during the timed regions (B200_PROFILING.md clocks line)."""

    FIELDS = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.path = f"/tmp/dcmt_clocks_{os.getpid()}.csv"
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(index)], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        self.windows = []

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        import datetime

        rows = []
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(p[2]), float(p[3]), p[5:9]))
            except Exception:
                continue
        try:
            os.unlink(self.path)
        except OSError:
            pass
        inwin = [r for r in rows if any(a <= r[0] <= b for a, b in self.windows)]
        used = inwin or rows
        if not used:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "no samples"}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in used for n, v in zip(names, r[3]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(r[1] for r in used), "sm_max_mhz": max(r[2] for r in used), "reasons": reasons,
                "samples": len(used), "samples_in_timed_regions": len(inwin)}


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and the pinned host buffers it allocates afterwards, first touch) to the CPUs of the NUMA node its
    GPU hangs off: the e2e leg is bound by host memory and PCIe, and cross-socket traffic halves it on multi-GPU boxes.
    Returns a short description for the JSON line; never fails the run."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return "numa node unknown"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return f"numa node {node}: no allowed cpus"
        os.sched_setaffinity(0, allowed)
        return f"numa node {node}, {len(allowed)} cpus"
    except Exception as exc:  # noqa: BLE001
        return f"not bound ({type(exc).__name__})"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload):
    """record of the committed ncu capture of this workload, if one exists (profiles/traffic.json): DRAM bytes and warp
    instructions per frame, and the launch configuration they were captured at (the bench's own chunk size)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(workload)
    except Exception:
        return None


DUMP_BYTES = 60 * 10**6  # payload of --dump-outputs: below 64 MB with the .npy header
DUMP_SEED = 0


def dump_outputs(directory, name, out):
    """Write `out` (frames first) as directory/name.npy in float32.  When the whole batch is over DUMP_BYTES, a seeded
    sample of whole frames in frame order (of single elements when one frame is already over it): the same arguments pick
    the same sample, so that two builds of the project can be compared output for output."""
    import numpy as np
    import torch

    os.makedirs(directory, exist_ok=True)
    n, frame_elems = out.shape[0], out[0].numel()
    keep = DUMP_BYTES // (4 * frame_elems)
    rng = np.random.default_rng(DUMP_SEED)
    if keep >= n:
        sample, what = out, f"all {n} frames"
    elif keep >= 1:
        idx = np.sort(rng.choice(n, keep, replace=False))
        sample, what = out[torch.from_numpy(idx).to(out.device)], f"frames {idx.tolist()} of {n}"
    else:
        idx = np.sort(rng.choice(out.numel(), DUMP_BYTES // 4, replace=False))
        sample, what = out.reshape(-1)[torch.from_numpy(idx).to(out.device)], f"{idx.size} seeded elements of {out.numel()}"
    path = os.path.join(directory, name + ".npy")
    np.save(path, sample.to(torch.float32).cpu().numpy())
    print(f"--dump-outputs: {path} = {what}", file=sys.stderr)


def run_ours(args):
    import numpy as np
    import torch

    from depth_completion_mt_b200 import _lib, api, sharding, synth

    rank, local_rank, world = sharding.init_process_group()
    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else "single rank: not bound"
    lib = _lib.load()
    rows, cols, n = args.rows, args.cols, args.frames
    reps = (n + UNIQUE - 1) // UNIQUE
    fpix = rows * cols

    # ---- synthetic inputs, device resident before timing
    holder = {}
    if args.workload == "lidar_only":
        if args.input == "float":
            d_in16 = None
            uniqf = np.stack([synth.sparse_depth_float(f, rows, cols, args.density) for f in range(UNIQUE)])
            d_in = torch.from_numpy(uniqf).to(dev).repeat(reps, 1, 1)[:n].contiguous()
        else:
            uniq16 = np.stack([synth.sparse_depth_q8(f, rows, cols, args.density) for f in range(UNIQUE)])
            d_in16 = torch.from_numpy(uniq16).to(dev).repeat(reps, 1, 1)[:n].contiguous()
            d_in = d_in16 if args.input == "u16" else (d_in16.to(torch.float32) / 256.0).contiguous()  # exact: convertTo(CV_32F, 1/256)
        d_out = torch.empty((n, rows, cols), dtype=torch.float32, device=dev)

        def step():
            api.img_completion(d_in, False, "gaussian", path=args.path, out=d_out, lib=lib)
        h2d, d2h = n * fpix * (2 if args.input == "u16" else 4), n * fpix * 4
    elif args.workload == "guided":
        uniq = np.stack([(synth.sparse_depth_float if args.input == "float" else synth.sparse_depth)(f, rows, cols, args.density) for f in range(UNIQUE)])
        if args.labels == "slic":
            k = lib.dcmt_slic_center_count(rows, cols, 18)
            labs = [(api.generate_superpixels(torch.from_numpy(synth.lab_image(f, rows, cols)).to(dev), 18, 50, lib=lib).cpu().numpy(), k)
                    for f in range(UNIQUE)]
        else:
            labs = [synth.superpixel_labels(f, rows, cols) for f in range(UNIQUE)]
            k = labs[0][1]
        d_in = torch.from_numpy(uniq).to(dev).repeat(reps, 1, 1)[:n].contiguous()
        d_lab = torch.from_numpy(np.stack([l[0] for l in labs])).to(dev).repeat(reps, 1, 1)[:n].contiguous()
        holder = {}

        def step():
            holder["out"] = api.interpolate_with_superpixels(d_lab, d_in, "gaussian", 1, n_clusters=k, path=args.path, lib=lib)
        h2d, d2h = n * fpix * 8, n * fpix * 4
    elif args.workload == "lidar_camera_chain":
        # what the camera program runs per frame (main_lc.cpp:184-220): Lab image -> SLIC superpixels -> guided completion of the
        # sparse depth with those labels; the labels never leave the device
        uniq = np.stack([synth.sparse_depth(f, rows, cols, args.density) for f in range(UNIQUE)])
        d_in = torch.from_numpy(uniq).to(dev).repeat(reps, 1, 1)[:n].contiguous()
        d_labimg = torch.from_numpy(np.stack([synth.lab_image(f, rows, cols) for f in range(UNIQUE)])).to(dev).repeat(reps, 1, 1, 1)[:n].contiguous()
        k = lib.dcmt_slic_center_count(rows, cols, 18)
        holder = {}
        CH = 256  # frames per SLIC call: bounds its per-frame work buffers

        def step():
            outs = []
            for c0 in range(0, n, CH):
                labels = api.generate_superpixels(d_labimg[c0:c0 + CH], 18, 50, lib=lib)
                outs.append(api.interpolate_with_superpixels(labels, d_in[c0:c0 + CH], "gaussian", 1, n_clusters=k, path=args.path, lib=lib))
            holder["out"] = torch.cat(outs) if len(outs) > 1 else outs[0]
        h2d, d2h = n * fpix * 7, n * fpix * 4
        args.no_e2e = True  # the chain has no single host entry point: its stages are the two calls above
    elif args.workload == "stereo_chain":
        # what the stereo program really runs per frame (main_sl.cpp:1150 withSuperPixels, :1162-1253): Velodyne cloud ->
        # projected depth image -> cv::normalize(0, 80) -> superpixel-guided completion of the normalised FLOATS (dictionary
        # path of the fused kernels) -> disparity refinement against the gray pair.  Labels are an input here (SLIC of the
        # left image is the f1 row, measured on its own).
        npts = 120000
        uniq_n = min(UNIQUE, n)
        clouds = np.stack([synth.velodyne_cloud(f, npts) for f in range(uniq_n)])
        reps_c = (n + uniq_n - 1) // uniq_n
        d_pts = torch.from_numpy(clouds).to(dev).repeat(reps_c, 1, 1)[:n].contiguous()
        labs = [synth.superpixel_labels(f, rows, cols, 65) for f in range(uniq_n)]  # ~100 superpixels, main_sl.cpp:443
        k = labs[0][1]
        d_lab = torch.from_numpy(np.stack([l[0] for l in labs])).to(dev).repeat(reps_c, 1, 1)[:n].contiguous()
        trip = [synth.stereo_pair(f, rows, cols) for f in range(uniq_n)]
        d_l, d_r = (torch.from_numpy(np.stack([t[i] for t in trip])).to(dev).repeat(reps_c, 1, 1)[:n].contiguous() for i in (1, 2))
        prm = api.stereo_params(lib=lib)
        holder = {}
        CH = 128  # clouds per projection call: bounds the 8-byte key plane per cloud (3.4 MB at 352x1216)

        def step():
            outs = []
            for c0 in range(0, n, CH):
                _, nrm, _ = api.lidar_project_batch(d_pts[c0:c0 + CH], None, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, rows, cols, lib=lib)
                dense = api.interpolate_with_superpixels(d_lab[c0:c0 + CH], nrm, "gaussian", 1, n_clusters=k, path="rank", lib=lib)
                outs.append(api.stereo_refine(dense, d_l[c0:c0 + CH], d_r[c0:c0 + CH], prm, lib=lib))
            holder["out"] = torch.cat(outs) if len(outs) > 1 else outs[0]
        h2d, d2h = n * (npts * 16 + fpix * 6), n * fpix * 4
        args.no_e2e = True  # the chain has no single host entry point: its stages are the three calls above
    else:
        trip = [synth.stereo_pair(f, rows, cols) for f in range(UNIQUE)]
        d_ig, d_l, d_r = (torch.from_numpy(np.stack([t[i] for t in trip])).to(dev).repeat(reps, 1, 1)[:n].contiguous() for i in range(3))
        prm = api.stereo_params(lib=lib)
        holder = {}

        def step():
            holder["out"] = api.stereo_refine(d_ig, d_l, d_r, prm, lib=lib)
        h2d, d2h = n * fpix * 6, n * fpix * 4

    def barrier():
        if world > 1:
            torch.distributed.barrier()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.dcmt_launch_count()
    torch.cuda.synchronize()
    w0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    w1 = time.time()
    barrier()
    launches = lib.dcmt_launch_count() - launches0
    if sampler:
        sampler.mark(w0, w1)
    elapsed_ms = ev0.elapsed_time(ev1)

    # ---- validation payload: checksums of the unique outputs (+ digests vs the committed golden file)
    out_t = d_out if args.workload == "lidar_only" else holder["out"]
    if args.dump_outputs and rank == 0:  # every rank computes the same frames
        dump_outputs(args.dump_outputs, "depth", out_t)
    sums = sharding.frame_checksums(out_t[: min(n, UNIQUE)])
    replicas_equal = all(bool(torch.equal(out_t[UNIQUE * k_:UNIQUE * (k_ + 1)], out_t[:UNIQUE][: max(0, min(UNIQUE, n - UNIQUE * k_))]))
                         for k_ in range(1, reps) if n - UNIQUE * k_ > 0)
    golden_ok = None
    if args.workload == "lidar_only" and args.input != "float" and (rows, cols, args.density) == (352, 1216, 0.05):
        golden_ok = True
        for l in open(os.path.join(ROOT, "tests", "golden", "lidar_only_352x1216.sha256")):
            p = l.split()
            if l.startswith("#") or len(p) != 5 or p[1] != "0" or p[2] != "gaussian":
                continue
            golden_ok &= hashlib.sha256(out_t[int(p[0])].cpu().numpy().tobytes()).hexdigest() == p[4]

    # ---- end to end through the host entry points: pinned host buffers, H2D + D2H inside the timed region; next to
    #      every leg the COPY-ONLY ceiling: the same buffers, chunking and streams with the kernels left out
    def timed_host(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        barrier()
        t0w = time.time()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        t1w = time.time()
        barrier()
        if sampler:
            sampler.mark(t0w, t1w)
        return ms

    import ctypes as C

    e2e_ms = e2e16_ms = ceil_ms = ceil16_ms = multi_ms = None
    latency = None
    if not args.no_e2e:
        if args.workload == "lidar_only" and args.input == "float":
            h_in = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
            h_in.copy_(d_in)
            h_out = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
            np_in, np_out = h_in.numpy(), h_out.numpy()
            e2e_ms = timed_host(lambda: api.img_completion(np_in, False, "gaussian", path=args.path, out=np_out, lib=lib))
            ceil_ms = timed_host(lambda: lib.check(lib.dcmt_debug_host_copy_f32(np_in.ctypes.data, np_out.ctypes.data, rows, cols, n, None, 0)))
        elif args.workload == "lidar_only":
            if args.host_input == "wc":
                hb = api.HostBuffer((n, rows, cols), np.float32, write_combined=True, lib=lib)
                holder["hb"] = hb
                hb.array[...] = (d_in16.to(torch.float32) / 256.0).cpu().numpy()
                np_in = hb.array
            else:
                h_in = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
                h_in.copy_(d_in16.to(torch.float32) / 256.0)
                np_in = h_in.numpy()
            h_in16 = torch.empty((n, rows, cols), dtype=torch.uint16, pin_memory=True)
            h_in16.copy_(d_in16)
            np_in16 = h_in16.numpy()
            h_out = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
            np_out = h_out.numpy()
            # the copy-only ceiling is measured before AND after each end-to-end leg and the faster of the two is reported: the
            # host side of a shared box drifts by 10-20 % within a run, and a ceiling must not be taken in a slower moment than
            # the thing it bounds
            copy_f32 = lambda: lib.check(lib.dcmt_debug_host_copy_f32(np_in.ctypes.data, np_out.ctypes.data, rows, cols, n, None, 0))
            copy_u16 = lambda: lib.check(lib.dcmt_debug_host_copy_u16(np_in16.ctypes.data, np_out.ctypes.data, rows, cols, n, None, 0))
            ceil_ms = timed_host(copy_f32)
            e2e_ms = timed_host(lambda: api.img_completion(np_in, False, "gaussian", path=args.path, out=np_out, lib=lib))
            assert bool(torch.equal(h_out[:UNIQUE].to(dev), out_t[:UNIQUE])), "host path and device path disagree"
            ceil_ms = min(ceil_ms, timed_host(copy_f32))
            # the same frames as the KITTI uint16 payload (dcmt_img_completion_u16_host, main.cpp:75-93): half the H2D bytes
            ceil16_ms = timed_host(copy_u16)
            h_out.zero_()
            e2e16_ms = timed_host(lambda: api.img_completion(np_in16, False, "gaussian", out=np_out, lib=lib))
            assert bool(torch.equal(h_out[:UNIQUE].to(dev), out_t[:UNIQUE])), "uint16 host path and device path disagree"
            ceil16_ms = min(ceil16_ms, timed_host(copy_u16))
            # one process, all visible GPUs: the multi-device host entry point (only where this rank sees several devices)
            if world == 1 and torch.cuda.device_count() > 1 and args.host_multi:
                h_out.zero_()
                multi_ms = timed_host(lambda: api.img_completion(np_in16, False, "gaussian", out=np_out, devices="all", lib=lib))
                assert bool(torch.equal(h_out[:UNIQUE].to(dev), out_t[:UNIQUE])), "multi-device host path and device path disagree"
            # single-frame latency (BASELINE configs[0], main.cpp:93 is called with ONE frame): median of 30 calls
            def med(fn, k=30):
                fn()
                ts = []
                for _ in range(k):
                    t0 = time.perf_counter()
                    fn()
                    ts.append(1e3 * (time.perf_counter() - t0))
                return statistics.median(ts)
            one_in, one_in16, one_out = np_in[:1], np_in16[:1], np_out[:1]
            d_one, d_one_out = d_in[:1].contiguous(), torch.empty((1, rows, cols), dtype=torch.float32, device=dev)

            def dev_one(path):
                api.img_completion(d_one, False, "gaussian", path=path, out=d_one_out, lib=lib)
                torch.cuda.synchronize()
            latency = {"unit": "ms", "calls": 30, "frames_per_call": 1,
                       "f32_host": med(lambda: api.img_completion(one_in, False, "gaussian", out=one_out, lib=lib)),
                       "u16_host": med(lambda: api.img_completion(one_in16, False, "gaussian", out=one_out, lib=lib)),
                       "device_auto": med(lambda: dev_one("auto")), "device_fused": med(lambda: dev_one("fused")),
                       "note": "one 352x1216 frame per call, median wall time incl. the synchronisation; *_host: pinned host buffers in "
                               "and out (dcmt_img_completion_f32_host / _u16_host); device_*: resident input, kernels + sync only"}
        elif args.workload == "guided":
            h_in = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
            h_in.copy_(d_in)
            h_lab = torch.empty((n, rows, cols), dtype=torch.int32, pin_memory=True)
            h_lab.copy_(d_lab)
            h_out = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
            np_in, np_lab, np_out = h_in.numpy(), h_lab.numpy(), h_out.numpy()

            def host_step():
                holder["h"] = api.interpolate_with_superpixels(np_lab, np_in, "gaussian", 1, n_clusters=k, path=args.path, out=np_out, lib=lib)
            e2e_ms = timed_host(host_step)
        else:
            hs = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (d_ig, d_l, d_r)]
            for a, b in zip(hs, (d_ig, d_l, d_r)):
                a.copy_(b)
            nps = [a.numpy() for a in hs]
            h_out = torch.empty((n, rows, cols), dtype=torch.float32, pin_memory=True)
            np_out = h_out.numpy()

            def host_step():
                holder["h"] = api.stereo_refine(nps[0], nps[1], nps[2], prm, out=np_out, lib=lib)
            e2e_ms = timed_host(host_step)

    # ---- per-kernel split of the fused path (CUDA events around each kernel, a few extra untimed steps)
    kernels = None
    if args.workload == "lidar_only" and args.input != "float":
        lib.check(lib.dcmt_profile_begin())
        for _ in range(3):
            step()
        fm, tm, ch = C.c_double(0), C.c_double(0), C.c_longlong(0)
        lib.check(lib.dcmt_profile_end(C.byref(fm), C.byref(tm), C.byref(ch)))
        if ch.value:
            peak_, _src = measured_peak()
            px = 3 * n * fpix
            fb = 4 if args.input == "u16" else 6
            kernels = {
                "k_q8_front": {"ms_per_step": fm.value / 3, "alg_bytes_per_px": fb, "achieved_GBps": fb * px / (fm.value * 1e6),
                               "frac": fb * px / (fm.value * 1e6) / peak_, "note": f"{args.input} in, uint16 intermediate out"},
                "k_q8_tail": {"ms_per_step": tm.value / 3, "alg_bytes_per_px": 6, "achieved_GBps": 6 * px / (tm.value * 1e6),
                              "frac": 6 * px / (tm.value * 1e6) / peak_, "note": "uint16 intermediate in, float32 out; dominant kernel"},
                "chunks_per_step": ch.value // 3,
                "how": "CUDA events around each kernel over 3 extra steps AFTER the timed region (dcmt_profile_begin / _end)",
            }
    res = sharding.gather_validation(elapsed_ms, n * args.steps, sums, device=dev)
    def gathered_fps(ms):
        if ms is None:
            return None
        g = sharding.gather_validation(ms, n * args.steps, sums, device=dev)
        return g["total_frames"] / (g["max_ms"] / 1e3)

    fps_e2e, fps_e2e16, fps_ceil, fps_ceil16 = (gathered_fps(m) for m in (e2e_ms, e2e16_ms, ceil_ms, ceil16_ms))
    clocks = sampler.stop() if sampler else None
    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    total_frames = res["total_frames"]
    secs = res["max_ms"] / 1e3
    fps = total_frames / secs
    bpp = 6 if (args.workload == "lidar_only" and args.input == "u16") else BYTES_PER_PX[args.workload]  # uint16 in + float32 out
    bytes_per_frame = bpp * fpix
    peak, peak_src = measured_peak()
    achieved = fps * bytes_per_frame / 1e9 / world  # per GPU
    traffic_rec = ncu_traffic(args.workload) or {}
    traffic = traffic_rec.get("dram_bytes_per_frame") if isinstance(traffic_rec, dict) else traffic_rec
    # the bound the kernels actually run against, next to the HBM one: warp instructions per frame (committed ncu counters)
    # over the issue rate of the chip (4 schedulers x SMs x SM clock)
    issue = None
    wi = traffic_rec.get("warp_instructions_per_frame") if isinstance(traffic_rec, dict) else None
    if wi and clocks and clocks.get("sm_mhz"):
        sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        rate = 4.0 * sms * clocks["sm_mhz"] * 1e6
        per_frame = float(sum(wi.values()))
        issue = {"warp_instructions_per_frame": wi, "issue_rate_per_s": rate, "floor_us_per_frame": 1e6 * per_frame / rate,
                 "achieved_us_per_frame": 1e6 * world / fps, "frac": (per_frame / rate) / (world / fps),
                 "source": traffic_rec.get("source"),
                 "note": "time the counted instructions would take if every scheduler issued every cycle / measured time per frame"}
    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": res["max_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, n),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_unit": "DRAM bytes per frame (read + write, front + tail)", "traffic_capture": traffic_rec.get("capture") if isinstance(traffic_rec, dict) else None,
                     "algorithmic_bytes_per_frame": bytes_per_frame, "peak_source": peak_src, "kernels": kernels, "issue": issue,
                     "note": f"whole hot path, {bpp} algorithmic B/px x {fpix} px x frames / CUDA-event time, per GPU"},
        "gpu_launches": int(launches), "clocks": clocks, "lib": {"path": lib.path, "build": lib.dcmt_build_info().decode(), "version": lib.dcmt_version()},
        "validation": {"ranks": world, "checksums_equal_across_ranks": all(bool(torch.equal(c, res["checksums"][0])) for c in res["checksums"]),
                       "replicas_equal": bool(replicas_equal), "golden_sha256_match": golden_ok, "ms_per_rank": res["ms_per_rank"]},
    }
    if not args.no_e2e:
        api_note = "dcmt_*_host via depth_completion_mt_b200.api with numpy views of pinned host buffers"
        if args.workload == "lidar_only" and args.input != "float":
            # headline: the reference program's own input format -- the uint16 payload of the KITTI depth PNG (main.cpp:75-82);
            # the call stands for convertTo(CV_32F, 1/256) + img_completion (main.cpp:79,93)
            line["e2e"] = {"value": fps_e2e16, "unit": "frames/s", "h2d_bytes_per_step": int(n * fpix * 2), "d2h_bytes_per_step": int(d2h),
                           "input": "uint16 KITTI depth payload (main.cpp:75-82), float32 out",
                           "api": "dcmt_img_completion_u16_host; " + api_note, "copy_ceiling": fps_ceil16,
                           "frac_of_copy_ceiling": fps_e2e16 / fps_ceil16 if fps_ceil16 else None,
                           "copy_ceiling_note": "dcmt_debug_host_copy_u16: the same pinned buffers, chunks and streams, kernels left out; the faster of a run before and a run after the e2e leg",
                           "host_binding_rank0": numa}
            line["e2e_f32_input"] = {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(n * fpix * 4), "d2h_bytes_per_step": int(d2h),
                                     "input": "float32 metres (the cv::Mat img_completion takes, img_completion.cpp:17)",
                                     "api": "dcmt_img_completion_f32_host", "copy_ceiling": fps_ceil,
                                     "frac_of_copy_ceiling": fps_e2e / fps_ceil if fps_ceil else None}
            if multi_ms is not None:
                line["e2e_host_multi"] = {"value": n * args.steps / (multi_ms / 1e3), "unit": "frames/s", "devices": torch.cuda.device_count(),
                                          "api": "dcmt_img_completion_u16_host_multi: one process, one thread, all visible GPUs"}
            if latency:
                line["latency"] = latency
        else:
            line["e2e"] = {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "api": api_note,
                           "copy_ceiling": fps_ceil, "host_binding_rank0": numa}
    if world == 1 and not args.no_cpu_baseline:
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1", "--workload", args.workload,
                   "--rows", str(rows), "--cols", str(cols), "--density", str(args.density)]
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
            ref = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
            line["cpu_baseline"] = ref["cpu_baseline"]
            if line.get("latency") and ref["cpu_baseline"].get("single_thread_ms"):
                line["latency"]["reference_single_thread_ms"] = ref["cpu_baseline"]["single_thread_ms"]
        except Exception as exc:  # never lose the GPU numbers because the CPU leg failed
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": None, "kind": "port", "sample": f"failed: {exc!r}"}
    emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    # libraries print to fd 1 behind Python's back (NCCL's version banner under torchrun): route fd 1 to stderr for the
    # whole run and keep the real stdout for the JSON line alone
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0  # rank 0 alone runs the CPU arm
        run_reference(args)
        return 0
    run_ours(args)
    return 0


if __name__ == "__main__":
    sys.exit(main())
