#!/usr/bin/env python
"""Throughput of the SURVEY.md 8(f) rows (SLIC, LiDAR projection, evaluation) and of cvtColor(BGR2Lab) at 352x1216 on
one GPU, next to the C oracle (the literal CPU loops, one core) or single-threaded cv2 on the same inputs.  One JSON line
per row; the first line names the GPU and its power limit.

    python tools/bench_rows.py [--reps 20]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from depth_completion_mt_b200 import _lib, api, synth
from oracle import c_oracle as co


def gpu_time(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def cpu_time(fn, reps=3):
    fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return 1e3 * (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    lib = _lib.load()
    rows, cols = 352, 1216
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks))["hbm_gbs"] if os.path.exists(peaks) else 6558.7  # measured B200 HBM peak (SURVEY.md)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True)
    out = [{"gpu": torch.cuda.get_device_name(), "nvidia_smi": smi.stdout.strip() or smi.stderr.strip(), "hbm_peak_GBps": peak}]
    # ---- cvtColor(COLOR_BGR2Lab): 1024 device-resident frames (1.3 GB in, 1.3 GB out: well above the 126 MB L2), 6 B/px
    nl = 1024
    bgr = torch.from_numpy(np.stack([synth.bgr_image(f, rows, cols) for f in range(8)])).cuda().repeat(nl // 8, 1, 1, 1).contiguous()
    labo = torch.empty_like(bgr)

    def convert(src, dst, n):
        lib.check(lib.dcmt_bgr2lab_u8(src.data_ptr(), dst.data_ptr(), rows, cols, 0, 0, n, torch.cuda.current_stream().cuda_stream))
    ms = gpu_time(lambda: convert(bgr, labo, nl), a.reps)
    ms1 = gpu_time(lambda: convert(bgr, labo, 1), 10 * a.reps)
    import cv2

    cv2.setNumThreads(1)
    b0 = bgr[0].cpu().numpy()
    cms = cpu_time(lambda: cv2.cvtColor(b0, cv2.COLOR_BGR2Lab), reps=20)
    byt = 6 * rows * cols * nl
    out.append({"row": "cvtColor(BGR2Lab) (main_lc.cpp:182-183), batch of 1024 frames (dcmt_bgr2lab_u8)", "frames": nl, "ms": ms,
                "frames_per_s": nl / ms * 1e3, "ms_per_frame": ms / nl, "achieved_GBps": byt / ms / 1e6, "frac_of_hbm_peak": byt / ms / 1e6 / peak,
                "single_frame_call_ms": ms1, "cv2_1thread_ms_per_frame": cms, "cv2_version": cv2.__version__,
                "note": "6 algorithmic B/px (3 in, 3 out); single_frame_call_ms: one frame per call, L2-resident"})
    del labo
    # ---- evaluation: batch of 256 frames, 8 B/px
    n = 256
    gt = torch.from_numpy(np.stack([synth.sparse_depth(f, rows, cols, 0.3) for f in range(8)])).cuda().repeat(n // 8, 1, 1).contiguous()
    dense = (gt * 1.01 + 0.5).contiguous()
    ms = gpu_time(lambda: api.evaluate(gt, dense, "lidar_camera", lib=lib), a.reps)
    g0, d0 = gt[0].cpu().numpy(), dense[0].cpu().numpy()
    cms = cpu_time(lambda: co.evaluate(g0, d0, 0, 1))
    out.append({"row": "8f#3 evaluate_performance (main_lc.cpp:85-116)", "frames": n, "ms": ms, "frames_per_s": n / ms * 1e3,
                "achieved_GBps": 8 * rows * cols * n / ms / 1e6, "frac_of_hbm_peak": 8 * rows * cols * n / ms / 1e6 / peak,
                "cpu_oracle_ms_per_frame": cms, "note": "includes the read-back of 256 result records"})
    # ---- projection: one 120k-point cloud per call
    pts = torch.from_numpy(synth.velodyne_cloud(0, 120000)).cuda()
    ms = gpu_time(lambda: api.lidar_project(pts, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, rows, cols, lib=lib), a.reps)
    pn = pts.cpu().numpy()
    cms = cpu_time(lambda: co.lidar_project(pn, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, rows, cols))
    out.append({"row": "8f#2 LiDAR projection + normalize (main_sl.cpp:478-523)", "points": 120000, "ms": ms, "clouds_per_s": 1e3 / ms,
                "cpu_oracle_ms_per_cloud": cms, "note": "4 small kernels per cloud: launch-latency bound at this size"})
    # ---- projection, batched: 128 clouds per call in the same four launches
    nb = 128
    clouds = torch.from_numpy(np.stack([synth.velodyne_cloud(f % 8, 120000) for f in range(nb)])).cuda()
    ms = gpu_time(lambda: api.lidar_project_batch(clouds, None, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, rows, cols, lib=lib), max(3, a.reps // 2))
    out.append({"row": "8f#2 LiDAR projection + normalize, batch of 128 clouds (dcmt_lidar_project_batch_f32)", "points": 120000, "ms": ms,
                "clouds_per_s": nb * 1e3 / ms})
    del clouds
    # ---- SLIC: one frame, step 18, 10 iterations
    lab = torch.from_numpy(synth.lab_image(0, rows, cols)).cuda()
    ms = gpu_time(lambda: api.generate_superpixels(lab, 18, 50, lib=lib), a.reps)
    ln = lab.cpu().numpy()
    cms = cpu_time(lambda: co.slic(ln, 18, 50), reps=1)
    out.append({"row": "8f#1 Slic::generate_superpixels (slic.cpp:101-182)", "step": 18, "iterations": 10, "ms": ms, "frames_per_s": 1e3 / ms,
                "cpu_oracle_ms_per_frame": cms})
    labs = torch.from_numpy(np.stack([synth.lab_image(f, rows, cols) for f in range(8)])).cuda().repeat(8, 1, 1, 1).contiguous()
    ms = gpu_time(lambda: api.generate_superpixels(labs, 18, 50, lib=lib), max(3, a.reps // 4))
    out.append({"row": "8f#1 Slic::generate_superpixels, batch of 64 frames", "step": 18, "iterations": 10, "ms": ms, "frames_per_s": 64e3 / ms})
    labs256 = labs.repeat(4, 1, 1, 1).contiguous()
    ms = gpu_time(lambda: api.generate_superpixels(labs256, 18, 50, lib=lib), 3)
    out.append({"row": "8f#1 Slic::generate_superpixels, batch of 256 frames", "step": 18, "iterations": 10, "ms": ms, "frames_per_s": 256e3 / ms})
    del labs256
    # ---- the DC_lidar_camera chain on device: SLIC -> guided completion -> evaluation, one frame (main_lc.cpp:184-225)
    sparse = torch.from_numpy(synth.sparse_depth(0, rows, cols, 0.05)).cuda()
    k = lib.dcmt_slic_center_count(rows, cols, 18)

    def chain():
        labels = api.generate_superpixels(lab, 18, 50, lib=lib)
        d = api.interpolate_with_superpixels(labels, sparse, "gaussian", 1, n_clusters=k, lib=lib)
        return api.evaluate(sparse, d, "lidar_camera", lib=lib)
    ms = gpu_time(chain, max(3, a.reps // 4))
    out.append({"row": "DC_lidar_camera chain: SLIC -> interpolate_with_superpixels -> evaluate_performance (main_lc.cpp:184-225)", "ms": ms,
                "frames_per_s": 1e3 / ms})
    sparse64 = torch.from_numpy(np.stack([synth.sparse_depth(f, rows, cols, 0.05) for f in range(8)])).cuda().repeat(8, 1, 1).contiguous()

    def chain64():
        labels = api.generate_superpixels(labs, 18, 50, lib=lib)
        d = api.interpolate_with_superpixels(labels, sparse64, "gaussian", 1, n_clusters=k, lib=lib)
        return api.evaluate(sparse64, d, "lidar_camera", lib=lib)
    ms = gpu_time(chain64, 3)
    out.append({"row": "DC_lidar_camera chain, batch of 64 frames", "ms": ms, "frames_per_s": 64e3 / ms})
    # ---- the same front from the BGR frame as read: cvtColor(BGR2Lab) -> SLIC -> guided completion -> evaluation
    # (main_lc.cpp:182-225), the conversion inside dcmt_slic_bgr_u8c3; next to the Lab-in chain on the same batches
    for nf in (64, 256):
        bgrs = bgr[:nf].contiguous()
        labs_n = api.bgr2lab(bgrs, lib=lib)
        sp = sparse64.repeat(nf // 64, 1, 1).contiguous()

        def chain_bgr():
            labels = api.generate_superpixels_bgr(bgrs, 18, 50, lib=lib)
            d = api.interpolate_with_superpixels(labels, sp, "gaussian", 1, n_clusters=k, lib=lib)
            return api.evaluate(sp, d, "lidar_camera", lib=lib)

        def chain_lab():
            labels = api.generate_superpixels(labs_n, 18, 50, lib=lib)
            d = api.interpolate_with_superpixels(labels, sp, "gaussian", 1, n_clusters=k, lib=lib)
            return api.evaluate(sp, d, "lidar_camera", lib=lib)
        ms_lab = gpu_time(chain_lab, 3)
        ms_bgr = gpu_time(chain_bgr, 3)
        out.append({"row": f"DC_lidar_camera chain from BGR: BGR2Lab -> SLIC -> interpolate_with_superpixels -> evaluate, batch of {nf} frames",
                    "ms": ms_bgr, "frames_per_s": nf * 1e3 / ms_bgr, "lab_in_chain_ms": ms_lab, "lab_in_chain_frames_per_s": nf * 1e3 / ms_lab,
                    "added_by_conversion": ms_bgr / ms_lab - 1})
    for o in out:
        print(json.dumps(o), flush=True)


if __name__ == "__main__":
    main()
