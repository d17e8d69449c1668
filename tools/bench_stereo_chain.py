"""The stereo program's per-frame chain in one call (dcmt_stereo_chain_f32*) against the calls it replaces.

Workload: 352x1216 frames, 120 000-point synth.velodyne_cloud clouds under the KITTI calibration of synth, synth.bgr_image
left frames with the right frame shifted by 3 columns, step 65 (100 superpixels), nc 40, 10 SLIC iterations, the main_sl.cpp
refinement parameters; 64 unique frames tiled.
  - device: 1024 device-resident frames per call (2 GB of clouds, 2.6 GB of BGR: well past the 126 MB L2); the device
    entry point against the device composition in 128-frame pieces (bench.py --workload stereo_chain's piece size):
    dcmt_lidar_project_batch_f32, dcmt_slic_bgr_u8c3, dcmt_interpolate_with_superpixels_ex_f32 (DCMT_PATH_RANK),
    dcmt_bgr2gray_u8 twice, dcmt_stereo_refine_f32.  frames/s from CUDA events over --steps calls after --warmup, best of
    three alternating rounds.
  - host: 512 frames in page-locked buffers (dcmt_host_alloc), copies inside the timed region (the calls return
    synchronised): _host against the six host calls (dcmt_lidar_project_f32_host per cloud, dcmt_slic_bgr_u8c3_host,
    dcmt_interpolate_with_superpixels_ex_f32_host, dcmt_bgr2gray_u8_host twice, dcmt_stereo_refine_f32_host).  Bytes over
    the host links per pixel from shapes: 10.5 in (cloud 4.5 + two BGR frames) and 4 out against 27.5 in and 18 out.
  - multi-device: _host_multi on 1 / 2 / 4 / 8 GPUs where the box has them, 1024 frames per call.
Checks in the same run: every chained result is byte-equal to its composition.  Prints one JSON line with the GPU's name,
power limit and SM clocks read in the same run.
Usage: python tools/bench_stereo_chain.py [--steps K] [--warmup W]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from depth_completion_mt_b200 import _lib, api, synth  # noqa: E402

ROWS, COLS, UNIQUE, N_DEV, N_HOST, STEP, NC, ITERS, NPTS, PIECE = 352, 1216, 64, 1024, 512, 65, 40, 10, 120000, 128
PX = ROWS * COLS
RANK = 3
CLOUD_B = NPTS * 16 / PX
LINK_BYTES = {"one_call": (CLOUD_B + 6, 4), "six_calls": (CLOUD_B + 23, 18)}  # per pixel over the host links: in, out


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines() if r.returncode == 0 and r.stdout.strip() else ["unavailable: " + r.stderr.strip()]


def best_of_three(fa, fb):
    a, b = [], []
    for _ in range(3):
        a.append(fa())
        b.append(fb())
    return a, b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "bench_stereo_chain needs a CUDA device"
    res = {"gpu": gpu_info(), "shape": [ROWS, COLS], "points": NPTS, "step": STEP, "nc": NC, "iterations": ITERS}
    lib = _lib.load()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    T = np.ascontiguousarray(synth.KITTI_T_VELO_TO_CAM, np.float32)
    P = np.ascontiguousarray(synth.KITTI_P_RECT_02, np.float32)
    pts_u = np.stack([synth.velodyne_cloud(f, NPTS) for f in range(UNIQUE)])
    left_u = np.stack([synth.bgr_image(f, ROWS, COLS) for f in range(UNIQUE)])
    right_u = np.roll(left_u, -3, axis=2).copy()
    k = lib.dcmt_slic_center_count(ROWS, COLS, STEP)
    prm = api.stereo_params(lib=lib)
    stream = torch.cuda.current_stream().cuda_stream
    pT, pP = T.ctypes.data, P.ctypes.data

    # ---- device-resident: one call against the device composition
    reps = N_DEV // UNIQUE
    tp = torch.from_numpy(pts_u).to(dev).repeat(reps, 1, 1).contiguous()
    tl = torch.from_numpy(left_u).to(dev).repeat(reps, 1, 1, 1).contiguous()
    tr = torch.from_numpy(right_u).to(dev).repeat(reps, 1, 1, 1).contiguous()
    o1 = torch.empty((N_DEV, ROWS, COLS), dtype=torch.float32, device=dev)
    o2 = torch.empty_like(o1)
    nrm = torch.empty((PIECE, ROWS, COLS), dtype=torch.float32, device=dev)
    dense = torch.empty_like(nrm)
    labels = torch.empty((PIECE, ROWS, COLS), dtype=torch.int32, device=dev)
    gl = torch.empty((PIECE, ROWS, COLS), dtype=torch.uint8, device=dev)
    gr = torch.empty_like(gl)

    def run_one():
        lib.check(lib.dcmt_stereo_chain_f32(tp.data_ptr(), None, NPTS, NPTS, pT, pP, 0.0, 80.0, tl.data_ptr(), tr.data_ptr(), 0, 0, o1.data_ptr(),
                                            None, ROWS, COLS, N_DEV, STEP, NC, ITERS, 1, 0, C.byref(prm), None, stream))

    def run_composition():
        for c0 in range(0, N_DEV, PIECE):
            n = min(PIECE, N_DEV - c0)
            lib.check(lib.dcmt_lidar_project_batch_f32(tp[c0].data_ptr(), None, NPTS, NPTS, n, pT, pP, ROWS, COLS, None, nrm.data_ptr(), 0.0, 80.0,
                                                       None, stream))
            lib.check(lib.dcmt_slic_bgr_u8c3(tl[c0].data_ptr(), ROWS, COLS, n, STEP, NC, ITERS, labels.data_ptr(), None, stream))
            lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32(nrm.data_ptr(), labels.data_ptr(), k, dense.data_ptr(), ROWS, COLS, 0, 0, n, 1,
                                                                   RANK, None, stream))
            lib.check(lib.dcmt_bgr2gray_u8(tl[c0].data_ptr(), gl.data_ptr(), ROWS, COLS, 0, 0, n, stream))
            lib.check(lib.dcmt_bgr2gray_u8(tr[c0].data_ptr(), gr.data_ptr(), ROWS, COLS, 0, 0, n, stream))
            lib.check(lib.dcmt_stereo_refine_f32(dense.data_ptr(), gl.data_ptr(), gr.data_ptr(), o2[c0].data_ptr(), None, ROWS, COLS, n,
                                                 C.byref(prm), stream))

    def timed_dev(fn):
        def run():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            e1.synchronize()
            return N_DEV * args.steps / (e0.elapsed_time(e1) / 1e3)
        return run

    for _ in range(args.warmup):
        run_one()
        run_composition()
    torch.cuda.synchronize()
    equal = bool(torch.equal(o1.view(torch.int32), o2.view(torch.int32)))
    a, b = best_of_three(timed_dev(run_one), timed_dev(run_composition))
    res["device_resident"] = {"frames": N_DEV, "one_call_fps": round(max(a)), "composition_fps": round(max(b)), "rounds_one": [round(v) for v in a],
                              "rounds_composition": [round(v) for v in b], "byte_equal": equal}
    print(f"device: one call {max(a):.0f} frames/s, composition {max(b):.0f} frames/s, equal {equal}", file=sys.stderr)
    del tp, tl, tr, o1, o2, nrm, dense, labels, gl, gr
    torch.cuda.empty_cache()
    lib.dcmt_release_workspaces()

    # ---- host end to end, page-locked buffers
    def tile(x, n):
        return np.concatenate([x] * ((n + len(x) - 1) // len(x)))[:n]

    bufs = {}

    def hbuf(name, shape, dt):
        bufs[name] = api.HostBuffer(shape, dt, lib=lib)
        return bufs[name].array

    hp, hl, hr = hbuf("p", (N_DEV, NPTS, 4), np.float32), hbuf("l", (N_DEV, ROWS, COLS, 3), np.uint8), hbuf("r", (N_DEV, ROWS, COLS, 3), np.uint8)
    hp[...], hl[...], hr[...] = tile(pts_u, N_DEV), tile(left_u, N_DEV), tile(right_u, N_DEV)
    h1, h2 = hbuf("o1", (N_DEV, ROWS, COLS), np.float32), hbuf("o2", (N_HOST, ROWS, COLS), np.float32)
    hn, hd = hbuf("n", (N_HOST, ROWS, COLS), np.float32), hbuf("d", (N_HOST, ROWS, COLS), np.float32)
    hlab = hbuf("lab", (N_HOST, ROWS, COLS), np.int32)
    hgl, hgr = hbuf("gl", (N_HOST, ROWS, COLS), np.uint8), hbuf("gr", (N_HOST, ROWS, COLS), np.uint8)
    fpx = PX

    def run_host_one(n=N_HOST):
        lib.check(lib.dcmt_stereo_chain_f32_host(hp.ctypes.data, None, NPTS, NPTS, pT, pP, 0.0, 80.0, hl.ctypes.data, hr.ctypes.data, 0, 0,
                                                 h1.ctypes.data, None, ROWS, COLS, n, STEP, NC, ITERS, 1, 0, C.byref(prm), None))

    def run_host_six():
        for f in range(N_HOST):
            lib.check(lib.dcmt_lidar_project_f32_host(hp[f].ctypes.data, NPTS, pT, pP, ROWS, COLS, None, hn.ctypes.data + f * fpx * 4, 0.0, 80.0,
                                                      None))
        lib.check(lib.dcmt_slic_bgr_u8c3_host(hl.ctypes.data, ROWS, COLS, N_HOST, STEP, NC, ITERS, hlab.ctypes.data, None))
        lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32_host(hn.ctypes.data, hlab.ctypes.data, k, hd.ctypes.data, ROWS, COLS, 0, 0, N_HOST,
                                                                    1, RANK, None))
        lib.check(lib.dcmt_bgr2gray_u8_host(hl.ctypes.data, hgl.ctypes.data, ROWS, COLS, 0, 0, N_HOST))
        lib.check(lib.dcmt_bgr2gray_u8_host(hr.ctypes.data, hgr.ctypes.data, ROWS, COLS, 0, 0, N_HOST))
        lib.check(lib.dcmt_stereo_refine_f32_host(hd.ctypes.data, hgl.ctypes.data, hgr.ctypes.data, h2.ctypes.data, None, ROWS, COLS, N_HOST,
                                                  C.byref(prm)))

    def timed_host(fn, n):
        def run():
            t0 = time.perf_counter()
            for _ in range(args.steps):
                fn()
            return n * args.steps / (time.perf_counter() - t0)
        return run

    for _ in range(args.warmup):
        run_host_one()
        run_host_six()
    equal = bool(np.array_equal(h1[:N_HOST].view(np.int32), h2.view(np.int32)))
    a, b = best_of_three(timed_host(run_host_one, N_HOST), timed_host(run_host_six, N_HOST))
    host = {"frames": N_HOST, "one_call_fps": round(max(a)), "six_calls_fps": round(max(b)), "rounds_one": [round(v) for v in a],
            "rounds_six": [round(v) for v in b], "byte_equal": equal,
            "link_bytes_per_px": {k2: {"in": round(v[0], 2), "out": v[1]} for k2, v in LINK_BYTES.items()}}
    host["one_call_link_GBps"] = round(max(a) * PX * sum(LINK_BYTES["one_call"]) / 1e9, 1)
    host["six_calls_link_GBps"] = round(max(b) * PX * sum(LINK_BYTES["six_calls"]) / 1e9, 1)
    res["host"] = host
    print(f"host: one call {max(a):.0f} frames/s, six calls {max(b):.0f} frames/s, equal {equal}", file=sys.stderr)

    # ---- multi-device, 1024 frames per call, against the one-device _host result of the same frames
    run_host_one(N_DEV)
    ref = h1.copy()
    multi = {}
    n_gpu = torch.cuda.device_count()
    for nd in (1, 2, 4, 8):
        if nd > n_gpu:
            multi[str(nd)] = "not measured: the box has %d GPU(s)" % n_gpu
            continue

        def run_multi():
            lib.check(lib.dcmt_stereo_chain_f32_host_multi(hp.ctypes.data, None, NPTS, NPTS, pT, pP, 0.0, 80.0, hl.ctypes.data, hr.ctypes.data, 0, 0,
                                                           h1.ctypes.data, None, ROWS, COLS, N_DEV, STEP, NC, ITERS, 1, 0, C.byref(prm), None, None,
                                                           nd))

        for _ in range(args.warmup):
            run_multi()
        equal = bool(np.array_equal(h1.view(np.int32), ref.view(np.int32)))
        t = [timed_host(run_multi, N_DEV)() for _ in range(3)]
        multi[str(nd)] = {"fps": round(max(t)), "rounds": [round(v) for v in t], "byte_equal": equal}
        print(f"multi {nd}: {max(t):.0f} frames/s, equal {equal}", file=sys.stderr)
    res["host_multi"] = multi
    for hb in bufs.values():
        hb.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
