"""KITTI uint16 output against float32 output: device-resident and host end-to-end rates, each next to its copy ceiling.

Workload: 352x1216 frames at 5 % valid pixels, gaussian blur, 1024 frames per step built as bench.py builds them (64 unique
frames x 16).  Legs:
  - device-resident a1: dcmt_img_completion_u16 (u16 -> f32) against dcmt_img_completion_u16_u16 (u16 -> u16), CUDA events;
  - host a1 with page-locked buffers: the *_host variants of the same, each with its copy ceiling (dcmt_debug_host_copy_u16 /
    _u16_u16: the same buffers, chunks and streams with the kernels left out; the faster of a run before and after the leg);
  - host guided: dcmt_interpolate_with_superpixels_ex_f32_host (f32 -> f32) against _u16_u16_host, grid superpixels.
Every uint16 output of a timed run is checked against the rule (round half to even, clamp, NaN -> 0) applied to the float32
output of the matching timed run, for the whole batch.  Prints one JSON line, with the GPU's name, power limit and maximum SM
clock read in the same run.  Usage: python tools/bench_kitti_io.py [--steps K] [--warmup W]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from depth_completion_mt_b200 import _lib, api, synth  # noqa: E402

ROWS, COLS, N, UNIQUE = 352, 1216, 1024, 64


def rule_u16(t):
    """the conversion rule on a float32 CUDA tensor, in torch (round half to even, clamp to [0, 65535], NaN -> 0)"""
    import torch

    s = t * 256.0
    return torch.where(torch.isnan(s), torch.zeros_like(s), torch.round(s).clamp(0, 65535)).to(torch.int32)


def as_i32(t):
    """uint16 tensor -> int32 values (through int16, whose casts every torch build has)"""
    import torch

    return t.view(torch.int16).to(torch.int32) & 0xFFFF


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable: " + r.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "bench_kitti_io needs a CUDA device"
    lib = _lib.load()
    dev = torch.device("cuda:0")
    reps = N // UNIQUE
    u16 = np.tile(np.stack([synth.sparse_depth_q8(f, ROWS, COLS, 0.05) for f in range(UNIQUE)]), (reps, 1, 1))
    labs = np.tile(np.stack([synth.superpixel_labels(f, ROWS, COLS)[0] for f in range(UNIQUE)]), (reps, 1, 1))
    k = synth.superpixel_labels(0, ROWS, COLS)[1]
    d_in = torch.from_numpy(u16).to(dev)
    out_f = torch.empty((N, ROWS, COLS), dtype=torch.float32, device=dev)
    out_u = torch.empty((N, ROWS, COLS), dtype=torch.uint16, device=dev)

    def dev_rate(fn):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return N * args.steps / (e0.elapsed_time(e1) / 1e3)

    res = {"gpu": gpu_info(), "workload": f"a1/a2 {N} frames of {ROWS}x{COLS} per step ({UNIQUE} unique x {reps}), 5 % valid, gaussian",
           "steps": args.steps, "warmup": args.warmup, "unit": "frames/s"}
    a1_f = lambda: api.img_completion(d_in, False, "gaussian", out=out_f, lib=lib)
    a1_u = lambda: api.img_completion(d_in, False, "gaussian", out=out_u, out_dtype=torch.uint16, lib=lib)
    fps_f, fps_u = [], []
    for _ in range(3):  # alternating
        fps_f.append(dev_rate(a1_f))
        fps_u.append(dev_rate(a1_u))
    res["device_u16_f32"], res["device_u16_u16"] = max(fps_f), max(fps_u)
    res["device_runs"] = {"u16_f32": fps_f, "u16_u16": fps_u}
    checks = {"device_a1": bool(torch.equal(rule_u16(out_f), as_i32(out_u)))}

    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype, pin_memory=True)

    def host_rate(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return N * args.steps / (time.perf_counter() - t0)

    h_in = pinned((N, ROWS, COLS), torch.uint16)
    h_in.copy_(d_in)
    h_out_f, h_out_u = pinned((N, ROWS, COLS), torch.float32), pinned((N, ROWS, COLS), torch.uint16)
    np_in, np_f, np_u = h_in.numpy(), h_out_f.numpy(), h_out_u.numpy()
    copy_f = lambda: lib.check(lib.dcmt_debug_host_copy_u16(np_in.ctypes.data, np_f.ctypes.data, ROWS, COLS, N, None, 0))
    copy_u = lambda: lib.check(lib.dcmt_debug_host_copy_u16_u16(np_in.ctypes.data, np_u.ctypes.data, ROWS, COLS, N, None, 0))
    # the copy-only ceilings overwrite the output buffers: the outputs of each timed leg are kept on the device first
    ceil_f = host_rate(copy_f)
    e2e_f = host_rate(lambda: api.img_completion(np_in, False, "gaussian", out=np_f, lib=lib))
    host_f = h_out_f.to(dev)
    ceil_f = max(ceil_f, host_rate(copy_f))
    ceil_u = host_rate(copy_u)
    checks["copy_u16_u16_echoes"] = bool(np.array_equal(np_u, np_in))
    e2e_u = host_rate(lambda: api.img_completion(np_in, False, "gaussian", out=np_u, out_dtype=np.uint16, lib=lib))
    host_u = as_i32(h_out_u.to(dev))
    ceil_u = max(ceil_u, host_rate(copy_u))
    res["host_u16_f32"] = {"e2e": e2e_f, "copy_ceiling": ceil_f, "frac_of_copy_ceiling": e2e_f / ceil_f, "api": "dcmt_img_completion_u16_host"}
    res["host_u16_u16"] = {"e2e": e2e_u, "copy_ceiling": ceil_u, "frac_of_copy_ceiling": e2e_u / ceil_u, "api": "dcmt_img_completion_u16_u16_host"}
    checks["host_a1"] = bool(torch.equal(rule_u16(host_f), host_u))
    checks["host_equals_device_a1"] = bool(torch.equal(host_u, as_i32(out_u)))
    del host_f, host_u

    h_f32 = pinned((N, ROWS, COLS), torch.float32)
    h_f32.numpy()[...] = u16.astype(np.float32) / np.float32(256)
    h_lab = pinned((N, ROWS, COLS), torch.int32)
    h_lab.copy_(torch.from_numpy(labs))
    np_f32, np_lab = h_f32.numpy(), h_lab.numpy()
    np_f[...] = 0
    np_u[...] = 0
    g_f = host_rate(lambda: api.interpolate_with_superpixels(np_lab, np_f32, "gaussian", 1, n_clusters=k, out=np_f, lib=lib))
    g_u = host_rate(lambda: api.interpolate_with_superpixels(np_lab, np_in, "gaussian", 1, n_clusters=k, out=np_u, out_dtype=np.uint16, lib=lib))
    res["host_guided_f32_f32"] = {"e2e": g_f, "api": "dcmt_interpolate_with_superpixels_ex_f32_host", "bytes_per_px_pcie": 12}
    res["host_guided_u16_u16"] = {"e2e": g_u, "api": "dcmt_interpolate_with_superpixels_u16_u16_host", "bytes_per_px_pcie": 8}
    checks["host_guided"] = bool(torch.equal(rule_u16(h_out_f.to(dev)), as_i32(h_out_u.to(dev))))
    res["outputs_follow_rule"] = checks
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if not all(checks.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
