"""Evaluation on KITTI uint16 ground truth against the float32 evaluation: device and host rates of the three instantiations of
k_eval_partial, next to each other.

Workload: 1024 frames of 352x1216 per call (64 unique frames x 16; 1.75 GB per float32 plane, well past the 126 MB L2),
GT at 30 % valid pixels (synth.sparse_depth_q8), results completed from 5 % sparse input with blur none and stored both as
float32 and as KITTI uint16, mode DCMT_EVAL_BOTH_VALID with tolerance 0 (main_lc.cpp:85-116).  Legs, alternating three
times:
  - device: dcmt_evaluate_f32 (GT u / 256, 8 B/px), dcmt_evaluate_u16 (6 B/px), dcmt_evaluate_u16_u16 (4 B/px); CUDA events;
    bytes/s from the bytes the planes hold, over the HBM peak of the data sheet (7.7 TB/s);
  - host, page-locked buffers: the *_host variants of the same, perf_counter around calls that synchronise.
Every timed call's records are checked: the uint16 calls must be byte-equal to the float32 call on the decoded planes.
With --parent-lib PATH (a libdcmt.so built from another commit), its dcmt_evaluate_f32 / _host are timed in the same
alternation, and its records must be byte-identical to this build's -- on the benchmark's frames and on the inputs of
tests/test_evaluate_u16.py.  Prints one JSON line with the GPU's name, power limit and maximum SM clock read in the same run.
Usage: python tools/bench_eval_u16.py [--steps K] [--warmup W] [--parent-lib PATH]"""
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

ROWS, COLS, N, UNIQUE = 352, 1216, 1024, 64
MODE, TOL = api.EVAL_VARIANTS["lidar_camera"]
HBM_PEAK = 7.7e12  # bytes/s, NVIDIA's HGX B200 data sheet, one GPU
REC_BYTES = C.sizeof(_lib.EvalResult)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable: " + r.stderr.strip()


def bind_parent_f32(path):
    """dcmt_evaluate_f32 and _host of another build (its binding may lack this build's entry points)"""
    cdll = C.CDLL(path)
    f, h = cdll.dcmt_evaluate_f32, cdll.dcmt_evaluate_f32_host
    f.restype = h.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p]
    h.argtypes = f.argtypes[:-1]
    return f, h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--parent-lib", default=None)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "bench_eval_u16 needs a CUDA device"
    lib = _lib.load()
    parent = bind_parent_f32(args.parent_lib) if args.parent_lib else None
    dev = torch.device("cuda:0")
    reps = N // UNIQUE
    gt16 = np.stack([synth.sparse_depth_q8(1000 + f, ROWS, COLS, 0.3) for f in range(UNIQUE)])
    sparse = np.stack([synth.sparse_depth_q8(f, ROWS, COLS, 0.05) for f in range(UNIQUE)])
    r16 = api.img_completion(sparse, False, "none", out_dtype=np.uint16, lib=lib)  # lossless with blur none: r32 = r16 / 256

    def pinned(unique):  # the 64 unique frames repeated to N, in page-locked memory
        t = torch.empty((N, ROWS, COLS), dtype=torch.uint16 if unique.dtype == np.uint16 else torch.float32, pin_memory=True)
        t.numpy().reshape(reps, UNIQUE, ROWS, COLS)[...] = unique
        return t

    h_g16, h_r16 = pinned(gt16), pinned(r16)
    h_g32, h_r32 = pinned(gt16.astype(np.float32) / np.float32(256)), pinned(r16.astype(np.float32) / np.float32(256))
    d_g16, d_r16, d_g32, d_r32 = (t.to(dev) for t in (h_g16, h_r16, h_g32, h_r32))
    st = lambda: int(torch.cuda.current_stream().cuda_stream)
    d_res = {k: torch.empty((N, REC_BYTES), dtype=torch.uint8, device=dev) for k in ("f32", "u16", "u16_u16", "parent_f32")}
    px = ROWS * COLS
    calls = {
        "f32": (8, lambda: lib.check(lib.dcmt_evaluate_f32(d_g32.data_ptr(), d_r32.data_ptr(), ROWS, COLS, 0, 0, N, TOL, MODE,
                                                             d_res["f32"].data_ptr(), st()))),
        "u16": (6, lambda: lib.check(lib.dcmt_evaluate_u16(d_g16.data_ptr(), d_r32.data_ptr(), ROWS, COLS, 0, 0, 0, 0, N, TOL, MODE,
                                                             d_res["u16"].data_ptr(), st()))),
        "u16_u16": (4, lambda: lib.check(lib.dcmt_evaluate_u16_u16(d_g16.data_ptr(), d_r16.data_ptr(), ROWS, COLS, 0, 0, 0, 0, N, TOL,
                                                                     MODE, d_res["u16_u16"].data_ptr(), st()))),
    }
    if parent:
        calls["parent_f32"] = (8, lambda: lib.check(parent[0](d_g32.data_ptr(), d_r32.data_ptr(), ROWS, COLS, 0, 0, N, TOL, MODE,
                                                              d_res["parent_f32"].data_ptr(), st())))

    def dev_seconds(fn):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / args.steps

    runs = {k: [] for k in calls}
    for _ in range(3):
        for k, (_, fn) in calls.items():
            runs[k].append(N / dev_seconds(fn))
    res = {"gpu": gpu_info(), "workload": f"{N} frames of {ROWS}x{COLS} per call ({UNIQUE} unique x {reps}), GT 30 % valid, "
           f"mode {MODE} tolerance {TOL:g}", "steps": args.steps, "warmup": args.warmup, "unit": "frames/s", "device": {}}
    for k, (bpp, _) in calls.items():
        fps = max(runs[k])
        res["device"][k] = {"frames_per_s": fps, "runs": runs[k], "bytes_per_px": bpp, "bytes_per_s": fps * px * bpp,
                            "frac_of_hbm_peak": fps * px * bpp / HBM_PEAK}
    rec = {k: v.cpu().numpy().tobytes() for k, v in d_res.items() if k in calls}
    checks = {"device_u16_equals_f32": rec["u16"] == rec["f32"], "device_u16_u16_equals_f32": rec["u16_u16"] == rec["f32"]}
    if parent:
        checks["device_f32_equals_parent"] = rec["parent_f32"] == rec["f32"]

    # host variants on page-locked buffers
    del d_g16, d_r16, d_g32, d_r32
    torch.cuda.empty_cache()
    h_res = {k: np.zeros(N * REC_BYTES, np.uint8) for k in calls}
    p = lambda t: t.data_ptr()
    hcalls = {
        "f32": lambda: lib.check(lib.dcmt_evaluate_f32_host(p(h_g32), p(h_r32), ROWS, COLS, 0, 0, N, TOL, MODE, h_res["f32"].ctypes.data)),
        "u16": lambda: lib.check(lib.dcmt_evaluate_u16_host(p(h_g16), p(h_r32), ROWS, COLS, 0, 0, 0, 0, N, TOL, MODE, h_res["u16"].ctypes.data)),
        "u16_u16": lambda: lib.check(lib.dcmt_evaluate_u16_u16_host(p(h_g16), p(h_r16), ROWS, COLS, 0, 0, 0, 0, N, TOL, MODE,
                                                                    h_res["u16_u16"].ctypes.data)),
    }
    if parent:
        hcalls["parent_f32"] = lambda: lib.check(parent[1](p(h_g32), p(h_r32), ROWS, COLS, 0, 0, N, TOL, MODE, h_res["parent_f32"].ctypes.data))
    hsteps = max(1, args.steps // 4)

    def host_seconds(fn):
        for _ in range(max(1, args.warmup // 2)):
            fn()
        t0 = time.perf_counter()
        for _ in range(hsteps):
            fn()
        return (time.perf_counter() - t0) / hsteps  # the *_host calls return after their device-to-host copy

    hruns = {k: [] for k in hcalls}
    for _ in range(3):
        for k, fn in hcalls.items():
            hruns[k].append(N / host_seconds(fn))
    res["host"] = {k: {"frames_per_s": max(v), "runs": v, "staged_bytes_per_px": calls[k][0]} for k, v in hruns.items()}
    res["host_steps"] = hsteps
    checks["host_u16_equals_f32"] = h_res["u16"].tobytes() == h_res["f32"].tobytes()
    checks["host_u16_u16_equals_f32"] = h_res["u16_u16"].tobytes() == h_res["f32"].tobytes()
    checks["host_equals_device"] = h_res["f32"].tobytes() == rec["f32"]
    if parent:
        checks["host_f32_equals_parent"] = h_res["parent_f32"].tobytes() == h_res["f32"].tobytes()
        checks["test_inputs_f32_equal_parent"] = parent_on_test_inputs(lib, parent, torch)
    res["checks"] = checks
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if not all(checks.values()):
        sys.exit(1)


def parent_on_test_inputs(lib, parent, torch):
    """dcmt_evaluate_f32 of both builds on the float32 planes of tests/test_evaluate_u16.py (layouts and all 65 536 codes)"""
    from tests import test_evaluate_u16 as t

    cases = []
    for k, (name, layout) in enumerate(t.LAYOUTS.items()):
        rows, cols, pitch, fstride, offset, n = layout()
        gt, r32, r16 = t.frames(100 + k, n, rows, cols, empty=3 if name == "batch_with_empty" else None)
        cases += [(t.decode(gt), r32, pitch, fstride, offset), (t.decode(gt), t.decode(r16), pitch, fstride, offset)]
    codes = np.arange(65536, dtype=np.uint16).reshape(1, 256, 256)
    cases.append((t.decode(codes), np.random.default_rng(3).uniform(0.0, 300.0, codes.shape).astype(np.float32), 256, 65536, 0))
    same = True
    for g, r, pitch, fstride, offset in cases:
        n, rows, cols = g.shape
        bg = t.Buf(t.place(g, pitch, fstride, offset), True, offset)
        br = t.Buf(t.place(r, pitch, fstride, offset), True, offset)
        for mode, tol in api.EVAL_VARIANTS.values():
            out = []
            for fn in (lib.dcmt_evaluate_f32, parent[0]):
                res = torch.zeros(n * REC_BYTES, dtype=torch.uint8, device="cuda")
                assert 0 == fn(bg.ptr, br.ptr, rows, cols, pitch * 4, fstride * 4, n, float(tol), mode, res.data_ptr(), None)
                torch.cuda.synchronize()
                out.append(res.cpu().numpy().tobytes())
            same = same and out[0] == out[1]
    return same


if __name__ == "__main__":
    main()
