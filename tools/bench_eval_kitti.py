"""The KITTI benchmark's figures (dcmt_evaluate_kitti_*) next to the reductions of the same type pair (dcmt_evaluate_*,
mode DCMT_EVAL_GT_VALID, tolerance 0): device rates of the three instantiations of k_kitti_partial and k_eval_partial.

Workload: 1024 device-resident frames of 352x1216 per call (64 unique frames x 16; 1.75 GB per float32 plane, well past
the 126 MB L2), KITTI-like GT at 30 % valid pixels (synth.sparse_depth_q8(..., kitti_like=True): the upper 35 % empty).
Two predictions:
  - dense: the library's own completed outputs (blur none, so the float32 plane is exactly the uint16 one / 256);
  - sparse: 5 %-valid maps, where nearly every GT pixel goes through the background interpolation.
Per call: frames/s from CUDA events over --steps calls after --warmup, best of three alternating rounds, and GB/s at the
algorithmic 8 / 6 / 4 bytes per pixel (float32 pair, uint16 GT with float32 prediction, uint16 pair) over the HBM peak of
the data sheet (7.7 TB/s).  Checks in the same run: the uint16 calls give the bytes of the float32 call on the decoded
planes, and on the dense prediction n_gt / sum_abs / sum_sq are the bytes of the reductions' count / sum_abs / sum_sq.
Prints one JSON line with the GPU's name, power limit and maximum SM clock read in the same run.
Usage: python tools/bench_eval_kitti.py [--steps K] [--warmup W]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from depth_completion_mt_b200 import _lib, api, synth  # noqa: E402

ROWS, COLS, N, UNIQUE = 352, 1216, 1024, 64
HBM_PEAK = 7.7e12  # bytes/s, NVIDIA's HGX B200 data sheet, one GPU
K_BYTES, E_BYTES = C.sizeof(_lib.KittiMetrics), C.sizeof(_lib.EvalResult)
PAIRS = {"f32": 8, "u16": 6, "u16_u16": 4}  # bytes per pixel the two planes hold


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable: " + r.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "bench_eval_kitti needs a CUDA device"
    res = {"gpu": gpu_info()}
    lib = _lib.load()
    dev = torch.device("cuda:0")
    reps = N // UNIQUE
    gt16 = np.stack([synth.sparse_depth_q8(1000 + f, ROWS, COLS, 0.3, kitti_like=True) for f in range(UNIQUE)])
    sparse_in = np.stack([synth.sparse_depth_q8(f, ROWS, COLS, 0.05, kitti_like=True) for f in range(UNIQUE)])
    preds16 = {
        "dense": api.img_completion(sparse_in, False, "none", out_dtype=np.uint16, lib=lib),
        "sparse": np.stack([synth.sparse_depth_q8(2000 + f, ROWS, COLS, 0.05) for f in range(UNIQUE)]),
    }

    def on_device(unique):  # the unique frames repeated to N
        t = torch.from_numpy(np.ascontiguousarray(unique)).to(dev)
        return t.repeat(reps, 1, 1)

    d_g16 = on_device(gt16)
    d_g32 = on_device(gt16.astype(np.float32) / np.float32(256))
    st = lambda: int(torch.cuda.current_stream().cuda_stream)
    px = ROWS * COLS
    k_res = {k: torch.empty((N, K_BYTES), dtype=torch.uint8, device=dev) for k in PAIRS}
    e_res = {k: torch.empty((N, E_BYTES), dtype=torch.uint8, device=dev) for k in PAIRS}

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

    res.update({"workload": f"{N} frames of {ROWS}x{COLS} per call ({UNIQUE} unique x {reps}), KITTI-like GT 30 % valid",
                "steps": args.steps, "warmup": args.warmup, "unit": "frames/s"})
    checks = {}
    for pname, p16 in preds16.items():
        d_r16 = on_device(p16)
        d_r32 = on_device(p16.astype(np.float32) / np.float32(256))
        planes = {"f32": (d_g32, d_r32), "u16": (d_g16, d_r32), "u16_u16": (d_g16, d_r16)}
        calls = {}
        for k, (g, r) in planes.items():
            kf = getattr(lib, "dcmt_evaluate_kitti_" + k)
            ef = getattr(lib, "dcmt_evaluate_" + k)
            calls["kitti_" + k] = lambda kf=kf, g=g, r=r, k=k: lib.check(
                kf(g.data_ptr(), r.data_ptr(), ROWS, COLS, 0, 0, 0, 0, N, k_res[k].data_ptr(), st()))
            if k == "f32":
                calls["eval_" + k] = lambda ef=ef, g=g, r=r, k=k: lib.check(
                    ef(g.data_ptr(), r.data_ptr(), ROWS, COLS, 0, 0, N, 0.0, 0, e_res[k].data_ptr(), st()))
            else:
                calls["eval_" + k] = lambda ef=ef, g=g, r=r, k=k: lib.check(
                    ef(g.data_ptr(), r.data_ptr(), ROWS, COLS, 0, 0, 0, 0, N, 0.0, 0, e_res[k].data_ptr(), st()))
        runs = {k: [] for k in calls}
        for _ in range(3):
            for k, fn in calls.items():
                runs[k].append(N / dev_seconds(fn))
        out = {}
        for k, v in runs.items():
            bpp = PAIRS[k.split("_", 1)[1]]
            fps = max(v)
            out[k] = {"frames_per_s": fps, "runs": v, "bytes_per_px": bpp, "GB_per_s": fps * px * bpp / 1e9,
                      "frac_of_hbm_peak": fps * px * bpp / HBM_PEAK}
        res[pname] = out
        torch.cuda.synchronize()
        krec = {k: v.cpu().numpy().view(api.KITTI_METRICS).reshape(N) for k, v in k_res.items()}
        erec = {k: v.cpu().numpy().view(np.dtype([("count", "f8"), ("sum_err", "f8"), ("sum_abs", "f8"), ("sum_sq", "f8"),
                                                   ("mean_err", "f4"), ("mae", "f4"), ("rmse", "f4"), ("pad", "i4")])).reshape(N)
                for k, v in e_res.items()}
        checks[f"{pname}_u16_equals_f32"] = krec["u16"].tobytes() == krec["f32"].tobytes()
        checks[f"{pname}_u16_u16_equals_f32"] = krec["u16_u16"].tobytes() == krec["f32"].tobytes()
        if pname == "dense":
            checks["dense_has_no_invalid_pixel"] = bool((p16 > 0).all())
            checks["dense_tie_to_reductions"] = all(
                krec[k]["n_gt"].tobytes() == erec[k]["count"].tobytes() and krec[k]["sum_abs"].tobytes() == erec[k]["sum_abs"].tobytes()
                and krec[k]["sum_sq"].tobytes() == erec[k]["sum_sq"].tobytes() for k in PAIRS)
        m = krec["f32"][:UNIQUE]
        res[pname]["benchmark_figures"] = {f: float(np.mean(m[f])) for f in ("mae_mm", "rmse_mm", "imae_per_km", "irmse_per_km", "density")}
        del d_r16, d_r32
    res["checks"] = checks
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if not all(checks.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
