"""The camera program's front in one call (dcmt_interpolate_with_superpixels_bgr_*: BGR -> Lab -> SLIC -> guided completion
of KITTI uint16 depth) against the two calls it replaces (dcmt_slic_bgr_u8c3 + dcmt_interpolate_with_superpixels_u16[_u16]).

Workload: 352x1216 frames, synth.bgr_image colour frames and KITTI-like q8 depth (synth.sparse_depth_q8(..., kitti_like=True),
5 % valid), step 18, nc 50, 10 iterations (main_lc.cpp:187-201); 64 unique frames tiled.
  - device: 1024 device-resident frames per call (1.3 GB of BGR, 0.9 GB of depth: well past the 126 MB L2); the new device
    entry point against the two device calls in 256-frame pieces, as bench.py --workload lidar_camera_chain runs its chain.
    frames/s from CUDA events over --steps calls after --warmup, best of three alternating rounds.
  - host: 512 frames in page-locked buffers (dcmt_host_alloc), H2D and D2H inside the timed region (the calls return
    synchronised): _host against dcmt_slic_bgr_u8c3_host + the guided _host call.  Bytes over the host links per frame
    from shapes: 3 + 2 in and 2 (uint16 out) or 4 (float32 out) out, against 3 + 2 + 4 in and 4 + 2 or 4 + 4 out for the two
    calls (the label map goes out and comes back): 7 / 9 against 15 / 17 B/px.
  - multi-device: _host_multi (uint16 out) on 1 / 2 / 4 / 8 GPUs where the box has them, 1024 frames per call.
Checks in the same run: every chained result is byte-equal to its composition.  Prints one JSON line with the GPU's name,
power limit and SM clocks read in the same run.
Usage: python tools/bench_superpixels_bgr.py [--steps K] [--warmup W]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from depth_completion_mt_b200 import _lib, api, synth  # noqa: E402

ROWS, COLS, UNIQUE, N_DEV, N_HOST, STEP, NC, ITERS, SLIC_CHUNK = 352, 1216, 64, 1024, 512, 18, 50, 10, 256
PX = ROWS * COLS
LINK_BYTES = {"u16": (7, 15), "f32": (9, 17)}  # per pixel over the host links: one call, two calls


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines() if r.returncode == 0 and r.stdout.strip() else ["unavailable: " + r.stderr.strip()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "bench_superpixels_bgr needs a CUDA device"
    res = {"gpu": gpu_info(), "shape": [ROWS, COLS], "step": STEP, "nc": NC, "iterations": ITERS}
    lib = _lib.load()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    bgr_u = np.stack([synth.bgr_image(f, ROWS, COLS) for f in range(UNIQUE)])
    s16_u = np.stack([synth.sparse_depth_q8(f, ROWS, COLS, 0.05, kitti_like=True) for f in range(UNIQUE)])
    k = lib.dcmt_slic_center_count(ROWS, COLS, STEP)
    stream = torch.cuda.current_stream().cuda_stream

    # ---- device-resident: one call against the two calls
    reps = N_DEV // UNIQUE
    tb = torch.from_numpy(bgr_u).to(dev).repeat(reps, 1, 1, 1).contiguous()
    ts = torch.from_numpy(s16_u).to(dev).repeat(reps, 1, 1).contiguous()
    labels = torch.empty((N_DEV, ROWS, COLS), dtype=torch.int32, device=dev)
    device = {}
    for out_name, tdt in (("u16", torch.uint16), ("f32", torch.float32)):
        o1 = torch.empty((N_DEV, ROWS, COLS), dtype=tdt, device=dev)
        o2 = torch.empty_like(o1)
        one = getattr(lib, "dcmt_interpolate_with_superpixels_bgr_" + ("u16_u16" if out_name == "u16" else "u16"))
        guided = getattr(lib, "dcmt_interpolate_with_superpixels_" + ("u16_u16" if out_name == "u16" else "u16"))

        def run_one():
            lib.check(one(tb.data_ptr(), 0, 0, ts.data_ptr(), o1.data_ptr(), ROWS, COLS, 0, 0, 0, 0, N_DEV, STEP, NC, ITERS, 1, 0, None, stream))

        def run_two():
            for c0 in range(0, N_DEV, SLIC_CHUNK):
                n = min(SLIC_CHUNK, N_DEV - c0)
                lib.check(lib.dcmt_slic_bgr_u8c3(tb[c0].data_ptr(), ROWS, COLS, n, STEP, NC, ITERS, labels[c0].data_ptr(), None, stream))
                lib.check(guided(ts[c0].data_ptr(), labels[c0].data_ptr(), k, o2[c0].data_ptr(), ROWS, COLS, 0, 0, 0, 0, n, 1, 0, None, stream))

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            e1.synchronize()
            return N_DEV * args.steps / (e0.elapsed_time(e1) / 1e3)

        for _ in range(args.warmup):
            run_one()
            run_two()
        torch.cuda.synchronize()
        equal = bool(torch.equal(o1.view(torch.int16) if tdt == torch.uint16 else o1.view(torch.int32),
                                 o2.view(torch.int16) if tdt == torch.uint16 else o2.view(torch.int32)))
        a, b = [], []
        for _ in range(3):
            a.append(timed(run_one))
            b.append(timed(run_two))
        device[out_name] = {"one_call_fps": round(max(a)), "two_calls_fps": round(max(b)), "rounds_one": [round(v) for v in a],
                            "rounds_two": [round(v) for v in b], "byte_equal": equal}
        print(f"device {out_name}: one call {max(a):.0f} frames/s, two calls {max(b):.0f} frames/s, equal {equal}", file=sys.stderr)
        del o1, o2
    res["device_resident"] = device
    del tb, ts, labels
    torch.cuda.empty_cache()
    lib.dcmt_release_workspaces()

    # ---- host end to end, page-locked buffers
    def tile(a, n):
        return np.concatenate([a] * ((n + len(a) - 1) // len(a)))[:n]

    hb = api.HostBuffer((N_DEV, ROWS, COLS, 3), np.uint8, lib=lib)
    hs = api.HostBuffer((N_DEV, ROWS, COLS), np.uint16, lib=lib)
    hl = api.HostBuffer((N_HOST, ROWS, COLS), np.int32, lib=lib)
    hb.array[...] = tile(bgr_u, N_DEV)
    hs.array[...] = tile(s16_u, N_DEV)
    host = {}
    for out_name, dt in (("u16", np.uint16), ("f32", np.float32)):
        h1 = api.HostBuffer((N_DEV, ROWS, COLS), dt, lib=lib)
        h2 = api.HostBuffer((N_HOST, ROWS, COLS), dt, lib=lib)
        sfx = "u16_u16" if out_name == "u16" else "u16"
        one = getattr(lib, f"dcmt_interpolate_with_superpixels_bgr_{sfx}_host")
        guided = getattr(lib, f"dcmt_interpolate_with_superpixels_{sfx}_host")
        pb, ps, pl = hb.array.ctypes.data, hs.array.ctypes.data, hl.array.ctypes.data

        def run_one():
            lib.check(one(pb, 0, 0, ps, h1.array.ctypes.data, ROWS, COLS, 0, 0, 0, 0, N_HOST, STEP, NC, ITERS, 1, 0, None))

        def run_two():
            lib.check(lib.dcmt_slic_bgr_u8c3_host(pb, ROWS, COLS, N_HOST, STEP, NC, ITERS, pl, None))
            lib.check(guided(ps, pl, k, h2.array.ctypes.data, ROWS, COLS, 0, 0, 0, 0, N_HOST, 1, 0, None))

        def timed(fn):
            t0 = time.perf_counter()
            for _ in range(args.steps):
                fn()
            return N_HOST * args.steps / (time.perf_counter() - t0)

        for _ in range(args.warmup):
            run_one()
            run_two()
        equal = bool(np.array_equal(h1.array[:N_HOST], h2.array))
        a, b = [], []
        for _ in range(3):
            a.append(timed(run_one))
            b.append(timed(run_two))
        one_b, two_b = LINK_BYTES[out_name]
        host[out_name] = {"one_call_fps": round(max(a)), "two_calls_fps": round(max(b)), "rounds_one": [round(v) for v in a],
                          "rounds_two": [round(v) for v in b], "link_bytes_per_px": {"one_call": one_b, "two_calls": two_b},
                          "one_call_link_GBps": round(max(a) * PX * one_b / 1e9, 1), "two_calls_link_GBps": round(max(b) * PX * two_b / 1e9, 1),
                          "byte_equal": equal}
        print(f"host {out_name}: one call {max(a):.0f} frames/s, two calls {max(b):.0f} frames/s, equal {equal}", file=sys.stderr)
        if out_name == "u16":
            # ---- multi-device, 1024 frames per call, against the one-device _host result of the same frames
            lib.check(one(pb, 0, 0, ps, h1.array.ctypes.data, ROWS, COLS, 0, 0, 0, 0, N_DEV, STEP, NC, ITERS, 1, 0, None))
            ref = h1.array.copy()
            multi = {}
            n_gpu = torch.cuda.device_count()
            fn = lib.dcmt_interpolate_with_superpixels_bgr_u16_u16_host_multi
            for nd in (1, 2, 4, 8):
                if nd > n_gpu:
                    multi[str(nd)] = "not measured: the box has %d GPU(s)" % n_gpu
                    continue

                def run_multi():
                    lib.check(fn(pb, 0, 0, ps, h1.array.ctypes.data, ROWS, COLS, 0, 0, 0, 0, N_DEV, STEP, NC, ITERS, 1, 0, None, None, nd))

                for _ in range(args.warmup):
                    run_multi()
                equal = bool(np.array_equal(h1.array, ref))
                t = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    for _ in range(args.steps):
                        run_multi()
                    t.append(N_DEV * args.steps / (time.perf_counter() - t0))
                multi[str(nd)] = {"fps": round(max(t)), "rounds": [round(v) for v in t], "byte_equal": equal}
                print(f"multi {nd}: {max(t):.0f} frames/s, equal {equal}", file=sys.stderr)
            res["host_multi_u16"] = multi
        h1.close()
        h2.close()
    res["host"] = host
    for b in (hb, hs, hl):
        b.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
