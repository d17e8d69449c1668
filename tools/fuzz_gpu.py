"""Randomised parity run of the product on the GPU against the C oracle: lidar-only (float32 / uint16 input, device and host
entry points) and the superpixel-guided variant, random shapes / densities / boundary codes.  Run on the GPU box:
    python tools/fuzz_gpu.py [seconds] [seed]"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from depth_completion_mt_b200 import _lib, api, synth  # noqa: E402
from oracle import c_oracle as co  # noqa: E402
from oracle import ref_oracle as ro  # noqa: E402

HAVE_REF = ro.available()  # the reference's own compiled sources (prebuilt oracle/_ref travels with the snapshot)

secs = float(sys.argv[1]) if len(sys.argv) > 1 else 60
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
rng = np.random.default_rng(seed)
lib = _lib.load()
t_end = time.time() + secs
n = ng = nr = ns = nf = 0
while time.time() < t_end:
    rows = int(rng.integers(32, 420))
    cols = int(rng.integers(32, 1400))
    p = float(rng.choice([0.001, 0.003, 0.01, 0.03, 0.05, 0.1, 0.2, 0.5]))
    kitti = bool(rng.integers(0, 2))
    blur = str(rng.choice(["gaussian", "none"]))
    u16 = bool(rng.integers(0, 2))
    host = bool(rng.integers(0, 2))
    fseed = int(rng.integers(0, 1 << 30))
    d16 = synth.sparse_depth_q8(fseed, rows, cols, p, kitti_like=kitti)
    if rng.random() < 0.3:  # sprinkle boundary codes
        ys, xs = rng.integers(0, rows, 20), rng.integers(0, cols, 20)
        d16[ys, xs] = rng.choice([1, 25, 26, 27, 25574, 25575, 25600, 30000, 65535], 20)
    s = d16.astype(np.float32) / np.float32(256)
    st = {}
    want = co.img_completion(s, blur, st)
    src = d16 if u16 else s
    if not host:
        src = torch.from_numpy(src).cuda()
    got, stats = api.img_completion(src, False, blur, return_stats=True, lib=lib)
    if not host:
        got, stats = got.cpu().numpy(), stats.cpu().numpy()
    ok = np.array_equal(got.view(np.uint32), want.view(np.uint32)) and int(stats[0, 0]) == st["loop_passes"]
    if not ok:
        print(f"MISMATCH lidar rows={rows} cols={cols} p={p} kitti={kitti} blur={blur} u16={u16} host={host} seed={fseed} diff={(got != want).sum()}", flush=True)
        sys.exit(1)
    n += 1
    if HAVE_REF and rows * cols < 150_000:  # ... and to the reference build itself
        if not np.array_equal(got.view(np.uint32), ro.img_completion(s, blur).view(np.uint32)):
            print(f"MISMATCH vs reference build rows={rows} cols={cols} p={p} blur={blur} seed={fseed}", flush=True)
            sys.exit(1)
        nr += 1
    if rng.random() < 0.4:  # arbitrary float frames: the per-frame dictionary path of the fused kernels, bit-exact with either blur
        hi = float(rng.choice([5.0, 50.0, 90.0, 99.95, 140.0]))
        f = synth.sparse_depth_float(fseed, rows, cols, min(p, 0.07), hi=hi)
        if rng.random() < 0.3:
            ys, xs = rng.integers(0, rows, 30), rng.integers(0, cols, 30)
            f[ys, xs] = rng.choice(np.array([-3.0, 0.0999, 0.1, 99.9, 99.95, 100.0, 17.123, 1e-30], np.float32), 30)
        srcf = f if host else torch.from_numpy(f).cuda()
        gotf, stf = api.img_completion(srcf, False, "none", return_stats=True, lib=lib)
        if not host:
            gotf, stf = gotf.cpu().numpy(), stf.cpu().numpy()
        nvalid = int(((f >= np.float32(0.1)) & ((np.float32(100) - f) >= np.float32(0.1))).sum())
        if int(stf[0, 3]) != (2 if nvalid <= 32768 else 0) or not np.array_equal(gotf.view(np.uint32), co.img_completion(f, "none").view(np.uint32)):
            print(f"MISMATCH float rows={rows} cols={cols} p={p} hi={hi} host={host} seed={fseed} path={stf[0, 3]}", flush=True)
            sys.exit(1)
        gotf = api.img_completion(srcf, False, "gaussian", lib=lib)
        gotf = gotf if host else gotf.cpu().numpy()
        if not np.array_equal(gotf.view(np.uint32), co.img_completion(f, "gaussian").view(np.uint32)):
            print(f"MISMATCH float gaussian rows={rows} cols={cols} p={p} hi={hi} seed={fseed}", flush=True)
            sys.exit(1)
        nf += 1
    if rng.random() < 0.15:  # stereo refinement (bit-exact without the final float Gaussian)
        dig, left, right = synth.stereo_pair(fseed % 1000, rows, cols)
        prm = api.stereo_params(final_gauss=0, lib=lib)
        gots = api.stereo_refine(torch.from_numpy(dig).cuda(), torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda(), prm, lib=lib).cpu().numpy()
        if not np.array_equal(gots.view(np.uint32), co.stereo_refine(dig, left, right, final_gauss=False).view(np.uint32)):
            print(f"MISMATCH stereo rows={rows} cols={cols} seed={fseed}", flush=True)
            sys.exit(1)
        ns += 1
    if rng.random() < 0.35 and rows * cols < 200_000:  # guided: the oracle's closed form is slower
        step = int(rng.choice([6, 9, 12, 18, 25]))
        lab, k = synth.superpixel_labels(fseed % 1000, rows, cols, step=step)
        lab = lab.copy()
        if rng.random() < 0.5:
            lab[:: int(rng.integers(3, 9)), :: int(rng.integers(3, 9))] = -1
        kk = k if rng.random() < 0.7 else max(1, k - int(rng.integers(1, 5)))
        wantg = co.interpolate_with_superpixels(s, lab, kk)
        gotg = api.interpolate_with_superpixels(torch.from_numpy(lab).cuda(), torch.from_numpy(s).cuda(), "gaussian", 1, n_clusters=kk, lib=lib).cpu().numpy()
        if not np.array_equal(gotg.view(np.uint32), wantg.view(np.uint32)):
            print(f"MISMATCH guided rows={rows} cols={cols} p={p} step={step} k={kk} seed={fseed} diff={(gotg != wantg).sum()}", flush=True)
            sys.exit(1)
        ng += 1
print(f"fuzz ok: {n} lidar-only ({nr} of them also against the reference build), {nf} float (dictionary path), {ng} guided and {ns} stereo random frames, seed {seed}")
