"""Every float32 path against the C restatement (oracle/dcmt_oracle.c), bit for bit.

The float32 Gaussians of the fused dictionary tail (k_q8_tail<true>), of the generic pipeline and of the stereo kernel are
written with explicit round-to-nearest operations in the C restatement's operation order, so on float input the kernels
must give the restatement's bytes, not merely come close (cv2 and the reference build sum in another order and stay
within 1e-4; that bar is checked in test_reference_build.py / test_oracle.py).  The cases sit where a float Gaussian goes
wrong: REFLECT_101 borders of frames narrower than the 5-tap kernel, ragged tile edges, values at the validity thresholds
and where 100 - v cancels, subnormals and signed zeros, duplicated values, the dictionary's capacity (32 768 valid pixels),
mixed batches and batches that span a chunk boundary.  Same bodies on the CPU emulator build and on the B200."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from tests.conftest import ROOT, assert_bit_equal
from tests.helpers import Backend

GENERIC_SHAPES = [(1, 1), (1, 9), (9, 1), (2, 2), (4, 5), (31, 31), (31, 200), (200, 31)]  # below the fused kernels' 32 x 32
DICT_SHAPES = [(32, 32), (33, 47), (97, 171), (100, 321), (193, 40)]  # ragged tile edges on both axes
RANK_CAP = 32768  # valid pixels the per-frame dictionary holds (rank_f32.cuh kRankMaxValid)


def f32(v):
    return np.float32(v)


def n_valid(f):
    """valid <=> v >= 0.1f and 100 - v >= 0.1f, in float32 (img_completion.cpp:55-67 and the `< 0.1` tests after it)"""
    return int(((f >= f32(0.1)) & ((f32(100) - f) >= f32(0.1))).sum())


def float_frame(seed, rows, cols, density=0.05):
    """non-q8 depths; tiny frames get a dense mix of holes and valid pixels so that there is something to blur"""
    if rows * cols >= 400:
        return synth.sparse_depth_float(seed, rows, cols, density)
    rng = np.random.default_rng(seed)
    f = rng.uniform(0.5, 90.0, (rows, cols)).astype(np.float32)
    f[rng.random((rows, cols)) < 0.4] = 0
    return f


def check(be, f, name, blur="gaussian", path="auto", want_path=None):
    out, st = be.img_completion(f, blur, path=path, return_stats=True)
    ref_st = {}
    assert_bit_equal(out, co.img_completion(f, blur, ref_st), f"{name} blur={blur} path={path}")
    assert int(st[0, 0]) == ref_st["loop_passes"], f"{name}: loop passes"
    assert int(st[0, 1]) == ref_st["holes_before_loop"], f"{name}: holes before the loop"
    assert int(st[0, 2]) == ref_st["holes_after_extrapolation"], f"{name}: holes after extrapolation"
    if want_path is not None:
        assert int(st[0, 3]) == want_path, f"{name} path={path}: took path {st[0, 3]}, want {want_path}"


def check_all_paths(be, f, name):
    """auto and rank take the dictionary (2) when the frame is at least 32 x 32 and its valid pixels fit, else the generic
    pipeline (0); generic is always 0"""
    rows, cols = f.shape
    dict_ok = rows >= 32 and cols >= 32 and n_valid(f) <= RANK_CAP
    for path in ("auto", "rank", "generic"):
        check(be, f, name, path=path, want_path=2 if dict_ok and path != "generic" else 0)


def body_shapes(be, shapes):
    for i, (rows, cols) in enumerate(shapes):
        check_all_paths(be, float_frame(700 + i, rows, cols), f"{rows}x{cols}")


def body_values(be, rows=64, cols=96):
    rng = np.random.default_rng(17)

    def sprinkle(values, n=80, seed=0):
        f = synth.sparse_depth_float(720 + seed, rows, cols, 0.05)
        ys, xs = rng.integers(0, rows, n), rng.integers(0, cols, n)
        f[ys, xs] = rng.choice(np.asarray(values, np.float32), n)
        return f

    def around(v, k=3):
        v = f32(v)
        out = [v]
        lo = hi = v
        for _ in range(k):
            lo, hi = np.nextafter(lo, f32(-np.inf)), np.nextafter(hi, f32(np.inf))
            out += [lo, hi]
        return out

    check_all_paths(be, sprinkle(around(0.1), seed=1), "nextafter neighbours of 0.1")
    check_all_paths(be, sprinkle(around(99.9), seed=2), "nextafter neighbours of 99.9")
    check_all_paths(be, sprinkle(around(0.1) + around(99.9), n=300, seed=3), "both thresholds, dense")
    # 100 - v cancels: every float32 in [99.8, 99.9] once, on a frame of its own (13 108 values, inside the dictionary)
    v = np.arange(np.float32(99.8).view(np.int32), np.float32(99.9).view(np.int32) + 1, dtype=np.int32).view(np.float32)
    f = np.zeros((160, 160), np.float32)
    f.ravel()[rng.permutation(f.size)[: v.size]] = v
    check_all_paths(be, f, "every float32 in [99.8, 99.9]")
    tiny = [1e-45, 1e-40, 1.1754942e-38, 1.1754944e-38, -1e-45, -1e-40, 0.0, -0.0]
    check_all_paths(be, sprinkle(tiny, n=200, seed=4), "subnormals and signed zeros")
    big = [-1e30, -3.4028235e38, -100.0, -0.1, 1e30, 3.4028235e38, 100.0, 1e4]
    check_all_paths(be, sprinkle(big, n=200, seed=5), "large magnitudes (all holes)")
    # heavy duplication: a handful of distinct values; then one value for every valid pixel
    f = synth.sparse_depth_float(730, rows, cols, 0.08)
    f[f > 0] = rng.choice(np.array([3.3, 47.77, 47.770004, 88.1], np.float32), int((f > 0).sum()))
    check_all_paths(be, f, "four distinct values")
    f = np.where(synth.sparse_depth_float(731, rows, cols, 0.05) > 0, f32(37.3), f32(0))
    check_all_paths(be, f, "every valid pixel equal")
    f = np.where(synth.sparse_depth_float(732, rows, cols, 0.02) > 0, f32(99.899994), f32(0))
    check_all_paths(be, f, "every valid pixel at the last valid value")


def capacity_frame(n, rows=192, cols=192, seed=740):
    """exactly n valid pixels (the rest holes), values not on the q8 grid"""
    rng = np.random.default_rng(seed)
    f = np.zeros((rows, cols), np.float32)
    f.ravel()[rng.permutation(rows * cols)[:n]] = rng.uniform(0.5, 90.0, n).astype(np.float32)
    assert n_valid(f) == n
    return f


def body_capacity(be):
    for n, want in ((RANK_CAP, 2), (RANK_CAP + 1, 0)):
        f = capacity_frame(n)
        for path in ("auto", "rank"):
            check(be, f, f"{n} valid pixels", path=path, want_path=want)
        check(be, f, f"{n} valid pixels", path="generic", want_path=0)


def mixed_batch(rows, cols, seed=750):
    """q8, float, float beyond the dictionary, float, q8: paths 1, 2, 0, 2, 1"""
    dense = synth.sparse_depth_float(seed + 2, rows, cols, 0.9)
    assert n_valid(dense) > RANK_CAP
    return np.stack([synth.sparse_depth(seed, rows, cols, 0.05), synth.sparse_depth_float(seed + 1, rows, cols, 0.05), dense,
                     synth.sparse_depth_float(seed + 3, rows, cols, 0.02), synth.sparse_depth(seed + 4, rows, cols, 0.03)])


def body_mixed_batch(be, rows, cols):
    b = mixed_batch(rows, cols)
    for path, want in (("auto", [1, 2, 0, 2, 1]), ("rank", [2, 2, 0, 2, 2]), ("generic", [0] * 5)):
        out, st = be.img_completion(b, "gaussian", path=path, return_stats=True)
        assert [int(v) for v in st[:, 3]] == want, f"mixed batch path={path}: {st[:, 3]}"
        for i in range(len(b)):
            ref_st = {}
            assert_bit_equal(out[i], co.img_completion(b[i], "gaussian", ref_st), f"mixed batch path={path} frame {i}")
            assert int(st[i, 0]) == ref_st["loop_passes"]


def body_guided(be, shapes):
    """guided completion of float frames: the dictionary path of the fused guided front, and the generic float kernel"""
    for i, (rows, cols, step) in enumerate(shapes):
        f = float_frame(760 + i, rows, cols, 0.06)
        lab, k = synth.superpixel_labels(760 + i, rows, cols, step)
        ref_st = {}
        want = co.interpolate_with_superpixels(f, lab, k, literal=False, stats=ref_st)
        fused = rows >= 32 and cols >= 32
        for path, want_path in (("auto", 2 if fused else 0), ("generic", 0)):
            got, st = be.interpolate_with_superpixels(lab, f, 1, n_clusters=k, path=path, return_stats=True)
            assert_bit_equal(got, want, f"float guided {rows}x{cols} step {step} path={path}")
            assert int(st[0, 3]) == want_path and int(st[0, 0]) == ref_st["loop_passes"], f"float guided {rows}x{cols}: {st[0]}"
    # a batch of q8 and float frames, each with its own labels
    rows, cols = 48, 80
    b = np.stack([synth.sparse_depth_float(770, rows, cols, 0.06), synth.sparse_depth(771, rows, cols, 0.06),
                  synth.sparse_depth_float(772, rows, cols, 0.03)])
    labs = np.stack([synth.superpixel_labels(770 + j, rows, cols, 9)[0] for j in range(3)])
    k = synth.superpixel_labels(770, rows, cols, 9)[1]
    got, st = be.interpolate_with_superpixels(labs, b, 1, n_clusters=k, return_stats=True)
    assert [int(v) for v in st[:, 3]] == [2, 1, 2]
    for j in range(3):
        assert_bit_equal(got[j], co.interpolate_with_superpixels(b[j], labs[j], k, literal=False), f"guided batch frame {j}")


def body_stereo(be, rows, cols):
    """stereo refinement ending in the float Gaussian (a9): default constants and the OFFICIAL ones with the blur switched
    on, one frame and a batch"""
    lib = be.lib
    frames = [synth.stereo_pair(780 + j, rows, cols) for j in range(3)]
    for name, prm in (("default", api.stereo_params(lib=lib)), ("official", api.stereo_params(official=True, num_iterations=10, lib=lib, final_gauss=1))):
        kw = dict(num_iterations=prm.num_iterations, damp_factor=prm.damp_factor, err_clip=prm.err_clip, depth_clip=prm.depth_clip,
                  final_gauss=True, baseline=prm.baseline, focal=prm.focal)
        wants = [co.stereo_refine(*fr, **kw) for fr in frames]
        assert_bit_equal(be.stereo_refine(*frames[0], prm), wants[0], f"stereo {name} single frame")
        dig, left, right = (np.stack([fr[i] for fr in frames]) for i in range(3))
        out = be.stereo_refine(dig, left, right, prm)
        for j in range(3):
            assert_bit_equal(out[j], wants[j], f"stereo {name} batch frame {j}")


_CHUNKED = r"""
import sys; sys.path.insert(0, %(root)r)
import numpy as np
from depth_completion_mt_b200 import _lib, synth
from tests.test_float_exact import body_guided, body_mixed_batch
from tests.helpers import Backend
if %(gpu)r:
    lib = _lib.load()
    modes = ["gpu_host", "gpu_device"]
else:
    from tests.emu import build_emu
    lib = _lib.bind(build_emu.build())
    modes = ["emu"]
for mode in modes:
    be = Backend(lib, mode)
    body_mixed_batch(be, %(rows)d, %(cols)d)
    body_guided(be, [])
print("CHUNKED_OK")
"""


def run_chunked(on_gpu, rows, cols):
    """the mixed batch and the guided batch in chunks of 2 frames (fused and generic pipelines) and, on the host entry
    points, in chunks of 1 Mpx; separate process: the chunk sizes are read once per process"""
    env = dict(os.environ, DCMT_FUSED_CHUNK="2", DCMT_GENERIC_CHUNK="2", DCMT_HOST_CHUNK_MPX="1")
    code = _CHUNKED % {"root": ROOT, "gpu": on_gpu, "rows": rows, "cols": cols}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert r.returncode == 0 and "CHUNKED_OK" in r.stdout, r.stdout + r.stderr


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_shapes(emu_lib):
    body_shapes(Backend(emu_lib, "emu"), GENERIC_SHAPES + DICT_SHAPES)


def test_emu_values(emu_lib):
    body_values(Backend(emu_lib, "emu"))


def test_emu_capacity(emu_lib):
    body_capacity(Backend(emu_lib, "emu"))


def test_emu_mixed_batch(emu_lib):
    body_mixed_batch(Backend(emu_lib, "emu"), 200, 200)


def test_emu_chunked():
    run_chunked(False, 200, 200)


def test_emu_guided(emu_lib):
    body_guided(Backend(emu_lib, "emu"), [(9, 31, 4), (31, 200, 9), (32, 32, 6), (33, 47, 8), (97, 171, 12), (64, 333, 18)])


def test_emu_stereo(emu_lib):
    body_stereo(Backend(emu_lib, "emu"), 40, 150)


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_shapes_values(gpu_lib, mode):
    be = Backend(gpu_lib, mode)
    body_shapes(be, GENERIC_SHAPES + DICT_SHAPES + [(352, 1216), (375, 1242), (1024, 2048)])
    body_values(be)
    body_values(be, 352, 1216)
    body_capacity(be)
    body_mixed_batch(be, 200, 200)
    body_mixed_batch(be, 352, 1216)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_guided_stereo(gpu_lib, mode):
    be = Backend(gpu_lib, mode)
    body_guided(be, [(9, 31, 4), (31, 200, 9), (32, 32, 6), (33, 47, 8), (97, 171, 12), (352, 1216, 18), (375, 1242, 65)])
    body_stereo(be, 40, 150)
    body_stereo(be, 352, 1216)


@pytest.mark.gpu
def test_gpu_chunked():
    run_chunked(True, 352, 1216)


@pytest.mark.gpu
def test_gpu_rank_equals_generic_on_a_large_batch(gpu_lib):
    """128 distinct float frames at KITTI size, densities 1-10 % (the densest beyond the dictionary): the dictionary path and
    the generic pipeline give the same bytes, and sampled frames the C restatement's"""
    import torch

    dens = (0.01, 0.02, 0.04, 0.07, 0.1)
    batch = np.stack([synth.sparse_depth_float(800 + f, 352, 1216, dens[f % 5]) for f in range(128)])
    dev = torch.from_numpy(batch).cuda()
    a, sa = api.img_completion(dev, False, "gaussian", path="rank", return_stats=True, lib=gpu_lib)
    b, sb = api.img_completion(dev, False, "gaussian", path="generic", return_stats=True, lib=gpu_lib)
    assert torch.equal(a, b)
    assert torch.equal(sa[:, :3], sb[:, :3]) and bool((sb[:, 3] == 0).all())
    want = [2 if n_valid(batch[f]) <= RANK_CAP else 0 for f in range(128)]
    assert sa[:, 3].cpu().tolist() == want and 2 in want and 0 in want
    for f in (0, 63, 127):
        assert_bit_equal(a[f].cpu().numpy(), co.img_completion(batch[f], "gaussian"), f"frame {f}")
