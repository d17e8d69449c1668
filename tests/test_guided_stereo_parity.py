"""(a2) interpolate_with_superpixels and (a3-a9) stereo refinement parity vs the oracle.

Bars (SURVEY.md 8c): a2 bit-exact on q8 input (the guided stage is pure select/min/max, the tail is the
a1 tail); a4, a5, a7, a8 bit-exact (explicit round-to-nearest float ops in source order); a2 on float input and the
a9 Gaussian bit-equal to the C restatement (same operation order), within 1e-4 of cv2 and the reference build."""
from __future__ import annotations

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from tests.conftest import assert_bit_equal
from tests.helpers import Backend

GAUSS_TOL = 1e-4  # float Gaussian against cv2 (the golden files)


def body_guided_golden(be, golden):
    g = golden["guided"]
    for name in sorted({k.split("__")[0] for k in g.files}):
        s, lab, k = g[name + "__in"], g[name + "__labels"], int(g[name + "__k"])
        assert_bit_equal(be.interpolate_with_superpixels(lab, s, 1, n_clusters=k), g[name + "__sp1"], f"{name} use_superpixel=1")
        assert_bit_equal(be.interpolate_with_superpixels(lab, s, 0, n_clusters=k), g[name + "__sp0"], f"{name} use_superpixel=0")


def body_guided_seeded(be, shapes):
    for i, (rows, cols, p, step) in enumerate(shapes):
        s = synth.sparse_depth(70 + i, rows, cols, p)
        lab, k = synth.superpixel_labels(70 + i, rows, cols, step)
        got, st = be.interpolate_with_superpixels(lab, s, 1, n_clusters=k, return_stats=True)
        ref_st = {}
        assert_bit_equal(got, co.interpolate_with_superpixels(s, lab, k, literal=False, stats=ref_st), f"guided {rows}x{cols}")
        assert int(st[0, 0]) == ref_st["loop_passes"]
        # n_clusters smaller than the label range: labels >= n_clusters are never processed (:78 loop bound)
        got = be.interpolate_with_superpixels(lab, s, 1, n_clusters=k // 2)
        assert_bit_equal(got, co.interpolate_with_superpixels(s, lab, k // 2, literal=False), "partial cluster range")


def body_guided_fused(be, shapes):
    """strict-q8 frames take the fused guided front (k_q8_guided_front) + the fused tail; any other frame, and
    path="generic", the float pipeline: same bytes as the oracle either way."""
    rng = np.random.default_rng(5)
    for i, (rows, cols, p, step) in enumerate(shapes):
        s = synth.sparse_depth(170 + i, rows, cols, p, kitti_like=bool(i & 1))
        lab, k = synth.superpixel_labels(170 + i, rows, cols, step)
        if i % 3 == 1:  # unassigned pixels and labels beyond n_clusters keep their own value
            lab = lab.copy()
            lab[rng.random(lab.shape) < 0.05] = -1
            lab[rng.random(lab.shape) < 0.02] = k + 7
        ref_st = {}
        ref = co.interpolate_with_superpixels(s, lab, k, literal=False, stats=ref_st)
        got, st = be.interpolate_with_superpixels(lab, s, 1, n_clusters=k, return_stats=True)
        assert_bit_equal(got, ref, f"fused guided {rows}x{cols} step {step}")
        assert int(st[0, 3]) == 1 and int(st[0, 0]) == ref_st["loop_passes"], f"{rows}x{cols}: path {st[0, 3]}"
        got, st = be.interpolate_with_superpixels(lab, s, 1, n_clusters=k, path="generic", return_stats=True)
        assert_bit_equal(got, ref, f"generic guided {rows}x{cols}")
        assert int(st[0, 3]) == 0
    # thousands of tiny superpixels: more labels per tile than the per-label kernel's table holds -> its tiles are left to
    # the word-by-word kernel
    rows, cols = 64, 96
    s = synth.sparse_depth(190, rows, cols, 0.1)
    yy, xx = np.mgrid[0:rows, 0:cols]
    lab = ((yy * cols + xx) // 2).astype(np.int32)
    k = int(lab.max()) + 1
    got, st = be.interpolate_with_superpixels(lab, s, 1, n_clusters=k, return_stats=True)
    assert_bit_equal(got, co.interpolate_with_superpixels(s, lab, k, literal=False), "label table overflow")
    assert int(st[0, 3]) == 1
    # a non-q8 frame in a batch is redone through the float32 dictionary (DCMT_PATH_RANK) with its own labels
    rows, cols = 48, 80
    b = np.stack([synth.sparse_depth(180, rows, cols, 0.06), synth.sparse_depth_float(181, rows, cols, 0.06), synth.sparse_depth(182, rows, cols, 0.06)])
    labs = np.stack([synth.superpixel_labels(180 + f, rows, cols, 9)[0] for f in range(3)])
    k = synth.superpixel_labels(180, rows, cols, 9)[1]
    got, st = be.interpolate_with_superpixels(labs, b, 1, n_clusters=k, return_stats=True)
    assert [int(v) for v in st[:, 3]] == [1, 2, 1]
    for f in (0, 2):
        assert_bit_equal(got[f], co.interpolate_with_superpixels(b[f], labs[f], k, literal=False), f"batch frame {f}")
    assert_bit_equal(got[1], co.interpolate_with_superpixels(b[1], labs[1], k, literal=False), "batch frame 1 (dictionary path)")
    # guided completion of float frames at the shapes given (the only form DC_stereo_lidar feeds it, main_sl.cpp:540)
    for i, (rows, cols, p, step) in enumerate(shapes[:3]):
        f = synth.sparse_depth_float(500 + i, rows, cols, p)
        lab, k = synth.superpixel_labels(500 + i, rows, cols, step)
        got, st = be.interpolate_with_superpixels(lab, f, 1, n_clusters=k, return_stats=True)
        assert int(st[0, 3]) == 2, f"float guided {rows}x{cols}: path {st[0, 3]}"
        assert_bit_equal(got, co.interpolate_with_superpixels(f, lab, k, literal=False), f"float guided {rows}x{cols}")


def body_stereo_golden(be, golden):
    g = golden["stereo"]
    for name in sorted({k.split("__")[0] for k in g.files}):
        dig, left, right = g[name + "__depth_ig"], g[name + "__left"], g[name + "__right"]
        lib = be.lib
        out, disp = be.stereo_refine(dig, left, right, api.stereo_params(lib=lib, final_gauss=0), return_disparity=True)
        assert_bit_equal(out, g[name + "__default_nogauss"], f"{name} depth (a5+a7+a8)")
        assert_bit_equal(disp, g[name + "__disp4"], f"{name} disparity (a7)")
        out = be.stereo_refine(dig, left, right)
        assert np.abs(out - g[name + "__default"]).max() <= GAUSS_TOL, f"{name} final Gaussian (a9)"
        out = be.stereo_refine(dig, left, right, api.stereo_params(official=True, num_iterations=10, lib=lib))
        assert_bit_equal(out, g[name + "__official10"], f"{name} OFFICIAL constants")


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_guided_golden(emu_lib, golden):
    body_guided_golden(Backend(emu_lib, "emu"), golden)


def test_emu_guided_seeded(emu_lib):
    body_guided_seeded(Backend(emu_lib, "emu"), [(40, 70, 0.06, 8)])


def test_emu_guided_fused(emu_lib):
    body_guided_fused(Backend(emu_lib, "emu"), [(40, 70, 0.06, 8), (97, 171, 0.05, 12), (64, 333, 0.03, 18), (130, 96, 0.1, 7), (33, 47, 0.08, 6)])


def test_emu_stereo_golden(emu_lib, golden):
    body_stereo_golden(Backend(emu_lib, "emu"), golden)


def test_emu_stereo_batch(emu_lib):
    frames = [synth.stereo_pair(f, 20, 70) for f in range(3)]
    dig, left, right = (np.stack([fr[i] for fr in frames]) for i in range(3))
    out = Backend(emu_lib, "emu").stereo_refine(dig, left, right, api.stereo_params(lib=emu_lib, final_gauss=0))
    for f in range(3):
        assert_bit_equal(out[f], co.stereo_refine(*frames[f], final_gauss=False), f"stereo frame {f}")


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_guided_golden(gpu_lib, golden, mode):
    body_guided_golden(Backend(gpu_lib, mode), golden)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_guided_fused(gpu_lib, mode):
    body_guided_fused(Backend(gpu_lib, mode), [(40, 70, 0.06, 8), (97, 171, 0.05, 12), (64, 333, 0.03, 18), (130, 96, 0.1, 7), (33, 47, 0.08, 6),
                                               (352, 1216, 0.05, 18), (375, 1242, 0.05, 18)])


@pytest.mark.gpu
def test_gpu_guided_seeded(gpu_lib):
    body_guided_seeded(Backend(gpu_lib, "gpu_device"), [(40, 70, 0.06, 8), (120, 200, 0.05, 18), (352, 1216, 0.05, 18)])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_stereo_golden(gpu_lib, golden, mode):
    body_stereo_golden(Backend(gpu_lib, mode), golden)


@pytest.mark.gpu
def test_gpu_stereo_full_size_and_functions(gpu_lib):
    """352 x 1216 stereo pair: fused kernel and the one-by-one functions (a4, a5, a7, a8) against the oracle."""
    import torch

    dig, left, right = synth.stereo_pair(1)
    want, want_disp = co.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)
    be = Backend(gpu_lib, "gpu_device")
    out, disp = be.stereo_refine(dig, left, right, api.stereo_params(lib=gpu_lib, final_gauss=0), return_disparity=True)
    assert_bit_equal(out, want, "fused depth")
    assert_bit_equal(disp, want_disp, "fused disparity")
    assert_bit_equal(be.stereo_refine(dig, left, right), co.stereo_refine(dig, left, right), "final Gaussian (a9)")
    vl = torch.from_numpy(left.astype(np.float32)).cuda()
    vr = torch.from_numpy(right.astype(np.float32)).cuda()
    dx, dy = api.calculateMeasuementDerivatives(vr, lib=gpu_lib)
    wdx, wdy = co.measurement_derivatives(right.astype(np.float32))
    assert_bit_equal(dx.cpu().numpy(), wdx, "a4 dx")
    assert_bit_equal(dy.cpu().numpy(), wdy, "a4 dy")
    d0 = api.get_initial_disparity(torch.from_numpy(dig).cuda(), lib=gpu_lib)
    d4 = api.optimize_IG(vl, vr, d0, lib=gpu_lib)
    assert_bit_equal(d4.cpu().numpy(), want_disp, "a7 optimize_IG")
    assert_bit_equal(api.retrieve_optimized_depth(d4, lib=gpu_lib).cpu().numpy(), want, "a8 depth")
