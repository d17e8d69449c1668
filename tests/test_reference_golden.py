"""The comparisons of tests/test_reference_build.py against stored values, so that they run where the reference build is
absent.  tests/golden/reference.npz holds, for the same inputs, what that module compares with the reference build
(oracle/make_reference_golden.py, which checks every value against the reference build wherever it exists).  Here the
C restatement, the cv2 transliteration and, on the B200, the product must reproduce those values with the tolerances of
that module; large arrays are compared through the sha256 of their bytes."""
from __future__ import annotations

import hashlib
import os

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from oracle import cv2_oracle as cvo
from oracle import make_reference_golden as mg
from tests.conftest import GOLDEN, assert_bit_equal

needs_cv2 = pytest.mark.skipif(not cvo.HAVE_CV2, reason="cv2 not importable")
T, P = mg.T, mg.P


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLDEN, "reference.npz"))


def check(ref, key, got, what=""):
    """got equals the stored value bit for bit (whole, or through its digest)."""
    want, got = ref[key], np.asarray(got)
    if want.dtype.kind == "U":
        assert mg.digest(got) == str(want), f"{key} {what}: sha256 differs"
    else:
        assert_bit_equal(got, want, f"{key} {what}")


def near(ref, key, got, tol):
    assert np.abs(np.asarray(got, np.float64) - ref[key]).max() <= tol, key


def test_golden_file_covers_every_case(ref):
    assert len(ref.files) == 98


@pytest.mark.parametrize("shape,density,kitti_like", mg.LIDAR_CASES)
def test_img_completion_restatements_vs_stored_reference(ref, shape, density, kitti_like):
    s = mg.lidar_input(shape, density, kitti_like)
    for bt in ("none", "gaussian"):
        key = f"lidar_{shape[0]}x{shape[1]}_{density}_{int(kitti_like)}_{bt}"
        check(ref, key, co.img_completion(s, bt), "C oracle")
        if cvo.HAVE_CV2:
            check(ref, key, cvo.img_completion(s, bt), "cv2 transliteration")


def test_img_completion_float_input_vs_stored_reference(ref):
    s = synth.sparse_depth_float(3, 97, 211, 0.05)
    check(ref, "float_none", co.img_completion(s, "none"))
    if cvo.HAVE_CV2:  # the float Gaussian is stored as a digest: the C port is held within 1e-4 of it through the transliteration
        t = cvo.img_completion(s, "gaussian")
        check(ref, "float_gaussian", t)
        assert np.abs(co.img_completion(s, "gaussian") - t).max() <= 1e-4


def test_img_completion_special_values_vs_stored_reference(ref):
    s = mg.special_values_frame()
    check(ref, "special_none", co.img_completion(s, "none"))
    near(ref, "special_gaussian", co.img_completion(s, "gaussian"), 1e-4)
    for name, frame in mg.CONSTANT_FRAMES.items():
        for bt in ("none", "gaussian"):
            check(ref, f"constant_{name}_{bt}", co.img_completion(frame, bt))


def test_full_size_digests_all_lines():
    """every line of the committed 352 x 1216 digests (the reference's outputs), by the C restatement"""
    lines = [l.split() for l in open(os.path.join(GOLDEN, "lidar_only_352x1216.sha256")) if not l.startswith("#")]
    assert len(lines) == 12
    for frame, kitti_like, blur, h_in, h_out in lines:
        s = synth.sparse_depth(int(frame), density=0.05, kitti_like=bool(int(kitti_like)))
        assert hashlib.sha256(s.tobytes()).hexdigest() == h_in
        assert hashlib.sha256(co.img_completion(s, blur).tobytes()).hexdigest() == h_out, (frame, kitti_like, blur)


@pytest.mark.parametrize("shape,step", mg.GUIDED_CASES)
def test_interpolate_with_superpixels_vs_stored_reference(ref, shape, step):
    s, lab, k = mg.guided_input(shape, step)
    for n in (k, k - 3):
        key = f"guided_{shape[0]}x{shape[1]}_n{n}_sp1"
        check(ref, key, co.interpolate_with_superpixels(s, lab, n, literal=True), "literal C loop")
        check(ref, key, co.interpolate_with_superpixels(s, lab, n, literal=False), "closed form")
        if cvo.HAVE_CV2:
            check(ref, key, cvo.interpolate_with_superpixels(s, lab, n), "cv2 transliteration")
    key = f"guided_{shape[0]}x{shape[1]}_n{k}_sp0"
    check(ref, key, co.interpolate_with_superpixels(s, lab, k, use_superpixel=0), "use_superpixel = 0")
    check(ref, key, co.img_completion(s, "gaussian"), "use_superpixel = 0 is img_completion with the gaussian blur")


@pytest.mark.parametrize("shape,step,nc", mg.SLIC_CASES)
def test_slic_vs_stored_reference(ref, shape, step, nc):
    lab, cen = co.slic(synth.lab_image(2, shape[0], shape[1]), step, nc)
    key = f"slic_{shape[0]}x{shape[1]}_{step}_{nc}"
    check(ref, key + "_labels", lab)
    check(ref, key + "_centers", cen)


def test_slic_flat_image_vs_stored_reference(ref):
    lab, cen = co.slic(np.full((48, 64, 3), 128, np.uint8), 9, 40)
    check(ref, "slic_flat_labels", lab)
    check(ref, "slic_flat_centers", cen)


@pytest.mark.parametrize("shape", mg.STEREO_SHAPES)
def test_stereo_chain_vs_stored_reference(ref, shape):
    dig, left, right = synth.stereo_pair(5, shape[0], shape[1])
    out, disp = co.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)
    key = f"stereo_{shape[0]}x{shape[1]}"
    check(ref, key + "_disp", disp, "disparity after 4 iterations")
    check(ref, key + "_depth", out, "depth")
    blurred = co.stereo_refine(dig, left, right)
    if min(shape) >= 5:
        if cvo.HAVE_CV2:
            t = np.asarray(cvo.stereo_refine(dig, left, right))
            check(ref, key + "_blurred", t, "transliteration")
            assert np.abs(blurred - t).max() <= 1e-4
    else:
        near(ref, key + "_blurred", blurred, 1e-4)


@needs_cv2
def test_stereo_functions_one_by_one_vs_stored_reference(ref):
    dig, left, right = synth.stereo_pair(6, 48, 80)
    dx, dy = co.measurement_derivatives(right.astype(np.float32))
    check(ref, "one_by_one_dx", dx)
    check(ref, "one_by_one_dy", dy)
    check(ref, "one_by_one_d0", np.asarray(cvo.get_initial_disparity(dig)))
    d4 = co.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)[1]
    check(ref, "one_by_one_d4", d4)
    check(ref, "one_by_one_depth", np.asarray(cvo.retrieve_optimized_depth(d4)))


def test_stereo_zero_and_far_depths_vs_stored_reference(ref):
    dig, left, right = mg.stereo_zero_far_input()
    out = co.stereo_refine(dig, left, right, final_gauss=False)
    check(ref, "stereo_zero_far", out)
    assert (out[:5] == 0).all() and (out[5:8] <= 100.0).all()


@pytest.mark.parametrize("shape", mg.EVAL_SHAPES)
def test_evaluation_loops_vs_stored_reference(ref, shape):
    gt, dense = mg.eval_input(shape)
    key = f"eval_{shape[0]}x{shape[1]}"
    if shape[0] < 100:
        check(ref, key + "_lidar_only", np.float32(co.evaluate(gt, dense, 0, 0)["mean_err"]))
    o = co.evaluate(gt, dense, 0, 1)
    check(ref, key + "_lidar_camera", np.float32([o["rmse"], o["mae"]]))
    o = co.evaluate(gt, dense, 2, 1)
    check(ref, key + "_stereo_lidar", np.float32([o["mae"], o["rmse"]]))


@pytest.mark.parametrize("rows,cols,n", mg.PROJ_CASES)
def test_projection_loop_vs_stored_reference(ref, rows, cols, n):
    cp, cn, cc = co.lidar_project(mg.proj_input(rows, cols, n), T, P, rows, cols)
    key = f"proj_{rows}x{cols}_{n}"
    assert cc == int(ref[key + "_count"]) and (cc > 1000 or cols < 1000)
    check(ref, key + "_projected", cp)
    check(ref, key + "_normalized", cn)


def test_projection_loop_degenerate_clouds_vs_stored_reference(ref):
    for name, pts in mg.degenerate_clouds().items():
        cp, cn, cc = co.lidar_project(pts, T, P, 40, 60)
        assert cc == int(ref[f"proj_{name}_count"]) == 0
        check(ref, f"proj_{name}_projected", cp)
        check(ref, f"proj_{name}_normalized", cn)


def test_raw_mat_format_vs_stored_reference(ref, tmp_path):
    m = mg.raw_mat()
    api.write_M(tmp_path / "pkg.bin", m)
    data = np.frombuffer(open(tmp_path / "pkg.bin", "rb").read(), np.uint8)
    check(ref, "raw_mat_bytes", data, "the bytes the reference's write_M writes")
    assert_bit_equal(api.read_M(tmp_path / "pkg.bin"), m, "package reads the reference's bytes")


# ---------------------------------------------------------------------------------------------------------------------
# the product against the stored reference values (B200, through the C ABI)


@pytest.mark.gpu
def test_gpu_img_completion_equals_stored_reference(ref, gpu_lib):
    import torch

    for frame, density, kitti_like in mg.GPU_LIDAR_CASES:
        d16 = synth.sparse_depth_q8(frame, density=density, kitti_like=kitti_like)
        s = d16.astype(np.float32) / np.float32(256)
        for bt in ("gaussian", "none"):
            key = f"gpu_lidar_{frame}_{bt}"
            check(ref, key, api.img_completion(torch.from_numpy(s).cuda(), False, bt, lib=gpu_lib).cpu().numpy(), "fused")
            check(ref, key, api.img_completion(torch.from_numpy(s).cuda(), False, bt, path="generic", lib=gpu_lib).cpu().numpy(), "generic")
        check(ref, f"gpu_lidar_{frame}_gaussian", api.img_completion(s, False, "gaussian", lib=gpu_lib), "host entry point")
        check(ref, f"gpu_lidar_{frame}_gaussian", api.img_completion(torch.from_numpy(d16).cuda(), False, "gaussian", lib=gpu_lib).cpu().numpy(),
              "uint16 input")


@pytest.mark.gpu
def test_gpu_guided_and_stereo_equal_stored_reference(ref, gpu_lib):
    import torch

    s, lab, k = mg.guided_gpu_input()
    for sp in (1, 0):
        got = api.interpolate_with_superpixels(torch.from_numpy(lab).cuda(), torch.from_numpy(s).cuda(), "gaussian", sp, n_clusters=k, lib=gpu_lib)
        check(ref, f"gpu_guided_sp{sp}", got.cpu().numpy(), f"guided sp={sp}")
    dig, left, right = synth.stereo_pair(4)
    prm = api.stereo_params(final_gauss=0, lib=gpu_lib)
    got = api.stereo_refine(torch.from_numpy(dig).cuda(), torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda(), prm, lib=gpu_lib)
    check(ref, "gpu_stereo_nogauss", got.cpu().numpy(), "stereo refinement at 352 x 1216")
    if cvo.HAVE_CV2:  # the final float Gaussian: within 1e-4 of the stored value, reproduced here by the transliteration
        blurred = np.asarray(cvo.stereo_refine(dig, left, right))
        check(ref, "gpu_stereo_blurred", blurred, "transliteration")
        got = api.stereo_refine(torch.from_numpy(dig).cuda(), torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda(), lib=gpu_lib)
        assert np.abs(got.cpu().numpy() - blurred).max() <= 1e-4


@pytest.mark.gpu
def test_gpu_slic_equals_stored_reference(ref, gpu_lib):
    import torch

    img = synth.lab_image(1)
    labels, centers = api.generate_superpixels(torch.from_numpy(img).cuda(), 18, 40, return_centers=True, lib=gpu_lib)
    check(ref, "gpu_slic_labels", labels.cpu().numpy())
    check(ref, "gpu_slic_centers", np.ascontiguousarray(centers.cpu().numpy(), dtype=np.float64))
