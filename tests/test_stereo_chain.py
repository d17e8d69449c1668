"""The chain the DC_stereo_lidar program runs per frame (main_sl.cpp:1150 withSuperPixels :474-540, then :1162-1253) as ONE
unit: Velodyne cloud -> projection + cv::normalize(0, 80) -> interpolate_with_superpixels on the normalised FLOATS ->
EntryType fill, derivatives, initial disparity, optimize_IG, depth, GaussianBlur.

Checked stage by stage on the reference chain's own intermediates, and end to end.  The reference chain is the reference's
own compiled sources (oracle/_ref) where they are available, else the C restatement (oracle/dcmt_oracle.c).

Against the C restatement every stage and the end-to-end result are bit-equal: its float Gaussians use the kernels'
operation order.  Against the reference build a float Gaussian is held within 1e-4 (OpenCV sums in another order), and
end to end the Gauss-Newton refinement amplifies those last-bit differences of the blurred depth at disparity
discontinuities (the bilinear tap index is a rounded float), so the bar there is statistical: stated below."""
from __future__ import annotations

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from oracle import ref_oracle as ro
from tests.conftest import assert_bit_equal
from tests.helpers import Backend

T, P = synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02


def reference_chain(impl_kind, pts, lab, k, left, right, rows, cols):
    if impl_kind == "ref":
        nrm = ro.lidar_project(pts, T, P, rows, cols)[1]
        dense = ro.interpolate_with_superpixels(lab, nrm, n_clusters=k)
        depth, disp = ro.stereo_refine(dense, left, right, return_disp=True)
    else:
        nrm = co.lidar_project(pts, T, P, rows, cols)[1]
        dense = co.interpolate_with_superpixels(nrm, lab, k)
        depth, disp = co.stereo_refine(dense, left, right, return_disp=True)
    return nrm, dense, depth, disp


def body_chain(be, rows, cols, npts, step, use_ref):
    lib = be.lib
    pts = synth.velodyne_cloud(11, npts)
    lab, k = synth.superpixel_labels(11, rows, cols, step)
    _, left, right = synth.stereo_pair(11, rows, cols)
    r_nrm, r_dense, r_depth, r_disp = reference_chain("ref" if use_ref else "c", pts, lab, k, left, right, rows, cols)
    assert (r_nrm >= 0.1).sum() > 200, "the cloud must land in the image"
    # stage 1: projection + normalize, bit-exact
    _, nrm = api.lidar_project(be._to(pts), T, P, rows, cols, lib=lib)
    nrm = be._from(nrm)
    assert_bit_equal(nrm, r_nrm, "chain stage 1: normalised projection")
    # stage 2: guided completion of the normalised floats (dictionary path of the fused kernels)
    dense, st = be.interpolate_with_superpixels(lab, nrm, 1, n_clusters=k, return_stats=True)
    if rows >= 32 and cols >= 32:
        assert int(st[0, 3]) == 2, f"float frame must take the dictionary path, took {st[0, 3]}"
    if use_ref:
        assert np.abs(dense - r_dense).max() <= 1e-4, "chain stage 2: guided completion"
    else:
        assert_bit_equal(dense, r_dense, "chain stage 2: guided completion")
    # stage 3 on the reference's own stage-2 output: bit-exact disparity; the depth includes the final Gaussian
    depth3, disp3 = be.stereo_refine(r_dense, left, right, None, return_disparity=True)
    assert_bit_equal(disp3, r_disp, "chain stage 3: refined disparity on the reference's dense depth")
    if use_ref:
        assert np.abs(depth3 - r_depth).max() <= 1e-4, "chain stage 3: depth"
    else:
        assert_bit_equal(depth3, r_depth, "chain stage 3: depth")
    # the whole chain on its own intermediates
    depth, disp = be.stereo_refine(dense, left, right, None, return_disparity=True)
    if use_ref:
        d = np.abs(depth - r_depth)
        assert np.median(d) <= 1e-5 and (d <= 1e-3).mean() >= 0.999, f"chain end to end: median {np.median(d)}, within 1e-3: {(d <= 1e-3).mean()}"
    else:
        assert_bit_equal(disp, r_disp, "chain end to end: disparity")
        assert_bit_equal(depth, r_depth, "chain end to end: depth")


def test_emu_stereo_chain(emu_lib):
    body_chain(Backend(emu_lib, "emu"), 200, 700, 40000, 40, use_ref=ro.available())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_stereo_chain(gpu_lib, mode):
    body_chain(Backend(gpu_lib, mode), 352, 1216, 120000, 65, use_ref=ro.available())
    body_chain(Backend(gpu_lib, mode), 375, 1242, 120000, 65, use_ref=False)
