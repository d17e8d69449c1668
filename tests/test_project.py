"""LiDAR projection + normalisation (SURVEY.md 8f #2) against the literal loop of main_sl.cpp:478-523 (C oracle) and
cv2.normalize.  Bar: bit-exact (float arithmetic in source order, last writer wins made deterministic)."""
from __future__ import annotations

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from tests.conftest import assert_bit_equal

T, P = synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02


def test_oracle_normalize_matches_cv2():
    cv2 = pytest.importorskip("cv2")
    pts = synth.velodyne_cloud(0, 60000)
    proj, nrm, cnt = co.lidar_project(pts, T, P, 352, 1216)
    assert cnt > 5000 and (proj > 0).sum() > 3000
    assert_bit_equal(nrm, cv2.normalize(proj, None, 0, 80, cv2.NORM_MINMAX), "normalize 0..80")
    proj2, nrm2, _ = co.lidar_project(pts, T, P, 352, 1216, norm=(1.0, 0.0))
    assert_bit_equal(nrm2, cv2.normalize(proj2, None, 1.0, 0.0, cv2.NORM_MINMAX), "normalize 1..0 (toColorImage, utils.cpp:8)")


def body(lib, to_backend, sizes):
    for k, (rows, cols, n) in enumerate(sizes):
        pts = synth.velodyne_cloud(k, n)
        if k == 1:  # many points per pixel: the last one in file order must win
            pts = np.concatenate([pts, pts[::-1] * np.float32(1.0001), pts[: n // 2]])
        proj, nrm, cnt = api.lidar_project(to_backend(pts), T, P, rows, cols, return_count=True, lib=lib)
        proj, nrm = (a if isinstance(a, np.ndarray) else a.cpu().numpy() for a in (proj, nrm))
        rp, rn, rc = co.lidar_project(pts, T, P, rows, cols)
        assert cnt == rc
        assert_bit_equal(proj, rp, f"projected {rows}x{cols}")
        assert_bit_equal(nrm, rn, f"normalized {rows}x{cols}")
    # no points at all / nothing in front of the camera: empty image, normalize of a constant image is all zeros
    empty = np.zeros((0, 4), np.float32)
    proj, nrm, cnt = api.lidar_project(to_backend(empty), T, P, 40, 60, return_count=True, lib=lib)
    proj, nrm = (a if isinstance(a, np.ndarray) else a.cpu().numpy() for a in (proj, nrm))
    assert cnt == 0 and not proj.any() and not nrm.any()
    behind = synth.velodyne_cloud(3, 2000)
    behind[:, 0] = -np.abs(behind[:, 0]) - 1.0
    proj, nrm, cnt = api.lidar_project(to_backend(behind), T, P, 40, 60, return_count=True, lib=lib)
    assert cnt == co.lidar_project(behind, T, P, 40, 60)[2] == 0
    # the projected image feeds the completion like main_sl.cpp:523 (float, not q8: the float32 dictionary path)
    pts = synth.velodyne_cloud(7, 40000)
    _, nrm = api.lidar_project(to_backend(pts), T, P, 96, 320, lib=lib)
    dense = api.img_completion(nrm, False, "gaussian", lib=lib)
    dn = dense if isinstance(dense, np.ndarray) else dense.cpu().numpy()
    ref = co.img_completion(co.lidar_project(pts, T, P, 96, 320)[1], "gaussian")
    assert_bit_equal(dn, ref, "completion of the normalised projection")


def test_emu_project(emu_lib):
    body(emu_lib, lambda a: a, [(64, 200, 20000), (48, 160, 30000), (352, 1216, 60000)])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
def test_gpu_project(gpu_lib, mode):
    import torch

    body(gpu_lib, (lambda a: a) if mode == "host" else (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()),
         [(64, 200, 20000), (48, 160, 30000), (352, 1216, 120000), (375, 1242, 120000)])


@pytest.mark.gpu
def test_gpu_project_batch(gpu_lib):
    """dcmt_lidar_project_batch_f32: clouds of different sizes in one call == the literal loop per cloud"""
    import torch

    rows, cols = 352, 1216
    sizes = [120000, 60000, 0, 99999, 1]
    clouds = [synth.velodyne_cloud(k, n) if n else np.zeros((0, 4), np.float32) for k, n in enumerate(sizes)]
    mp = max(sizes)
    buf = np.zeros((len(sizes), mp, 4), np.float32)
    for k, c in enumerate(clouds):
        buf[k, : len(c)] = c
    proj, nrm, cnt = api.lidar_project_batch(torch.from_numpy(buf).cuda(), torch.tensor(sizes, dtype=torch.int32).cuda(), T, P, rows, cols,
                                             lib=gpu_lib)
    for k, c in enumerate(clouds):
        rp, rn, rc = co.lidar_project(c, T, P, rows, cols)
        assert int(cnt[k]) == rc
        assert_bit_equal(proj[k].cpu().numpy(), rp, f"cloud {k} projected")
        assert_bit_equal(nrm[k].cpu().numpy(), rn, f"cloud {k} normalized")
