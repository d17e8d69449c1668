"""The front of the lidar-camera program from the colour image as read (main_lc.cpp:182-220): cvtColor(COLOR_BGR2Lab),
generate_superpixels and interpolate_with_superpixels of q8 sparse depth, with the conversion on the device.  Checked
bit for bit against the C oracle chain started from OpenCV's Lab and, where it exists, the reference build.  Also the
OpenCV-free C++ shim's dcmt::bgr2lab."""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from oracle import lab_oracle
from oracle import ref_oracle as ro
from tests.conftest import ROOT, assert_bit_equal


def _cv2():
    try:
        import cv2
    except ImportError:
        return None
    return cv2


def oracle_lab(bgr):
    """OpenCV's Lab of one frame: cv2 where installed (and the C oracle must agree), else the C oracle (pinned to cv2 on
    all 2^24 colours by tests/test_color_lab.py)."""
    lab = lab_oracle.bgr2lab(bgr)
    cv2 = _cv2()
    if cv2 is not None:
        assert np.array_equal(lab, cv2.cvtColor(bgr, cv2.COLOR_BGR2Lab))
    return lab


def chain(lib, bgr, sparse, step, nc, to_backend, fused_entry):
    """main_lc.cpp:182-220 on the device: Lab, superpixels, guided completion; returns (labels, dense) as numpy."""
    x = to_backend(bgr)
    if fused_entry:
        labels = api.generate_superpixels_bgr(x, step, nc, lib=lib)
    else:
        labels = api.generate_superpixels(api.bgr2lab(x, lib=lib), step, nc, lib=lib)
    k = lib.dcmt_slic_center_count(bgr.shape[-3], bgr.shape[-2], int(step))
    dense = api.interpolate_with_superpixels(labels, to_backend(sparse), "gaussian", 1, n_clusters=k, lib=lib)
    as_np = lambda a: a if isinstance(a, np.ndarray) else a.cpu().numpy()  # noqa: E731
    return as_np(labels), as_np(dense)


def check_chain(lib, n, rows, cols, step, nc, to_backend, fused_entry):
    bgr = np.stack([synth.bgr_image(f, rows, cols) for f in range(n)])
    sparse = np.stack([synth.sparse_depth(f, rows, cols, kitti_like=True) for f in range(n)])
    labels, dense = chain(lib, bgr, sparse, step, nc, to_backend, fused_entry)
    have_ref = ro.available()
    for f in range(n):
        lab = oracle_lab(bgr[f])
        want_l, _ = co.slic(lab, int(step), nc)
        assert_bit_equal(labels[f], want_l, f"frame {f}: labels")
        want_d = co.interpolate_with_superpixels(sparse[f], want_l, lib.dcmt_slic_center_count(rows, cols, int(step)))
        assert_bit_equal(dense[f], want_d, f"frame {f}: dense depth")
        if have_ref and f == 0:
            ref_l, _, _ = ro.generate_superpixels(lab, int(step), nc)
            assert_bit_equal(labels[f], ref_l, "labels vs the reference build")
            assert_bit_equal(dense[f], ro.interpolate_with_superpixels(want_l, sparse[f], "gaussian", 1), "dense vs the reference build")


@pytest.mark.parametrize("fused_entry", [False, True], ids=["bgr2lab_then_slic", "slic_bgr"])
def test_emu_camera_chain_from_bgr(emu_lib, fused_entry):
    check_chain(emu_lib, 2, 48, 80, 9, 50, lambda a: a, fused_entry)


@pytest.mark.gpu
@pytest.mark.parametrize("fused_entry", [False, True], ids=["bgr2lab_then_slic", "slic_bgr"])
@pytest.mark.parametrize("mode", ["host", "device"])
def test_gpu_camera_chain_from_bgr(gpu_lib, mode, fused_entry):
    import torch

    to_backend = (lambda a: a) if mode == "host" else (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda())
    # main_lc.cpp:187-201: step = sqrt(rows * cols / 1200) = 18.9 -> 18 as an int parameter, nc = 50
    check_chain(gpu_lib, 2, synth.KITTI_ROWS, synth.KITTI_COLS, np.sqrt(synth.KITTI_ROWS * synth.KITTI_COLS / 1200.0), 50, to_backend,
                fused_entry)


# ---- dcmt::bgr2lab of include/img_completion.h (the OpenCV-free MatView half) ------------------------------------------
def compile_lab_shim(tmp_path, lib_path):
    exe = str(tmp_path / "shim_lab_main")
    libdir, libname = os.path.dirname(lib_path), os.path.basename(lib_path)[3:-3]
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "shim_lab_main.cpp"), "-o", exe, "-L", libdir, "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def run_lab_shim(exe, tmp_path, bgr, pad):
    fin, fout = tmp_path / "bgr.u8", tmp_path / "lab.u8"
    bgr.tofile(fin)
    r = subprocess.run([exe, str(bgr.shape[0]), str(bgr.shape[1]), str(fin), str(fout), str(pad)], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (r.returncode, r.stderr)
    return np.fromfile(fout, np.uint8).reshape(bgr.shape)


def test_shim_bgr2lab_on_emulator(tmp_path, emu_lib):
    exe = compile_lab_shim(tmp_path, emu_lib.path)
    bgr = synth.bgr_image(5, 31, 45)
    for pad in (0, 5, 16):
        assert np.array_equal(run_lab_shim(exe, tmp_path, bgr, pad), oracle_lab(bgr)), pad


@pytest.mark.gpu
def test_shim_bgr2lab_on_gpu(tmp_path, gpu_lib):
    exe = compile_lab_shim(tmp_path, gpu_lib.path)
    bgr = synth.bgr_image(6)
    for pad in (0, 7):
        assert np.array_equal(run_lab_shim(exe, tmp_path, bgr, pad), oracle_lab(bgr)), pad
