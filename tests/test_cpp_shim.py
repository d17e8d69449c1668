"""include/img_completion.h (the header the reference includes but never shipped) compiles without OpenCV and a C++
caller written like src/DC_lidar_only/main.cpp:93 gets the oracle's bytes.  CPU: linked against the emulator
build; GPU: against libdcmt.so.  Without a GPU the product library makes the call fail loudly."""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

from depth_completion_mt_b200 import build, synth
from oracle import c_oracle as co
from oracle import ref_oracle as ro
from tests.conftest import ROOT, assert_bit_equal


def compile_shim(tmp_path, lib_path):
    exe = str(tmp_path / "shim_main")
    libdir, libname = os.path.dirname(lib_path), os.path.basename(lib_path)[3:-3]
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "shim_main.cpp"), "-o", exe, "-L", libdir, "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def run_shim(exe, tmp_path, s, blur):
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    s.tofile(fin)
    r = subprocess.run([exe, str(s.shape[0]), str(s.shape[1]), fin, fout, blur], capture_output=True, text=True, timeout=600)
    return r, (np.fromfile(fout, np.float32).reshape(s.shape) if r.returncode == 0 else None)


def check_eval(stdout, gt, dense):
    """the shim's evaluate_performance / evaluate_performances against the literal float32 loops"""
    mse, rmse, mae, mae2, rmse2 = (float(v) for v in stdout.split())
    assert abs(mse - co.evaluate(gt, dense, 0, 0)["mean_err"]) < 1e-4
    ref = co.evaluate(gt, dense, 0, 1)
    assert abs(rmse - ref["rmse"]) < 1e-3 and abs(mae - ref["mae"]) < 1e-3
    ref = co.evaluate(gt, dense, 2, 1)
    assert abs(rmse2 - ref["rmse"]) < 1e-3 and abs(mae2 - ref["mae"]) < 1e-3


def test_shim_on_emulator_matches_oracle(tmp_path, emu_lib):
    exe = compile_shim(tmp_path, emu_lib.path)
    for blur in ("gaussian", "none", "something else"):
        s = synth.sparse_depth(17, 60, 100, 0.05)
        r, out = run_shim(exe, tmp_path, s, blur)
        assert r.returncode == 0, r.stderr
        assert_bit_equal(out, co.img_completion(s, blur if blur in ("gaussian", "none") else "none"), f"shim {blur}")
        check_eval(r.stdout, s, out)


def test_shim_with_product_library_fails_loudly_without_gpu(tmp_path):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    exe = compile_shim(tmp_path, build.build_library())
    r, _ = run_shim(exe, tmp_path, synth.sparse_depth(17, 40, 48, 0.05), "gaussian")
    assert r.returncode == 4 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_shim_with_product_library_on_gpu(tmp_path, gpu_lib):
    exe = compile_shim(tmp_path, gpu_lib.path)
    s = synth.sparse_depth(3)
    r, out = run_shim(exe, tmp_path, s, "gaussian")
    assert r.returncode == 0, r.stderr
    assert_bit_equal(out, co.img_completion(s, "gaussian"), "shim on the GPU")
    check_eval(r.stdout, s, out)


# ---- the cv::Mat half of the header: the reference's own signatures on cv::Mat / Slic / EntryType ---------------------
# Compiled against the stand-in OpenCV / Eigen headers of oracle/refshim (containers only, test infrastructure); the
# program (tests/cpp/shim_cv_main.cpp) makes the calls of main.cpp:93, main_lc.cpp:219-220 and main_sl.cpp:1162-1246 the
# way the reference writes them.  Checked against the C restatement and -- where the prebuilt oracle/_ref travelled --
# against the reference's own compiled sources.
REFSHIM = os.path.join(ROOT, "oracle", "refshim")
REF_SLIC_DIR = os.path.join(ro._REF, "src", "DC_lidar_camera")  # the reference checkout ref_oracle builds from (DCMT_REFERENCE_DIR)


def compile_cv_shim(tmp_path, lib_path, reference_slic_h=False):
    exe = str(tmp_path / ("shim_cv_main_ref" if reference_slic_h else "shim_cv_main"))
    libdir, libname = os.path.dirname(lib_path), os.path.basename(lib_path)[3:-3]
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), "-I", REFSHIM]
    if reference_slic_h:  # the reference's class Slic: its declaration and its own slic.cpp, compiled where they lie
        cmd = [c for c in cmd if c not in ("-Wall", "-Wextra", "-Werror")]
        cmd += ["-w", "-DDCMT_TEST_REFERENCE_SLIC_H", "-I", REF_SLIC_DIR, os.path.join(REF_SLIC_DIR, "slic.cpp")]
    cmd += [os.path.join(ROOT, "tests", "cpp", "shim_cv_main.cpp"), "-o", exe, "-L", libdir, "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def _run(cmd):
    r = subprocess.run([str(c) for c in cmd], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.returncode, r.stderr)
    return r.stdout


def body_cv_shim(exe, tmp_path, rows, cols):
    from oracle import ref_oracle as ro

    have_ref = ro.available()
    # main.cpp:93 (float Mat) and main.cpp:75-93 (the uint16 PNG payload)
    d16 = synth.sparse_depth_q8(21, rows, cols, 0.05)
    s = d16.astype(np.float32) / np.float32(256)
    s.tofile(tmp_path / "s.f32")
    d16.tofile(tmp_path / "s.u16")
    for blur in ("gaussian", "none"):
        out = _run([exe, "lidar", rows, cols, tmp_path / "s.f32", tmp_path / "o.f32", blur])
        got = np.fromfile(tmp_path / "o.f32", np.float32).reshape(rows, cols)
        assert_bit_equal(got, co.img_completion(s, blur), f"cv::Mat img_completion {blur}")
        if have_ref:
            assert_bit_equal(got, ro.img_completion(s, blur), f"cv::Mat img_completion {blur} vs the reference build")
        assert abs(float(out.split()[0]) - co.evaluate(s, got, 0, 0)["mean_err"]) < 1e-4
        _run([exe, "lidar16", rows, cols, tmp_path / "s.u16", tmp_path / "o16.f32", blur])
        assert_bit_equal(np.fromfile(tmp_path / "o16.f32", np.float32).reshape(rows, cols), got, f"CV_16UC1 input {blur}")
    # main_lc.cpp:219-220: Slic::clusters is [col][row]
    lab, k = synth.superpixel_labels(21, rows, cols, 9)
    np.ascontiguousarray(lab.T).astype(np.int32).tofile(tmp_path / "lab.i32")
    _run([exe, "guided", rows, cols, tmp_path / "s.f32", tmp_path / "lab.i32", k, tmp_path / "g0.f32", tmp_path / "g1.f32"])
    assert_bit_equal(np.fromfile(tmp_path / "g0.f32", np.float32).reshape(rows, cols), co.img_completion(s, "gaussian"), "main_lc.cpp:219")
    g1 = np.fromfile(tmp_path / "g1.f32", np.float32).reshape(rows, cols)
    assert_bit_equal(g1, co.interpolate_with_superpixels(s, lab, k), "main_lc.cpp:220")
    if have_ref and rows * cols <= 64 * 96:  # the reference's per-superpixel loop is slow
        assert_bit_equal(g1, ro.interpolate_with_superpixels(lab, s, n_clusters=k), "main_lc.cpp:220 vs the reference build")
    # main_sl.cpp:1162-1246 on EntryType matrices
    dig, left, right = synth.stereo_pair(22, rows, cols)
    dig.tofile(tmp_path / "dig.f32")
    left.tofile(tmp_path / "l.u8")
    right.tofile(tmp_path / "r.u8")
    out = _run([exe, "stereo", rows, cols, tmp_path / "dig.f32", tmp_path / "l.u8", tmp_path / "r.u8", tmp_path / "disp.f32",
                tmp_path / "depth.f32", tmp_path / "er.f32"])
    disp = np.fromfile(tmp_path / "disp.f32", np.float32).reshape(rows, cols)
    depth = np.fromfile(tmp_path / "depth.f32", np.float32).reshape(rows, cols)
    er = np.fromfile(tmp_path / "er.f32", np.float32).reshape(rows, cols, 3)
    want_depth, want_disp = co.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)
    assert_bit_equal(disp, want_disp, "optimize_IG on EntryType matrices")
    assert_bit_equal(depth, want_depth, "retrieve_optimized_depth")
    dx, dy = co.measurement_derivatives(right.astype(np.float32))
    assert_bit_equal(er[..., 0], right.astype(np.float32), "entry values untouched")
    assert_bit_equal(er[..., 1], dx, "calculateMeasuementDerivatives dx")
    assert_bit_equal(er[..., 2], dy, "calculateMeasuementDerivatives dy")
    if have_ref:
        rdepth, rdisp = ro.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)
        assert_bit_equal(disp, rdisp, "optimize_IG vs the reference build")
        assert_bit_equal(depth, rdepth, "retrieve_optimized_depth vs the reference build")
    # the probe of calculateObservationDerivatives at (rows / 2, cols / 2 - 0.25): dr = 0, dc = -0.25 after rounding
    ok, value, gx, gy = out.split()
    r0, c = rows // 2, np.float32(cols // 2 - 0.25)
    c0 = int(np.float64(c) + 0.5)
    dc = np.float32(c - np.float32(c0))
    dc1 = np.float32(1.0 - np.float64(dc))
    v = right.astype(np.float32)
    assert int(ok) == 1
    assert np.float32(value) == np.float32(np.float32(v[r0, c0] * dc1) + np.float32(v[r0, c0 + 1] * dc))
    assert np.float32(gx) == np.float32(np.float32(dx[r0, c0] * dc1) + np.float32(dx[r0, c0 + 1] * dc))
    assert np.float32(gy) == np.float32(np.float32(dy[r0, c0] * dc1) + np.float32(dy[r0, c0 + 1] * dc))


def test_cv_shim_on_emulator(tmp_path, emu_lib):
    body_cv_shim(compile_cv_shim(tmp_path, emu_lib.path), tmp_path, 48, 80)


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_SLIC_DIR, "slic.h")), reason="reference tree not present")
def test_cv_shim_compiles_against_the_reference_slic_h(tmp_path, emu_lib):
    """the template in the header binds to the reference's own class Slic (src/DC_lidar_camera/slic.h:30-71)"""
    body_cv_shim(compile_cv_shim(tmp_path, emu_lib.path, reference_slic_h=True), tmp_path, 40, 64)


@pytest.mark.gpu
def test_cv_shim_with_product_library_on_gpu(tmp_path, gpu_lib):
    body_cv_shim(compile_cv_shim(tmp_path, gpu_lib.path), tmp_path, 352, 1216)
