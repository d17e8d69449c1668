"""The camera program's front in one call (dcmt_interpolate_with_superpixels_bgr_*, main_lc.cpp:159-220): BGR frame ->
Lab -> SLIC -> guided completion of KITTI uint16 depth, with the Lab frames and labels kept on the device.  Checked byte
for byte against the two calls it replaces (dcmt_slic_bgr_u8c3 + dcmt_interpolate_with_superpixels_u16[_u16]) and
against the C oracle chain, on every entry point, layout, chunking and device list; plus the argument errors and the
C++ shim's overloads."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, api, synth
from oracle import c_oracle as co
from oracle import lab_oracle
from tests.conftest import ROOT, assert_bit_equal
from tests.test_kitti_u16 import rule_u16

AUTO, GENERIC = 0, 1
STEP, NC = 9, 50


def frames(n, rows, cols, seed=0):
    bgr = np.stack([synth.bgr_image(seed + f, rows, cols) for f in range(n)])
    s16 = np.stack([synth.sparse_depth_q8(seed + f, rows, cols, 0.06, kitti_like=True) for f in range(n)])
    return bgr, s16


def composition(lib, bgr, s16, step, nc, use_sp=1, flags=AUTO, u16_out=False, iterations=10):
    """the two host calls the chain replaces: SLIC from BGR, then the guided uint16 call on its labels"""
    n, rows, cols = s16.shape
    labels = np.empty((n, rows, cols), np.int32)
    lib.check(lib.dcmt_slic_bgr_u8c3_host(bgr.ctypes.data, rows, cols, n, step, nc, iterations, labels.ctypes.data, None))
    k = lib.dcmt_slic_center_count(rows, cols, step)
    out = np.empty((n, rows, cols), np.uint16 if u16_out else np.float32)
    stats = np.zeros((n, _lib.STATS_STRIDE), np.int32)
    fn = lib.dcmt_interpolate_with_superpixels_u16_u16_host if u16_out else lib.dcmt_interpolate_with_superpixels_u16_host
    lib.check(fn(s16.ctypes.data, labels.ctypes.data, k, out.ctypes.data, rows, cols, 0, 0, 0, 0, n, use_sp, flags, stats.ctypes.data))
    return out, stats


def chain(lib, bgr, s16, step, nc, use_sp=1, flags=AUTO, u16_out=False, form="_host", iterations=10, devices=(0,)):
    """one chained call on dense numpy planes; form "" is the device entry point (host memory is device memory on the
    emulator)"""
    n, rows, cols = s16.shape
    out = np.empty((n, rows, cols), np.uint16 if u16_out else np.float32)
    stats = np.zeros((n, _lib.STATS_STRIDE), np.int32)
    fn = getattr(lib, "dcmt_interpolate_with_superpixels_bgr_" + ("u16_u16" if u16_out else "u16") + form)
    args = [bgr.ctypes.data, 0, 0, s16.ctypes.data, out.ctypes.data, rows, cols, 0, 0, 0, 0, n, step, nc, iterations, use_sp, flags,
            stats.ctypes.data]
    if form == "_host_multi":
        args += [(C.c_int * len(devices))(*devices), len(devices)]
    elif form == "":
        args += [None]
    lib.check(fn(*args))
    return out, stats


def oracle_chain(lib, bgr, s16, step, nc, use_sp=1, u16_out=False):
    """lab_oracle.bgr2lab -> co.slic -> co.interpolate_with_superpixels on u16 / 256, per frame"""
    rows, cols = s16.shape[1:]
    k = lib.dcmt_slic_center_count(rows, cols, step)
    outs = []
    for f in range(len(s16)):
        labels, _ = co.slic(lab_oracle.bgr2lab(bgr[f]), step, nc)
        d = co.interpolate_with_superpixels(s16[f].astype(np.float32) / np.float32(256), labels, k, use_superpixel=use_sp)
        outs.append(rule_u16(d) if u16_out else d)
    return np.stack(outs)


# ---- emulator: every form, both outputs, both label modes, both paths --------------------------------------------------
@pytest.mark.parametrize("u16_out", [False, True], ids=["f32", "u16"])
def test_emu_chain_equals_composition_and_oracle(emu_lib, u16_out):
    bgr, s16 = frames(3, 48, 80, 11)
    for use_sp in (1, 0):
        want = oracle_chain(emu_lib, bgr, s16, STEP, NC, use_sp, u16_out)
        for flags in (AUTO, GENERIC):
            ref, ref_st = composition(emu_lib, bgr, s16, STEP, NC, use_sp, flags, u16_out)
            assert_bit_equal(ref, want, f"composition vs oracle, use_superpixel {use_sp}, flags {flags}")
            for form in ("", "_host", "_host_multi"):
                what = f"form {form or 'device'}, use_superpixel {use_sp}, flags {flags}"
                got, st = chain(emu_lib, bgr, s16, STEP, NC, use_sp, flags, u16_out, form)
                assert_bit_equal(got, ref, what)
                assert_bit_equal(st, ref_st, what + ": stats")
            assert [int(v) for v in ref_st[:, 3]] == [0 if flags == GENERIC else 1] * 3


def test_emu_layouts_and_odd_shapes(emu_lib):
    """a pitched BGR ROI, pitched and gapped depth planes, and frames down to 1 x N / N x 1"""
    rows, cols, n = 37, 53, 2
    bgr, s16 = frames(n, rows, cols, 21)
    for u16_out in (False, True):
        ref, ref_st = composition(emu_lib, bgr, s16, STEP, NC, u16_out=u16_out)
        et = np.uint16 if u16_out else np.float32
        # the BGR frames as an ROI (rows 2.., columns 3..) of larger frames with a gap between frames
        big = np.zeros((n, rows + 5, cols + 7, 3), np.uint8)
        big[:, 2:2 + rows, 3:3 + cols] = bgr
        fb = big.strides[0] + 96
        bgr_buf = np.zeros(n * fb, np.uint8)
        for f in range(n):
            bgr_buf[f * fb:f * fb + big[f].nbytes] = big[f].ravel()
        roi = bgr_buf.ctypes.data + 2 * big.strides[1] + 3 * 3
        # depth planes: rows padded by 6 elements, frames 40 bytes apart beyond that; the output padded differently
        sp, sf = (cols + 6) * 2, (cols + 6) * 2 * rows + 40
        s_buf = np.zeros(n * sf // 2, np.uint16)
        for f in range(n):
            s_buf.view(np.uint8)[f * sf:f * sf + rows * sp].view(np.uint16).reshape(rows, cols + 6)[:, :cols] = s16[f]
        op = (cols + 3) * np.dtype(et).itemsize
        of = op * rows + 64
        o_buf = np.full(n * of, 0xA5, np.uint8)
        st = np.zeros((n, _lib.STATS_STRIDE), np.int32)
        for form in ("", "_host", "_host_multi"):
            o_buf[:] = 0xA5
            fn = getattr(emu_lib, "dcmt_interpolate_with_superpixels_bgr_" + ("u16_u16" if u16_out else "u16") + form)
            args = [roi, big.strides[1], fb, s_buf.ctypes.data, o_buf.ctypes.data, rows, cols, sp, sf, op, of, n, STEP, NC, 10, 1, AUTO,
                    st.ctypes.data]
            args += {"": [None], "_host": [], "_host_multi": [(C.c_int * 1)(0), 1]}[form]
            emu_lib.check(fn(*args))
            for f in range(n):
                plane = o_buf[f * of:f * of + op * rows].reshape(rows, op)
                assert_bit_equal(plane[:, :cols * np.dtype(et).itemsize].copy().view(et), ref[f], f"pitched {form or 'device'} frame {f}")
                assert (plane[:, cols * np.dtype(et).itemsize:] == 0xA5).all(), "row padding written"
                assert (o_buf[f * of + op * rows:(f + 1) * of] == 0xA5).all(), "frame gap written"
            assert_bit_equal(st, ref_st, f"pitched {form or 'device'} stats")
    for shape in ((1, 41), (33, 1), (5, 7), (9, 9)):
        bgr, s16 = frames(2, *shape, seed=31)
        s16[:, ::2, ::3] = 1000  # dense enough that tiny frames have something to complete
        for u16_out in (False, True):
            ref, _ = composition(emu_lib, bgr, s16, 4, NC, u16_out=u16_out)
            assert_bit_equal(ref, oracle_chain(emu_lib, bgr, s16, 4, NC, 1, u16_out), f"{shape}: composition vs oracle")
            for form in ("", "_host", "_host_multi"):
                assert_bit_equal(chain(emu_lib, bgr, s16, 4, NC, u16_out=u16_out, form=form)[0], ref, f"{shape} {form or 'device'}")


_CHUNKED = r"""
import sys; sys.path.insert(0, %(root)r)
from tests.emu import build_emu
from depth_completion_mt_b200 import _lib
from tests.test_superpixels_bgr import frames, composition, chain, oracle_chain, STEP, NC
from tests.conftest import assert_bit_equal
lib = _lib.bind(build_emu.build())
bgr, s16 = frames(3, 48, 80, 41)
for u16_out in (False, True):
    ref, ref_st = composition(lib, bgr, s16, STEP, NC, u16_out=u16_out)
    assert_bit_equal(ref, oracle_chain(lib, bgr, s16, STEP, NC, 1, u16_out), "composition vs oracle")
    got, st = chain(lib, bgr, s16, STEP, NC, u16_out=u16_out, form="")
    assert_bit_equal(got, ref, "device entry in chunks of 2 + 1 frames")
    assert_bit_equal(st, ref_st, "stats in chunks")
print("CHUNKED_OK")
"""


def test_emu_device_entry_in_chunks(emu_lib):
    """chunks of 2 + 1 frames (the chunk size is read once per process): the last chunk is a single frame, which SLIC
    segments with its tile kernel instead of the band kernel -- same bytes"""
    env = dict(os.environ, DCMT_FUSED_CHUNK="2", DCMT_GENERIC_CHUNK="2")
    r = subprocess.run([sys.executable, "-c", _CHUNKED % {"root": ROOT}], capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert r.returncode == 0 and "CHUNKED_OK" in r.stdout, r.stdout + r.stderr


# ---- argument errors: exact codes, before any device work, outputs untouched -------------------------------------------
def test_emu_argument_errors(emu_lib):
    lib = emu_lib
    rows, cols, n = 24, 40, 2
    bgr, s16 = frames(n, rows, cols, 51)
    out = np.full((n, rows, cols), 0x5A5A, np.uint16)
    stats = np.full((n, _lib.STATS_STRIDE), 7, np.int32)
    B, U = _lib.DCMT_E_BADARG, _lib.DCMT_E_UNSUPPORTED
    good = dict(bgr=bgr.ctypes.data, bp=0, bf=0, s=s16.ctypes.data, o=out.ctypes.data, rows=rows, cols=cols, ip=0, if_=0, op=0, of=0,
                n=n, step=STEP, nc=NC, it=10, sp=1, flags=AUTO, st=stats.ctypes.data)
    cases = [
        ("null bgr", dict(bgr=None), B), ("null sparse", dict(s=None), B), ("null output", dict(o=None), B),
        ("step 3", dict(step=3), U), ("nc 0", dict(nc=0), B), ("iterations -1", dict(it=-1), B),
        ("bgr pitch below cols * 3", dict(bp=cols * 3 - 1), B), ("bgr frame stride too small", dict(bp=cols * 3 + 4, bf=(cols * 3 + 4) * rows - 5), B),
        ("output overlaps the depth input", dict(o=s16.ctypes.data + 2), B), ("output overlaps the BGR input", dict(o=bgr.ctypes.data + 3), B),
        ("flags", dict(flags=4), B), ("rows 0", dict(rows=0), B), ("n_frames -1", dict(n=-1), B),
        ("depth pitch below cols", dict(ip=cols * 2 - 2), B), ("2^24 columns", dict(rows=1, cols=1 << 24, n=0), U),
    ]
    for form in ("", "_host", "_host_multi"):
        fn = getattr(lib, "dcmt_interpolate_with_superpixels_bgr_u16_u16" + form)
        extra = {"": [None], "_host": [], "_host_multi": [(C.c_int * 1)(0), 1]}[form]
        for what, change, code in cases:
            a = dict(good, **change)
            rc = fn(a["bgr"], a["bp"], a["bf"], a["s"], a["o"], a["rows"], a["cols"], a["ip"], a["if_"], a["op"], a["of"], a["n"], a["step"],
                    a["nc"], a["it"], a["sp"], a["flags"], a["st"], *extra)
            assert rc == code, (form, what, rc, lib.dcmt_last_error())
            assert (out == 0x5A5A).all() and (stats == 7).all(), (form, what, "output written")
            assert (s16 == frames(n, rows, cols, 51)[1]).all()
    a = good
    for devs, nd in (([1], 1), ([0, 0], 2), ([0], 0), ([-1], 1)):
        rc = lib.dcmt_interpolate_with_superpixels_bgr_u16_u16_host_multi(
            a["bgr"], 0, 0, a["s"], a["o"], rows, cols, 0, 0, 0, 0, n, STEP, NC, 10, 1, AUTO, a["st"], (C.c_int * len(devs))(*devs), nd)
        assert rc == B, (devs, nd, rc)
        assert (out == 0x5A5A).all() and (stats == 7).all()
    # the float32 entry has no one-call form; a float32 `sparse` points to the two calls
    with pytest.raises(ValueError, match="generate_superpixels_bgr"):
        api.interpolate_with_superpixels_bgr(bgr, s16.astype(np.float32) / 256, STEP, NC, lib=lib)
    with pytest.raises(ValueError):
        api.interpolate_with_superpixels_bgr(bgr[:, :-1], s16, STEP, NC, lib=lib)


def test_emu_python_api(emu_lib):
    bgr, s16 = frames(2, 48, 80, 61)
    for out_dtype in (np.float32, np.uint16):
        u16_out = out_dtype is np.uint16
        ref, ref_st = composition(emu_lib, bgr, s16, STEP, NC, u16_out=u16_out)
        got, st = api.interpolate_with_superpixels_bgr(bgr, s16, STEP + 0.9, NC, out_dtype=out_dtype, return_stats=True, lib=emu_lib)
        assert_bit_equal(got, ref, "api, step truncated")
        assert_bit_equal(st, ref_st, "api stats")
        assert_bit_equal(api.interpolate_with_superpixels_bgr(bgr, s16, STEP, NC, out_dtype=out_dtype, devices=[0], lib=emu_lib), ref, "api devices")
        assert_bit_equal(api.interpolate_with_superpixels_bgr(bgr[1], s16[1], STEP, NC, out_dtype=out_dtype, lib=emu_lib), ref[1], "api one frame")


# ---- GPU at KITTI size: 81 frames = host chunks of 40 + 40 + 1 ---------------------------------------------------------
@pytest.mark.gpu
def test_gpu_chain_at_kitti_size(gpu_lib):
    import torch

    lib = gpu_lib
    rows, cols, n = synth.KITTI_ROWS, synth.KITTI_COLS, 81
    step = int(np.sqrt(rows * cols / 1200.0))  # main_lc.cpp:187-201: 18
    assert step == 18
    bgr, s16 = frames(n, rows, cols, 71)
    torch.cuda.set_device(0)
    tb, ts = torch.from_numpy(bgr).cuda(), torch.from_numpy(s16).cuda()
    n_dev = torch.cuda.device_count()
    for out_dtype in (np.float32, np.uint16):
        u16_out = out_dtype is np.uint16
        tdt = torch.uint16 if u16_out else torch.float32
        # the two-call device composition (what bench.py's lidar_camera_chain runs)
        k = lib.dcmt_slic_center_count(rows, cols, step)
        labels = api.generate_superpixels_bgr(tb, step, 50, lib=lib)
        dev_ref = api.interpolate_with_superpixels(labels, ts, n_clusters=k, out_dtype=tdt, lib=lib).cpu().numpy()
        ref, ref_st = composition(lib, bgr, s16, step, 50, u16_out=u16_out)
        assert_bit_equal(ref, dev_ref, "host and device compositions")
        want = oracle_chain(lib, bgr[[0, n - 1]], s16[[0, n - 1]], step, 50, 1, u16_out)
        assert_bit_equal(ref[[0, n - 1]], want, "composition vs oracle")
        s = torch.cuda.Stream()
        got, st = api.interpolate_with_superpixels_bgr(tb, ts, step, 50, out_dtype=tdt, return_stats=True, stream=s, lib=lib)
        s.synchronize()
        assert_bit_equal(got.cpu().numpy(), ref, f"device entry on a side stream {out_dtype.__name__}")
        assert_bit_equal(st.cpu().numpy(), ref_st, "device stats")
        got, st = api.interpolate_with_superpixels_bgr(bgr, s16, step, 50, out_dtype=out_dtype, return_stats=True, lib=lib)
        assert_bit_equal(got, ref, f"_host {out_dtype.__name__}")
        assert_bit_equal(st, ref_st, "_host stats")
        for devices in ([0], "all", list(range(n_dev))[::-1]):
            got, st = api.interpolate_with_superpixels_bgr(bgr, s16, step, 50, out_dtype=out_dtype, return_stats=True, devices=devices, lib=lib)
            assert_bit_equal(got, ref, f"_host_multi {devices} {out_dtype.__name__}")
            assert_bit_equal(st, ref_st, f"_host_multi {devices} stats")
        assert torch.cuda.current_device() == 0  # the caller's device is restored
    # use_superpixel 0 and the generic path on the device entry
    for use_sp, flags in ((0, AUTO), (1, GENERIC)):
        ref, _ = composition(lib, bgr[:3], s16[:3], step, 50, use_sp, flags)
        got = api.interpolate_with_superpixels_bgr(tb[:3], ts[:3], step, 50, use_superpixel=use_sp, path="generic" if flags else "auto",
                                                   lib=lib).cpu().numpy()
        assert_bit_equal(got, ref, f"device use_superpixel {use_sp} flags {flags}")


# ---- C++ shim: the MatView overloads (emulator, GPU) and the cv::Mat overloads (stand-in OpenCV headers) -----------------
REFSHIM = os.path.join(ROOT, "oracle", "refshim")


def compile_shim(tmp_path, lib_path, with_cv):
    exe = str(tmp_path / ("shim_bgr_cv" if with_cv else "shim_bgr"))
    libdir, libname = os.path.dirname(lib_path), os.path.basename(lib_path)[3:-3]
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include")]
    cmd += ["-I", REFSHIM] if with_cv else ["-DDCMT_NO_OPENCV"]
    cmd += [os.path.join(ROOT, "tests", "cpp", "shim_bgr_main.cpp"), "-o", exe, "-L", libdir, "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def body_shim(lib, tmp_path, rows, cols, step):
    bgr, s16 = frames(1, rows, cols, 81)
    ref32, _ = composition(lib, bgr, s16, step, NC)
    ref16, _ = composition(lib, bgr, s16, step, NC, u16_out=True)
    bgr[0].tofile(tmp_path / "bgr.u8")
    s16[0].tofile(tmp_path / "in.u16")
    for with_cv in (False, True):
        exe = compile_shim(tmp_path, lib.path, with_cv)
        r = subprocess.run([exe, str(rows), str(cols), str(tmp_path / "bgr.u8"), str(tmp_path / "in.u16"), str(step), str(NC), str(tmp_path / "o"), "12"],
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
        outs = ["view"] + (["mat"] if with_cv else [])
        for kind in outs:
            assert_bit_equal(np.fromfile(tmp_path / f"o_{kind}.f32", np.float32).reshape(rows, cols), ref32[0], f"shim {kind} float32")
            assert_bit_equal(np.fromfile(tmp_path / f"o_{kind}.u16", np.uint16).reshape(rows, cols), ref16[0], f"shim {kind} uint16")
        if with_cv:
            assert "type errors thrown: 3" in r.stdout, r.stdout


def test_shim_on_emulator(tmp_path, emu_lib):
    body_shim(emu_lib, tmp_path, 48, 80, STEP)


@pytest.mark.gpu
def test_shim_on_gpu(tmp_path, gpu_lib):
    body_shim(gpu_lib, tmp_path, synth.KITTI_ROWS, synth.KITTI_COLS, 18)
