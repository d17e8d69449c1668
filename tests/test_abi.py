"""The C-ABI boundary (include/dcmt.h): the library loads, exports every declared symbol, validates
arguments with the documented codes and -- on a machine without a GPU -- refuses to compute instead
of falling back to the CPU."""
from __future__ import annotations

import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, build
from tests.conftest import ROOT


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "dcmt.h")).read()
    return sorted(set(re.findall(r"DCMT_API\s+[\w\s\*]+?\b(dcmt_\w+)\s*\(", text)))


@pytest.fixture(scope="module")
def product_lib():
    return _lib.bind(build.build_library())


def test_header_symbols_match_binding():
    assert declared_symbols() == sorted(_lib.EXPORTED_SYMBOLS)


def test_library_exports_every_declared_symbol(product_lib):
    out = subprocess.run(["nm", "-D", "--defined-only", product_lib.path], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (dcmt_\w+)", out))
    assert set(declared_symbols()) <= exported
    assert not [s for s in exported if "oracle" in s], "the product must not link the oracle"
    assert product_lib.dcmt_version() == 200


def test_product_is_sm100a_cuda_and_does_not_link_oracle(product_lib):
    sass = subprocess.run(["cuobjdump", "-lelf", product_lib.path], capture_output=True, text=True).stdout
    assert "sm_100a" in sass, sass
    ldd = subprocess.run(["ldd", product_lib.path], capture_output=True, text=True).stdout
    assert "oracle" not in ldd and "opencv" not in ldd.lower()


def test_no_cpu_fallback_without_gpu(product_lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    s = np.zeros((8, 8), np.float32)
    out = np.empty_like(s)
    rc = product_lib.dcmt_img_completion_f32_host(s.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), 8, 8, 0, 0, 1, 1, 0, None)
    assert rc == _lib.DCMT_E_CUDA
    assert b"no CPU fallback" in product_lib.dcmt_last_error()
    with pytest.raises(_lib.DcmtError):
        from depth_completion_mt_b200 import api

        api.img_completion(s, lib=product_lib)


def test_argument_validation(emu_lib):
    """error behaviour of the ABI (validated before any device work; exercised on the emulator build)."""
    lib = emu_lib
    s = np.zeros((8, 8), np.float32)
    o = np.empty_like(s)
    sp, op = s.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p)
    call = lib.dcmt_img_completion_f32_host
    assert call(None, op, 8, 8, 0, 0, 1, 1, 0, None) == _lib.DCMT_E_BADARG
    assert call(sp, op, 0, 8, 0, 0, 1, 1, 0, None) == _lib.DCMT_E_BADARG
    assert call(sp, op, 8, 8, 0, 0, -1, 1, 0, None) == _lib.DCMT_E_BADARG
    assert call(sp, op, 8, 8, 30, 0, 1, 1, 0, None) == _lib.DCMT_E_BADARG  # pitch not a multiple of 4
    assert call(sp, op, 8, 8, 16, 0, 1, 1, 0, None) == _lib.DCMT_E_BADARG  # pitch < cols*4
    assert call(sp, op, 8, 8, 0, 0, 1, 7, 0, None) == _lib.DCMT_E_BADARG   # blur type
    assert call(sp, op, 8, 8, 0, 0, 1, 1, 9, None) == _lib.DCMT_E_BADARG   # flags
    assert call(sp, sp, 8, 8, 0, 0, 1, 1, 0, None) == _lib.DCMT_E_BADARG   # aliasing
    assert b"overlap" in lib.dcmt_last_error()
    assert call(sp, op, 8, 8, 0, 0, 0, 1, 0, None) == _lib.DCMT_OK          # empty batch is a no-op
    assert lib.dcmt_interpolate_with_superpixels_f32_host(sp, None, 4, op, 8, 8, 0, 0, 1, 1, None) == _lib.DCMT_E_BADARG
    assert lib.dcmt_stereo_refine_f32_host(sp, None, None, op, None, 8, 8, 1, None) == _lib.DCMT_E_BADARG
    assert lib.dcmt_status_string(_lib.DCMT_E_CUDA) == b"CUDA error"
    assert lib.dcmt_workspace_bytes(352, 1216, 1024) > 0


def test_python_api_rejects_wrong_types(emu_lib):
    from depth_completion_mt_b200 import api

    with pytest.raises(TypeError):
        api.img_completion(np.zeros((4, 4), np.float64), lib=emu_lib)
    with pytest.raises(ValueError):
        api.img_completion(np.zeros((4,), np.float32), lib=emu_lib)
    # any blur string other than gaussian/bilateral means "no blur" (img_completion.cpp:172-189)
    s = np.zeros((6, 6), np.float32)
    s[2, 3] = 5.0
    assert np.array_equal(api.img_completion(s, False, "whatever", lib=emu_lib), api.img_completion(s, False, "none", lib=emu_lib))


def test_raw_mat_file_roundtrip(tmp_path):
    """utils.cpp:15-58: `int rows, cols, depth, type, channels, nbytes` + payload (CV_32FC1 = type 5, CV_16UC1 = 2, CV_8UC3 = 16)."""
    import numpy as np

    from depth_completion_mt_b200 import api, synth

    for a, want_type in ((synth.sparse_depth(1, 20, 30), 5), (synth.sparse_depth_q8(1, 20, 30), 2), (synth.lab_image(1, 12, 16), 16)):
        f = str(tmp_path / "m.bin")
        api.write_M(f, a)
        hdr = np.fromfile(f, np.int32, 6)
        assert list(hdr[:2]) == [a.shape[0], a.shape[1]] and hdr[3] == want_type and hdr[5] == a.nbytes
        b = api.read_M(f)
        assert b.dtype == a.dtype and np.array_equal(a, b)


# ---- the multi-device host entry points (SURVEY 8e for a C-ABI caller): one call, frames split over the listed GPUs ---------
@pytest.mark.gpu
def test_host_multi_entry_points(gpu_lib):
    """dcmt_img_completion_{f32,u16}_host_multi: same bytes as the single-device call, for an explicit device list, for
    `all visible devices`, with more devices than frames, and with a non-q8 frame in the batch (redo on the device that
    served it).  Runs on one GPU (the list [0]); uses every GPU of the box when there are several."""
    import torch

    from depth_completion_mt_b200 import api, synth
    from oracle import c_oracle as co

    n_dev = torch.cuda.device_count()
    rows, cols = 97, 171
    d16 = np.stack([synth.sparse_depth_q8(600 + f, rows, cols, 0.05) for f in range(7)])
    s = d16.astype(np.float32) / np.float32(256)
    s[3] = synth.sparse_depth_float(603, rows, cols, 0.05)  # not strict q8: dictionary path, on whichever device got frame 3
    want = np.stack([co.img_completion(f, "none") for f in s])
    want16 = np.stack([co.img_completion(f.astype(np.float32) / np.float32(256), "none") for f in d16])
    for devices in ([0], "all", list(range(n_dev))[::-1]):
        got, st = api.img_completion(s, False, "none", devices=devices, return_stats=True, lib=gpu_lib)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"f32 multi {devices}"
        assert [int(v) for v in st[:, 3]] == [1, 1, 1, 2, 1, 1, 1]
        got = api.img_completion(d16, False, "none", devices=devices, lib=gpu_lib)
        assert np.array_equal(got.view(np.uint32), want16.view(np.uint32)), f"u16 multi {devices}"
    assert torch.cuda.current_device() == 0  # the caller's device is restored
    # argument errors: an ordinal out of range, a repeated ordinal
    import ctypes as C

    out = np.empty_like(s)
    for bad in ([n_dev], [0, 0]):
        arr = (C.c_int * len(bad))(*bad)
        rc = gpu_lib.dcmt_img_completion_f32_host_multi(s.ctypes.data, out.ctypes.data, rows, cols, 0, 0, len(s), 0, 0, None, arr, len(bad))
        assert rc == _lib.DCMT_E_BADARG, bad
    # the copy-only ceiling leg echoes the input
    echo = np.zeros_like(s)
    gpu_lib.check(gpu_lib.dcmt_debug_host_copy_f32(s.ctypes.data, echo.ctypes.data, rows, cols, len(s), None, 0))
    assert np.array_equal(echo, s)


def test_host_multi_rejects_bad_device_lists_without_gpu(product_lib):
    """argument validation happens before any device work"""
    import ctypes as C

    s = np.zeros((2, 8, 8), np.float32)
    out = np.empty_like(s)
    rc = product_lib.dcmt_img_completion_f32_host_multi(s.ctypes.data, out.ctypes.data, 8, 8, 0, 0, 2, 0, 0, None, (C.c_int * 1)(0), 0)
    assert rc in (_lib.DCMT_E_BADARG, _lib.DCMT_E_CUDA)


def test_host_multi_on_emulator(emu_lib):
    """the lane / redo logic of the multi-device host driver (one emulated device): same bytes as the plain host call,
    incl. a frame that falls through strict q8 -> dictionary and one that falls through to the generic pipeline"""
    from depth_completion_mt_b200 import api, synth
    from oracle import c_oracle as co

    rows, cols = 64, 96
    s = np.stack([synth.sparse_depth(700 + f, rows, cols, 0.05) for f in range(4)])
    s[1] = synth.sparse_depth_float(701, rows, cols, 0.05)
    s[2] = synth.sparse_depth_float(702, rows, cols, 0.05)
    s[2, 5, 5] = np.nan  # outside the parity domain: must still be routed to the generic pipeline, not crash
    got, st = api.img_completion(s, False, "none", devices=[0], return_stats=True, lib=emu_lib)
    assert [int(v) for v in st[:, 3]] == [1, 2, 0, 1]
    for f in (0, 1, 3):
        assert np.array_equal(got[f].view(np.uint32), co.img_completion(s[f], "none").view(np.uint32)), f
    plain = api.img_completion(s, False, "none", lib=emu_lib)
    assert np.array_equal(got.view(np.uint32), plain.view(np.uint32))
    # the copy-only ceiling leg echoes the input
    echo = np.zeros_like(s)
    emu_lib.check(emu_lib.dcmt_debug_host_copy_f32(s.ctypes.data, echo.ctypes.data, rows, cols, len(s), None, 0))
    assert np.array_equal(echo.view(np.uint32), s.view(np.uint32))


def test_q8_phase_cycles_on_emulator(emu_lib):
    """dcmt_debug_q8_phase_cycles runs the fused kernels with Gaussian blur: same bytes as DCMT_PATH_FUSED"""
    from depth_completion_mt_b200 import synth

    rows, cols = 64, 100
    s = synth.sparse_depth(710, rows, cols, 0.05)
    want = np.zeros_like(s)
    emu_lib.check(emu_lib.dcmt_img_completion_f32(s.ctypes.data, want.ctypes.data, rows, cols, 0, 0, 1, _lib.BLUR["gaussian"],
                                                  _lib.PATH["fused"], None, None))
    got = np.zeros_like(s)
    stamps = [np.zeros(1 << 12, np.int64) for _ in range(2)]
    tiles = C.c_int(0)
    rc = emu_lib.dcmt_debug_q8_phase_cycles(s.ctypes.data, got.ctypes.data, rows, cols, 1, stamps[0].ctypes.data,
                                            stamps[1].ctypes.data, C.byref(tiles), None)
    assert rc == _lib.DCMT_OK, emu_lib.dcmt_last_error()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert tiles.value == 1  # 64 x 100 fits one tile of at most 96 x 160
