"""KITTI uint16 output (uint16 = metres * 256, 0 = empty) and KITTI uint16 input on the guided path.

The rule is cv::Mat::convertTo(CV_16U, 256.0) of the float32 result: u = saturate_cast<uint16_t>(cvRound(v * 256)) -- round
half to even, clamp to [0, 65535], NaN -> 0.  dcmt_depth_to_u16 applies it on the device; every uint16-output entry point
must equal that rule applied to the float32-output entry point's result, bit for bit, whichever path (fused tail with its
uint16 store, generic pipeline with the conversion kernel) served the frame.  The guided uint16-input entry points must equal
dcmt_interpolate_with_superpixels_ex_f32 on u16 / 256, which tests/test_completion_parity.py pins to the C oracle.  Device
entry points are called directly so that pitches and offsets reach the kernels as given; on the emulator build the same
calls run on host memory."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, api, synth
from tests.conftest import ROOT, assert_bit_equal

NONE, GAUSSIAN, BILATERAL = 0, 1, 2
AUTO, GENERIC, FUSED, RANK = 0, 1, 2, 3


def rule_u16(v) -> np.ndarray:
    """numpy restatement of the rule: rint (half to even) of the exact product, clipped to [0, 65535], NaN -> 0"""
    v = np.asarray(v, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        s = v * np.float32(256)
        return np.where(np.isnan(s), 0, np.clip(np.rint(s), 0, 65535)).astype(np.uint16)


CRAFTED = np.array(
    [k / 256 + 0.5 / 256 for k in range(8)]  # ties k + 0.5 for even and odd k
    + [np.nextafter(np.float32(k / 256 + 0.5 / 256), np.float32(d)) for k in (0, 1, 2, 3, 100, 25599) for d in (-1, 1)]
    + [-0.0, 0.0, -1.0, -1e-30, -np.float32(0.5 / 256), 1e-45, 1e-40, 1.1754942e-38, 255.998, 255.998046875, 255.99609375, 256.0,
       256.00390625, 1e30, np.inf, -np.inf, np.nan, 100.0, 0.1015625, 80.0, 65535.0, 8388607.5, 2.0**31 / 256],
    np.float32)


class Dev:
    """a buffer in device memory (GPU) or host memory (emulator) with a host copy that reads it back"""

    def __init__(self, a: np.ndarray, on_gpu: bool):
        self.on_gpu = on_gpu
        if on_gpu:
            import torch

            self.t = torch.from_numpy(np.ascontiguousarray(a).copy()).cuda()
            self.ptr = self.t.data_ptr()
        else:
            self.a = np.ascontiguousarray(a).copy()
            self.ptr = self.a.ctypes.data

    def get(self) -> np.ndarray:
        if self.on_gpu:
            import torch

            torch.cuda.synchronize()
            return self.t.cpu().numpy()
        return self.a


def place(frames: np.ndarray, pitch: int, offset: int, fill):
    """frames (n, rows, cols) in a buffer with rows of `pitch` elements, frames of (rows + 1) * pitch, `offset` elements in"""
    n, rows, cols = frames.shape
    fstride = (rows + 1) * pitch
    buf = np.full(offset + n * fstride, fill, frames.dtype)
    buf[offset:].reshape(n, rows + 1, pitch)[:, :rows, :cols] = frames
    return buf, fstride


def unplace(buf: np.ndarray, shape, pitch: int, offset: int, fill, what: str):
    n, rows, cols = shape
    v = buf[offset:].reshape(n, rows + 1, pitch)
    outside = np.concatenate([v[:, :, cols:].ravel(), v[:, rows:].ravel(), buf[:offset]])
    assert (outside == fill).all(), f"{what}: elements outside the frames were written"
    return v[:, :rows, :cols].copy()


# ------------------------------------------------------------------ 1. the rule
def body_rule(lib, on_gpu):
    rng = np.random.default_rng(5)
    for (rows, cols, n), in_pitch, in_off, out_pitch, out_off in (
            ((3, 64, 2), 64, 0, 64, 0),     # dense and aligned: 16-byte loads, 8-byte stores
            ((4, 70, 3), 72, 0, 72, 0),     # ragged row end
            ((5, 45, 2), 47, 1, 49, 1),     # pitched and unaligned: pixel by pixel
            ((2, 33, 2), 36, 0, 40, 3)):    # loads aligned, stores not
        f = rng.uniform(-2, 300, (n, rows, cols)).astype(np.float32)
        flat = f.reshape(-1)
        flat[: len(CRAFTED)] = CRAFTED[: flat.size]
        src, in_fs = place(f, in_pitch, in_off, np.float32(7))
        dst, out_fs = place(np.zeros((n, rows, cols), np.uint16), out_pitch, out_off, np.uint16(0xBEEF))
        dst[:] = 0xBEEF
        d_src, d_dst = Dev(src, on_gpu), Dev(dst, on_gpu)
        lib.check(lib.dcmt_depth_to_u16(d_src.ptr + in_off * 4, d_dst.ptr + out_off * 2, rows, cols, in_pitch * 4, in_fs * 4, out_pitch * 2,
                                        out_fs * 2, n, None))
        got = unplace(d_dst.get(), (n, rows, cols), out_pitch, out_off, 0xBEEF, "depth_to_u16")
        assert_bit_equal(got, rule_u16(f), f"depth_to_u16 {rows}x{cols} pitches {in_pitch}/{out_pitch}")


def test_rule_restatement():
    """the numpy restatement itself on the values the format turns on: ties to even, saturation (65535.5 ties to 65536 and
    saturates), NaN, signed zero, infinities"""
    m = np.array([0.5, 1.5, 2.5, 3.5, 65535.488, 65535.5], np.float32) / np.float32(256)
    assert list(rule_u16(m)) == [0, 2, 2, 4, 65535, 65535]
    m = np.array([-0.0, -3.0, np.nan, np.inf, -np.inf, 1e30, 256.0], np.float32)
    assert list(rule_u16(m)) == [0, 0, 0, 65535, 0, 65535, 65535]


def test_rule_matches_opencv():
    """cv2.multiply(v, 256, dtype=CV_16U) goes through saturate_cast<ushort>(float) = saturate_cast<ushort>(cvRound(v)), the
    conversion of convertTo(CV_16U, 256).  It agrees with the rule wherever v * 256 fits an int; beyond that (and at +inf)
    OpenCV's x86 cvRound overflows to INT_MIN and gives 0, where the rule -- and the library -- saturate to 65535."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(11)
    v = np.concatenate([CRAFTED, rng.uniform(-5, 300, 20000).astype(np.float32),
                        (rng.integers(0, 1 << 17, 20000) / np.float32(512)).astype(np.float32)])[None, :]
    ref = cv2.multiply(v, np.full_like(v, 256.0), dtype=cv2.CV_16U)
    with np.errstate(over="ignore", invalid="ignore"):
        in_int = np.abs(v * np.float32(256)) < np.float32(2.0**31)
    assert in_int.sum() > 40000
    assert_bit_equal(rule_u16(v)[in_int], ref[in_int], "rule vs cv2 inside the int range")


# ------------------------------------------------------------------ 2. a1: img_completion
def run_a1(lib, on_gpu, u16, blur, flags, u16_out, out_pitch=None, out_off=0):
    """dcmt_img_completion_u16[_u16] on device buffers; returns (output frames, stats)"""
    n, rows, cols = u16.shape
    out_pitch = out_pitch or cols
    et = np.uint16 if u16_out else np.float32
    fill = et(0xBEEF) if u16_out else et(-3.0)
    dst, out_fs = place(np.zeros(u16.shape, et), out_pitch, out_off, fill)
    dst[:] = fill
    d_src, d_dst = Dev(u16, on_gpu), Dev(dst, on_gpu)
    d_st = Dev(np.zeros((n, _lib.STATS_STRIDE), np.int32), on_gpu)
    fn = lib.dcmt_img_completion_u16_u16 if u16_out else lib.dcmt_img_completion_u16
    esz = np.dtype(et).itemsize
    lib.check(fn(d_src.ptr, d_dst.ptr + out_off * esz, rows, cols, 0, 0, out_pitch * esz, out_fs * esz, n, blur, flags, d_st.ptr, None))
    return unplace(d_dst.get(), u16.shape, out_pitch, out_off, fill, "a1 output"), d_st.get()


def check_a1(lib, on_gpu, u16, blur, flags, what, want_path):
    f32, st_f = run_a1(lib, on_gpu, u16, blur, flags, False)
    got, st_u = run_a1(lib, on_gpu, u16, blur, flags, True)
    assert_bit_equal(got, rule_u16(f32), f"{what}: u16 output vs the rule on the float output")
    assert np.array_equal(st_u, st_f), f"{what}: stats differ"
    assert list(st_u[:, 3]) == [want_path] * len(u16), f"{what}: paths {list(st_u[:, 3])}"
    if blur == NONE:  # lossless: u / 256 is the float output
        assert_bit_equal(got.astype(np.float32) / np.float32(256), f32, f"{what}: u / 256 vs float output")
    # pitched and unaligned output: the per-pixel store of the tail / the scalar path of the conversion kernel
    got_p, _ = run_a1(lib, on_gpu, u16, blur, flags, True, out_pitch=u16.shape[2] + 3, out_off=1)
    assert_bit_equal(got_p, got, f"{what}: pitched, unaligned output")


def body_a1(lib, on_gpu, rows, cols):
    big = lambda d, kl, s: np.stack([synth.sparse_depth_q8(s + f, rows, cols, d, kitti_like=kl) for f in range(2)])
    for d, kl, name in ((0.05, False, "5 %"), (0.01, False, "1 %"), (0.05, True, "KITTI-like")):
        for blur in (GAUSSIAN, NONE):
            check_a1(lib, on_gpu, big(d, kl, 800), blur, AUTO, f"{rows}x{cols} {name} blur={blur}", 1)
    check_a1(lib, on_gpu, big(0.05, False, 810), GAUSSIAN, GENERIC, "DCMT_PATH_GENERIC", 0)
    ragged = np.stack([synth.sparse_depth_q8(820 + f, 45, 70, 0.06) for f in range(3)])
    check_a1(lib, on_gpu, ragged, GAUSSIAN, FUSED, "45x70", 1)
    check_a1(lib, on_gpu, ragged, BILATERAL, AUTO, "45x70 bilateral", 0)
    small = np.stack([synth.sparse_depth_q8(830 + f, 20, 30, 0.2) for f in range(2)])
    check_a1(lib, on_gpu, small, GAUSSIAN, RANK, "20x30", 0)
    one = np.array([[[1000]], [[0]]], np.uint16)
    check_a1(lib, on_gpu, one, NONE, AUTO, "1x1", 0)


# ------------------------------------------------------------------ 3. a2: interpolate_with_superpixels
def run_a2(lib, on_gpu, sparse, labels, k, use_sp, flags, kind, host=False):
    """kind: "f32" (ex_f32 on float input), "u16" or "u16_u16"; host=True: the *_host entry point on host arrays"""
    n, rows, cols = sparse.shape
    et = np.uint16 if kind == "u16_u16" else np.float32
    out = np.zeros(sparse.shape, et)
    st = np.zeros((n, _lib.STATS_STRIDE), np.int32)
    if host:
        args = (sparse.ctypes.data, labels.ctypes.data, k, out.ctypes.data, rows, cols)
        tail = (n, use_sp, flags, st.ctypes.data)
        if kind == "f32":
            lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32_host(*args, 0, 0, *tail))
        else:
            fn = lib.dcmt_interpolate_with_superpixels_u16_u16_host if kind == "u16_u16" else lib.dcmt_interpolate_with_superpixels_u16_host
            lib.check(fn(*args, 0, 0, 0, 0, *tail))
        return out, st
    d_s, d_l, d_o, d_st = Dev(sparse, on_gpu), Dev(labels, on_gpu), Dev(out, on_gpu), Dev(st, on_gpu)
    args = (d_s.ptr, d_l.ptr, k, d_o.ptr, rows, cols)
    tail = (n, use_sp, flags, d_st.ptr, None)
    if kind == "f32":
        lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32(*args, 0, 0, *tail))
    else:
        fn = lib.dcmt_interpolate_with_superpixels_u16_u16 if kind == "u16_u16" else lib.dcmt_interpolate_with_superpixels_u16
        lib.check(fn(*args, 0, 0, 0, 0, *tail))
    return d_o.get(), d_st.get()


def check_a2(lib, on_gpu, u16, labels, k, use_sp, what, want_path, flags=AUTO):
    f32 = u16.astype(np.float32) / np.float32(256)
    ref, st_ref = run_a2(lib, on_gpu, f32, labels, k, use_sp, AUTO, "f32")
    got, st = run_a2(lib, on_gpu, u16, labels, k, use_sp, flags, "u16")
    assert_bit_equal(got, ref, f"{what}: u16 input vs float input")
    assert list(st[:, 3]) == [want_path] * len(u16), f"{what}: paths {list(st[:, 3])}"
    assert np.array_equal(st[:, :3], st_ref[:, :3]), f"{what}: stats differ"
    got16, st16 = run_a2(lib, on_gpu, u16, labels, k, use_sp, flags, "u16_u16")
    assert_bit_equal(got16, rule_u16(ref), f"{what}: u16 output vs the rule")
    assert np.array_equal(st16, st), f"{what}: stats of the u16-output call differ"
    return got, got16


def body_a2(lib, on_gpu, rows, cols):
    u16 = np.stack([synth.sparse_depth_q8(900 + f, rows, cols, 0.05, kitti_like=bool(f & 1)) for f in range(2)])
    lab18 = np.stack([synth.superpixel_labels(900 + f, rows, cols, 18)[0] for f in range(2)])
    k18 = synth.superpixel_labels(900, rows, cols, 18)[1]
    check_a2(lib, on_gpu, u16, lab18, k18, 1, "per-label front", 1)
    # step 4: more labels per tile than the per-label table holds -- the word-by-word front
    lab4, k4 = synth.superpixel_labels(901, rows, cols, 4)
    lab4 = np.stack([lab4, lab4])
    check_a2(lib, on_gpu, u16, lab4, k4, 1, "word-by-word front", 1)
    unassigned = lab18.copy()
    unassigned[:, ::7, ::5] = -1
    unassigned[:, rows // 2:, : cols // 3] = -1
    check_a2(lib, on_gpu, u16, unassigned, k18, 1, "unassigned labels", 1)
    check_a2(lib, on_gpu, u16, lab18, 70000, 1, "n_clusters > 65535", 0)
    check_a2(lib, on_gpu, u16, lab18, k18, 1, "DCMT_PATH_GENERIC", 0, flags=GENERIC)
    check_a2(lib, on_gpu, u16, lab18, k18, 0, "use_superpixel = 0", 1)


# ------------------------------------------------------------------ 4. host variants
def body_host(lib, rows, cols, multi_devices):
    u16 = np.stack([synth.sparse_depth_q8(950 + f, rows, cols, 0.05) for f in range(5)])
    u16[3] = synth.sparse_depth_q8(953, rows, cols, 0.01)
    for blur in (GAUSSIAN, BILATERAL):
        f32 = api.img_completion(u16, False, blur, lib=lib)
        got, st = api.img_completion(u16, False, blur, out_dtype=np.uint16, return_stats=True, lib=lib)
        assert_bit_equal(got, rule_u16(f32), f"host a1 blur={blur}")
        _, st_f = api.img_completion(u16, False, blur, return_stats=True, lib=lib)
        assert np.array_equal(st, st_f)
        multi = api.img_completion(u16, False, blur, out_dtype=np.uint16, devices=multi_devices, lib=lib)
        assert_bit_equal(multi, got, f"host_multi a1 blur={blur}")
    lab, k = synth.superpixel_labels(950, rows, cols, 18)
    labs = np.stack([lab] * 5)
    ref = api.interpolate_with_superpixels(labs, u16.astype(np.float32) / np.float32(256), lib=lib)
    got = api.interpolate_with_superpixels(labs, u16, lib=lib)
    assert_bit_equal(got, ref, "host a2 u16 input")
    got16 = api.interpolate_with_superpixels(labs, u16, out_dtype=np.uint16, lib=lib)
    assert_bit_equal(got16, rule_u16(ref), "host a2 u16 output")
    n, rows_, cols_ = u16.shape
    for fn, et, want in ((lib.dcmt_interpolate_with_superpixels_u16_host_multi, np.float32, ref),
                         (lib.dcmt_interpolate_with_superpixels_u16_u16_host_multi, np.uint16, got16)):
        out = np.zeros(u16.shape, et)
        dev = (C.c_int * len(multi_devices))(*multi_devices)
        lib.check(fn(u16.ctypes.data, labs.ctypes.data, k, out.ctypes.data, rows_, cols_, 0, 0, 0, 0, n, 1, AUTO, None, dev, len(multi_devices)))
        assert_bit_equal(out, want, f"host_multi a2 {np.dtype(et).name}")
    # pitched host output
    out = np.full((n, rows + 1, cols + 5), 0xBEEF, np.uint16)
    lib.check(lib.dcmt_img_completion_u16_u16_host(u16.ctypes.data, out.ctypes.data, rows, cols, 0, 0, (cols + 5) * 2, (rows + 1) * (cols + 5) * 2,
                                                   n, GAUSSIAN, AUTO, None))
    assert_bit_equal(out[:, :rows, :cols], api.img_completion(u16, False, "gaussian", out_dtype=np.uint16, lib=lib), "pitched host output")
    assert (out[:, rows:] == 0xBEEF).all() and (out[:, :, cols:] == 0xBEEF).all()
    echo = np.zeros_like(u16)
    lib.check(lib.dcmt_debug_host_copy_u16_u16(u16.ctypes.data, echo.ctypes.data, rows, cols, n, None, 0))
    assert np.array_equal(echo, u16), "dcmt_debug_host_copy_u16_u16 must echo its input"
    zeros = np.full(u16.shape, 7.0, np.float32)
    lib.check(lib.dcmt_debug_host_copy_u16(u16.ctypes.data, zeros.ctypes.data, rows, cols, n, None, 0))
    assert not zeros.any(), "dcmt_debug_host_copy_u16 must leave a float output all zeros"


# ------------------------------------------------------------------ 5. argument errors
def body_errors(lib, on_gpu):
    rows, cols, n = 8, 10, 2
    buf = Dev(np.zeros(4096, np.uint16), on_gpu)
    p = buf.ptr
    lab = Dev(np.zeros(n * rows * cols, np.int32), on_gpu)
    BAD = _lib.DCMT_E_BADARG
    a1 = lib.dcmt_img_completion_u16_u16
    ok_out = p + 2048  # far enough from the input at p
    assert a1(None, ok_out, rows, cols, 0, 0, 0, 0, n, 1, 0, None, None) == BAD
    assert a1(p, None, rows, cols, 0, 0, 0, 0, n, 1, 0, None, None) == BAD
    assert a1(p, ok_out, rows, cols, 21, 0, 0, 0, n, 1, 0, None, None) == BAD, "odd input pitch"
    assert a1(p, ok_out, rows, cols, 18, 0, 0, 0, n, 1, 0, None, None) == BAD, "input pitch shorter than a row"
    assert a1(p, ok_out, rows, cols, 0, 0, 19, 0, n, 1, 0, None, None) == BAD, "odd output pitch"
    assert a1(p, ok_out, rows, cols, 0, 0, 18, 0, n, 1, 0, None, None) == BAD, "output pitch shorter than a row"
    assert a1(p, p + 100, rows, cols, 0, 0, 0, 0, n, 1, 0, None, None) == BAD, "overlap"
    assert a1(p, p, rows, cols, 0, 0, 0, 0, 0, 1, 0, None, None) == 0, "n_frames = 0 is a no-op"
    assert lib.dcmt_img_completion_u16_u16_host(None, None, rows, cols, 0, 0, 0, 0, n, 1, 0, None) == BAD
    for fn in (lib.dcmt_interpolate_with_superpixels_u16, lib.dcmt_interpolate_with_superpixels_u16_u16):
        assert fn(p, None, 4, ok_out, rows, cols, 0, 0, 0, 0, n, 1, 0, None, None) == BAD, "null labels"
        assert fn(p, lab.ptr, 4, None, rows, cols, 0, 0, 0, 0, n, 1, 0, None, None) == BAD
        assert fn(p, lab.ptr, 4, ok_out, rows, cols, 0, 0, 6, 0, n, 1, 0, None, None) == BAD, "short output pitch"
        assert fn(p, lab.ptr, 4, p + 20, rows, cols, 0, 0, 0, 0, n, 1, 0, None, None) == BAD, "overlap"
        assert fn(p, lab.ptr, 4, p, rows, cols, 0, 0, 0, 0, 0, 1, 0, None, None) == 0
    assert lib.dcmt_interpolate_with_superpixels_u16_host(p, None, 4, ok_out, rows, cols, 0, 0, 0, 0, n, 1, 0, None) == BAD
    d2u = lib.dcmt_depth_to_u16
    assert d2u(None, ok_out, rows, cols, 0, 0, 0, 0, n, None) == BAD
    assert d2u(p, None, rows, cols, 0, 0, 0, 0, n, None) == BAD
    assert d2u(p, ok_out, rows, cols, 42, 0, 0, 0, n, None) == BAD, "float pitch not a multiple of 4"
    assert d2u(p, ok_out, rows, cols, 36, 0, 0, 0, n, None) == BAD, "float pitch shorter than a row"
    assert d2u(p, ok_out, rows, cols, 0, 0, 21, 0, n, None) == BAD, "odd output pitch"
    assert d2u(p, p + 300, rows, cols, 0, 0, 0, 0, n, None) == BAD, "overlap"
    assert d2u(p, p, rows, cols, 0, 0, 0, 0, 0, None) == 0


# ------------------------------------------------------------------ 6. Python API
def body_python(lib, on_gpu):
    rows, cols = 40, 64
    u16 = np.stack([synth.sparse_depth_q8(990 + f, rows, cols, 0.05) for f in range(2)])
    f32 = u16.astype(np.float32) / np.float32(256)
    lab, k = synth.superpixel_labels(990, rows, cols, 9)
    labs = np.stack([lab, lab])
    if on_gpu:
        import torch

        dev = lambda a: torch.from_numpy(a).cuda()
        host = lambda t: t.cpu().numpy()
        u16_types = (np.uint16, torch.uint16, "uint16")
    else:
        dev = host = lambda a: a
        u16_types = (np.uint16, "uint16")
    ref = host(api.img_completion(dev(u16), lib=lib))
    assert ref.dtype == np.float32
    assert_bit_equal(host(api.img_completion(dev(u16), out_dtype=np.float32, lib=lib)), ref, "out_dtype float32")
    for t in u16_types:
        got = host(api.img_completion(dev(u16), out_dtype=t, lib=lib))
        assert_bit_equal(got, rule_u16(ref), f"out_dtype {t}")
        got2 = host(api.img_completion(dev(u16[0]), out_dtype=t, lib=lib))
        assert got2.shape == (rows, cols) and np.array_equal(got2, got[0])
    with pytest.raises(ValueError):
        api.img_completion(dev(f32), out_dtype=np.uint16, lib=lib)  # uint16 output needs uint16 input
    with pytest.raises(ValueError):
        api.img_completion(dev(u16), out_dtype=np.int32, lib=lib)
    with pytest.raises(ValueError):  # `out` must match the chosen dtype
        api.img_completion(dev(u16), out=dev(np.zeros(u16.shape, np.float32)), out_dtype=np.uint16, lib=lib)
    with pytest.raises(ValueError):
        api.img_completion(dev(u16), out=dev(np.zeros(u16.shape, np.uint16)), lib=lib)
    out = dev(np.zeros(u16.shape, np.uint16))
    api.img_completion(dev(u16), out=out, out_dtype=np.uint16, lib=lib)
    assert_bit_equal(host(out), rule_u16(ref), "caller-supplied uint16 out")
    g_ref = host(api.interpolate_with_superpixels(dev(labs), dev(f32), n_clusters=k, lib=lib))
    assert_bit_equal(host(api.interpolate_with_superpixels(dev(labs), dev(u16), n_clusters=k, lib=lib)), g_ref, "a2 uint16 input")
    assert_bit_equal(host(api.interpolate_with_superpixels(dev(labs), dev(u16), n_clusters=k, out_dtype=np.uint16, lib=lib)),
                     rule_u16(g_ref), "a2 uint16 output")
    with pytest.raises(ValueError):
        api.interpolate_with_superpixels(dev(labs), dev(f32), out_dtype=np.uint16, lib=lib)
    if on_gpu:
        got = host(api.depth_to_u16(dev(ref), lib=lib))
        assert_bit_equal(got, rule_u16(ref), "api.depth_to_u16")
        assert host(api.depth_to_u16(dev(ref[0]), lib=lib)).shape == (rows, cols)
        with pytest.raises(TypeError):
            api.depth_to_u16(dev(u16), lib=lib)
    with pytest.raises(TypeError):
        api.depth_to_u16(ref, lib=lib)  # host arrays: convert with numpy / OpenCV


# ------------------------------------------------------------------ multi-chunk (chunk size is read once per process)
_CHUNKED = r"""
import sys; sys.path.insert(0, %(root)r)
import numpy as np
from depth_completion_mt_b200 import _lib, synth
from tests.test_kitti_u16 import check_a1, check_a2, GAUSSIAN, NONE, BILATERAL, AUTO
on_gpu = %(gpu)r
if on_gpu:
    lib = _lib.load()
else:
    from tests.emu import build_emu
    lib = _lib.bind(build_emu.build())
rows, cols = %(shape)s
u16 = np.stack([synth.sparse_depth_q8(970 + f, rows, cols, 0.04) for f in range(5)])
check_a1(lib, on_gpu, u16, GAUSSIAN, AUTO, "chunked gaussian", 1)
check_a1(lib, on_gpu, u16, NONE, AUTO, "chunked none", 1)
check_a1(lib, on_gpu, u16, BILATERAL, AUTO, "chunked generic", 0)
lab, k = synth.superpixel_labels(970, rows, cols, 18)
check_a2(lib, on_gpu, u16, np.stack([lab] * 5), k, 1, "chunked guided", 1)
print("CHUNKED_OK")
"""


def run_chunked(on_gpu, shape):
    env = dict(os.environ, DCMT_FUSED_CHUNK="2", DCMT_GENERIC_CHUNK="2")
    code = _CHUNKED % {"root": ROOT, "gpu": on_gpu, "shape": shape}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert r.returncode == 0 and "CHUNKED_OK" in r.stdout, r.stdout + r.stderr


# ------------------------------------------------------------------ C++ shim (the OpenCV-free MatView half)
def body_shim(lib, tmp_path, rows, cols):
    libdir, libname = os.path.dirname(lib.path), os.path.basename(lib.path)[3:-3]
    exe = str(tmp_path / "shim_kitti_main")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "shim_kitti_main.cpp"), "-o", exe, "-L", libdir, "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    u16 = synth.sparse_depth_q8(995, rows, cols, 0.05)
    lab, k = synth.superpixel_labels(995, rows, cols, 18)
    u16.tofile(tmp_path / "in.u16")
    lab.tofile(tmp_path / "lab.i32")
    r = subprocess.run([exe, str(rows), str(cols), str(tmp_path / "in.u16"), str(tmp_path / "lab.i32"), str(k), str(tmp_path / "out"), "8"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.returncode, r.stderr)
    a1 = np.fromfile(tmp_path / "out_a1.raw", np.uint16).reshape(rows, cols)
    a2 = np.fromfile(tmp_path / "out_a2.raw", np.float32).reshape(rows, cols)
    a2u = np.fromfile(tmp_path / "out_a2u.raw", np.uint16).reshape(rows, cols)
    assert_bit_equal(a1, rule_u16(api.img_completion(u16, False, "gaussian", lib=lib)), "shim img_completion_u16_u16")
    ref = api.interpolate_with_superpixels(lab, u16.astype(np.float32) / np.float32(256), n_clusters=k, lib=lib)
    assert_bit_equal(a2, ref, "shim interpolate_with_superpixels_u16")
    assert_bit_equal(a2u, rule_u16(ref), "shim interpolate_with_superpixels_u16_u16")


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_shim(emu_lib, tmp_path):
    body_shim(emu_lib, tmp_path, 48, 72)


def test_emu_depth_to_u16(emu_lib):
    body_rule(emu_lib, False)


def test_emu_a1(emu_lib):
    body_a1(emu_lib, False, 64, 96)


def test_emu_a2(emu_lib):
    body_a2(emu_lib, False, 64, 96)


def test_emu_host_variants(emu_lib):
    body_host(emu_lib, 48, 72, [0])
    body_host(emu_lib, 45, 77, [0])  # width not a multiple of 8: device staging rows are padded past the host's


def test_emu_argument_errors(emu_lib):
    body_errors(emu_lib, False)


def test_emu_python_api(emu_lib):
    body_python(emu_lib, False)


def test_emu_chunked():
    run_chunked(False, "(48, 72)")


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
def test_gpu_depth_to_u16(gpu_lib):
    body_rule(gpu_lib, True)


@pytest.mark.gpu
def test_gpu_a1(gpu_lib):
    body_a1(gpu_lib, True, 352, 1216)


@pytest.mark.gpu
def test_gpu_a2(gpu_lib):
    body_a2(gpu_lib, True, 352, 1216)


@pytest.mark.gpu
def test_gpu_host_variants(gpu_lib):
    body_host(gpu_lib, 352, 1216, [0])
    body_host(gpu_lib, 45, 77, [0])


@pytest.mark.gpu
def test_gpu_argument_errors(gpu_lib):
    body_errors(gpu_lib, True)


@pytest.mark.gpu
def test_gpu_python_api(gpu_lib):
    body_python(gpu_lib, True)


@pytest.mark.gpu
def test_gpu_shim(gpu_lib, tmp_path):
    body_shim(gpu_lib, tmp_path, 352, 1216)


@pytest.mark.gpu
def test_gpu_chunked():
    run_chunked(True, "(352, 1216)")
