"""Evaluation on KITTI uint16 ground truth (dcmt_evaluate_u16, dcmt_evaluate_u16_u16 and their *_host variants).

A uint16 value u is decoded to (float)u * (1.0f / 256.0f), which is exact, so the records must be byte-equal to those of
dcmt_evaluate_f32 on the decoded planes whenever the float32 planes have the same pitch, frame stride and base alignment
counted in elements: both calls then make the same choice between the 4-pixel vector loads and the scalar loop, and
accumulate the same values in the same order.  Device entry points are called directly so that pitches and offsets reach
the kernel as given; on the emulator build the same calls run on host memory.  tests/test_evaluate.py pins the float32
call to the reference's loops."""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, api, synth
from oracle import c_oracle as co
from tests.conftest import ROOT

REC = np.dtype([("count", "f8"), ("sum_err", "f8"), ("sum_abs", "f8"), ("sum_sq", "f8"), ("mean_err", "f4"), ("mae", "f4"),
                ("rmse", "f4"), ("pad", "i4")])
SENTINEL = 0xA7


def decode(u: np.ndarray) -> np.ndarray:
    return u.astype(np.float32) / np.float32(256)


def aligned(n_elems: int, dtype) -> np.ndarray:
    """a zeroed host array whose first element is 256-byte aligned"""
    itemsize = np.dtype(dtype).itemsize
    raw = np.zeros(n_elems * itemsize + 256, np.uint8)
    off = (-raw.ctypes.data) % 256
    return raw[off:off + n_elems * itemsize].view(dtype)


class Buf:
    """an array in device memory (GPU) or host memory (emulator, host entry points); .ptr is what the call gets"""

    def __init__(self, a: np.ndarray, on_device: bool, offset: int = 0):
        self.on_device = on_device
        if on_device:
            import torch

            self.t = torch.from_numpy(a.view(np.uint8).copy()).cuda()  # the caching allocator's blocks are 512-byte aligned
            self.ptr = self.t.data_ptr() + offset * a.itemsize
        else:
            self.a = a
            self.ptr = a.ctypes.data + offset * a.itemsize

    def get(self) -> np.ndarray:
        if self.on_device:
            import torch

            torch.cuda.synchronize()
            return self.t.cpu().numpy()
        return self.a.view(np.uint8)


def place(frames: np.ndarray, pitch: int, fstride: int, offset: int) -> np.ndarray:
    """frames (n, rows, cols) at `offset` elements into an aligned buffer, rows `pitch` and frames `fstride` elements apart"""
    n, rows, cols = frames.shape
    buf = aligned(offset + (n - 1) * fstride + (rows - 1) * pitch + cols, frames.dtype)
    for f in range(n):
        for y in range(rows):
            s = offset + f * fstride + y * pitch
            buf[s:s + cols] = frames[f, y]
    return buf


class Caller:
    """the entry points of one library through one kind of pointer: "device" (the buffers live where the library computes)
    or "host" (the *_host variants on host arrays)"""

    def __init__(self, lib, kind: str, on_gpu: bool):
        self.lib, self.kind = lib, kind
        self.on_device = kind == "device" and on_gpu

    def results(self, n):
        return Buf(np.full(n * REC.itemsize, SENTINEL, np.uint8), self.on_device)

    def call(self, name, g, r, rows, cols, geo, n, tol, mode, res):
        fn = getattr(self.lib, name + ("_host" if self.kind == "host" else ""))
        args = [g.ptr, r.ptr, rows, cols] + list(geo) + [n, float(tol), mode, res.ptr]
        if self.kind == "device":
            args.append(None)
        return fn(*args)

    def records(self, name, gt, r, geo_g, geo_r, offset, tol, mode):
        """records of entry `name` on frames gt / r placed with geometries (pitch, frame stride) in elements"""
        n, rows, cols = gt.shape
        g = Buf(place(gt, *geo_g, offset), self.on_device, offset)
        q = Buf(place(r, *geo_r, offset), self.on_device, offset)
        res = self.results(n)
        if name == "dcmt_evaluate_f32":
            assert geo_g == geo_r
            geo = (geo_g[0] * 4, geo_g[1] * 4)
        else:
            geo = (geo_g[0] * gt.itemsize, geo_g[1] * gt.itemsize, geo_r[0] * r.itemsize, geo_r[1] * r.itemsize)
        self.lib.check(self.call(name, g, q, rows, cols, geo, n, tol, mode, res))
        return res.get().view(REC)


def frames(seed: int, n: int, rows: int, cols: int, empty: int | None = None):
    """KITTI-like GT codes (30 % valid, 0.5-80 m plus codes around 2 m), a float32 result and a uint16 result"""
    rng = np.random.default_rng(seed)
    shape = (n, rows, cols)
    gt = rng.integers(128, 20481, shape).astype(np.uint16)
    gt = np.where(rng.random(shape) < 0.1, rng.integers(500, 530, shape), gt).astype(np.uint16)
    gt = np.where(rng.random(shape) < 0.3, gt, 0).astype(np.uint16)
    if empty is not None:
        gt[empty] = 0
    r32 = (rng.uniform(0.0, 85, shape) * (rng.random(shape) < 0.9)).astype(np.float32)
    r16 = (rng.integers(0, 21761, shape) * (rng.random(shape) < 0.9)).astype(np.uint16)
    return gt, r32, r16


# (rows, cols, pitch, frame stride, offset, n frames) in elements; both planes and the float32 reference share them
LAYOUTS = {
    "dense_cols4": lambda: (9, 64, 64, 9 * 64, 0, 2),
    "ragged_1x1": lambda: (1, 1, 1, 1, 0, 3),
    "ragged_3": lambda: (9, 3, 3, 27, 0, 2),
    "ragged_13": lambda: (7, 13, 13, 7 * 13, 0, 2),
    "ragged_wide": lambda: (6, 1218, 1220, 6 * 1220, 0, 1),  # 304 4-pixel items per row, then a 2-pixel tail
    "pitch_not_8_bytes": lambda: (7, 64, 67, 7 * 67, 0, 2),  # 134-byte uint16 rows: scalar loop
    "base_offset_1": lambda: (5, 64, 64, 5 * 64, 1, 2),
    "frame_gaps": lambda: (5, 40, 44, 7 * 44, 0, 3),
    "batch_with_empty": lambda: (6, 72, 72, 6 * 72, 0, 5),
}


def check_bit_equal(got, want, what):
    assert got.tobytes() == want.tobytes(), f"{what}: records differ\n{got}\n{want}"


def body_layouts(caller, names=tuple(LAYOUTS)):
    for k, (name, layout) in enumerate(LAYOUTS.items()):
        if name not in names:
            continue
        rows, cols, pitch, fstride, offset, n = layout()
        gt, r32, r16 = frames(100 + k, n, rows, cols, empty=3 if name == "batch_with_empty" else None)
        geo = (pitch, fstride)
        for variant, (mode, tol) in api.EVAL_VARIANTS.items():
            got = caller.records("dcmt_evaluate_u16", gt, r32, geo, geo, offset, tol, mode)
            want = caller.records("dcmt_evaluate_f32", decode(gt), r32, geo, geo, offset, tol, mode)
            check_bit_equal(got, want, f"u16/f32 {name} {variant}")
            got = caller.records("dcmt_evaluate_u16_u16", gt, r16, geo, geo, offset, tol, mode)
            want = caller.records("dcmt_evaluate_f32", decode(gt), decode(r16), geo, geo, offset, tol, mode)
            check_bit_equal(got, want, f"u16/u16 {name} {variant}")
            if name == "batch_with_empty":
                assert got["count"][3] == 0
                for fld in ("mean_err", "mae", "rmse"):
                    assert np.isnan(got[fld][3]) and np.isnan(want[fld][3])
    # GT and result each with a geometry of its own (ragged columns: the packed float32 reference takes the scalar loop too)
    gt, r32, r16 = frames(7, 2, 11, 13)
    packed = (13, 11 * 13)
    for mode, tol in api.EVAL_VARIANTS.values():
        want = caller.records("dcmt_evaluate_f32", decode(gt), r32, packed, packed, 0, tol, mode)
        check_bit_equal(caller.records("dcmt_evaluate_u16", gt, r32, (18, 12 * 18), (15, 11 * 15), 0, tol, mode), want, "own geometries")
        want = caller.records("dcmt_evaluate_f32", decode(gt), decode(r16), packed, packed, 0, tol, mode)
        check_bit_equal(caller.records("dcmt_evaluate_u16_u16", gt, r16, (17, 11 * 17), (20, 13 * 20), 0, tol, mode), want, "own geometries")


def body_all_codes(caller):
    """one frame holding all 65 536 codes: 512 is exactly 2.0 and fails `gt > 2`, 513 passes"""
    gt = np.arange(65536, dtype=np.uint16).reshape(1, 256, 256)
    rng = np.random.default_rng(3)
    r32 = rng.uniform(0.0, 300.0, gt.shape).astype(np.float32)
    r16 = rng.integers(0, 65536, gt.shape).astype(np.uint16)
    geo = (256, 65536)
    for mode in (0, 1):
        for tol in (0, 2):
            for name, r, rf in (("dcmt_evaluate_u16", r32, r32), ("dcmt_evaluate_u16_u16", r16, decode(r16))):
                rec = caller.records(name, gt, r, geo, geo, 0, tol, mode)[0]
                g = decode(gt[0])
                mask = (g > tol) if mode == 0 else (g > tol) & (rf[0] > tol)
                assert int(rec["count"]) == co.evaluate(g, rf[0], tol, mode)["count"] == int(mask.sum())
                if mode == 0:
                    assert int(rec["count"]) == 65535 - 512 * tol // 2
                d = (g - rf[0])[mask].astype(np.float64)  # float32 subtraction, then exact sums
                for got, want in ((rec["sum_err"], d.sum()), (rec["sum_abs"], np.abs(d).sum()), (rec["sum_sq"], (d * d).sum())):
                    assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (name, mode, tol, got, want)


def body_arguments(caller):
    """every bad argument is DCMT_E_BADARG before any device work, with the results untouched"""
    rows, cols = 6, 10
    g16 = Buf(aligned(rows * cols, np.uint16), caller.on_device)
    r32 = Buf(aligned(rows * cols, np.float32), caller.on_device)
    r16 = Buf(aligned(rows * cols, np.uint16), caller.on_device)
    res = caller.results(1)
    null = type("Null", (), {"ptr": None})()
    for name, r, re in (("dcmt_evaluate_u16", r32, 4), ("dcmt_evaluate_u16_u16", r16, 2)):
        bad = [
            (null, r, rows, cols, (0, 0, 0, 0), 1, 0, res),
            (g16, null, rows, cols, (0, 0, 0, 0), 1, 0, res),
            (g16, r, rows, cols, (0, 0, 0, 0), 1, 0, null),
            (g16, r, rows, cols, (0, 0, 0, 0), 1, 2, res),  # mode
            (g16, r, rows, cols, (0, 0, 0, 0), 1, -1, res),
            (g16, r, 0, cols, (0, 0, 0, 0), 1, 0, res),
            (g16, r, rows, 0, (0, 0, 0, 0), 1, 0, res),
            (g16, r, rows, cols, (0, 0, 0, 0), -1, 0, res),
            (g16, r, rows, cols, (2 * cols + 1, 0, 0, 0), 1, 0, res),  # GT pitch not a multiple of 2
            (g16, r, rows, cols, (2 * cols - 2, 0, 0, 0), 1, 0, res),  # GT pitch too small
            (g16, r, rows, cols, (0, 2 * rows * cols + 1, 0, 0), 1, 0, res),  # GT frame stride not a multiple of 2
            (g16, r, rows, cols, (0, 2 * rows * cols - 2, 0, 0), 1, 0, res),  # GT frame stride too small
            (g16, r, rows, cols, (0, 0, re * cols + re // 2, 0), 1, 0, res),  # result pitch not a multiple of its element
            (g16, r, rows, cols, (0, 0, re * (cols - 1), 0), 1, 0, res),  # result pitch too small
            (g16, r, rows, cols, (0, 0, 0, re * rows * cols + re // 2), 1, 0, res),
            (g16, r, rows, cols, (0, 0, 0, re * (rows * cols - 1)), 1, 0, res),
        ]
        for i, (g, q, rr, cc, geo, n, mode, out) in enumerate(bad):
            assert caller.call(name, g, q, rr, cc, geo, n, 0.0, mode, out) == _lib.DCMT_E_BADARG, (name, i)
        assert caller.call(name, g16, r, rows, cols, (0, 0, 0, 0), 0, 0.0, 0, res) == _lib.DCMT_OK  # an empty batch is a no-op
    assert (res.get() == SENTINEL).all(), "results written by a rejected call"


def body_python(lib, to_backend, u16_dtype):
    """the reference flow main.cpp:75-101 on the PNG payloads: completion from uint16 input, scored against uint16 GT"""
    sparse = synth.sparse_depth_q8(11, 64, 96, 0.05)
    gt = synth.sparse_depth_q8(12, 64, 96, 0.3)
    d16 = api.img_completion(to_backend(sparse), False, "gaussian", out_dtype=u16_dtype, lib=lib)
    d32 = api.img_completion(to_backend(sparse), False, "gaussian", lib=lib)
    host = lambda x: x if isinstance(x, np.ndarray) else x.cpu().numpy()
    for dense, dense_f in ((d16, decode(host(d16))), (d32, host(d32))):
        for variant in api.EVAL_VARIANTS:
            got = api.evaluate(to_backend(gt), dense, variant, lib=lib)
            want = api.evaluate(to_backend(decode(gt)), to_backend(dense_f), variant, lib=lib)
            check_bit_equal(got, want, f"reference flow {variant}")
        assert api.evaluate_performance(to_backend(gt), dense, "lidar_only", lib=lib) == \
            api.evaluate_performance(to_backend(decode(gt)), to_backend(dense_f), "lidar_only", lib=lib)
        assert api.evaluate_performance(to_backend(gt), dense, lib=lib) == \
            api.evaluate_performance(to_backend(decode(gt)), to_backend(dense_f), lib=lib)
        assert api.evaluate_performances(to_backend(gt), dense, lib=lib) == \
            api.evaluate_performances(to_backend(decode(gt)), to_backend(dense_f), lib=lib)
    with pytest.raises(ValueError, match="uint16"):
        api.evaluate(to_backend(decode(gt)), d16, lib=lib)


def test_emu_layouts(emu_lib):
    body_layouts(Caller(emu_lib, "device", on_gpu=False))
    # the host variants stage each plane into device memory: the layouts whose bytes differ from a packed batch
    body_layouts(Caller(emu_lib, "host", on_gpu=False), ("pitch_not_8_bytes", "base_offset_1", "frame_gaps", "batch_with_empty"))


def test_emu_all_codes(emu_lib):
    for kind in ("device", "host"):
        body_all_codes(Caller(emu_lib, kind, on_gpu=False))


def test_emu_arguments(emu_lib):
    for kind in ("device", "host"):
        body_arguments(Caller(emu_lib, kind, on_gpu=False))


def test_emu_python(emu_lib):
    body_python(emu_lib, lambda a: a, np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["host", "device"])
def test_gpu_evaluate_u16(gpu_lib, kind):
    import torch

    caller = Caller(gpu_lib, kind, on_gpu=True)
    body_layouts(caller)
    body_all_codes(caller)
    body_arguments(caller)
    if kind == "host":
        body_python(gpu_lib, lambda a: a, np.uint16)
    else:
        body_python(gpu_lib, lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.uint16)


# ---- the cv::Mat overloads of include/img_completion.h on CV_16UC1 GT (tests/cpp/shim_eval_u16_main.cpp), compiled against
# the stand-in OpenCV headers of oracle/refshim
def compile_eval_shim(tmp_path, lib_path):
    exe = str(tmp_path / "shim_eval_u16_main")
    libdir, libname = os.path.dirname(lib_path), os.path.basename(lib_path)[3:-3]
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), "-I",
           os.path.join(ROOT, "oracle", "refshim"), os.path.join(ROOT, "tests", "cpp", "shim_eval_u16_main.cpp"), "-o", exe, "-L", libdir,
           "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def body_shim(exe, tmp_path, rows, cols):
    sparse = synth.sparse_depth_q8(31, rows, cols, 0.05)
    gt = synth.sparse_depth_q8(32, rows, cols, 0.3)
    sparse.tofile(tmp_path / "s.u16")
    gt.tofile(tmp_path / "gt.u16")
    r = subprocess.run([exe, str(rows), str(cols), str(tmp_path / "s.u16"), str(tmp_path / "gt.u16")], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, (r.returncode, r.stderr)
    lines = dict(l.split(":", 1) for l in r.stdout.strip().splitlines())
    # the figures of the CV_16UC1 GT equal those of the float32 Mats, for a float32 and for a uint16 result
    assert lines["u16 gt, f32 result"] == lines["f32 gt, f32 result"]
    assert lines["u16 gt, u16 result"] == lines["f32 gt, f32 of u16 result"]
    assert lines["f32 gt, u16 result"].strip() == "throws"
    mse, rmse, mae, mae2, rmse2 = (float(v) for v in lines["u16 gt, f32 result"].split())
    dense = co.img_completion(decode(sparse), "gaussian")
    assert abs(mse - co.evaluate(decode(gt), dense, 0, 0)["mean_err"]) < 1e-4
    ref = co.evaluate(decode(gt), dense, 0, 1)
    assert abs(rmse - ref["rmse"]) < 1e-3 and abs(mae - ref["mae"]) < 1e-3
    ref = co.evaluate(decode(gt), dense, 2, 1)
    assert abs(rmse2 - ref["rmse"]) < 1e-3 and abs(mae2 - ref["mae"]) < 1e-3


def test_eval_shim_on_emulator(tmp_path, emu_lib):
    body_shim(compile_eval_shim(tmp_path, emu_lib.path), tmp_path, 48, 80)


@pytest.mark.gpu
def test_eval_shim_with_product_library_on_gpu(tmp_path, gpu_lib):
    body_shim(compile_eval_shim(tmp_path, gpu_lib.path), tmp_path, 352, 1216)
