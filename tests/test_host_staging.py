"""The single-shot host entry points: SLIC, the LiDAR projection, BGR2GRAY / BGR2Lab, the evaluations, the EntryType and
the CV_32FC1 Mat operations.

* A bad argument comes back as the status and message of the device entry point, before any byte of the caller's buffers
  is read: every case runs in a child process on buffers mapped PROT_NONE, so a read shows up as a signal, not a status.
* On pitched host layouts each one returns what its device entry point returns, leaves the padding between host rows
  alone, and keeps the caller's value where the Mat kernels skip a pixel."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BADARG, UNSUP = _lib.DCMT_E_BADARG, _lib.DCMT_E_UNSUPPORTED

# ------------------------------------------------------------------------------------------- rejection before any read
# One argument of a valid call replaced at a time.  "B" stands for the PROT_NONE mapping, ["B", k] for k bytes into it.
_B2 = ["B", 1 << 19]
_SLIC = ["B", 32, 32, 1, 8, 10, 10, _B2, None]
_PROJECT = ["B", 1, ["B", 4096], ["B", 8192], 64, 64, _B2, _B2, 1.0, 0.0, ["B", 12288]]
_COLOR = ["B", _B2, 8, 8, 0, 0, 1]
_EVAL_F32 = ["B", _B2, 8, 8, 0, 0, 1, 0.0, 0, ["B", 1 << 20]]
_EVAL_2 = ["B", _B2, 8, 8, 0, 0, 0, 0, 1, 0.0, 0, ["B", 1 << 20]]
_KITTI = ["B", _B2, 8, 8, 0, 0, 0, 0, 1, ["B", 1 << 20]]
_ENTRIES = ["B", 8, 8, 96, 12]
_OPT_IG = ["B", 96, ["B", 4096], 96, 12, _B2, 0, 8, 8, 4, 500.0, 255.0]
_MAT = ["B", 0, _B2, 0, 8, 8, 0.54, 959.0]


def _with(base, **at):
    a = list(base)
    for i, v in at.items():
        a[int(i[1:])] = v
    return a


def _cases():
    out = []
    for name in ("dcmt_slic_u8c3_host", "dcmt_slic_bgr_u8c3_host"):
        for what, st, kw in [("null image", BADARG, {"a0": None}), ("null labels", BADARG, {"a7": None}),
                             ("zero rows", BADARG, {"a1": 0}), ("negative frames", BADARG, {"a3": -1}),
                             ("step 2", UNSUP, {"a4": 2}), ("nc 0", BADARG, {"a5": 0}), ("iterations -1", BADARG, {"a6": -1}),
                             ("2^24 rows", UNSUP, {"a1": 1 << 24, "a2": 1}), ("over 2^30 pixels", UNSUP, {"a1": 32768, "a2": 32769}),
                             ("65536 frames", UNSUP, {"a3": 65536})]:
            out.append((f"{name}-{what}", name, _with(_SLIC, **kw), st))
    name = "dcmt_lidar_project_f32_host"
    for what, st, kw in [("null points", BADARG, {"a0": None}), ("null T", BADARG, {"a2": None}), ("null P", BADARG, {"a3": None}),
                         ("negative n_points", BADARG, {"a1": -1}), ("zero cols", BADARG, {"a5": 0}),
                         ("40000 x 40000", UNSUP, {"a4": 40000, "a5": 40000})]:
        out.append((f"{name}-{what}", name, _with(_PROJECT, **kw), st))
    name = "dcmt_bgr2gray_u8_host"
    for what, st, kw in [("null input", BADARG, {"a0": None}), ("null output", BADARG, {"a1": None}), ("zero rows", BADARG, {"a2": 0}),
                         ("negative frames", BADARG, {"a6": -1}), ("65536 rows", UNSUP, {"a2": 65536}),
                         ("65536 frames", UNSUP, {"a6": 65536}), ("input pitch", BADARG, {"a4": 23}), ("output pitch", BADARG, {"a5": 7})]:
        out.append((f"{name}-{what}", name, _with(_COLOR, **kw), st))
    name = "dcmt_bgr2lab_u8_host"
    for what, st, kw in [("null input", BADARG, {"a0": None}), ("null output", BADARG, {"a1": None}), ("zero rows", BADARG, {"a2": 0}),
                         ("negative frames", BADARG, {"a6": -1}), ("65536 frames", UNSUP, {"a6": 65536}),
                         ("2^31 pixels", UNSUP, {"a2": 46341, "a3": 46341}), ("input pitch", BADARG, {"a4": 23}),
                         ("output pitch", BADARG, {"a5": 23}), ("in place", BADARG, {"a1": "B"})]:
        out.append((f"{name}-{what}", name, _with(_COLOR, **kw), st))
    for name, base, pitch, mode in [("dcmt_evaluate_f32_host", _EVAL_F32, 4, 8), ("dcmt_evaluate_u16_host", _EVAL_2, 4, 10),
                                    ("dcmt_evaluate_u16_u16_host", _EVAL_2, 4, 10), ("dcmt_evaluate_kitti_f32_host", _KITTI, 4, None),
                                    ("dcmt_evaluate_kitti_u16_host", _KITTI, 4, None),
                                    ("dcmt_evaluate_kitti_u16_u16_host", _KITTI, 4, None)]:
        n_at = 6 if base is _EVAL_F32 else 8
        cases = [("null gt", BADARG, {"a0": None}), ("null result plane", BADARG, {"a1": None}),
                 ("null records", BADARG, {f"a{len(base) - 1}": None}), ("zero rows", BADARG, {"a2": 0}),
                 ("negative frames", BADARG, {f"a{n_at}": -1}), ("over 2^30 pixels", UNSUP, {"a2": 32768, "a3": 32769}),
                 ("gt pitch", BADARG, {"a4": 5}), ("gt frame stride", BADARG, {"a5": pitch})]
        if base is not _EVAL_F32:
            cases.append(("result pitch", BADARG, {"a6": 3}))
        if mode is not None:
            cases.append(("mode", BADARG, {f"a{mode}": 7}))
        out += [(f"{name}-{what}", name, _with(base, **kw), st) for what, st, kw in cases]
    name = "dcmt_entries_measurement_derivatives_host"
    for what, st, kw in [("null", BADARG, {"a0": None}), ("zero rows", BADARG, {"a1": 0}), ("65536 rows", UNSUP, {"a1": 65536}),
                         ("elem_stride 8", BADARG, {"a4": 8}), ("elem_stride 14", BADARG, {"a4": 14}),
                         ("row_step 95", BADARG, {"a3": 95}), ("row_step below the row", BADARG, {"a3": 84}),
                         ("misaligned", BADARG, {"a0": ["B", 2]})]:
        out.append((f"{name}-{what}", name, _with(_ENTRIES, **kw), st))
    name = "dcmt_entries_optimize_ig_host"
    for what, st, kw in [("null left", BADARG, {"a0": None}), ("right row_step", BADARG, {"a3": 95}), ("null disp", BADARG, {"a5": None}),
                         ("disp pitch", BADARG, {"a6": 30}), ("iterations -1", BADARG, {"a9": -1}), ("65536 rows", UNSUP, {"a7": 65536})]:
        out.append((f"{name}-{what}", name, _with(_OPT_IG, **kw), st))
    for name, base in [("dcmt_get_initial_disparity_mat_f32_host", _MAT), ("dcmt_retrieve_optimized_depth_mat_f32_host", _MAT + [80.0])]:
        for what, st, kw in [("zero rows", BADARG, {"a4": 0}), ("65536 rows", UNSUP, {"a4": 65536}), ("null input", BADARG, {"a0": None}),
                             ("null output", BADARG, {"a2": None}), ("input pitch", BADARG, {"a1": 30}),
                             ("output pitch", BADARG, {"a3": 33})]:
            out.append((f"{name}-{what}", name, _with(base, **kw), st))
    return out


# Binds the library without importing the package (and torch), maps the PROT_NONE buffer, calls the device entry point
# and then the host entry point with the same arguments (the device one with the default stream), and prints both
# statuses and messages.
_CHILD = r"""
import ctypes as C, importlib.util, json, sys
spec = importlib.util.spec_from_file_location("dcmt_lib", sys.argv[1])
m = importlib.util.module_from_spec(spec)
spec.loader.exec_module(m)
lib = m.bind(sys.argv[2])
libc = C.CDLL(None, use_errno=True)
libc.mmap.restype = C.c_void_p
libc.mmap.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_long]
buf = libc.mmap(None, 1 << 21, 0, 0x22, -1, 0)  # PROT_NONE, MAP_PRIVATE | MAP_ANONYMOUS
assert buf and buf != C.c_void_p(-1).value
name, args = json.loads(sys.argv[3])
args = [buf if a == "B" else buf + a[1] if isinstance(a, list) else a for a in args]
dev = getattr(lib, name[: -len("_host")])(*args, None)
dev_msg = lib.dcmt_last_error().decode()
host = getattr(lib, name)(*args)
print(json.dumps([dev, dev_msg, host, lib.dcmt_last_error().decode()]))
"""


@pytest.mark.parametrize("case", _cases(), ids=lambda c: c[0])
def test_emu_rejects_before_reading(emu_lib, case):
    what, name, args, want = case
    r = subprocess.run([sys.executable, "-c", _CHILD, os.path.join(ROOT, "depth_completion_mt_b200", "_lib.py"), emu_lib.path,
                        json.dumps([name, args])], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, f"{what}: child exited with {r.returncode} (a negative code is the signal that killed it)\n{r.stderr[-2000:]}"
    dev, dev_msg, host, host_msg = json.loads(r.stdout.strip().splitlines()[-1])
    assert dev == want, f"{what}: device entry point returned {dev} ({dev_msg})"
    assert (host, host_msg) == (dev, dev_msg), what


# ------------------------------------------------------------------------------------- host and device twins agree
class _Emu:
    """the emulator's device pointers are host pointers"""

    def put(self, a):
        c = np.array(a, copy=True)
        return c, c.ctypes.data

    def get(self, c):
        return c


class _Gpu:
    def put(self, a):
        import torch

        t = torch.from_numpy(np.array(a, copy=True)).cuda()
        return t, t.data_ptr()

    def get(self, t):
        import torch

        torch.cuda.synchronize()
        return t.cpu().numpy()


def _twins(lib, be, name, bufs, args, ro=()):
    """Runs `name` (host) and its device twin on copies of `bufs` ({key: array}); an argument that is a key of `bufs` is that
    buffer's pointer.  Returns {key: (host result, device result)} for the buffers not listed in `ro`."""
    host = {k: np.array(v, copy=True) for k, v in bufs.items()}
    dev = {k: be.put(v) for k, v in bufs.items()}
    lib.check(getattr(lib, name)(*[host[a].ctypes.data if isinstance(a, str) and a in host else a for a in args]))
    lib.check(getattr(lib, name[: -len("_host")])(*[dev[a][1] if isinstance(a, str) and a in dev else a for a in args], None))
    return {k: (host[k], be.get(dev[k][0])) for k in bufs if k not in ro}


def _same(pairs, what):
    for k, (h, d) in pairs.items():
        assert h.tobytes() == d.tobytes(), f"{what}: {k} differs between the host and the device entry point"


def body_twins(lib, be):
    rng = np.random.default_rng(11)
    u8 = lambda *s: rng.integers(0, 256, s, dtype=np.uint8)  # noqa: E731

    # BGR2GRAY: input pitch 47 for 13 * 3 bytes, output pitch 20 for 13; the padding of both starts at 7
    rows, cols, n = 9, 13, 2
    src, dst = u8(n * rows, 47), np.full((n * rows, 20), 7, np.uint8)
    r = _twins(lib, be, "dcmt_bgr2gray_u8_host", {"s": src, "d": dst}, ["s", "d", rows, cols, 47, 20, n], ro="s")
    _same(r, "bgr2gray")
    assert (r["d"][0][:, cols:] == 7).all()

    # EntryType planes of 16-byte elements in rows of row_step > cols * 16 bytes, random bytes in the row padding
    rows, cols = 7, 11
    step_l, step_r = cols * 16 + 20, cols * 16 + 36
    ent = rng.standard_normal((rows, step_l // 4)).astype(np.float32)
    r = _twins(lib, be, "dcmt_entries_measurement_derivatives_host", {"e": ent}, ["e", rows, cols, step_l, 16])
    _same(r, "entries derivatives")
    assert np.array_equal(r["e"][0][:, cols * 4:].view(np.uint32), ent[:, cols * 4:].view(np.uint32)), "row padding was written"
    assert not np.array_equal(r["e"][0], ent)
    left = r["e"][0]
    right = rng.standard_normal((rows, step_r // 4)).astype(np.float32)
    right[:, : cols * 4] = np.roll(left[:, : cols * 4], 4, axis=1)
    disp = np.abs(rng.standard_normal((rows, cols + 5))).astype(np.float32) * 2
    r = _twins(lib, be, "dcmt_entries_optimize_ig_host", {"l": left, "r": right, "d": disp},
               ["l", step_l, "r", step_r, 16, "d", (cols + 5) * 4, rows, cols, 3, 500.0, 255.0], ro="lr")
    _same(r, "entries optimize_IG")
    assert np.array_equal(r["d"][0][:, cols:], disp[:, cols:]) and not np.array_equal(r["d"][0], disp)

    # Mats with pitch > cols * 4; pixels <= 0 are skipped by both kernels and keep what the output held
    rows, cols = 6, 21
    src = rng.uniform(0.5, 80.0, (rows, cols + 3)).astype(np.float32)
    src[rng.random((rows, cols + 3)) < 0.3] = 0.0
    src[0, :3] = -1.0
    out = rng.uniform(-5.0, 5.0, (rows, cols + 9)).astype(np.float32)
    skip = src[:, :cols] <= 0
    for name, extra in [("dcmt_get_initial_disparity_mat_f32_host", [0.54, 959.0]),
                        ("dcmt_retrieve_optimized_depth_mat_f32_host", [0.54, 959.0, 80.0])]:
        r = _twins(lib, be, name, {"i": src, "o": out}, ["i", (cols + 3) * 4, "o", (cols + 9) * 4, rows, cols, *extra], ro="i")
        _same(r, name)
        got = r["o"][0]
        assert np.array_equal(got[:, cols:], out[:, cols:]), name
        assert np.array_equal(got[:, :cols][skip], out[:, :cols][skip]) and not np.array_equal(got[:, :cols][~skip], out[:, :cols][~skip]), name

    # SLIC on dense Lab and BGR frames, labels and centres
    rows, cols, n, step, nc, it = 24, 30, 2, 8, 10, 3
    img = u8(n, rows, cols, 3)
    k = lib.dcmt_slic_center_count(rows, cols, step)
    for name in ("dcmt_slic_u8c3_host", "dcmt_slic_bgr_u8c3_host"):
        bufs = {"i": img, "l": np.full((n, rows, cols), -7, np.int32), "c": np.full((n, k, 5), -7.0)}
        r = _twins(lib, be, name, bufs, ["i", rows, cols, n, step, nc, it, "l", "c"], ro="i")
        _same(r, name)
        assert (r["l"][0] >= 0).all()

    # the projection: the host entry point takes points at any address, the device one 16-byte aligned points
    rows, cols = 376, 1242
    pts = np.c_[rng.uniform(2, 60, 3000), rng.uniform(-20, 20, 3000), rng.uniform(-2, 1, 3000), rng.uniform(0, 1, 3000)].astype(np.float32)
    raw = np.zeros(pts.size * 4 + 8, np.uint8)
    unaligned = raw[4: 4 + pts.nbytes].view(np.float32).reshape(pts.shape)
    unaligned[...] = pts
    T = np.ascontiguousarray(synth.KITTI_T_VELO_TO_CAM, np.float32)
    P = np.ascontiguousarray(synth.KITTI_P_RECT_02, np.float32)
    planes = {"j": np.full((rows, cols), -3.0, np.float32), "n": np.full((rows, cols), -3.0, np.float32), "c": np.zeros(1, np.int32)}
    host = {k: v.copy() for k, v in planes.items()}
    lib.check(lib.dcmt_lidar_project_f32_host(unaligned.ctypes.data, len(pts), T.ctypes.data, P.ctypes.data, rows, cols,
                                              host["j"].ctypes.data, host["n"].ctypes.data, 1.0, 0.0, host["c"].ctypes.data))
    dev = {k: be.put(v) for k, v in planes.items()}
    d_pts = be.put(pts)
    lib.check(lib.dcmt_lidar_project_f32(d_pts[1], len(pts), T.ctypes.data, P.ctypes.data, rows, cols, dev["j"][1], dev["n"][1], 1.0, 0.0,
                                         dev["c"][1], None))
    _same({k: (host[k], be.get(dev[k][0])) for k in planes}, "lidar projection")
    assert host["c"][0] > 0


def test_emu_host_device_twins(emu_lib):
    body_twins(emu_lib, _Emu())


@pytest.mark.gpu
def test_gpu_host_device_twins(gpu_lib):
    body_twins(gpu_lib, _Gpu())
