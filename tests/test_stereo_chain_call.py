"""The stereo program's per-frame chain in one call (dcmt_stereo_chain_f32*, main_sl.cpp:435-563 withSuperPixels and
:1162-1253): Velodyne clouds + BGR stereo pairs -> projection + cv::normalize(0, 80) -> SLIC of the left frame -> guided
completion of the normalised floats -> BGR2GRAY of both frames -> stereo refinement, with nothing in between leaving the
device.  Checked byte for byte against the five device calls it replaces and against the C oracle chain, on every form,
cloud layout, BGR layout, chunking and device list, including the redo of frames the dictionary cannot serve; plus every
argument error (before any read of the caller's buffers) and the C++ shim's overloads."""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, api, synth
from oracle import c_oracle as co
from oracle import lab_oracle
from oracle import ref_oracle as ro
from tests.conftest import ROOT, assert_bit_equal
from tests.test_host_staging import _Emu, _Gpu

AUTO, GENERIC, FUSED, RANK = 0, 1, 2, 3
STEP, NC = 9, 40
B, U = _lib.DCMT_E_BADARG, _lib.DCMT_E_UNSUPPORTED


def pinhole(rows, cols):
    """T = identity (the cloud is in camera coordinates), P a pinhole with f = cols at the image centre"""
    T = np.eye(4, dtype=np.float32)
    P = np.array([[cols, 0, cols / 2, 0], [0, cols, rows / 2, 0], [0, 0, 1, 0]], np.float32)
    return T, P


def back_project(rng, rows, cols, m=None, behind=False):
    """points that project onto pixel centres under pinhole(): m random pixels, or every pixel once (m None)"""
    if m is None:
        v, u = np.divmod(np.arange(rows * cols), cols)
    else:
        v, u = np.divmod(rng.integers(0, rows * cols, m), cols)
    z = rng.uniform(4.0, 40.0, len(u))
    x, y = (u + 0.5 - cols / 2) * z / cols, (v + 0.5 - rows / 2) * z / cols
    pts = np.c_[x, y, z, rng.uniform(0, 1, len(u))].astype(np.float32)
    if behind:
        pts[:, 2] *= -1
    return pts


class Scene:
    """n frames: clouds laid out cloud_stride points apart (max_points each, counts[f] used), BGR pairs"""

    def __init__(self, clouds, rows, cols, seed, extra_stride=0, with_counts=True):
        self.rows, self.cols, self.n = rows, cols, len(clouds)
        self.T, self.P = pinhole(rows, cols)
        self.max_points = max([len(c) for c in clouds] + [1])
        self.stride = self.max_points + extra_stride
        self.points = np.full((self.n, self.stride, 4), np.nan, np.float32)  # unread padding
        for f, c in enumerate(clouds):
            self.points[f, :len(c)] = c
        self.counts = np.array([len(c) for c in clouds], np.int32) if with_counts else None
        if not with_counts:
            assert all(len(c) == self.max_points for c in clouds)
        self.left = np.stack([synth.bgr_image(seed + f, rows, cols) for f in range(self.n)])
        self.right = np.roll(self.left, -3, axis=2).copy()

    def cloud(self, f):
        return self.points[f, :self.max_points if self.counts is None else self.counts[f]]


def scene(n, rows, cols, seed, m=300, **kw):
    rng = np.random.default_rng(seed)
    return Scene([back_project(rng, rows, cols, m + 37 * f) for f in range(n)], rows, cols, seed, **kw)


def gray(bgr):
    b, g, r = (bgr[..., i].astype(np.int32) for i in range(3))
    return ((3735 * b + 19235 * g + 9798 * r + 16384) >> 15).astype(np.uint8)


def params(lib):
    return api.stereo_params(lib=lib)


def composition(lib, be, sc, step=STEP, nc=NC, use_sp=1, flags=AUTO):
    """the five device calls the chain replaces (on the emulator, host memory is device memory): depth, disparity, stats"""
    n, rows, cols = sc.n, sc.rows, sc.cols
    held = []  # the device copies live until the results are read

    def put(a):
        held.append(be.put(a))
        return held[-1][1]

    plane = lambda dt: put(np.zeros((n, rows, cols), dt))  # noqa: E731
    pts, cnt = put(sc.points), (put(sc.counts) if sc.counts is not None else None)
    left, right = put(sc.left), put(sc.right)
    nrm, lab, dense, gl, gr = plane(np.float32), plane(np.int32), plane(np.float32), plane(np.uint8), plane(np.uint8)
    depth, disp, stats = plane(np.float32), plane(np.float32), put(np.zeros((n, _lib.STATS_STRIDE), np.int32))
    outs = held[-3:]
    lib.check(lib.dcmt_lidar_project_batch_f32(pts, cnt, sc.max_points, sc.stride, n, sc.T.ctypes.data, sc.P.ctypes.data, rows, cols, None, nrm,
                                               0.0, 80.0, None, None))
    lib.check(lib.dcmt_slic_bgr_u8c3(left, rows, cols, n, step, nc, 10, lab, None, None))
    k = lib.dcmt_slic_center_count(rows, cols, step)
    lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32(nrm, lab, k, dense, rows, cols, 0, 0, n, use_sp, GENERIC if flags == GENERIC else RANK,
                                                           stats, None))
    lib.check(lib.dcmt_bgr2gray_u8(left, gl, rows, cols, 0, 0, n, None))
    lib.check(lib.dcmt_bgr2gray_u8(right, gr, rows, cols, 0, 0, n, None))
    lib.check(lib.dcmt_stereo_refine_f32(dense, gl, gr, depth, disp, rows, cols, n, C.byref(params(lib)), None))
    return tuple(be.get(h) for h, _ in outs)


def chain(lib, sc, form, step=STEP, nc=NC, use_sp=1, flags=AUTO, devices=(0,), be=None):
    """one chained call; form "" is the device entry point (host memory on the emulator, `be` on the GPU)"""
    n, rows, cols = sc.n, sc.rows, sc.cols
    depth, disp = np.full((n, rows, cols), -7.0, np.float32), np.full((n, rows, cols), -7.0, np.float32)
    stats = np.full((n, _lib.STATS_STRIDE), -7, np.int32)
    bufs = dict(points=sc.points, counts=sc.counts, left=sc.left, right=sc.right, depth=depth, disp=disp, stats=stats)
    if form == "" and be is not None:
        held = {k: be.put(v) for k, v in bufs.items() if v is not None}
        ptr = {k: held[k][1] if k in held else None for k in bufs}
    else:
        ptr = {k: v.ctypes.data if v is not None else None for k, v in bufs.items()}
    args = [ptr["points"], ptr["counts"], sc.max_points, sc.stride, sc.T.ctypes.data, sc.P.ctypes.data, 0.0, 80.0, ptr["left"], ptr["right"], 0, 0,
            ptr["depth"], ptr["disp"], rows, cols, n, step, nc, 10, use_sp, flags, C.byref(params(lib)), ptr["stats"]]
    args += {"": [None], "_host": [], "_host_multi": [(C.c_int * len(devices))(*devices), len(devices)]}[form]
    lib.check(getattr(lib, "dcmt_stereo_chain_f32" + form)(*args))
    if form == "" and be is not None:
        return tuple(be.get(held[k][0]) for k in ("depth", "disp", "stats"))
    return depth, disp, stats


def oracle_chain(lib, sc, frames, step=STEP, nc=NC, use_sp=1):
    """lab_oracle.bgr2lab -> co.slic, co.lidar_project -> co.interpolate_with_superpixels, the gray formula, co.stereo_refine"""
    k = lib.dcmt_slic_center_count(sc.rows, sc.cols, step)
    depths, disps = [], []
    for f in frames:
        nrm = co.lidar_project(sc.cloud(f), sc.T, sc.P, sc.rows, sc.cols)[1]
        labels = co.slic(lab_oracle.bgr2lab(sc.left[f]), step, nc)[0] if use_sp else np.zeros((sc.rows, sc.cols), np.int32)
        dense = co.interpolate_with_superpixels(nrm, labels, k, use_superpixel=use_sp)
        d, p = co.stereo_refine(dense, gray(sc.left[f]), gray(sc.right[f]), return_disp=True)
        depths.append(d)
        disps.append(p)
    return np.stack(depths), np.stack(disps)


def same(got, want, what):
    for g, w, name in zip(got, want, ("depth", "disparity", "stats")):
        assert_bit_equal(g, w, f"{what}: {name}")


FORMS = ("", "_host", "_host_multi")


# ---- emulator ------------------------------------------------------------------------------------------------------------
def test_emu_chain_equals_composition_and_oracle(emu_lib):
    sc = scene(3, 40, 72, 11)
    for use_sp in (1, 0):
        want = oracle_chain(emu_lib, sc, range(sc.n), use_sp=use_sp)
        for flags in (AUTO, RANK, GENERIC):
            ref = composition(emu_lib, _Emu(), sc, use_sp=use_sp, flags=flags)
            assert_bit_equal(ref[0], want[0], f"composition vs oracle: depth, use_superpixel {use_sp}, flags {flags}")
            assert_bit_equal(ref[1], want[1], f"composition vs oracle: disparity, use_superpixel {use_sp}, flags {flags}")
            assert [int(v) for v in ref[2][:, 3]] == [0 if flags == GENERIC else 2] * 3
            for form in FORMS:
                same(chain(emu_lib, sc, form, use_sp=use_sp, flags=flags), ref, f"form {form or 'device'}, use_superpixel {use_sp}, flags {flags}")


def test_emu_ragged_clouds(emu_lib):
    """different sizes, a cloud of 0 points, a cloud entirely behind the camera, cloud_stride_points > max_points"""
    rows, cols = 36, 64
    rng = np.random.default_rng(5)
    clouds = [back_project(rng, rows, cols, 500), np.zeros((0, 4), np.float32), back_project(rng, rows, cols, 80, behind=True),
              back_project(rng, rows, cols, 120)]
    sc = Scene(clouds, rows, cols, 5, extra_stride=13)
    assert sc.stride > sc.max_points and list(sc.counts) == [500, 0, 80, 120]
    want = oracle_chain(emu_lib, sc, range(sc.n))
    ref = composition(emu_lib, _Emu(), sc)
    assert_bit_equal(ref[0], want[0], "composition vs oracle")
    for form in FORMS:
        same(chain(emu_lib, sc, form), ref, f"ragged {form or 'device'}")
    # no count array: max_points each, one 2-D copy of the clouds on the host forms
    sc = Scene([back_project(rng, rows, cols, 200) for _ in range(2)], rows, cols, 6, extra_stride=3, with_counts=False)
    ref = composition(emu_lib, _Emu(), sc)
    for form in FORMS:
        same(chain(emu_lib, sc, form), ref, f"no counts {form or 'device'}")


def body_redo(lib, be, forms):
    """sparse clouds around a dense one that lands on more than 32 768 distinct pixels: the dictionary serves the sparse
    frames (stats[3] 2) and the dense one is redone on the generic pipeline (stats[3] 0)"""
    rows, cols = 160, 224
    rng = np.random.default_rng(7)
    sc = Scene([back_project(rng, rows, cols, 1500), back_project(rng, rows, cols), back_project(rng, rows, cols, 900)], rows, cols, 7)
    assert rows * cols > 32768 + 1
    ref = composition(lib, be, sc)
    assert [int(v) for v in ref[2][:, 3]] == [2, 0, 2]
    for form in forms:
        same(chain(lib, sc, form, be=be), ref, f"redo {form or 'device'}")
    return sc, ref


def test_emu_redo_of_dense_frames(emu_lib):
    sc, ref = body_redo(emu_lib, _Emu(), ("", "_host"))
    assert_bit_equal(ref[0][1:2], oracle_chain(emu_lib, sc, [1])[0], "dense frame vs oracle")


def test_emu_layouts_and_odd_shapes(emu_lib):
    """a pitched BGR ROI with gapped frames, and frames of 1 x N / N x 1"""
    rows, cols, n = 37, 53, 2
    sc = scene(n, rows, cols, 21)
    ref = composition(emu_lib, _Emu(), sc)
    big_l, big_r = (np.zeros((n, rows + 5, cols + 7, 3), np.uint8) for _ in range(2))
    big_l[:, 2:2 + rows, 3:3 + cols], big_r[:, 2:2 + rows, 3:3 + cols] = sc.left, sc.right
    fb = big_l.strides[0] + 96
    bufs = []
    for big in (big_l, big_r):
        b = np.zeros(n * fb, np.uint8)
        for f in range(n):
            b[f * fb:f * fb + big[f].nbytes] = big[f].ravel()
        bufs.append(b)
    roi = [b.ctypes.data + 2 * big_l.strides[1] + 3 * 3 for b in bufs]
    for form in FORMS:
        depth, disp = np.full((n, rows, cols), -7.0, np.float32), np.full((n, rows, cols), -7.0, np.float32)
        st = np.zeros((n, _lib.STATS_STRIDE), np.int32)
        args = [sc.points.ctypes.data, sc.counts.ctypes.data, sc.max_points, sc.stride, sc.T.ctypes.data, sc.P.ctypes.data, 0.0, 80.0, roi[0], roi[1],
                big_l.strides[1], fb, depth.ctypes.data, disp.ctypes.data, rows, cols, n, STEP, NC, 10, 1, AUTO, C.byref(params(emu_lib)), st.ctypes.data]
        args += {"": [None], "_host": [], "_host_multi": [(C.c_int * 1)(0), 1]}[form]
        emu_lib.check(getattr(emu_lib, "dcmt_stereo_chain_f32" + form)(*args))
        same((depth, disp, st), ref, f"pitched BGR {form or 'device'}")
    for shape in ((1, 41), (33, 1)):
        rng = np.random.default_rng(31)
        sc = Scene([back_project(rng, *shape, 30) for _ in range(2)], *shape, 31)
        ref = composition(emu_lib, _Emu(), sc, step=4)
        assert_bit_equal(ref[0], oracle_chain(emu_lib, sc, range(2), step=4)[0], f"{shape}: composition vs oracle")
        for form in FORMS:
            same(chain(emu_lib, sc, form, step=4), ref, f"{shape} {form or 'device'}")


_CHUNKED = r"""
import sys; sys.path.insert(0, %(root)r)
from tests.emu import build_emu
from depth_completion_mt_b200 import _lib
from tests.test_stereo_chain_call import scene, composition, chain, same, body_redo, _Emu
lib = _lib.bind(build_emu.build())
sc = scene(3, 40, 72, 41)
ref = composition(lib, _Emu(), sc)
same(chain(lib, sc, ""), ref, "device entry in chunks of 2 + 1 frames")
body_redo(lib, _Emu(), ("",))
print("CHUNKED_OK")
"""


def test_emu_device_entry_in_chunks(emu_lib):
    """chunks of 2 + 1 frames (the chunk size is read once per process), the redo run crossing a chunk boundary"""
    env = dict(os.environ, DCMT_FUSED_CHUNK="2", DCMT_GENERIC_CHUNK="2")
    r = subprocess.run([sys.executable, "-c", _CHUNKED % {"root": ROOT}], capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert r.returncode == 0 and "CHUNKED_OK" in r.stdout, r.stdout + r.stderr


_HOST_CHUNKED = r"""
import sys; sys.path.insert(0, %(root)r)
import numpy as np
import torch
from depth_completion_mt_b200 import _lib, api, synth
from tests.conftest import assert_bit_equal
from tests.test_stereo_chain_call import Scene, back_project, chain, gray, params, same, _Gpu
lib = _lib.load()
rows, cols = synth.KITTI_ROWS, synth.KITTI_COLS
rng = np.random.default_rng(17)
# 8 frames: host chunks of 3 + 3 + 2.  Frames 2-5 land on every pixel, beyond the dictionary: their redo on the generic
# pipeline crosses the boundary of the first two chunks and runs in host chunks of 3 + 1.
sc = Scene([back_project(rng, rows, cols, None if 2 <= f <= 5 else 3000) for f in range(8)], rows, cols, 17)
ref = chain(lib, sc, "", step=65, be=_Gpu())
assert [int(v) for v in ref[2][:, 3]] == [2, 2, 0, 0, 0, 0, 2, 2], ref[2][:, 3]
for form in ("_host", "_host_multi"):
    same(chain(lib, sc, form, step=65), ref, form)
dig = rng.uniform(2.0, 60.0, (sc.n, rows, cols)).astype(np.float32)
lg, rg = gray(sc.left), gray(sc.right)
want = [t.cpu().numpy() for t in api.stereo_refine(*(torch.from_numpy(a).cuda() for a in (dig, lg, rg)), params(lib), return_disparity=True,
                                                  lib=lib)]
got = api.stereo_refine(dig, lg, rg, params(lib), return_disparity=True, lib=lib)
assert_bit_equal(got[0], want[0], "stereo refinement host form: depth")
assert_bit_equal(got[1], want[1], "stereo refinement host form: disparity")
print("HOST_CHUNKED_OK")
"""


@pytest.mark.gpu
def test_gpu_host_forms_in_chunks():
    """the chain's host forms and the stereo refinement's in host chunks of 3 frames at 352 x 1216 (1 Mpx, read once per
    process), with a run of dense frames redone on the generic pipeline across a chunk boundary: byte-equal to the device forms"""
    env = dict(os.environ, DCMT_HOST_CHUNK_MPX="1")
    r = subprocess.run([sys.executable, "-c", _HOST_CHUNKED % {"root": ROOT}], capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert r.returncode == 0 and "HOST_CHUNKED_OK" in r.stdout, r.stdout + r.stderr


# ---- argument errors ------------------------------------------------------------------------------------------------------
# One argument of a valid call (2 frames of 8 x 8, 16 points a cloud) replaced at a time; "B" stands for a PROT_NONE mapping,
# ["B", k] for k bytes into it, "PRM" for valid parameters, "PRM-1" for parameters with num_iterations -1.
_BASE = ["B", None, 16, 16, ["B", 4096], ["B", 8192], 0.0, 80.0, ["B", 1 << 18], ["B", 1 << 19], 0, 0, ["B", 1 << 20], ["B", 3 << 19], 8, 8, 2,
         4, 40, 10, 1, AUTO, "PRM", ["B", 7 << 18]]
_ERRORS = [
    ("null points", {0: None}, B), ("null T", {4: None}, B), ("null P", {5: None}, B), ("max_points -1", {2: -1}, B),
    ("n_frames -1", {16: -1}, B), ("cloud stride below max_points", {3: 15}, B), ("zero rows", {14: 0}, B),
    ("over 2^30 pixels", {14: 32768, 15: 32769}, U), ("null left", {8: None}, B), ("null right", {9: None}, B), ("null depth", {12: None}, B),
    ("null params", {22: None}, B), ("flags 4", {21: 4}, B), ("DCMT_PATH_FUSED", {21: FUSED}, B), ("num_iterations -1", {22: "PRM-1"}, B),
    ("step 3", {17: 3}, U), ("nc 0", {18: 0}, B), ("iterations -1", {19: -1}, B), ("65536 rows", {14: 65536, 15: 1}, U),
    ("bgr pitch below cols * 3", {10: 23}, B), ("bgr frame stride too small", {11: 100}, B),
    ("depth overlaps the clouds", {12: ["B", 256]}, B), ("depth overlaps the left frames", {12: ["B", (1 << 18) + 8]}, B),
    ("disparity overlaps the right frames", {13: ["B", 1 << 19]}, B), ("disparity overlaps depth", {13: ["B", (1 << 20) + 16]}, B),
]

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
prm, bad = m.StereoParams(), m.StereoParams()
lib.dcmt_stereo_params_default(C.byref(prm))
lib.dcmt_stereo_params_default(C.byref(bad))
bad.num_iterations = -1
special = {"B": buf, "PRM": C.byref(prm), "PRM-1": C.byref(bad)}
args = [special[a] if isinstance(a, str) else buf + a[1] if isinstance(a, list) else a for a in json.loads(sys.argv[3])]
out = []
for form, extra in (("", [None]), ("_host", []), ("_host_multi", [(C.c_int * 1)(0), 1])):
    out += [getattr(lib, "dcmt_stereo_chain_f32" + form)(*args, *extra), lib.dcmt_last_error().decode()]
print(json.dumps(out))
"""


@pytest.mark.parametrize("case", _ERRORS, ids=lambda c: c[0])
def test_emu_rejects_before_reading(emu_lib, case):
    """every form returns the check's code and the device form's message on buffers it cannot read or write"""
    what, change, want = case
    args = [change.get(i, a) for i, a in enumerate(_BASE)]
    r = subprocess.run([sys.executable, "-c", _CHILD, os.path.join(ROOT, "depth_completion_mt_b200", "_lib.py"), emu_lib.path, json.dumps(args)],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, f"{what}: child exited with {r.returncode} (a negative code is the signal that killed it)\n{r.stderr[-2000:]}"
    dev, dev_msg, host, host_msg, multi, multi_msg = json.loads(r.stdout.strip().splitlines()[-1])
    assert dev == want, f"{what}: device entry point returned {dev} ({dev_msg})"
    assert (host, host_msg) == (dev, dev_msg) and (multi, multi_msg) == (dev, dev_msg), what


def test_emu_host_only_checks_and_device_lists(emu_lib):
    """the host forms check the cloud sizes, the device form the points' alignment; bad device lists; outputs untouched"""
    lib = emu_lib
    sc = scene(2, 36, 40, 51)
    depth = np.full((2, 36, 40), -7.0, np.float32)
    stats = np.full((2, _lib.STATS_STRIDE), 7, np.int32)
    prm = params(lib)

    def call(form, pts=None, counts=None, extra=()):
        extra = list(extra) or {"": [None], "_host": [], "_host_multi": [(C.c_int * 1)(0), 1]}[form]
        return getattr(lib, "dcmt_stereo_chain_f32" + form)(pts or sc.points.ctypes.data, counts, sc.max_points, sc.stride, sc.T.ctypes.data,
                                                             sc.P.ctypes.data, 0.0, 80.0, sc.left.ctypes.data, sc.right.ctypes.data, 0, 0,
                                                             depth.ctypes.data, None, 36, 40, 2, STEP, NC, 10, 1, AUTO, C.byref(prm),
                                                             stats.ctypes.data, *extra)

    for bad in ([sc.max_points + 1, 3], [3, -1]):
        counts = np.array(bad, np.int32)
        for form in ("_host", "_host_multi"):
            assert call(form, counts=counts.ctypes.data) == B, (form, bad, lib.dcmt_last_error())
            assert b"n_points" in lib.dcmt_last_error()
    raw = np.zeros(sc.points.size + 4, np.float32)
    unaligned = raw[1:1 + sc.points.size]
    unaligned[:] = sc.points.ravel()
    assert call("", pts=unaligned.ctypes.data) == B and b"aligned" in lib.dcmt_last_error()
    for devs, nd in (([1], 1), ([0, 0], 2), ([0], 0), ([-1], 1)):
        assert call("_host_multi", extra=[(C.c_int * len(devs))(*devs), nd]) == B, (devs, nd)
    assert (depth == -7.0).all() and (stats == 7).all(), "output written"
    # the host forms take points at any address
    ref = composition(lib, _Emu(), sc)
    lib.check(call("_host", pts=unaligned.ctypes.data, counts=sc.counts.ctypes.data))
    assert_bit_equal(depth, ref[0], "host form on unaligned points")


def test_emu_python_api(emu_lib):
    sc = scene(2, 40, 72, 61, extra_stride=0)
    ref = composition(emu_lib, _Emu(), sc)
    got = api.stereo_chain(sc.points, sc.counts, sc.T, sc.P, sc.left, sc.right, STEP + 0.9, NC, return_disparity=True, return_stats=True,
                           lib=emu_lib)
    same(got, ref, "api, step truncated")
    same(api.stereo_chain(sc.points, sc.counts, sc.T, sc.P, sc.left, sc.right, STEP, NC, return_disparity=True, return_stats=True,
                          devices=[0], lib=emu_lib), ref, "api devices")
    one = api.stereo_chain(sc.cloud(1), None, sc.T, sc.P, sc.left[1], sc.right[1], STEP, NC, lib=emu_lib)
    assert_bit_equal(one, ref[0][1], "api one frame")
    with pytest.raises(ValueError):
        api.stereo_chain(sc.points, sc.counts, sc.T, sc.P, sc.left[:, :-1], sc.right, STEP, NC, lib=emu_lib)
    with pytest.raises(ValueError):
        api.stereo_chain(sc.points[..., :3], sc.counts, sc.T, sc.P, sc.left, sc.right, STEP, NC, lib=emu_lib)
    with pytest.raises(ValueError):
        api.stereo_chain(sc.points, sc.counts[:1], sc.T, sc.P, sc.left, sc.right, STEP, NC, lib=emu_lib)
    with pytest.raises(ValueError):
        api.stereo_chain(sc.points, sc.counts, sc.T, sc.P, sc.left, sc.right, STEP, NC, path="fused", lib=emu_lib)


# ---- GPU at KITTI size: 81 frames = host chunks of 40 + 40 + 1 -----------------------------------------------------------
def kitti_scene(n, rows, cols, seed):
    sc = Scene([synth.velodyne_cloud(seed + f, 120000) for f in range(n)], rows, cols, seed, with_counts=False)
    sc.T = np.ascontiguousarray(synth.KITTI_T_VELO_TO_CAM, np.float32)
    sc.P = np.ascontiguousarray(synth.KITTI_P_RECT_02, np.float32)
    return sc


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(352, 1216, 65, 81), (375, 1242, 68, 3)], ids=["352x1216", "375x1242"])
def test_gpu_chain_at_kitti_size(gpu_lib, shape):
    import torch

    lib = gpu_lib
    rows, cols, step, n = shape
    assert step == int(np.sqrt(rows * cols / 100.0))  # 100 superpixels, truncated like main_lc.cpp:187-201
    sc = kitti_scene(n, rows, cols, 71)
    torch.cuda.set_device(0)
    ref = composition(lib, _Gpu(), sc, step=step)
    assert (ref[2][:, 3] == 2).all()
    want = oracle_chain(lib, sc, [0, n - 1], step=step)
    assert_bit_equal(ref[0][[0, n - 1]], want[0], "composition vs oracle: depth")
    assert_bit_equal(ref[1][[0, n - 1]], want[1], "composition vs oracle: disparity")
    s = torch.cuda.Stream()
    tp, tl, tr = (torch.from_numpy(a).cuda() for a in (sc.points, sc.left, sc.right))
    got = api.stereo_chain(tp, None, sc.T, sc.P, tl, tr, step, NC, return_disparity=True, return_stats=True, stream=s, lib=lib)
    s.synchronize()
    same([g.cpu().numpy() for g in got], ref, "device entry on a side stream")
    same(api.stereo_chain(sc.points, None, sc.T, sc.P, sc.left, sc.right, step, NC, return_disparity=True, return_stats=True, lib=lib), ref, "_host")
    for devices in ([0], "all", list(range(torch.cuda.device_count()))[::-1]):
        got = api.stereo_chain(sc.points, None, sc.T, sc.P, sc.left, sc.right, step, NC, return_disparity=True, return_stats=True, devices=devices,
                               lib=lib)
        same(got, ref, f"_host_multi {devices}")
    assert torch.cuda.current_device() == 0  # the caller's device is restored
    if ro.available() and rows == synth.KITTI_ROWS:
        # the reference build end to end on the first frame, with the statistical bar of test_stereo_chain.py
        lab = lab_oracle.bgr2lab(sc.left[0])
        labels, centers = ro.generate_superpixels(lab, step, NC)[:2]
        nrm = ro.lidar_project(sc.cloud(0), sc.T, sc.P, rows, cols)[1]
        dense = ro.interpolate_with_superpixels(labels, nrm, n_clusters=len(centers))
        d = np.abs(ref[0][0] - ro.stereo_refine(dense, gray(sc.left[0]), gray(sc.right[0])))
        assert np.median(d) <= 1e-5 and (d <= 1e-3).mean() >= 0.999, f"median {np.median(d)}, within 1e-3: {(d <= 1e-3).mean()}"


@pytest.mark.gpu
def test_gpu_redo_and_generic(gpu_lib):
    body_redo(gpu_lib, _Gpu(), FORMS)
    sc = kitti_scene(3, synth.KITTI_ROWS, synth.KITTI_COLS, 81)
    for use_sp, flags in ((0, AUTO), (1, GENERIC)):
        ref = composition(gpu_lib, _Gpu(), sc, step=65, use_sp=use_sp, flags=flags)
        for form in FORMS:
            same(chain(gpu_lib, sc, form, step=65, use_sp=use_sp, flags=flags, be=_Gpu()), ref, f"{form or 'device'} {use_sp} {flags}")


# ---- C++ shim: the MatView overloads (emulator, GPU) and the cv::Mat overloads (stand-in OpenCV headers) -----------------
REFSHIM = os.path.join(ROOT, "oracle", "refshim")


def body_shim(lib, tmp_path, sc, step):
    ref = composition(lib, _Gpu() if lib.dcmt_build_info().startswith(b"cuda") else _Emu(), sc, step=step)
    sc.cloud(0).tofile(tmp_path / "pts.f32")
    sc.left[0].tofile(tmp_path / "left.u8")
    sc.right[0].tofile(tmp_path / "right.u8")
    np.concatenate([sc.T.ravel()[:16], sc.P.ravel()[:12]]).astype(np.float32).tofile(tmp_path / "tp.f32")
    libdir, libname = os.path.dirname(lib.path), os.path.basename(lib.path)[3:-3]
    for with_cv in (False, True):
        exe = str(tmp_path / ("shim_chain_cv" if with_cv else "shim_chain"))
        cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include")]
        cmd += ["-I", REFSHIM] if with_cv else ["-DDCMT_NO_OPENCV"]
        cmd += [os.path.join(ROOT, "tests", "cpp", "shim_stereo_chain_main.cpp"), "-o", exe, "-L", libdir, "-l" + libname, "-Wl,-rpath," + libdir]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        r = subprocess.run([exe, str(sc.rows), str(sc.cols), str(tmp_path / "pts.f32"), str(len(sc.cloud(0))), str(tmp_path / "tp.f32"),
                            str(tmp_path / "left.u8"), str(tmp_path / "right.u8"), str(step), str(NC), str(tmp_path / "o"), "12"],
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
        for kind in ["view"] + (["mat"] if with_cv else []):
            assert_bit_equal(np.fromfile(tmp_path / f"o_{kind}.depth", np.float32).reshape(sc.rows, sc.cols), ref[0][0], f"shim {kind} depth")
            assert_bit_equal(np.fromfile(tmp_path / f"o_{kind}.disp", np.float32).reshape(sc.rows, sc.cols), ref[1][0], f"shim {kind} disparity")
        if with_cv:
            assert "type errors thrown: 3" in r.stdout, r.stdout


def test_shim_on_emulator(tmp_path, emu_lib):
    body_shim(emu_lib, tmp_path, scene(1, 40, 72, 91), STEP)


@pytest.mark.gpu
def test_shim_on_gpu(tmp_path, gpu_lib):
    body_shim(gpu_lib, tmp_path, kitti_scene(1, synth.KITTI_ROWS, synth.KITTI_COLS, 91), 65)
