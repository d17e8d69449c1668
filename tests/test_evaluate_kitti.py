"""The KITTI depth-completion benchmark's figures (dcmt_evaluate_kitti_f32 / _u16 / _u16_u16 and their *_host variants).

include/dcmt.h states the rule: the devkit's background interpolation of the prediction, then the error terms at every
GT-valid pixel.  `kitti_oracle` below restates that text in numpy and is checked on hand-computed frames; the library is
checked against it (counts exact, sums within 1e-12 relative, figures within one float32 ulp), the uint16 calls against
the float32 call on the decoded planes (byte-equal), and on dense predictions n_gt / sum_abs / sum_sq against the pinned
dcmt_evaluate_* reductions in mode DCMT_EVAL_GT_VALID with tolerance 0 (byte-equal)."""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, api, synth
from tests.conftest import ROOT
from tests.test_evaluate_u16 import REC, SENTINEL, Buf, aligned, decode, place

KREC = api.KITTI_METRICS
SUMS = ("sum_abs", "sum_sq", "sum_iabs", "sum_isq")
COUNTS = ("n_gt", "n_pred", "n_unfilled")
FIGURES = ("mae_mm", "rmse_mm", "imae_per_km", "irmse_per_km", "density")


# ---- the contract in numpy
def background_fill(p: np.ndarray) -> np.ndarray:
    """the devkit's interpolateBackground as include/dcmt.h states it: float32 (rows, cols) -> filled plane, -1 = unfilled"""
    rows, cols = p.shape
    valid = p > 0
    rowpass = np.full(p.shape, -1.0, np.float32)
    has = np.zeros(rows, bool)
    x = np.arange(cols)
    for y in range(rows):
        idx = np.flatnonzero(valid[y])
        if idx.size == 0:
            continue
        has[y] = True
        vals = p[y, idx]
        li = np.searchsorted(idx, x, side="right") - 1  # nearest valid at or left of x
        ri = np.searchsorted(idx, x, side="left")  # nearest valid at or right of x
        left = np.where(li >= 0, vals[np.clip(li, 0, None)], np.inf)
        right = np.where(ri < idx.size, vals[np.clip(ri, None, idx.size - 1)], np.inf)
        rowpass[y] = np.minimum(left, right)
    out = rowpass.copy()
    if has.any():
        first, last = np.flatnonzero(has)[[0, -1]]
        out[:first] = rowpass[first]
        out[last + 1:] = rowpass[last]
    return out


def kitti_oracle(g: np.ndarray, p: np.ndarray) -> np.ndarray:
    """one record of the contract for float32 metre planes g (GT) and p (prediction)"""
    g = np.asarray(g, np.float32)
    p = np.asarray(p, np.float32)
    filled = background_fill(p)
    gv = g > 0
    gg, pp = g[gv], filled[gv]
    e = np.abs(gg - pp).astype(np.float64)  # float32 subtraction, then widened
    ie = np.abs(1.0 / gg.astype(np.float64) - 1.0 / pp.astype(np.float64))
    rec = np.zeros(1, KREC)[0]
    n = float(gv.sum())
    rec["n_gt"], rec["n_pred"], rec["n_unfilled"] = n, float((gv & (p > 0)).sum()), float((pp < 0).sum())
    rec["sum_abs"], rec["sum_sq"], rec["sum_iabs"], rec["sum_isq"] = e.sum(), (e * e).sum(), ie.sum(), (ie * ie).sum()
    with np.errstate(invalid="ignore", divide="ignore"):
        rec["mae_mm"] = np.float32(1000.0 * (rec["sum_abs"] / n))
        rec["rmse_mm"] = np.float32(1000.0 * np.sqrt(rec["sum_sq"] / n))
        rec["imae_per_km"] = np.float32(1000.0 * (rec["sum_iabs"] / n))
        rec["irmse_per_km"] = np.float32(1000.0 * np.sqrt(rec["sum_isq"] / n))
        rec["density"] = np.float32(rec["n_pred"] / n)
    return rec


def check_against_oracle(got, want, what):
    for f in COUNTS:
        assert got[f] == want[f], (what, f, got[f], want[f])
    for f in SUMS:
        g, w = float(got[f]), float(want[f])
        assert abs(g - w) <= 1e-12 * abs(w), (what, f, g, w)
    for f in FIGURES:
        g, w = np.float32(got[f]), np.float32(want[f])
        if np.isnan(w):
            assert np.isnan(g), (what, f, g)
        else:
            assert abs(int(g.view(np.int32)) - int(w.view(np.int32))) <= 1, (what, f, g, w)


# ---- 1. the oracle on hand-computed frames
def test_oracle_row_gaps():
    # left-border gap, interior gap, right-border gap: [., 2, ., ., 5, .] -> [2, 2, 2, 2, 5, 5]
    p = np.array([[0, 2, 0, 0, 5, 0]], np.float32)
    assert background_fill(p).tolist() == [[2, 2, 2, 2, 5, 5]]
    rec = kitti_oracle(np.ones_like(p), p)
    assert (rec["n_gt"], rec["n_pred"], rec["n_unfilled"]) == (6, 2, 0)
    assert rec["sum_abs"] == 12 and rec["sum_sq"] == 4 * 1 + 2 * 16
    assert abs(rec["sum_iabs"] - (4 * 0.5 + 2 * 0.8)) < 1e-15
    assert rec["mae_mm"] == np.float32(2000) and rec["rmse_mm"] == np.float32(1000 * np.sqrt(36 / 6))
    assert rec["imae_per_km"] == np.float32(600) and rec["density"] == np.float32(2 / 6)
    # interior gap takes the smaller neighbour, whichever side it is on
    assert background_fill(np.array([[7, 0, 0, 3]], np.float32)).tolist() == [[7, 3, 3, 3]]


def test_oracle_empty_rows():
    p = np.array([[0, 0, 0], [1, 0, 3], [0, 0, 0], [4, 4, 0], [0, 0, 0]], np.float32)
    want = [[1, 1, 3], [1, 1, 3], [-1, -1, -1], [4, 4, 4], [4, 4, 4]]
    assert background_fill(p).tolist() == want
    rec = kitti_oracle(np.full(p.shape, 2, np.float32), p)
    assert (rec["n_gt"], rec["n_pred"], rec["n_unfilled"]) == (15, 4, 3)
    assert rec["sum_abs"] == 3 + 3 + 9 + 6 + 6
    # the unfilled row counts with p = -1: |1/2 - 1/(-1)| = 1.5
    assert abs(rec["sum_iabs"] - (4 * 0.5 + 2 * (1 / 2 - 1 / 3) + 3 * 1.5 + 6 * 0.25)) < 1e-15


def test_oracle_all_empty_and_tiny():
    g = np.array([[0, 2, 4]], np.float32)
    rec = kitti_oracle(g, np.zeros_like(g))
    assert (rec["n_gt"], rec["n_pred"], rec["n_unfilled"]) == (2, 0, 2)
    assert rec["sum_abs"] == 3 + 5 and rec["sum_iabs"] == 1.5 + 1.25 and rec["density"] == 0
    # 1x1
    assert kitti_oracle(np.float32([[2]]), np.float32([[0]]))["sum_abs"] == 3
    assert kitti_oracle(np.float32([[2]]), np.float32([[4]]))["sum_abs"] == 2
    # N x 1: the column pass copies only above the first and below the last valid row
    p = np.float32([[0], [3], [0], [0], [5], [0]])
    assert background_fill(p)[:, 0].tolist() == [3, 3, -1, -1, 5, 5]
    # no GT: every figure NaN
    rec = kitti_oracle(np.zeros((2, 2), np.float32), np.ones((2, 2), np.float32))
    assert rec["n_gt"] == 0 and all(np.isnan(rec[f]) for f in FIGURES)
    # float32 invalid values: 0, negatives and NaN alike
    p = np.float32([[0, 2, -3, np.nan, 5, -0.0]])
    assert background_fill(p).tolist() == [[2, 2, 2, 2, 5, 5]]


# ---- the library
NAMES = {("f32", "f32"): "dcmt_evaluate_kitti_f32", ("u16", "f32"): "dcmt_evaluate_kitti_u16", ("u16", "u16"): "dcmt_evaluate_kitti_u16_u16"}


class Caller:
    """the KITTI entry points through one kind of pointer: "device" (buffers where the library computes) or "host" (*_host)"""

    def __init__(self, lib, kind: str, on_gpu: bool):
        self.lib, self.kind = lib, kind
        self.on_device = kind == "device" and on_gpu

    def results(self, n, rec=KREC):
        return Buf(np.full(n * rec.itemsize, SENTINEL, np.uint8), self.on_device)

    def call(self, name, g, r, rows, cols, geo, n, res):
        fn = getattr(self.lib, name + ("_host" if self.kind == "host" else ""))
        args = [g.ptr, r.ptr, rows, cols] + list(geo) + [n, res.ptr]
        if self.kind == "device":
            args.append(None)
        return fn(*args)

    def records(self, gt, pred, geo_g, geo_r, offset=0):
        """records of gt / pred (n, rows, cols) placed with geometries (pitch, frame stride) in elements"""
        n, rows, cols = gt.shape
        name = NAMES[("u16" if gt.dtype == np.uint16 else "f32", "u16" if pred.dtype == np.uint16 else "f32")]
        g = Buf(place(gt, *geo_g, offset), self.on_device, offset)
        q = Buf(place(pred, *geo_r, offset), self.on_device, offset)
        res = self.results(n)
        geo = (geo_g[0] * gt.itemsize, geo_g[1] * gt.itemsize, geo_r[0] * pred.itemsize, geo_r[1] * pred.itemsize)
        self.lib.check(self.call(name, g, q, rows, cols, geo, n, res))
        return res.get().view(KREC)

    def reductions(self, gt, pred, geo, offset=0):
        """dcmt_evaluate_* in mode DCMT_EVAL_GT_VALID, tolerance 0, both planes with geometry `geo` (elements)"""
        n, rows, cols = gt.shape
        g = Buf(place(gt, *geo, offset), self.on_device, offset)
        q = Buf(place(pred, *geo, offset), self.on_device, offset)
        res = self.results(n, REC)
        if gt.dtype == np.float32:
            name, bgeo = "dcmt_evaluate_f32", [geo[0] * 4, geo[1] * 4]
        else:
            name = "dcmt_evaluate_u16_u16" if pred.dtype == np.uint16 else "dcmt_evaluate_u16"
            bgeo = [geo[0] * 2, geo[1] * 2, geo[0] * pred.itemsize, geo[1] * pred.itemsize]
        fn = getattr(self.lib, name + ("_host" if self.kind == "host" else ""))
        args = [g.ptr, q.ptr, rows, cols] + bgeo + [n, 0.0, 0, res.ptr] + ([None] if self.kind == "device" else [])
        self.lib.check(fn(*args))
        return res.get().view(REC)


def kitti_gt(seed, n, rows, cols, density=0.3):
    return np.stack([synth.sparse_depth_q8(seed + f, rows, cols, density, kitti_like=True) for f in range(n)])


def sparse_pred(seed, n, rows, cols, kinds):
    """uint16 predictions, frame f of kind kinds[f % len]: a valid density, "rows" (5 % with whole empty rows above, inside
    and below) or "empty" (no valid pixel)"""
    out = np.zeros((n, rows, cols), np.uint16)
    for f in range(n):
        kind = kinds[f % len(kinds)]
        if kind == "empty":
            continue
        if kind == "rows":
            p = synth.sparse_depth_q8(seed + 1000 + f, rows, cols, 0.05)
            keep = np.random.default_rng(seed + f).random(rows) < 0.5
            keep[: rows // 4] = False
            keep[-(rows // 5):] = False if rows >= 5 else keep[-(rows // 5):]
            p[~keep] = 0
            out[f] = p
        else:
            out[f] = synth.sparse_depth_q8(seed + 1000 + f, rows, cols, kind)
    return out


# (rows, cols, (GT pitch, GT frame stride), (pred pitch, pred frame stride), offset, n frames) in elements
LAYOUTS = {
    "dense_cols4": lambda: (24, 64, (64, 24 * 64), (64, 24 * 64), 0, 3),
    "ragged_13": lambda: (17, 13, (13, 17 * 13), (13, 17 * 13), 0, 2),
    "own_pitches": lambda: (20, 64, (67, 20 * 67), (72, 21 * 72), 0, 2),
    "base_offset_1": lambda: (16, 64, (64, 16 * 64), (64, 16 * 64), 1, 2),
    "frame_gaps": lambda: (12, 40, (44, 15 * 44), (44, 15 * 44), 0, 3),
    "one_by_one": lambda: (1, 1, (1, 1), (1, 1), 0, 4),
    "one_row": lambda: (1, 50, (50, 50), (50, 50), 0, 3),
    "one_col": lambda: (40, 1, (1, 40), (1, 40), 0, 3),
    "wide_4096": lambda: (6, 4096, (4096, 6 * 4096), (4100, 6 * 4100), 0, 6),
    "batch_6": lambda: (30, 72, (72, 30 * 72), (72, 30 * 72), 0, 6),
}
KINDS = (0.01, 0.05, 0.2, "rows", "empty", 0.05)


def check_types_and_oracle(caller, gt16, p16, geo_g, geo_r, offset, what):
    """the three type pairs byte-equal on the decoded planes, each frame against the oracle; returns the records"""
    uu = caller.records(gt16, p16, geo_g, geo_r, offset)
    uf = caller.records(gt16, decode(p16), geo_g, geo_r, offset)
    ff = caller.records(decode(gt16), decode(p16), geo_g, geo_r, offset)
    assert uu.tobytes() == ff.tobytes(), f"{what}: u16/u16 differs from f32 on the decoded planes\n{uu}\n{ff}"
    assert uf.tobytes() == ff.tobytes(), f"{what}: u16/f32 differs from f32 on the decoded planes\n{uf}\n{ff}"
    for f in range(gt16.shape[0]):
        check_against_oracle(ff[f], kitti_oracle(decode(gt16[f]), decode(p16[f])), f"{what} frame {f}")
    return ff


def body_layouts(caller, names=tuple(LAYOUTS)):
    for k, (name, layout) in enumerate(LAYOUTS.items()):
        if name not in names:
            continue
        rows, cols, geo_g, geo_r, offset, n = layout()
        gt16 = kitti_gt(100 * k, n, rows, cols)
        if name in ("one_by_one", "one_row", "one_col"):
            gt16 = np.stack([synth.sparse_depth_q8(100 * k + f, rows, cols, 0.6) for f in range(n)])  # no empty upper band
        p16 = sparse_pred(100 * k, n, rows, cols, KINDS)
        recs = check_types_and_oracle(caller, gt16, p16, geo_g, geo_r, offset, name)
        if name == "batch_6":
            assert recs["n_unfilled"][4] == recs["n_gt"][4] > 0 and recs["n_pred"][4] == 0  # the empty prediction
            assert recs["n_unfilled"][3] > 0  # empty rows between the first and the last valid row


def body_float_invalid(caller):
    """float32 0, negatives and NaN are all invalid predictions: the records equal those with 0 in their place"""
    gt = decode(kitti_gt(7, 2, 16, 40))
    p = decode(sparse_pred(7, 2, 16, 40, (0.3,)))
    rng = np.random.default_rng(1)
    junk = p.copy()
    hole = p == 0
    junk[hole & (rng.random(p.shape) < 0.3)] = -1.5
    junk[hole & (rng.random(p.shape) < 0.3)] = np.nan
    junk[hole & (rng.random(p.shape) < 0.2)] = -0.0
    geo = (40, 16 * 40)
    assert caller.records(gt, junk, geo, geo).tobytes() == caller.records(gt, p, geo, geo).tobytes()


def body_tie(caller, preds16, gt16, what):
    """on dense predictions n_gt, sum_abs and sum_sq are the bytes of dcmt_evaluate_* (GT_VALID, tolerance 0)"""
    assert (preds16 > 0).all()
    n, rows, cols = gt16.shape
    for geo, offset in (((cols, rows * cols), 0), ((cols + 3, rows * (cols + 3) + 5), 1)):
        for g, p in ((gt16, preds16), (gt16, decode(preds16)), (decode(gt16), decode(preds16))):
            k = caller.records(g, p, geo, geo, offset)
            e = caller.reductions(g, p, geo, offset)
            for kf, ef in (("n_gt", "count"), ("sum_abs", "sum_abs"), ("sum_sq", "sum_sq")):
                assert k[kf].tobytes() == e[ef].tobytes(), (what, g.dtype, p.dtype, geo, kf, k[kf], e[ef])
            assert (k["n_pred"] == k["n_gt"]).all() and (k["n_unfilled"] == 0).all()


def body_own_outputs(caller, lib, rows, cols, n):
    """the library's own completion outputs (uint16 and float32) as predictions: against the oracle, and the tie"""
    sparse = np.stack([synth.sparse_depth_q8(40 + f, rows, cols, 0.05, kitti_like=True) for f in range(n)])
    gt16 = kitti_gt(60, n, rows, cols)
    d16 = api.img_completion(sparse, False, "gaussian", out_dtype=np.uint16, lib=lib)
    d32 = api.img_completion(sparse, False, "gaussian", lib=lib)
    geo = (cols, rows * cols)
    check_types_and_oracle(caller, gt16, d16, geo, geo, 0, "own u16 outputs")
    ff = caller.records(gt16, d32, geo, geo)
    for f in range(n):
        check_against_oracle(ff[f], kitti_oracle(decode(gt16[f]), d32[f]), f"own f32 outputs frame {f}")
    body_tie(caller, d16, gt16, "own outputs")
    rng = np.random.default_rng(5)
    body_tie(caller, rng.integers(1, 65536, (3, 9, 37)).astype(np.uint16), kitti_gt(70, 3, 9, 37), "random dense")


def body_very_wide(caller):
    """rows of more than 262 144 columns keep their validity bits in device memory instead of shared memory"""
    rows, cols, n = 3, 263000, 2
    gt16 = np.stack([synth.sparse_depth_q8(80 + f, rows, cols, 0.1) for f in range(n)])
    p16 = np.stack([synth.sparse_depth_q8(90 + f, rows, cols, 0.05) for f in range(n)])
    p16[0, 0] = 0  # a row above the first valid row
    p16[1, 1] = 0  # an unfilled row between the first and the last
    geo = (cols, rows * cols)
    recs = check_types_and_oracle(caller, gt16, p16, geo, geo, 0, "very wide")
    assert recs["n_unfilled"][1] > 0 and recs["n_unfilled"][0] == 0


def body_arguments(caller):
    """every bad argument is DCMT_E_BADARG before any device work, with the results untouched; n_frames == 0 is DCMT_OK"""
    rows, cols = 6, 10
    g16 = Buf(aligned(rows * cols, np.uint16), caller.on_device)
    g32 = Buf(aligned(rows * cols, np.float32), caller.on_device)
    r32 = Buf(aligned(rows * cols, np.float32), caller.on_device)
    r16 = Buf(aligned(rows * cols, np.uint16), caller.on_device)
    res = caller.results(1)
    null = type("Null", (), {"ptr": None})()
    for name, g, ge, r, re in (("dcmt_evaluate_kitti_f32", g32, 4, r32, 4), ("dcmt_evaluate_kitti_u16", g16, 2, r32, 4),
                               ("dcmt_evaluate_kitti_u16_u16", g16, 2, r16, 2)):
        bad = [
            (null, r, rows, cols, (0, 0, 0, 0), 1, res),
            (g, null, rows, cols, (0, 0, 0, 0), 1, res),
            (g, r, rows, cols, (0, 0, 0, 0), 1, null),
            (g, r, 0, cols, (0, 0, 0, 0), 1, res),
            (g, r, rows, 0, (0, 0, 0, 0), 1, res),
            (g, r, rows, cols, (0, 0, 0, 0), -1, res),
            (g, r, rows, cols, (ge * cols + 1, 0, 0, 0), 1, res),  # GT pitch not a multiple of its element
            (g, r, rows, cols, (ge * (cols - 1), 0, 0, 0), 1, res),  # GT pitch too small
            (g, r, rows, cols, (0, ge * rows * cols + 1, 0, 0), 1, res),
            (g, r, rows, cols, (0, ge * (rows * cols - 1), 0, 0), 1, res),
            (g, r, rows, cols, (0, 0, re * cols + 1, 0), 1, res),  # prediction pitch not a multiple of its element
            (g, r, rows, cols, (0, 0, re * (cols - 1), 0), 1, res),
            (g, r, rows, cols, (0, 0, 0, re * rows * cols + 1), 1, res),
            (g, r, rows, cols, (0, 0, 0, re * (rows * cols - 1)), 1, res),
        ]
        for i, (gg, q, rr, cc, geo, n, out) in enumerate(bad):
            assert caller.call(name, gg, q, rr, cc, geo, n, out) == _lib.DCMT_E_BADARG, (name, i)
        assert caller.call(name, g, r, rows, cols, (0, 0, 0, 0), 0, res) == _lib.DCMT_OK
    assert (res.get() == SENTINEL).all(), "results written by a rejected call"


def body_host_device(lib, on_gpu):
    """the *_host and the device entry points return the same bytes"""
    gt16 = kitti_gt(300, 4, 33, 120)
    p16 = sparse_pred(300, 4, 33, 120, KINDS)
    geo_g, geo_r = (124, 33 * 124), (121, 34 * 121)
    for g, p in ((gt16, p16), (gt16, decode(p16)), (decode(gt16), decode(p16))):
        h = Caller(lib, "host", on_gpu).records(g, p, geo_g, geo_r)
        d = Caller(lib, "device", on_gpu).records(g, p, geo_g, geo_r)
        assert h.tobytes() == d.tobytes()


def body_python(lib, to_backend, u16_dtype):
    sparse = synth.sparse_depth_q8(11, 64, 96, 0.05, kitti_like=True)
    gt = np.stack([synth.sparse_depth_q8(12 + f, 64, 96, 0.3, kitti_like=True) for f in range(2)])
    d16 = api.img_completion(to_backend(sparse), False, "gaussian", out_dtype=u16_dtype, lib=lib)
    host = lambda x: x if isinstance(x, np.ndarray) else x.cpu().numpy()
    d16h = host(d16)
    preds = np.stack([d16h, synth.sparse_depth_q8(13, 64, 96, 0.05)])
    got = api.evaluate_kitti(to_backend(gt), to_backend(preds), lib=lib)
    assert got.dtype == KREC and got.shape == (2,)
    for f in range(2):
        check_against_oracle(got[f], kitti_oracle(decode(gt[f]), decode(preds[f])), f"api frame {f}")
    want = api.evaluate_kitti(to_backend(decode(gt)), to_backend(decode(preds)), lib=lib)
    assert got.tobytes() == want.tobytes()
    assert api.evaluate_kitti(to_backend(gt), to_backend(decode(preds)), lib=lib).tobytes() == want.tobytes()
    one = api.evaluate_kitti(to_backend(gt[0]), d16, lib=lib)  # (rows, cols) is one frame
    assert one.shape == (1,) and one.tobytes() == want[:1].tobytes()
    with pytest.raises(ValueError, match="uint16"):
        api.evaluate_kitti(to_backend(decode(gt)), to_backend(preds), lib=lib)
    with pytest.raises(ValueError, match="shapes"):
        api.evaluate_kitti(to_backend(gt), to_backend(preds[:, :32]), lib=lib)


def test_emu_layouts(emu_lib):
    body_layouts(Caller(emu_lib, "device", on_gpu=False))
    body_layouts(Caller(emu_lib, "host", on_gpu=False), ("own_pitches", "base_offset_1", "frame_gaps", "batch_6"))
    body_float_invalid(Caller(emu_lib, "device", on_gpu=False))


def test_emu_own_outputs(emu_lib):
    body_own_outputs(Caller(emu_lib, "device", on_gpu=False), emu_lib, 64, 96, 2)


def test_emu_very_wide(emu_lib):
    body_very_wide(Caller(emu_lib, "device", on_gpu=False))


def test_emu_arguments(emu_lib):
    for kind in ("device", "host"):
        body_arguments(Caller(emu_lib, kind, on_gpu=False))


def test_emu_host_device(emu_lib):
    body_host_device(emu_lib, on_gpu=False)


def test_emu_python(emu_lib):
    body_python(emu_lib, lambda a: a, np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["host", "device"])
def test_gpu_evaluate_kitti(gpu_lib, kind):
    import torch

    caller = Caller(gpu_lib, kind, on_gpu=True)
    body_layouts(caller)
    body_float_invalid(caller)
    body_own_outputs(caller, gpu_lib, 352, 1216, 3)
    body_very_wide(caller)
    body_arguments(caller)
    if kind == "host":
        body_host_device(gpu_lib, on_gpu=True)
        body_python(gpu_lib, lambda a: a, np.uint16)
    else:
        body_python(gpu_lib, lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.uint16)


# ---- the cv::Mat overload of include/img_completion.h (tests/cpp/shim_eval_kitti_main.cpp), compiled against the stand-in
# OpenCV headers of oracle/refshim
def compile_kitti_shim(tmp_path, lib_path):
    exe = str(tmp_path / "shim_eval_kitti_main")
    libdir, libname = os.path.dirname(lib_path), os.path.basename(lib_path)[3:-3]
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), "-I",
           os.path.join(ROOT, "oracle", "refshim"), os.path.join(ROOT, "tests", "cpp", "shim_eval_kitti_main.cpp"), "-o", exe, "-L",
           libdir, "-l" + libname, "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def body_shim(exe, tmp_path, lib, rows, cols):
    gt = synth.sparse_depth_q8(32, rows, cols, 0.3, kitti_like=True)
    pred = synth.sparse_depth_q8(33, rows, cols, 0.05)
    gt.tofile(tmp_path / "gt.u16")
    pred.tofile(tmp_path / "pred.u16")
    r = subprocess.run([exe, str(rows), str(cols), str(tmp_path / "gt.u16"), str(tmp_path / "pred.u16")], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, (r.returncode, r.stderr)
    lines = dict(l.split(":", 1) for l in r.stdout.strip().splitlines())
    want = api.evaluate_kitti(gt, pred, lib=lib)[0]
    for key in ("u16 gt, u16 pred", "u16 gt, f32 pred", "f32 gt, f32 pred"):
        vals = lines[key].split()
        assert len(vals) == 12, (key, vals)
        for f, v in zip(COUNTS + SUMS + FIGURES, vals):
            got = np.float32(v) if f in FIGURES else float(v)  # printed with enough digits to round-trip
            assert (np.isnan(got) and np.isnan(want[f])) or got == want[f], (key, f, v, want[f])
    assert lines["f32 gt, u16 pred"].strip() == "throws"


def test_kitti_shim_on_emulator(tmp_path, emu_lib):
    body_shim(compile_kitti_shim(tmp_path, emu_lib.path), tmp_path, emu_lib, 48, 80)


@pytest.mark.gpu
def test_kitti_shim_with_product_library_on_gpu(tmp_path, gpu_lib):
    body_shim(compile_kitti_shim(tmp_path, gpu_lib.path), tmp_path, gpu_lib, 352, 1216)
