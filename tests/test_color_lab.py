"""cv::cvtColor(COLOR_BGR2Lab) (main_lc.cpp:182-183, main_sl.cpp:438), the conversion in front of SLIC: OpenCV's 8-bit
path, bit-equal to cv2 4.13 on all 2^24 colours.  The C oracle is pinned to cv2 and to a sha256 of the Lab image of
every colour, so the checks below run without cv2 too; the kernel runs on the CPU emulator and on the GPU."""
from __future__ import annotations

import hashlib

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, api, synth
from oracle import lab_oracle
from oracle.make_lab_tables import OUT as TABLES_HEADER
from oracle.make_lab_tables import all_colours

# sha256 of cv2.cvtColor(all_colours(), COLOR_BGR2Lab) with cv2 4.13.0: every (B, G, R) once, 4096 x 4096 x 3 bytes
ALL_COLOURS_LAB_SHA256 = "b3067516fa862bb008af4ffb4da5555722524a70776bf7ffd523a90f4331480c"


def _cv2():
    try:
        import cv2
    except ImportError:
        return None
    return cv2


def want_lab(img: np.ndarray) -> np.ndarray:
    """Lab of (rows, cols, 3) or (n, rows, cols, 3) BGR by the C oracle."""
    return np.stack([lab_oracle.bgr2lab(f) for f in img]) if img.ndim == 4 else lab_oracle.bgr2lab(img)


def colour_cube() -> np.ndarray:
    vals = np.array(list(range(0, 256, 5)) + [255], np.uint8)
    B, G, R = np.meshgrid(vals, vals, vals, indexing="ij")
    return np.stack([B, G, R], -1).reshape(len(vals), len(vals) * len(vals), 3)


def images():
    rng = np.random.default_rng(0)
    return [colour_cube(), rng.integers(0, 256, (1, 1, 3), dtype=np.uint8), rng.integers(0, 256, (5, 1, 3), dtype=np.uint8),
            rng.integers(0, 256, (97, 171, 3), dtype=np.uint8), rng.integers(0, 256, (3, 4, 33, 3), dtype=np.uint8),
            synth.bgr_image(0, 64, 80)]


def body(lib, to_backend):
    for img in images():
        got = api.bgr2lab(to_backend(np.ascontiguousarray(img)), lib=lib)
        got = got if isinstance(got, np.ndarray) else got.cpu().numpy()
        assert got.shape == img.shape and np.array_equal(got, want_lab(img)), img.shape


# ---------------------------------------------------------------------------------------------- tables and oracle
def test_make_lab_tables_regenerates_header(tmp_path):
    pytest.importorskip("cv2")
    from oracle import make_lab_tables

    out = tmp_path / "lab_tables.cuh"
    assert make_lab_tables.main(["--out", str(out)]) == 0
    with open(TABLES_HEADER, "rb") as fh:
        assert out.read_bytes() == fh.read()


def test_oracle_all_colours():
    img = all_colours()
    got = lab_oracle.bgr2lab(img)
    assert hashlib.sha256(got.tobytes()).hexdigest() == ALL_COLOURS_LAB_SHA256
    cv2 = _cv2()
    if cv2 is not None:
        assert np.array_equal(got, cv2.cvtColor(img, cv2.COLOR_BGR2Lab))


# ---------------------------------------------------------------------------------------------- kernel on the emulator
def test_emu_bgr2lab(emu_lib):
    body(emu_lib, lambda a: a)


def test_emu_bgr2lab_pitched_rows(emu_lib):
    rng = np.random.default_rng(1)
    rows, cols, bp, lp, n = 9, 37, 131, 120, 2
    src = rng.integers(0, 256, (n, rows, bp), dtype=np.uint8)
    for entry in ("dcmt_bgr2lab_u8_host", "dcmt_bgr2lab_u8"):  # the emulator's device pointers are host pointers
        dst = np.full((n, rows, lp), 7, np.uint8)
        extra = (None,) if entry == "dcmt_bgr2lab_u8" else ()
        emu_lib.check(getattr(emu_lib, entry)(src.ctypes.data, dst.ctypes.data, rows, cols, bp, lp, n, *extra))
        want = want_lab(np.ascontiguousarray(src[:, :, : cols * 3]).reshape(n, rows, cols, 3))
        assert np.array_equal(dst[:, :, : cols * 3].reshape(n, rows, cols, 3), want), entry
        assert (dst[:, :, cols * 3:] == 7).all(), entry


@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 3), (5, 7), (16, 16)])
def test_emu_bgr2lab_unaligned(emu_lib, in_off, out_off):
    rng = np.random.default_rng(2)
    rows, cols = 6, 70  # 70 columns: four full 16-pixel groups and a ragged end per row
    src = np.zeros(rows * cols * 3 + 64, np.uint8)
    img = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
    src[in_off:in_off + img.size] = img.ravel()
    dst = np.full(rows * cols * 3 + 64, 7, np.uint8)
    emu_lib.check(emu_lib.dcmt_bgr2lab_u8(src.ctypes.data + in_off, dst.ctypes.data + out_off, rows, cols, 0, 0, 1, None))
    assert np.array_equal(dst[out_off:out_off + img.size].reshape(img.shape), want_lab(img))
    assert (dst[:out_off] == 7).all() and (dst[out_off + img.size:] == 7).all()


def badarg_cases(lib, buf: int, other: int):
    """(description, status) of calls that must fail, on the device entry point; buf / other: separate buffers of at
    least 4 KB."""
    d = lib.dcmt_bgr2lab_u8
    return [
        ("null input", d(None, other, 4, 4, 0, 0, 1, None)),
        ("null output", d(buf, None, 4, 4, 0, 0, 1, None)),
        ("zero rows", d(buf, other, 0, 4, 0, 0, 1, None)),
        ("negative cols", d(buf, other, 4, -1, 0, 0, 1, None)),
        ("negative frames", d(buf, other, 4, 4, 0, 0, -1, None)),
        ("input pitch below cols * 3", d(buf, other, 4, 4, 11, 0, 1, None)),
        ("output pitch below cols * 3", d(buf, other, 4, 4, 0, 11, 1, None)),
        ("in place", d(buf, buf, 4, 4, 0, 0, 1, None)),
        ("output starts inside the input", d(buf, buf + 47, 4, 4, 0, 0, 1, None)),
        ("input starts inside the output", d(buf + 30, buf, 4, 4, 0, 0, 1, None)),
        ("overlap in a later frame", d(buf, buf + 4 * 12 * 2, 4, 4, 0, 0, 3, None)),
    ]


def test_emu_bgr2lab_bad_arguments(emu_lib):
    a = np.zeros(4096, np.uint8)
    b = np.zeros(4096, np.uint8)
    for what, rc in badarg_cases(emu_lib, a.ctypes.data, b.ctypes.data):
        assert rc == _lib.DCMT_E_BADARG, what
    h = emu_lib.dcmt_bgr2lab_u8_host
    assert h(None, b.ctypes.data, 4, 4, 0, 0, 1) == _lib.DCMT_E_BADARG
    assert h(a.ctypes.data, a.ctypes.data + 8, 4, 4, 0, 0, 1) == _lib.DCMT_E_BADARG
    assert h(a.ctypes.data, b.ctypes.data, 4, 4, 11, 0, 1) == _lib.DCMT_E_BADARG
    # adjacent ranges do not overlap; zero frames read and write nothing
    emu_lib.check(emu_lib.dcmt_bgr2lab_u8(a.ctypes.data, a.ctypes.data + 48, 4, 4, 0, 0, 1, None))
    emu_lib.check(emu_lib.dcmt_bgr2lab_u8(a.ctypes.data, a.ctypes.data, 4, 4, 0, 0, 0, None))


def test_emu_slic_bgr_equals_slic_on_lab(emu_lib):
    """cvtColor + generate_superpixels in one call == generate_superpixels on OpenCV's Lab of the same frames."""
    bgr = np.stack([synth.bgr_image(f, 40, 58) for f in range(2)])
    lab = want_lab(bgr)
    for step, nc in ((8, 50), (13, 40)):
        got_l, got_c = api.generate_superpixels_bgr(bgr, step, nc, return_centers=True, lib=emu_lib)
        want_l, want_c = api.generate_superpixels(lab, step, nc, return_centers=True, lib=emu_lib)
        assert np.array_equal(got_l, want_l) and np.array_equal(got_c.view(np.uint64), want_c.view(np.uint64)), (step, nc)
        # the device entry point (emulator pointers are host pointers)
        k = emu_lib.dcmt_slic_center_count(40, 58, step)
        labels = np.empty((2, 40, 58), np.int32)
        centers = np.empty((2, k, 5), np.float64)
        emu_lib.check(emu_lib.dcmt_slic_bgr_u8c3(bgr.ctypes.data, 40, 58, 2, step, nc, 10, labels.ctypes.data, centers.ctypes.data, None))
        assert np.array_equal(labels, want_l) and np.array_equal(centers.view(np.uint64), want_c.view(np.uint64)), (step, nc)
    assert emu_lib.dcmt_slic_bgr_u8c3_host(None, 40, 58, 1, 8, 50, 10, labels.ctypes.data, None) == _lib.DCMT_E_BADARG


# ---------------------------------------------------------------------------------------------- the product on the GPU
def _to_cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
def test_gpu_bgr2lab(gpu_lib, mode):
    to_backend = (lambda a: a) if mode == "host" else _to_cuda
    got = api.bgr2lab(to_backend(all_colours()), lib=gpu_lib)
    got = got if isinstance(got, np.ndarray) else got.cpu().numpy()
    assert hashlib.sha256(got.tobytes()).hexdigest() == ALL_COLOURS_LAB_SHA256
    body(gpu_lib, to_backend)


@pytest.mark.gpu
def test_gpu_bgr2lab_pitched_unaligned_batched(gpu_lib):
    import torch

    rng = np.random.default_rng(3)
    n, rows, cols = 3, 17, 1216 + 5
    img = rng.integers(0, 256, (n, rows, cols, 3), dtype=np.uint8)
    want = want_lab(img)
    for bp, lp, in_off, out_off in ((0, 0, 0, 0), (cols * 3 + 13, cols * 3 + 32, 0, 0), (0, 0, 3, 1), (cols * 3 + 16, 0, 16, 5)):
        bpe, lpe = bp or cols * 3, lp or cols * 3
        src = torch.zeros(n * rows * bpe + 64, dtype=torch.uint8, device="cuda")
        src_rows = src[in_off:in_off + n * rows * bpe].view(n, rows, bpe)
        src_rows[:, :, : cols * 3] = torch.from_numpy(img.reshape(n, rows, cols * 3)).cuda()
        dst = torch.full((n * rows * lpe + 64,), 7, dtype=torch.uint8, device="cuda")
        gpu_lib.check(gpu_lib.dcmt_bgr2lab_u8(src.data_ptr() + in_off, dst.data_ptr() + out_off, rows, cols, bp, lp, n,
                                              int(torch.cuda.current_stream().cuda_stream)))
        out = dst.cpu().numpy()
        body_ = out[out_off:out_off + n * rows * lpe].reshape(n, rows, lpe)
        assert np.array_equal(body_[:, :, : cols * 3].reshape(img.shape), want), (bp, lp, in_off, out_off)
        assert (out[:out_off] == 7).all() and (body_[:, :, cols * 3:] == 7).all() and (out[out_off + n * rows * lpe:] == 7).all()
    # the host entry point with pitched rows
    src = rng.integers(0, 256, (n, rows, cols * 3 + 9), dtype=np.uint8)
    dst = np.full((n, rows, cols * 3 + 4), 7, np.uint8)
    gpu_lib.check(gpu_lib.dcmt_bgr2lab_u8_host(src.ctypes.data, dst.ctypes.data, rows, cols, src.shape[2], dst.shape[2], n))
    assert np.array_equal(dst[:, :, : cols * 3].reshape(n, rows, cols, 3), want_lab(np.ascontiguousarray(src[:, :, : cols * 3]).reshape(n, rows, cols, 3)))
    assert (dst[:, :, cols * 3:] == 7).all()
    a = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    b = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    for what, rc in badarg_cases(gpu_lib, a.data_ptr(), b.data_ptr()):
        assert rc == _lib.DCMT_E_BADARG, what
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("step,nc", [(18, 50), (65, 40)])  # main_lc.cpp:197-201 (1200 superpixels); main_sl.cpp:438-450 (100, nc 40)
def test_gpu_slic_bgr_equals_slic_on_lab(gpu_lib, mode, step, nc):
    bgr = np.stack([synth.bgr_image(f) for f in range(2)])
    lab = want_lab(bgr)
    cv2 = _cv2()
    if cv2 is not None:
        assert np.array_equal(lab, np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2Lab) for f in bgr]))
    to_backend = (lambda a: a) if mode == "host" else _to_cuda
    got_l, got_c = api.generate_superpixels_bgr(to_backend(bgr), step, nc, return_centers=True, lib=gpu_lib)
    want_l, want_c = api.generate_superpixels(to_backend(lab), step, nc, return_centers=True, lib=gpu_lib)
    if mode == "device":
        got_l, got_c, want_l, want_c = (t.cpu().numpy() for t in (got_l, got_c, want_l, want_c))
    assert np.array_equal(got_l, want_l)
    assert np.array_equal(got_c.view(np.uint64), want_c.view(np.uint64))
    assert (got_l >= 0).any()
