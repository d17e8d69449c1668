"""(a1) img_completion parity: CUDA path through the C ABI vs the oracle.

Bar (SURVEY.md 8c): bit-exact for the whole pipeline on q8 input in none/gaussian mode and for every
min/max/median/fill/extrapolation/invert stage on arbitrary finite float input (blur "none");
Gaussian on non-q8 input bit-equal to the C restatement (same operation order), max-abs <= 1e-4 against cv2 (the golden
files); bilateral max-abs <= 2e-4.
The same bodies run on the CPU emulator build (not gpu) and on the B200 (gpu)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, synth
from oracle import c_oracle as co
from tests.conftest import GOLDEN, assert_bit_equal
from tests.helpers import Backend

GAUSS_TOL = 1e-4  # float Gaussian against cv2 (the golden files)
BILATERAL_TOL = 2e-4


def check_case(be: Backend, name: str, s: np.ndarray, want_none, want_gauss, want_bilat, want_passes=None, c_port=False):
    """c_port: the expected values come from the C restatement, so the float Gaussian must match it bit for bit."""
    q8 = not name.startswith("float")
    got, st = be.img_completion(s, "none", return_stats=True)
    assert_bit_equal(got, want_none, f"{name} blur=none")
    if want_passes is not None:
        assert int(st[0, 0]) == want_passes, f"{name}: loop passes {st[0, 0]} != {want_passes}"
    got = be.img_completion(s, "gaussian")
    if q8 or c_port:
        assert_bit_equal(got, want_gauss, f"{name} blur=gaussian")
    else:
        assert np.abs(got - want_gauss).max() <= GAUSS_TOL, name
    got = be.img_completion(s, "bilateral")
    assert np.abs(got - want_bilat).max() <= BILATERAL_TOL, f"{name} bilateral {np.abs(got - want_bilat).max()}"


def golden_cases(golden):
    g = golden["lidar_only"]
    for name in sorted({k.split("__")[0] for k in g.files}):
        yield name, g[name + "__in"], g[name + "__none"], g[name + "__gaussian"], g[name + "__bilateral"], int(g[name + "__passes"])


def body_golden(be, golden):
    for case in golden_cases(golden):
        check_case(be, *case)


def body_seeded(be, shapes):
    for i, (rows, cols, p) in enumerate(shapes):
        s = synth.sparse_depth(40 + i, rows, cols, p, kitti_like=bool(i & 1))
        st = {}
        want_none = co.img_completion(s, "none", st)
        check_case(be, f"q8_{rows}x{cols}", s, want_none, co.img_completion(s, "gaussian"), co.img_completion(s, "bilateral"),
                   st["loop_passes"])
        f = synth.sparse_depth_float(40 + i, rows, cols, p)
        check_case(be, f"float_{rows}x{cols}", f, co.img_completion(f, "none"), co.img_completion(f, "gaussian"),
                   co.img_completion(f, "bilateral"), c_port=True)


def body_batch(be, rows, cols, n):
    """frames are independent: a batch equals its frames processed one by one; stats come back per frame."""
    batch = np.stack([synth.sparse_depth(60 + f, rows, cols, 0.05 if f % 3 else 0.01) for f in range(n)])
    out, st = be.img_completion(batch, "gaussian", return_stats=True)
    assert out.shape == batch.shape and st.shape == (n, 4)
    for f in range(n):
        ref_st = {}
        assert_bit_equal(out[f], co.img_completion(batch[f], "gaussian", ref_st), f"batch frame {f}")
        assert int(st[f, 0]) == ref_st["loop_passes"]
        assert int(st[f, 1]) == ref_st["holes_before_loop"]
        assert int(st[f, 2]) == ref_st["holes_after_extrapolation"]


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_golden(emu_lib, golden):
    body_golden(Backend(emu_lib, "emu"), golden)


def test_emu_seeded(emu_lib):
    body_seeded(Backend(emu_lib, "emu"), [(40, 70, 0.05), (65, 33, 0.02), (33, 129, 0.1)])


def test_emu_batch_and_chunking(emu_lib, monkeypatch):
    body_batch(Backend(emu_lib, "emu"), 36, 70, 5)


def test_emu_pitched_rows_and_frame_stride(emu_lib):
    """pitch_bytes / frame_stride_bytes of the C ABI (cv::Mat step semantics); padding is preserved."""
    rows, cols, n, pitch, extra = 20, 37, 3, 48, 5
    fstride = rows * pitch + extra
    src = np.zeros(n * fstride, np.float32)
    dst = np.full(n * fstride, -7.0, np.float32)
    frames = [synth.sparse_depth(80 + f, rows, cols, 0.1) for f in range(n)]
    for f in range(n):
        v = src[f * fstride:f * fstride + rows * pitch].reshape(rows, pitch)
        v[:, :cols] = frames[f]
    st = np.zeros((n, 4), np.int32)
    rc = emu_lib.dcmt_img_completion_f32_host(src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), rows, cols,
                                              pitch * 4, fstride * 4, n, 1, 0, st.ctypes.data_as(C.c_void_p))
    assert rc == 0, emu_lib.dcmt_last_error()
    for f in range(n):
        v = dst[f * fstride:f * fstride + rows * pitch].reshape(rows, pitch)
        assert_bit_equal(v[:, :cols].copy(), co.img_completion(frames[f], "gaussian"), f"pitched frame {f}")
        assert (v[:, cols:] == -7.0).all(), "row padding must not be written"


def test_emu_stage_snapshots(emu_lib):
    """the debugging entry point exposes the intermediates the kernels materialise; each equals the oracle's."""
    s = synth.sparse_depth(3, 50, 90, 0.03)
    out = np.empty_like(s)
    stages = np.zeros((_lib.N_STAGES,) + s.shape, np.float32)
    mask = C.c_uint32(0)
    rc = emu_lib.dcmt_img_completion_stages_f32(s.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), 50, 90, 1,
                                                stages.ctypes.data_as(C.c_void_p), _lib.N_STAGES, C.byref(mask), None)
    assert rc == 0, emu_lib.dcmt_last_error()
    want, want_stages = co.img_completion(s, "gaussian", stages=True)
    assert_bit_equal(out, want, "final")
    assert mask.value & (1 << 3) and mask.value & (1 << 9)
    for i in range(_lib.N_STAGES):
        if mask.value & (1 << i):
            assert_bit_equal(stages[i], want_stages[i], f"stage {i} ({co.STAGE_NAMES[i]})")


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_golden(gpu_lib, golden, mode):
    body_golden(Backend(gpu_lib, mode), golden)


@pytest.mark.gpu
def test_gpu_seeded(gpu_lib):
    body_seeded(Backend(gpu_lib, "gpu_device"), [(40, 70, 0.05), (65, 33, 0.02), (33, 129, 0.1), (200, 333, 0.01), (352, 1216, 0.05)])


@pytest.mark.gpu
def test_gpu_batch(gpu_lib):
    body_batch(Backend(gpu_lib, "gpu_device"), 36, 70, 5)
    body_batch(Backend(gpu_lib, "gpu_device"), 352, 1216, 6)


@pytest.mark.gpu
def test_gpu_full_size_digests(gpu_lib):
    """352 x 1216: sha256 of the GPU output equals the digest of OpenCV's output recorded in tests/golden."""
    be = Backend(gpu_lib, "gpu_device")
    lines = [l.split() for l in open(os.path.join(GOLDEN, "lidar_only_352x1216.sha256")) if not l.startswith("#")]
    for frame, kitti_like, blur, h_in, h_out in lines:
        s = synth.sparse_depth(int(frame), density=0.05, kitti_like=bool(int(kitti_like)))
        assert hashlib.sha256(s.tobytes()).hexdigest() == h_in
        assert hashlib.sha256(be.img_completion(s, blur).tobytes()).hexdigest() == h_out, (frame, kitti_like, blur)


@pytest.mark.gpu
def test_gpu_large_batch_properties(gpu_lib):
    """BASELINE-size batch (1024 frames = 64 unique x 16): every copy of a frame gives the same bytes, and the
    64 unique results equal the oracle's.  Size-independent check: xor-fold of all frames == fold of unique ones."""
    import torch

    from depth_completion_mt_b200 import api

    uniq = np.stack([synth.sparse_depth(f) for f in range(64)])
    dev = torch.from_numpy(uniq).cuda().repeat(16, 1, 1)
    out = api.img_completion(dev, False, "gaussian", lib=gpu_lib)
    first = out[:64]
    for k in range(1, 16):
        assert torch.equal(out[64 * k:64 * (k + 1)], first), f"replica {k} differs"
    host = first.cpu().numpy()
    for f in (0, 7, 31, 63):
        assert_bit_equal(host[f], co.img_completion(uniq[f], "gaussian"), f"frame {f}")


@pytest.mark.gpu
def test_gpu_sweep_sizes(gpu_lib):
    """resolution / density sweep of BASELINE configs[4], one frame each (oracle finishes in seconds)."""
    be = Backend(gpu_lib, "gpu_device")
    for rows, cols, p in [(512, 1760, 0.02), (1024, 2048, 0.01), (2048, 4096, 0.01), (2048, 4096, 0.2)]:
        s = synth.sparse_depth(5, rows, cols, p)
        st = {}
        want = co.img_completion(s, "gaussian", st)
        got, gst = be.img_completion(s, "gaussian", return_stats=True)
        assert_bit_equal(got, want, f"{rows}x{cols} p={p}")
        assert int(gst[0, 0]) == st["loop_passes"]


@pytest.mark.gpu
def test_gpu_fused_path_is_graph_capturable(gpu_lib):
    """DCMT_PATH_FUSED never synchronises or allocates once the workspace exists: a call can be captured into a CUDA graph
    and replayed on new data (include/dcmt.h, path flags)."""
    import torch

    from depth_completion_mt_b200 import api, synth
    from oracle import c_oracle as co

    frames = np.stack([synth.sparse_depth(300 + f, 96, 160, 0.05) for f in range(4)])
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.empty_like(d_in)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        api.img_completion(d_in, False, "gaussian", path="fused", out=d_out, lib=gpu_lib)  # sizes the workspace of this stream
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            api.img_completion(d_in, False, "gaussian", path="fused", out=d_out, lib=gpu_lib)
    new = np.stack([synth.sparse_depth(310 + f, 96, 160, 0.08) for f in range(4)])
    d_in.copy_(torch.from_numpy(new))
    d_out.zero_()
    graph.replay()
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    for f in range(4):
        assert_bit_equal(got[f], co.img_completion(new[f], "gaussian"), f"graph replay frame {f}")
