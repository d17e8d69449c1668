"""The region load of k_q8_front: one TMA box copy of the region when the input layout can be mapped (base, row pitch and
frame stride multiples of 16 bytes), per-thread loads otherwise.  Both must give the C oracle's bytes: pitched and
unaligned batches (per-thread loads), aligned batches whose width is not a multiple of 8 (the quad straddling the right
edge decoded from the zero-filled box), multi-chunk batches (one map per chunk) and the same batches with the TMA load
switched off.  The device entry points are called directly so that the input layout reaches the kernel as given; on the
emulator build the same calls run on host memory."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import _lib, synth
from oracle import c_oracle as co
from tests.conftest import ROOT, assert_bit_equal

GAUSSIAN, NONE = _lib.BLUR["gaussian"], 0


def run_device_entry(lib, on_gpu, frames, pitch, offset, blur, flags=0):
    """frames (n, rows, cols) placed `offset` elements into a buffer with rows of `pitch` elements and frames of
    (rows + 1) * pitch elements; returns the output frames and the per-frame path (stats column 3)."""
    n, rows, cols = frames.shape
    fstride = (rows + 1) * pitch
    src = np.full(offset + n * fstride, 7, frames.dtype)
    view = src[offset:].reshape(n, rows + 1, pitch)
    view[:, :rows, :cols] = frames
    dst = np.full(offset + n * fstride, -3.0, np.float32)
    esz = frames.dtype.itemsize
    u16 = frames.dtype == np.uint16
    if on_gpu:
        import torch

        d_src, d_dst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
        stats = torch.zeros((n, _lib.STATS_STRIDE), dtype=torch.int32, device="cuda")
        sp, dp, stp, stream = d_src.data_ptr() + offset * esz, d_dst.data_ptr() + offset * 4, stats.data_ptr(), None
    else:
        stats = np.zeros((n, _lib.STATS_STRIDE), np.int32)
        sp, dp, stp, stream = src.ctypes.data + offset * esz, dst.ctypes.data + offset * 4, stats.ctypes.data, None
    if u16:
        rc = lib.dcmt_img_completion_u16(C.c_void_p(sp), C.c_void_p(dp), rows, cols, pitch * 2, fstride * 2, pitch * 4, fstride * 4, n,
                                         blur, flags, C.c_void_p(stp), stream)
    else:
        rc = lib.dcmt_img_completion_f32(C.c_void_p(sp), C.c_void_p(dp), rows, cols, pitch * 4, fstride * 4, n, blur, flags,
                                         C.c_void_p(stp), stream)
    assert rc == 0, lib.dcmt_last_error()
    if on_gpu:
        dst, stats = d_dst.cpu().numpy(), stats.cpu().numpy()
    out = dst[offset:].reshape(n, rows + 1, pitch)
    assert (out[:, :, cols:] == -3.0).all() and (out[:, rows:] == -3.0).all(), "pixels outside the frames were written"
    return out[:, :rows, :cols].copy(), stats[:, 3].copy()


def check_layout(lib, on_gpu, frames, pitch, offset, want_paths, what):
    q8 = frames.dtype == np.uint16
    ref_in = frames.astype(np.float32) / np.float32(256) if q8 else frames
    for blur, name in ((GAUSSIAN, "gaussian"), (NONE, "none")):
        out, paths = run_device_entry(lib, on_gpu, frames, pitch, offset, blur)
        assert list(paths) == want_paths, f"{what}: paths {list(paths)}"
        for f in range(len(frames)):  # frames that are not strict q8 take the dictionary path: bit-exact as well
            assert_bit_equal(out[f], co.img_completion(ref_in[f], name), f"{what} frame {f} blur={name}")


def body_layouts(lib, on_gpu):
    rows, cols = 45, 70  # 70 = 8 * 8 + 6: one quad straddles the right edge
    f32 = np.stack([synth.sparse_depth(600 + f, rows, cols, 0.06, kitti_like=bool(f & 1)) for f in range(3)])
    f32[1, 9, 13] = np.float32(12.3)  # one valid pixel off the q8 grid: the in-kernel validation sends frame 1 elsewhere
    u16 = np.stack([synth.sparse_depth_q8(610 + f, rows, cols, 0.06) for f in range(3)])
    # rows of 72 floats / 80 uint16 (288 / 160 bytes), aligned base: the TMA box copy
    check_layout(lib, on_gpu, f32, 72, 0, [1, 2, 1], "f32 mapped, ragged width")
    check_layout(lib, on_gpu, u16, 80, 0, [1, 1, 1], "u16 mapped, ragged width")
    # rows of 75 floats / 77 uint16 and a base one element past 16-byte alignment: per-thread loads
    check_layout(lib, on_gpu, f32, 75, 1, [1, 2, 1], "f32 pitched and unaligned")
    check_layout(lib, on_gpu, u16, 77, 1, [1, 1, 1], "u16 pitched and unaligned")
    # aligned rows but a base 4 bytes off: per-thread loads (scalar: the rows are not 16-byte aligned either)
    check_layout(lib, on_gpu, f32[:, :, :64].copy(), 64, 1, [1, 2, 1], "f32 unaligned base")


_CHUNKED = r"""
import sys; sys.path.insert(0, %(root)r)
import numpy as np
from depth_completion_mt_b200 import _lib, api, synth
from oracle import c_oracle as co
from tests.test_front_tma import body_layouts
on_gpu = %(gpu)r
if on_gpu:
    lib = _lib.load()
else:
    from tests.emu import build_emu
    lib = _lib.bind(build_emu.build())
if on_gpu:
    import torch
    dev = lambda a: torch.from_numpy(a).cuda()
    host = lambda t: t.cpu().numpy()
else:
    dev = host = lambda a: a
rows, cols = %(shape)s
f32 = np.stack([synth.sparse_depth(620 + f, rows, cols, 0.04, kitti_like=bool(f & 1)) for f in range(5)])
u16 = np.stack([synth.sparse_depth_q8(630 + f, rows, cols, 0.04) for f in range(5)])
flt = np.stack([synth.sparse_depth_float(640 + f, rows, cols, 0.04) for f in range(5)])
for name, batch, ref, path, blur in (("f32", f32, f32, "auto", "gaussian"), ("u16", u16, u16.astype(np.float32) / np.float32(256), "auto", "gaussian"),
                                     ("rank", flt, flt, "rank", "none")):
    out, st = api.img_completion(dev(batch), False, blur, path=path, return_stats=True, lib=lib)
    out, st = host(out), host(st)
    assert list(st[:, 3]) == [2 if path == "rank" else 1] * 5, (name, st[:, 3])
    for f in range(5):
        assert np.array_equal(out[f].view(np.uint32), co.img_completion(ref[f], blur).view(np.uint32)), (name, f)
if %(layouts)r:
    body_layouts(lib, on_gpu)
print("CHUNKED_OK")
"""


def run_chunked(on_gpu, no_tma, shape):
    """5 frames in chunks of 2 (a tensor map per chunk, each with its own base), in a separate process: the chunk size
    and the TMA switch are read once per process.  With the TMA load switched off, the layouts of body_layouts as well."""
    env = dict(os.environ, DCMT_FUSED_CHUNK="2")
    if no_tma:
        env["DCMT_NO_TMA"] = "1"
    code = _CHUNKED % {"root": ROOT, "gpu": on_gpu, "shape": shape, "layouts": no_tma}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800, env=env, cwd=ROOT)
    assert r.returncode == 0 and "CHUNKED_OK" in r.stdout, r.stdout + r.stderr


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_front_layouts(emu_lib):
    body_layouts(emu_lib, False)


@pytest.mark.parametrize("no_tma", [False, True], ids=["tma", "no_tma"])
def test_emu_front_chunked(no_tma):
    run_chunked(False, no_tma, "(64, 90)")


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
def test_gpu_front_layouts(gpu_lib):
    body_layouts(gpu_lib, True)


@pytest.mark.gpu
@pytest.mark.parametrize("no_tma", [False, True], ids=["tma", "no_tma"])
def test_gpu_front_chunked(no_tma):
    run_chunked(True, no_tma, "(352, 1216)")
