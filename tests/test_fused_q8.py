"""The strict-q8 fused path (fused_q8.cu) against the oracle: bit-exact end to end (none / gaussian), for odd
sizes, tile-edge cases, boundary q8 values, pitched input, multi-pass frames (fix-up kernel) and the routing
of non-q8 frames to the generic pipeline.  Same bodies on the CPU emulator build and on the B200."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from oracle.make_golden import multipass_frame
from tests.conftest import assert_bit_equal
from tests.helpers import Backend


def check(be, s, name, blur="gaussian", path="auto", want_path=1):
    out, st = be.img_completion(s, blur, path=path, return_stats=True)
    ref_st = {}
    assert_bit_equal(out, co.img_completion(s, blur, ref_st), f"{name} blur={blur} path={path}")
    assert int(st[0, 0]) == ref_st["loop_passes"], name
    assert int(st[0, 1]) == ref_st["holes_before_loop"], name
    assert int(st[0, 2]) == ref_st["holes_after_extrapolation"], name
    if want_path is not None:
        assert int(st[0, 3]) == want_path, f"{name}: path {st[0, 3]}"


def body_shapes(be, shapes):
    for i, (rows, cols, p) in enumerate(shapes):
        s = synth.sparse_depth(90 + i, rows, cols, p, kitti_like=bool(i & 1))
        check(be, s, f"{rows}x{cols}")
        check(be, s, f"{rows}x{cols}", blur="none", path="fused")


def body_boundary_values(be):
    """q8 codes around the thresholds: 26/256 is the smallest valid depth; 25574/256 inverts to 26/256 (still valid);
    25575/256 .. 25600/256 invert to < 0.1 and become holes again; 1/256 .. 25/256 are holes from the start.  Hole
    VALUES never reach the output (every stage only tests `< 0.1f`), so all of these stay on the fused path and
    must still match the oracle bit for bit.  Negative and > 100 m pixels are holes too."""
    rng = np.random.default_rng(3)
    base = synth.sparse_depth_q8(5, 48, 72, 0.08)
    for codes in ((26, 27, 25574, 25573, 300), (25,), (25575,), (25600,), (1,), (1, 25, 26, 25574, 25575, 25599, 25600, 30000, 65535)):
        d16 = base.copy()
        ys, xs = rng.integers(0, 48, 30), rng.integers(0, 72, 30)
        d16[ys, xs] = rng.choice(codes, 30)
        s = d16.astype(np.float32) / np.float32(256)
        check(be, s, f"codes {codes}", want_path=1)
    s = base.astype(np.float32) / np.float32(256)
    s[rng.integers(0, 48, 10), rng.integers(0, 72, 10)] = np.float32(-3.25)
    s[rng.integers(0, 48, 10), rng.integers(0, 72, 10)] = np.float32(0.05)
    s[rng.integers(0, 48, 10), rng.integers(0, 72, 10)] = np.float32(1e-30)
    check(be, s, "negative / tiny / sub-threshold values are holes", want_path=1)
    s2 = s.copy()
    s2[7, 9] = np.float32(12.3)  # a valid pixel that is not a multiple of 1/256: generic pipeline
    check(be, s2, "one non-q8 valid pixel", want_path=2)  # the float32 dictionary (DCMT_PATH_RANK) serves it
    # slivers next to the thresholds where a non-q8 value is valid for the reference: must be caught, not mapped to a hole
    for v in (0.1, np.nextafter(np.float32(0.1015625), np.float32(0)), 99.899, 99.8999, np.nextafter(np.float32(99.9), np.float32(0)),
              np.nextafter(np.float32(36.00390625), np.float32(0)), np.nextafter(np.float32(12.5), np.float32(100))):
        s3 = base.astype(np.float32) / np.float32(256)
        s3[11, 13] = np.float32(v)
        check(be, s3, f"sliver value {v!r}", want_path=2)
    # ... and just outside them the pixel is a hole for the reference too (either path is fine, the bytes must match)
    for v in (0.0999, 99.9, 99.95, 100.0, 250.0):
        s3 = base.astype(np.float32) / np.float32(256)
        s3[11, 13] = np.float32(v)
        check(be, s3, f"hole-class value {v!r}", want_path=None)


def body_routing(be):
    s = synth.sparse_depth(6, 64, 96, 0.05)
    check(be, s, "forced generic", path="generic", want_path=0)
    f = synth.sparse_depth_float(6, 64, 96, 0.05)
    check(be, f, "float frame via auto", want_path=2)
    check(be, f, "float frame, dictionary path asked for", path="rank", want_path=2)
    check(be, f, "float frame, blur none: bit-exact", blur="none", want_path=2)
    # DCMT_PATH_FUSED trusts the caller (no validation, no synchronisation): only meaningful for strict q8 frames
    check(be, s, "forced fused", path="fused", want_path=1)
    # bilateral and tiny frames are served by the generic pipeline whatever the flag says
    out, st = be.img_completion(s, "bilateral", path="fused", return_stats=True)
    assert int(st[0, 3]) == 0 and np.abs(out - co.img_completion(s, "bilateral")).max() <= 2e-4
    t = synth.sparse_depth(6, 20, 24, 0.2)
    check(be, t, "tiny frame", path="fused", want_path=0)
    # mixed batch: only the non-q8 frame is redone
    b = np.stack([synth.sparse_depth(7, 64, 96, 0.05), f, synth.sparse_depth(8, 64, 96, 0.02)])
    out, st = be.img_completion(b, "gaussian", return_stats=True)
    assert [int(v) for v in st[:, 3]] == [1, 2, 1]
    for i in (0, 2):
        assert_bit_equal(out[i], co.img_completion(b[i], "gaussian"), f"mixed batch frame {i}")
    assert_bit_equal(out[1], co.img_completion(b[1], "gaussian"), "mixed batch frame 1 (dictionary path)")


def body_multipass(be, big=False):
    # very sparse frames: many holes survive the first 31x31 fill and are resolved by the growing-square search
    # (list path and, past 256 words per tile, the visit-everything path); up to 4-5 loop passes
    for seed, (rows, cols, p) in enumerate(((160, 260, 0.004), (97, 171, 0.001), (64, 400, 0.002))):
        check(be, synth.sparse_depth(70 + seed, rows, cols, p), f"very sparse {rows}x{cols} p={p}")
        check(be, synth.sparse_depth(70 + seed, rows, cols, p, kitti_like=True), f"very sparse kitti-like {rows}x{cols}", blur="none")
    if big:
        check(be, synth.sparse_depth(80, 352, 1216, 0.01), "352x1216 at 1 %")
        check(be, synth.sparse_depth(81, 352, 1216, 0.003, kitti_like=True), "352x1216 at 0.3 %")
    check(be, multipass_frame(), "multipass 120x64")
    check(be, multipass_frame(150, 200), "multipass 150x200", blur="none")
    b = np.stack([synth.sparse_depth(9, 120, 64, 0.05), multipass_frame(), synth.sparse_depth(10, 120, 64, 0.05)])
    out, st = be.img_completion(b, "gaussian", return_stats=True)
    assert [int(v) for v in st[:, 0]] == [1, 4, 1]
    for i in range(3):
        assert_bit_equal(out[i], co.img_completion(b[i], "gaussian"), f"frame {i}")


def body_u16(be, shapes):
    """KITTI uint16 input (main.cpp:75-82: PNG payload, convertTo(CV_32F, 1/256), img_completion): same bytes as the
    float32 call on d16 / 256, for every uint16 code, aligned and unaligned widths, fused and generic routing."""
    for i, (rows, cols, p) in enumerate(shapes):
        d16 = synth.sparse_depth_q8(300 + i, rows, cols, p, kitti_like=bool(i & 1))
        s = d16.astype(np.float32) / np.float32(256)
        for blur in ("gaussian", "none"):
            out, st = be.img_completion(d16, blur, return_stats=True)
            ref_st = {}
            assert_bit_equal(out, co.img_completion(s, blur, ref_st), f"u16 {rows}x{cols} {blur}")
            assert int(st[0, 0]) == ref_st["loop_passes"] and int(st[0, 2]) == ref_st["holes_after_extrapolation"]
            assert int(st[0, 3]) == (1 if rows >= 32 and cols >= 32 else 0)
    # every uint16 code once (256 x 256), then sparsified so that the pipeline has holes to fill
    codes = np.arange(65536, dtype=np.uint16).reshape(256, 256)
    rng = np.random.default_rng(12)
    codes = np.where(rng.random(codes.shape) < 0.15, rng.permutation(codes.ravel()).reshape(256, 256), 0).astype(np.uint16)
    s = codes.astype(np.float32) / np.float32(256)
    assert_bit_equal(be.img_completion(codes, "gaussian"), co.img_completion(s, "gaussian"), "all uint16 codes")
    assert_bit_equal(be.img_completion(codes, "gaussian", path="generic"), co.img_completion(s, "gaussian"), "all codes, generic")
    # bilateral is served by the generic pipeline behind the conversion kernel
    d16 = synth.sparse_depth_q8(17, 64, 96, 0.05)
    out = be.img_completion(d16, "bilateral")
    assert np.abs(out - co.img_completion(d16.astype(np.float32) / np.float32(256), "bilateral")).max() <= 2e-4
    # batch
    b16 = np.stack([synth.sparse_depth_q8(400 + f, 64, 96, 0.05) for f in range(5)])
    outb = be.img_completion(b16, "gaussian")
    for f in range(5):
        assert_bit_equal(outb[f], co.img_completion(b16[f].astype(np.float32) / np.float32(256), "gaussian"), f"u16 batch frame {f}")


def body_u16_pitched(lib):
    rows, cols, ipitch, opitch = 40, 70, 77, 75  # odd pitches: neither side is 16-byte aligned
    d16 = synth.sparse_depth_q8(21, rows, cols, 0.06)
    src = np.full((2, rows + 1, ipitch), 7, np.uint16)
    src[0, :rows, :cols] = d16
    src[1, :rows, :cols] = d16[::-1]
    dst = np.full((2, rows + 2, opitch), -3.0, np.float32)
    rc = lib.dcmt_img_completion_u16_host(src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), rows, cols, ipitch * 2,
                                          (rows + 1) * ipitch * 2, opitch * 4, (rows + 2) * opitch * 4, 2, 1, 0, None)
    assert rc == 0, lib.dcmt_last_error()
    assert_bit_equal(dst[0, :rows, :cols].copy(), co.img_completion(d16.astype(np.float32) / np.float32(256), "gaussian"), "pitched u16 f0")
    assert_bit_equal(dst[1, :rows, :cols].copy(), co.img_completion(d16[::-1].astype(np.float32) / np.float32(256), "gaussian"), "pitched u16 f1")
    assert (dst[:, :, cols:] == -3.0).all() and (dst[:, rows:] == -3.0).all()
    # argument errors: pitch too small for uint16 columns, aliasing
    assert lib.dcmt_img_completion_u16_host(src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), rows, cols, cols * 2 - 2, 0,
                                            0, 0, 1, 1, 0, None) == -1
    assert lib.dcmt_img_completion_u16_host(dst.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), rows, cols, 0, 0, 0, 0, 1, 1,
                                            0, None) == -1


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_u16(emu_lib):
    body_u16(Backend(emu_lib, "emu"), [(32, 32, 0.1), (33, 47, 0.05), (97, 171, 0.03), (20, 24, 0.2), (96, 160, 0.2)])
    body_u16_pitched(emu_lib)


def test_emu_shapes(emu_lib):
    body_shapes(Backend(emu_lib, "emu"), [(32, 32, 0.1), (33, 47, 0.05), (97, 171, 0.03), (100, 321, 0.02), (193, 40, 0.05), (96, 160, 0.2)])


def test_emu_boundary_values(emu_lib):
    body_boundary_values(Backend(emu_lib, "emu"))


def test_emu_routing(emu_lib):
    body_routing(Backend(emu_lib, "emu"))


def test_emu_multipass(emu_lib):
    body_multipass(Backend(emu_lib, "emu"))


def test_emu_kitti_frame(emu_lib):
    check(Backend(emu_lib, "emu"), synth.sparse_depth(1, kitti_like=True), "352x1216")


def test_emu_reverse_block_and_thread_order():
    """The emulator normally runs blocks and threads in ascending order, which hides write conflicts between tiles
    and missing barriers.  Re-run a multi-tile frame whose tile height is not a multiple of the 4-row Gaussian
    items with both orders reversed (separate process: the order is read once)."""
    import subprocess
    import sys

    from tests.conftest import ROOT

    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from depth_completion_mt_b200 import _lib, api, synth\n"
        "from oracle import c_oracle as co\n"
        "from tests.emu import build_emu\n"
        "lib = _lib.bind(build_emu.build())\n"
        "for (r, c, p, k) in ((200, 333, 0.01, True), (97, 171, 0.05, False), (120, 64, 0.03, False)):\n"
        "    s = synth.sparse_depth(43, r, c, p, kitti_like=k)\n"
        "    for blur in ('gaussian', 'none'):\n"
        "        out = api.img_completion(s, False, blur, lib=lib)\n"
        "        assert np.array_equal(out.view(np.uint32), co.img_completion(s, blur).view(np.uint32)), (r, c, blur)\n"
        "    g = api.img_completion(s, False, 'gaussian', path='generic', lib=lib)\n"
        "    assert np.array_equal(g.view(np.uint32), co.img_completion(s, 'gaussian').view(np.uint32)), (r, c, 'generic')\n"
        "for (r, c, p) in ((97, 171, 0.05), (64, 200, 0.01)):\n"
        "    f = synth.sparse_depth_float(44, r, c, p)\n"
        "    out = api.img_completion(f, False, 'none', path='rank', lib=lib)\n"
        "    assert np.array_equal(out.view(np.uint32), co.img_completion(f, 'none').view(np.uint32)), (r, c, 'rank')\n"
        "    out = api.img_completion(f, False, 'gaussian', lib=lib)\n"
        "    assert np.array_equal(out.view(np.uint32), co.img_completion(f, 'gaussian').view(np.uint32)), (r, c, 'rank gaussian')\n"
        "import os\n"
        "os.environ['DCMT_SLIC_BAND_MIN_FRAMES'] = '1'\n"
        "lab = np.stack([synth.lab_image(k, 64, 96) for k in range(2)])\n"
        "labels = api.generate_superpixels(lab, 10, 40, lib=lib)\n"
        "for k in range(2):\n"
        "    assert np.array_equal(labels[k], co.slic(lab[k], 10, 40)[0]), 'band SLIC'\n"
        "print('REVERSE_OK')\n" % ROOT
    )
    env = dict(os.environ, DCMT_EMU_ORDER="reverse")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "REVERSE_OK" in r.stdout, r.stdout + r.stderr


def test_emu_pitched_input_takes_scalar_loads(emu_lib):
    rows, cols, pitch = 40, 70, 75  # odd pitch: rows are not 16-byte aligned
    s = synth.sparse_depth(11, rows, cols, 0.06)
    src = np.zeros((rows, pitch), np.float32)
    src[:, :cols] = s
    dst = np.full((rows, pitch), -3.0, np.float32)
    st = np.zeros((1, 4), np.int32)
    rc = emu_lib.dcmt_img_completion_f32_host(src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), rows, cols, pitch * 4, 0, 1, 1,
                                              0, st.ctypes.data_as(C.c_void_p))
    assert rc == 0, emu_lib.dcmt_last_error()
    assert int(st[0, 3]) == 1
    assert_bit_equal(dst[:, :cols].copy(), co.img_completion(s, "gaussian"), "pitched")
    assert (dst[:, cols:] == -3.0).all()


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_shapes(gpu_lib, mode):
    body_shapes(Backend(gpu_lib, mode), [(32, 32, 0.1), (33, 47, 0.05), (97, 171, 0.03), (100, 321, 0.02), (193, 40, 0.05), (96, 160, 0.2),
                                         (352, 1216, 0.05), (375, 1242, 0.05), (512, 1760, 0.02)])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_u16(gpu_lib, mode):
    body_u16(Backend(gpu_lib, mode), [(32, 32, 0.1), (33, 47, 0.05), (97, 171, 0.03), (20, 24, 0.2), (352, 1216, 0.05), (375, 1242, 0.05)])
    body_u16_pitched(gpu_lib)


@pytest.mark.gpu
def test_gpu_boundary_routing_multipass(gpu_lib):
    be = Backend(gpu_lib, "gpu_device")
    body_boundary_values(be)
    body_routing(be)
    body_multipass(be, big=True)
    body_routing(Backend(gpu_lib, "gpu_host"))


@pytest.mark.gpu
def test_gpu_fused_equals_generic_on_a_large_batch(gpu_lib):
    """256 distinct frames at KITTI size, densities 1-20 %: the fused and the generic pipeline give the same bytes."""
    import torch

    dens = (0.01, 0.02, 0.05, 0.1, 0.2)
    batch = np.stack([synth.sparse_depth(200 + f, density=dens[f % 5], kitti_like=bool(f & 1)) for f in range(256)])
    dev = torch.from_numpy(batch).cuda()
    a, sa = api.img_completion(dev, False, "gaussian", path="fused", return_stats=True, lib=gpu_lib)
    b, sb = api.img_completion(dev, False, "gaussian", path="generic", return_stats=True, lib=gpu_lib)
    assert torch.equal(a, b)
    assert torch.equal(sa[:, :3], sb[:, :3]) and bool((sa[:, 3] == 1).all()) and bool((sb[:, 3] == 0).all())
    for f in (0, 101, 255):
        assert_bit_equal(a[f].cpu().numpy(), co.img_completion(batch[f], "gaussian"), f"frame {f}")


@pytest.mark.gpu
def test_gpu_large_shapes(gpu_lib):
    """BASELINE configs[4] shapes: 1024x2048 against the oracle, 2048x4096 fused == generic (the oracle needs seconds there)
    plus one oracle frame; densities 1 % and 20 %."""
    import torch

    for rows, cols, p in ((1024, 2048, 0.01), (1024, 2048, 0.2)):
        s = synth.sparse_depth(500, rows, cols, p)
        out, st = api.img_completion(torch.from_numpy(s).cuda(), False, "gaussian", return_stats=True, lib=gpu_lib)
        assert int(st[0, 3]) == 1
        assert_bit_equal(out.cpu().numpy(), co.img_completion(s, "gaussian"), f"{rows}x{cols} p={p}")
    big = np.stack([synth.sparse_depth(510 + f, 2048, 4096, 0.05, kitti_like=bool(f)) for f in range(2)])
    dev = torch.from_numpy(big).cuda()
    a = api.img_completion(dev, False, "gaussian", path="fused", lib=gpu_lib)
    b = api.img_completion(dev, False, "gaussian", path="generic", lib=gpu_lib)
    assert torch.equal(a, b)
    assert_bit_equal(a[0].cpu().numpy(), co.img_completion(big[0], "gaussian"), "2048x4096")


def body_rank(be, shapes, big=False):
    """DCMT_PATH_RANK (rank_f32.cu): float32 frames that are not strict q8 -- what the stereo program completes after
    cv::normalize (main_sl.cpp:522-540) -- run on the fused kernels through a per-frame order-preserving dictionary.
    Bit-exact against the C restatement for any finite input: with blur none every stage only selects, and the float32
    Gaussian uses the C restatement's operation order (it stays within 1e-4 of cv2 and the reference build)."""
    for i, (rows, cols, p) in enumerate(shapes):
        f = synth.sparse_depth_float(400 + i, rows, cols, p)
        if i % 3 == 1:  # negatives, sub-threshold, > 99.9 (inverts to a hole), exactly 100, duplicates
            rng = np.random.default_rng(i)
            f = f.copy()
            f[rng.integers(0, rows, 20), rng.integers(0, cols, 20)] = np.float32(-2.5)
            f[rng.integers(0, rows, 20), rng.integers(0, cols, 20)] = np.float32(0.0999)
            f[rng.integers(0, rows, 20), rng.integers(0, cols, 20)] = np.float32(99.95)
            f[rng.integers(0, rows, 20), rng.integers(0, cols, 20)] = np.float32(100.0)
            f[rng.integers(0, rows, 40), rng.integers(0, cols, 40)] = np.float32(17.123)
        for path in ("rank", "auto"):
            out, st = be.img_completion(f, "none", path=path, return_stats=True)
            ref_st = {}
            assert_bit_equal(out, co.img_completion(f, "none", ref_st), f"rank {rows}x{cols} p={p} none {path}")
            assert int(st[0, 3]) == 2 and int(st[0, 0]) == ref_st["loop_passes"] and int(st[0, 2]) == ref_st["holes_after_extrapolation"]
            out = be.img_completion(f, "gaussian", path=path)
            assert_bit_equal(out, co.img_completion(f, "gaussian"), f"rank {rows}x{cols} gaussian {path}")
    # a frame with more valid pixels than the dictionary holds (32768) goes to the generic pipeline; so does a NaN
    rows, cols = (352, 1216) if big else (200, 400)
    dense = synth.sparse_depth_float(420, rows, cols, 0.5)
    assert (dense >= 0.1).sum() > 32768
    out, st = be.img_completion(dense, "none", path="rank", return_stats=True)
    assert int(st[0, 3]) == 0
    assert_bit_equal(out, co.img_completion(dense, "none"), "dictionary overflow -> generic")
    b = np.stack([synth.sparse_depth_float(421, 64, 96, 0.05), synth.sparse_depth(422, 64, 96, 0.05), synth.sparse_depth_float(423, 64, 96, 0.05)])
    out, st = be.img_completion(b, "none", return_stats=True)
    assert [int(v) for v in st[:, 3]] == [2, 1, 2]
    for i in range(3):
        assert_bit_equal(out[i], co.img_completion(b[i], "none"), f"mixed batch frame {i}")
    # the normalised projection of a LiDAR cloud (main_sl.cpp:522-540): the input the stereo program really feeds
    pts = synth.velodyne_cloud(7, 60000 if big else 30000)
    r2, c2 = (352, 1216) if big else (200, 700)
    nrm = co.lidar_project(pts, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, r2, c2)[1]
    out, st = be.img_completion(nrm, "none", return_stats=True)
    assert (nrm >= 0.1).sum() > 300 and int(st[0, 3]) == 2
    assert_bit_equal(out, co.img_completion(nrm, "none"), "normalised projection, blur none")
    assert_bit_equal(be.img_completion(nrm, "gaussian"), co.img_completion(nrm, "gaussian"), "normalised projection, gaussian")


def test_emu_rank(emu_lib):
    body_rank(Backend(emu_lib, "emu"), [(64, 96, 0.05), (97, 171, 0.05), (120, 200, 0.01), (80, 136, 0.3), (50, 333, 0.002)])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_rank(gpu_lib, mode):
    body_rank(Backend(gpu_lib, mode), [(352, 1216, 0.05), (375, 1242, 0.05), (352, 1216, 0.01), (97, 171, 0.05), (512, 1760, 0.02),
                                       (1024, 2048, 0.005)], big=True)
