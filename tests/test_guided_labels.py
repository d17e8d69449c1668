"""The fused guided front (k_q8_guided_front) on label maps built to reach each of its branches, bit for bit against the C
restatement's closed form (co.interpolate_with_superpixels(literal=False)).

The per-label kernel gathers the labels of a tile into a 512-slot hash table (LabelTable: slot = label * 40503 mod 512,
linear probing), falls back to the word-by-word kernel when more than 384 (3/4) distinct labels meet its scanned area
(core rows +- 3, words 2 .. tw / 2 + 5), and runs one warp per label over the label's bounding box: a half warp when both
boxes of a pair are narrower than 11 words, else a whole warp in chunks of 27 output words.  Labels are kept as uint16
with 0xffff meaning "no label", so n_clusters 65535 is the last count the fused front takes.  Each generator below is
named for the branch it targets; every one runs on q8 float, KITTI uint16 and arbitrary float input (the dictionary
path), with the word-by-word kernel serving every tile, and on the emulator with blocks and threads in reverse order."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from tests.conftest import ROOT, assert_bit_equal
from tests.helpers import Backend


def grid(rows, cols, step):
    yy, xx = np.mgrid[0:rows, 0:cols]
    return ((yy // step) * ((cols + step - 1) // step) + xx // step).astype(np.int32)


def gen_wide(rows, cols):
    """boxes 54 px (27 words: one chunk), 55 and 56 px (two chunks), 110 px and the whole frame (several chunks)"""
    yy, xx = np.mgrid[0:rows, 0:cols]
    for w, off in ((54, 0), (55, 0), (55, 1), (56, 0), (110, 3)):
        yield f"wide {w} px, offset {off}", ((yy // 20) * 100 + (xx + off) // w).astype(np.int32), None
    yield "one label per band of rows, full width", (yy // 24).astype(np.int32), None


def gen_narrow(rows, cols):
    """boxes of 20..26 px (10..13 words, either side of the half-warp bound) mixed in every tile, so that narrow boxes are
    paired with narrow and with wide ones"""
    widths = np.resize(np.array([20, 22, 24, 26, 21, 23, 25]), cols)
    edges = np.cumsum(widths)
    col_lab = np.searchsorted(edges, np.arange(cols), side="right")
    yy = np.arange(rows)[:, None]
    yield "boxes of 20..26 px", ((yy // 16) * (int(col_lab.max()) + 1) + col_lab[None, :]).astype(np.int32), None


def gen_collisions(rows, cols):
    """labels congruent mod 512 share a hash slot (40503 is odd): c + 512 j, up to 65534 for c = 510"""
    cells = grid(rows, cols, 6) % 128
    for c in (3, 510):
        yield f"collisions at {c} + 512 j", (c + 512 * cells).astype(np.int32), 65535


def gen_edge_values(rows, cols):
    """label 65534 encodes as 0xfffe, next to the 0xffff sentinel; n_clusters 65536 no longer fits uint16 labels"""
    lab = grid(rows, cols, 12)
    lab[rows // 4: rows // 2, cols // 3: cols // 3 + 40] = 65534
    lab[-5:, -7:] = 65533
    yield "label 65534, n_clusters 65535", lab, 65535
    yield "label 65534, n_clusters 65536 (generic)", lab, 65536


def gen_shapes(rows, cols):
    """disconnected labels whose boxes cover every tile; two labels alternating pixel by pixel (both lanes of a word differ)"""
    yy, xx = np.mgrid[0:rows, 0:cols]
    yield "disconnected (x // 8 + y // 8) % 5", ((xx // 8 + yy // 8) % 5).astype(np.int32), 5
    yield "pixel checkerboard of two labels", ((xx + yy) & 1).astype(np.int32), 2


def gen_border(rows, cols):
    """labels that occur only on the image border: one-pixel rows and columns, and the four corner pixels"""
    lab = grid(rows, cols, 12)
    k = int(lab.max()) + 1
    lab[0, 1:-1], lab[-1, 1:-1], lab[1:-1, 0], lab[1:-1, -1] = k, k + 1, k + 2, k + 3
    lab[0, 0], lab[0, -1], lab[-1, 0], lab[-1, -1] = k + 4, k + 5, k + 6, k + 7
    yield "labels only on the image border", lab, k + 8


def gen_out_of_range(rows, cols):
    """negative labels and labels >= n_clusters: no superpixel, the pixel keeps its own value"""
    lab = grid(rows, cols, 10)
    k = int(lab.max()) + 1
    rng = np.random.default_rng(9)
    for v in (-1, -7, -(2 ** 31), k, k + 7, 65535, 65536, 2 ** 31 - 1):
        lab[rng.random(lab.shape) < 0.01] = v
    yield "negative and out-of-range labels", lab, k


GENERATORS = (gen_wide, gen_narrow, gen_collisions, gen_edge_values, gen_shapes, gen_border, gen_out_of_range)

# ---- fixed guided tiles (DCMT_GUIDED_TILE_H / _W) so that a label map can be placed relative to them
TILE_H, TILE_W = 32, 64
FIXED_ROWS, FIXED_COLS = 64, 128


def scanned_area(ty, tx, rows, cols):
    """image rows and columns whose labels the per-label kernel gathers for tile (ty, tx): core rows +- 3, and region
    words 2 .. tw / 2 + 5, i.e. columns x0 - 4 .. x0 + tw + 3"""
    y0, x0 = ty * TILE_H, tx * TILE_W
    return slice(max(0, y0 - 3), min(rows, y0 + TILE_H + 3)), slice(max(0, x0 - 4), min(cols, x0 + TILE_W + 4))


def table_limit_labels(n):
    """exactly n distinct labels in the scanned area of tile (0, 0): 2 x 2 blocks in raster order, the last label taking
    the rest of the area; a coarse grid of other labels outside it"""
    lab = grid(FIXED_ROWS, FIXED_COLS, 16)
    ys, xs = scanned_area(0, 0, FIXED_ROWS, FIXED_COLS)
    h, w = ys.stop - ys.start, xs.stop - xs.start
    yy, xx = np.mgrid[0:h, 0:w]
    block = (yy // 2) * ((w + 1) // 2) + xx // 2
    lab[ys, xs] = 1000 + np.minimum(block, n - 1)
    assert len(np.unique(lab[ys, xs])) == n
    return lab


def gen_fixed_tiles(rows=FIXED_ROWS, cols=FIXED_COLS):
    """the 3/4 table limit (384 labels stay on the per-label kernel, 385 fall back), and labels that occur only in a tile's
    halo rows or columns (the 3 rows / 4 columns next to a tile boundary)"""
    assert (rows, cols) == (FIXED_ROWS, FIXED_COLS)
    for n in (384, 385):
        lab = table_limit_labels(n)
        yield f"{n} labels in tile (0, 0)", lab, int(lab.max()) + 1
    lab = grid(rows, cols, 10)
    k = int(lab.max()) + 1
    yy, xx = np.mgrid[0:rows, 0:cols]
    seg = xx // 7
    lab[TILE_H - 3: TILE_H] = k + seg[TILE_H - 3: TILE_H]                       # rows of tile 0 seen by tile 1 as halo
    lab[TILE_H: TILE_H + 3] = k + 100 + seg[TILE_H: TILE_H + 3]                # rows of tile 1 seen by tile 0 as halo
    lab[:, TILE_W - 4: TILE_W] = k + 200 + yy[:, TILE_W - 4: TILE_W] // 5      # columns of tile 0 seen by tile 1 as halo
    lab[:, TILE_W: TILE_W + 4] = k + 300 + yy[:, TILE_W: TILE_W + 4] // 5      # columns of tile 1 seen by tile 0 as halo
    yield "labels only in the halo of a neighbouring tile", lab, k + 400


def inputs(seed, rows, cols):
    """(name, input, the float32 frame the oracle sees, fused path code): q8 float, KITTI uint16, arbitrary float"""
    d16 = synth.sparse_depth_q8(seed, rows, cols, 0.06)
    s = d16.astype(np.float32) / np.float32(256)
    f = synth.sparse_depth_float(seed, rows, cols, 0.06)
    return (("q8", s, s, 1), ("u16", d16, s, 1), ("float", f, f, 2))


def check_generator(be, gen, rows, cols, literal):
    for i, (name, lab, k) in enumerate(gen(rows, cols)):
        k = int(lab.max()) + 1 if k is None else k
        fused = k <= 65535
        for kind, sparse, ref_in, path in inputs(900 + i, rows, cols):
            ref_st = {}
            want = co.interpolate_with_superpixels(ref_in, lab, k, literal=False, stats=ref_st)
            if literal and kind == "q8" and k <= 4096:
                # the closed form must hold for the shape before it can judge the kernel
                assert_bit_equal(co.interpolate_with_superpixels(ref_in, lab, k, literal=True), want, f"{name}: literal loop")
            got, st = be.interpolate_with_superpixels(lab, sparse, 1, n_clusters=k, return_stats=True)
            assert_bit_equal(got, want, f"{name} {rows}x{cols} {kind}")
            assert int(st[0, 0]) == ref_st["loop_passes"], f"{name} {kind}: loop passes {st[0, 0]} != {ref_st['loop_passes']}"
            assert int(st[0, 3]) == (path if fused else 0), f"{name} {kind}: path {st[0, 3]}"


def body_labels(be, rows=64, cols=240, literal=False):
    for gen in GENERATORS:
        check_generator(be, gen, rows, cols, literal)


def body_fixed_tiles(be, literal=False):
    check_generator(be, gen_fixed_tiles, FIXED_ROWS, FIXED_COLS, literal)


_SUB = r"""
import sys; sys.path.insert(0, %(root)r)
from depth_completion_mt_b200 import _lib
from tests.helpers import Backend
from tests.test_guided_labels import body_fixed_tiles, body_labels
if %(gpu)r:
    lib = _lib.load()
    modes = ["gpu_host", "gpu_device"]
else:
    from tests.emu import build_emu
    lib = _lib.bind(build_emu.build())
    modes = ["emu"]
for mode in modes:
    %(body)s
print("LABELS_OK")
"""


def run_sub(on_gpu, env, body):
    """in a separate process: the switches are read once per process"""
    code = _SUB % {"root": ROOT, "gpu": on_gpu, "body": body}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800, env=dict(os.environ, **env), cwd=ROOT)
    assert r.returncode == 0 and "LABELS_OK" in r.stdout, r.stdout + r.stderr


FIXED_ENV = {"DCMT_GUIDED_TILE_H": str(TILE_H), "DCMT_GUIDED_TILE_W": str(TILE_W)}
FIXED_BODY = "body_fixed_tiles(Backend(lib, mode), literal=mode == 'emu')"
ALL_BODY = "body_labels(Backend(lib, mode)); body_fixed_tiles(Backend(lib, mode))"


# ------------------------------------------------------------------ CPU: emulator build
def test_emu_labels(emu_lib):
    body_labels(Backend(emu_lib, "emu"), literal=True)


def test_emu_fixed_tiles():
    run_sub(False, FIXED_ENV, FIXED_BODY)


def test_emu_word_by_word_kernel():
    """DCMT_GUIDED_PER_LABEL=0: the word-by-word kernel serves every tile"""
    run_sub(False, {"DCMT_GUIDED_PER_LABEL": "0"}, ALL_BODY)


def test_emu_reverse_order():
    """blocks and threads in reverse order: the table atomics and the per-label writes must not depend on the order"""
    run_sub(False, {"DCMT_EMU_ORDER": "reverse"}, ALL_BODY)


# ------------------------------------------------------------------ GPU: the product
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gpu_host", "gpu_device"])
def test_gpu_labels(gpu_lib, mode):
    be = Backend(gpu_lib, mode)
    body_labels(be)
    body_labels(be, 96, 400)
    body_labels(be, 352, 1216)


@pytest.mark.gpu
def test_gpu_fixed_tiles():
    run_sub(True, FIXED_ENV, FIXED_BODY)


@pytest.mark.gpu
def test_gpu_word_by_word_kernel():
    run_sub(True, {"DCMT_GUIDED_PER_LABEL": "0"}, ALL_BODY)


@pytest.mark.gpu
@pytest.mark.parametrize("step", [18, 65], ids=["main_lc", "main_sl"])
def test_gpu_slic_labels_large_batch(gpu_lib, step):
    """256 KITTI-size frames with the product's own SLIC labels (step 18 as main_lc, 65 as main_sl; nc 50): the labels equal
    the C restatement's on 2 frames, the fused guided path equals the generic one on every frame, and the C restatement
    on 3 frames"""
    import torch

    n_lab = 64
    lab_imgs = np.stack([synth.lab_image(950 + f, 352, 1216) for f in range(n_lab)])
    labels = api.generate_superpixels(torch.from_numpy(lab_imgs).cuda(), step, 50, lib=gpu_lib)
    for f in (0, n_lab - 1):
        assert_bit_equal(labels[f].cpu().numpy(), co.slic(lab_imgs[f], step, 50)[0], f"SLIC labels frame {f}")
    k = gpu_lib.dcmt_slic_center_count(352, 1216, step)
    labels = labels.repeat(256 // n_lab, 1, 1)
    batch = np.stack([synth.sparse_depth(960 + f, 352, 1216, (0.01, 0.05, 0.1)[f % 3], kitti_like=bool(f & 1)) for f in range(256)])
    dev = torch.from_numpy(batch).cuda()
    a, sa = api.interpolate_with_superpixels(labels, dev, "gaussian", 1, n_clusters=k, return_stats=True, lib=gpu_lib)
    b, sb = api.interpolate_with_superpixels(labels, dev, "gaussian", 1, n_clusters=k, path="generic", return_stats=True, lib=gpu_lib)
    assert bool((sa[:, 3] == 1).all()) and bool((sb[:, 3] == 0).all())
    assert torch.equal(a, b) and torch.equal(sa[:, :3], sb[:, :3])
    host_labels = labels.cpu().numpy()
    for f in (0, 129, 255):
        assert_bit_equal(a[f].cpu().numpy(), co.interpolate_with_superpixels(batch[f], host_labels[f], k, literal=False), f"frame {f}")
