"""Host-side mirror of the reference's call surface on top of the C ABI (include/dcmt.h).

Function names, argument meaning and error behaviour follow the reference:

    img_completion(sparse, extr, blur_type)                         src/DC_lidar_only/img_completion.cpp:17
    interpolate_with_superpixels(labels, sparse, blur_type, use_superpixel)
                                                                    src/DC_lidar_camera/img_completion_lc.cpp:34
    calculateMeasuementDerivatives / get_initial_disparity / optimize_IG /
    retrieve_optimized_depth / stereo_refine                        src/DC_stereo_lidar/main_sl.cpp:715-885,1165-1253

Inputs may be ``torch`` CUDA tensors (device entry points, asynchronous on the current stream) or
``numpy`` arrays (``*_host`` entry points: H2D, compute, D2H, synchronous).  A leading batch dimension
is optional everywhere: (rows, cols) or (n, rows, cols).  Outputs are returned (the reference's
``cv::Mat&`` out-parameter).  All compute happens in libdcmt.so on the GPU; nothing here falls back.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import BLUR, PATH, STATS_STRIDE, StereoParams

try:
    import torch
except Exception:  # pragma: no cover - torch is part of the image
    torch = None


def _is_torch(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor)


def _batch3(x, what: str):
    if x.ndim == 2:
        return x[None], True
    if x.ndim == 3:
        return x, False
    raise ValueError(f"{what} must be (rows, cols) or (n, rows, cols), got shape {tuple(x.shape)}")


def _blur_code(blur_type) -> int:
    # img_completion.cpp:172-189: exactly "bilateral" / "gaussian", anything else means no blur
    return BLUR.get(blur_type, 0) if isinstance(blur_type, str) else int(blur_type)


def _stream_ptr(stream) -> int:
    if stream is None:
        return int(torch.cuda.current_stream().cuda_stream)
    return int(getattr(stream, "cuda_stream", stream))


def _prep_torch(x, dtype, what: str):
    if not x.is_cuda:
        raise ValueError(f"{what}: torch tensors must live on a CUDA device (use numpy arrays for host data)")
    if x.dtype != dtype:
        raise TypeError(f"{what} must be {dtype}, got {x.dtype}")
    return x.contiguous()


def _prep_numpy(x, dtype, what: str):
    if not isinstance(x, np.ndarray):
        raise TypeError(f"{what} must be a numpy array or a torch CUDA tensor")
    if x.dtype != dtype:
        raise TypeError(f"{what} must be {np.dtype(dtype)}, got {x.dtype}")
    return np.ascontiguousarray(x)


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _device_list(devices):
    """devices=None -> (NULL, 0); "all" -> (NULL, -1) = every visible device; a sequence of ordinals -> (int[], n)."""
    if devices is None:
        return None, None, 0
    if isinstance(devices, str):
        if devices != "all":
            raise ValueError("devices must be None, 'all' or a sequence of CUDA device ordinals")
        return None, None, -1
    arr = (C.c_int * len(devices))(*[int(d) for d in devices])
    return arr, arr, len(devices)


def img_completion(sparse, extr: bool = False, blur_type="gaussian", *, path: str = "auto", return_stats: bool = False,
                   out=None, stream=None, devices=None, lib: _lib.Library | None = None):
    """img_completion(sparse_r_img, dense_r_img, extr, blur_type) -- img_completion.cpp:17-204.

    ``extr`` is accepted and ignored exactly like the reference (:103 ``int densify = true``).
    ``sparse`` is float32 metres, or uint16 = metres * 256 -- the payload of a KITTI depth PNG, in which case the call
    also stands for the ``convertTo(CV_32F, 1.0 / 256.0)`` of main.cpp:79 in front of it (``dcmt_img_completion_u16``).
    Returns ``dense`` (and an int32 (n, 4) stats array when ``return_stats``).  ``out`` optionally supplies the
    output buffer (same type/shape as ``sparse``, contiguous) so that steady-state callers allocate nothing.
    ``devices`` (host arrays only): "all" or a list of CUDA device ordinals -- the frames of the batch are partitioned
    over those GPUs inside the one call (``dcmt_img_completion_*_host_multi``)."""
    del extr
    lib = lib or _lib.load()
    blur = _blur_code(blur_type)
    if _is_torch(sparse):
        if devices is not None:
            raise ValueError("devices= applies to host (numpy) input; a CUDA tensor already lives on one device")
        u16 = sparse.dtype == torch.uint16
        s = _prep_torch(sparse, torch.uint16 if u16 else torch.float32, "sparse")
        s3, squeeze = _batch3(s, "sparse")
        n, rows, cols = s3.shape
        if out is None:
            out = torch.empty(s3.shape, dtype=torch.float32, device=s.device)
        else:
            if not (_is_torch(out) and out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.numel() == s3.numel()):
                raise ValueError("out must be a contiguous float32 CUDA tensor of the input's size")
            out = out.view(s3.shape)
        stats = torch.zeros((n, STATS_STRIDE), dtype=torch.int32, device=s.device) if return_stats else None
        st_ptr = stats.data_ptr() if return_stats else None
        with torch.cuda.device(s.device):
            if u16:
                lib.check(lib.dcmt_img_completion_u16(s3.data_ptr(), out.data_ptr(), rows, cols, 0, 0, 0, 0, n, blur, PATH[path],
                                                      st_ptr, _stream_ptr(stream)))
            else:
                lib.check(lib.dcmt_img_completion_f32(s3.data_ptr(), out.data_ptr(), rows, cols, 0, 0, n, blur, PATH[path],
                                                      st_ptr, _stream_ptr(stream)))
    else:
        u16 = isinstance(sparse, np.ndarray) and sparse.dtype == np.uint16
        s = _prep_numpy(sparse, np.uint16 if u16 else np.float32, "sparse")
        s3, squeeze = _batch3(s, "sparse")
        n, rows, cols = s3.shape
        if out is None:
            out = np.empty(s3.shape, np.float32)
        else:
            if not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.flags.c_contiguous and out.size == s3.size):
                raise ValueError("out must be a C-contiguous float32 array of the input's size")
            out = out.reshape(s3.shape)
        stats = np.zeros((n, STATS_STRIDE), np.int32) if return_stats else None
        st_ptr = _np_ptr(stats) if return_stats else None
        keep, dev_ptr, n_dev = _device_list(devices)
        if devices is not None and u16:
            lib.check(lib.dcmt_img_completion_u16_host_multi(_np_ptr(s3), _np_ptr(out), rows, cols, 0, 0, 0, 0, n, blur, PATH[path], st_ptr,
                                                             dev_ptr, n_dev))
        elif devices is not None:
            lib.check(lib.dcmt_img_completion_f32_host_multi(_np_ptr(s3), _np_ptr(out), rows, cols, 0, 0, n, blur, PATH[path], st_ptr,
                                                             dev_ptr, n_dev))
        elif u16:
            lib.check(lib.dcmt_img_completion_u16_host(_np_ptr(s3), _np_ptr(out), rows, cols, 0, 0, 0, 0, n, blur, PATH[path], st_ptr))
        else:
            lib.check(lib.dcmt_img_completion_f32_host(_np_ptr(s3), _np_ptr(out), rows, cols, 0, 0, n, blur, PATH[path], st_ptr))
        del keep
    out = out[0] if squeeze else out
    return (out, stats) if return_stats else out


def interpolate_with_superpixels(labels, sparse, blur_type="gaussian", use_superpixel: int = 1, *, n_clusters=None,
                                 path: str = "auto", return_stats: bool = False, out=None, stream=None,
                                 lib: _lib.Library | None = None):
    """interpolate_with_superpixels(slic, sparse, dense, blur_type, use_superpixel) -- img_completion_lc.cpp:34-203.

    ``labels`` stands for ``slic.clusters`` as an int32 [row][col] map (the reference indexes [col][row], :83);
    ``n_clusters`` for ``slic.centers.size()`` (default: max label + 1).  ``blur_type`` is ignored, as in the
    reference (:183-192 blurs unconditionally)."""
    del blur_type
    lib = lib or _lib.load()
    if _is_torch(sparse):
        s = _prep_torch(sparse, torch.float32, "sparse")
        s3, squeeze = _batch3(s, "sparse")
        n, rows, cols = s3.shape
        lab_ptr = None
        if use_superpixel:
            lab = _prep_torch(labels, torch.int32, "labels")
            lab3, _ = _batch3(lab, "labels")
            if lab3.shape != s3.shape:
                raise ValueError("labels and sparse shapes differ")
            if n_clusters is None:
                n_clusters = int(lab3.max().item()) + 1
            lab_ptr = lab3.data_ptr()
        if out is None:
            out = torch.empty_like(s3)
        else:
            if not (_is_torch(out) and out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.numel() == s3.numel()):
                raise ValueError("out must be a contiguous float32 CUDA tensor of the input's size")
            out = out.view(s3.shape)
        stats = torch.zeros((n, STATS_STRIDE), dtype=torch.int32, device=s.device) if return_stats else None
        with torch.cuda.device(s.device):
            lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32(
                s3.data_ptr(), lab_ptr, int(n_clusters or 0), out.data_ptr(), rows, cols, 0, 0, n, int(use_superpixel), PATH[path],
                stats.data_ptr() if return_stats else None, _stream_ptr(stream)))
    else:
        s = _prep_numpy(sparse, np.float32, "sparse")
        s3, squeeze = _batch3(s, "sparse")
        n, rows, cols = s3.shape
        lab_ptr = None
        if use_superpixel:
            lab3, _ = _batch3(_prep_numpy(labels, np.int32, "labels"), "labels")
            if lab3.shape != s3.shape:
                raise ValueError("labels and sparse shapes differ")
            if n_clusters is None:
                n_clusters = int(lab3.max()) + 1
            lab_ptr = _np_ptr(lab3)
        if out is None:
            out = np.empty_like(s3)
        else:
            if not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.flags.c_contiguous and out.size == s3.size):
                raise ValueError("out must be a C-contiguous float32 array of the input's size")
            out = out.reshape(s3.shape)
        stats = np.zeros((n, STATS_STRIDE), np.int32) if return_stats else None
        lib.check(lib.dcmt_interpolate_with_superpixels_ex_f32_host(
            _np_ptr(s3), lab_ptr, int(n_clusters or 0), _np_ptr(out), rows, cols, 0, 0, n, int(use_superpixel), PATH[path],
            _np_ptr(stats) if return_stats else None))
    out = out[0] if squeeze else out
    return (out, stats) if return_stats else out


def stereo_params(official: bool = False, num_iterations: int | None = None, lib: _lib.Library | None = None,
                  **overrides) -> StereoParams:
    """main_sl.cpp literals (baseline .54, focal 959.791, damp 500, clip 255/100, 4 iterations, final blur) or the
    main_sl_OFFICIAL.cpp set (damp 1370, clip 221/80, caller-supplied iterations, no blur)."""
    lib = lib or _lib.load()
    p = StereoParams()
    if official:
        lib.dcmt_stereo_params_official(C.byref(p), int(num_iterations if num_iterations is not None else 4))
    else:
        lib.dcmt_stereo_params_default(C.byref(p))
        if num_iterations is not None:
            p.num_iterations = int(num_iterations)
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown stereo parameter {k!r}")
        setattr(p, k, v)
    return p


def stereo_refine(depth_ig, left_gray, right_gray, params: StereoParams | None = None, *, return_disparity: bool = False,
                  out=None, stream=None, lib: _lib.Library | None = None):
    """main_sl.cpp:1165-1253: gray images + initial dense depth -> refined (and blurred) depth."""
    lib = lib or _lib.load()
    prm = params or stereo_params(lib=lib)
    if _is_torch(depth_ig):
        d3, squeeze = _batch3(_prep_torch(depth_ig, torch.float32, "depth_ig"), "depth_ig")
        l3, _ = _batch3(_prep_torch(left_gray, torch.uint8, "left_gray"), "left_gray")
        r3, _ = _batch3(_prep_torch(right_gray, torch.uint8, "right_gray"), "right_gray")
        if l3.shape != d3.shape or r3.shape != d3.shape:
            raise ValueError("depth_ig, left_gray and right_gray shapes differ")
        n, rows, cols = d3.shape
        out = torch.empty_like(d3) if out is None else out.view(d3.shape)
        disp = torch.empty_like(d3) if return_disparity else None
        with torch.cuda.device(d3.device):
            lib.check(lib.dcmt_stereo_refine_f32(d3.data_ptr(), l3.data_ptr(), r3.data_ptr(), out.data_ptr(),
                                                 disp.data_ptr() if return_disparity else None, rows, cols, n,
                                                 C.byref(prm), _stream_ptr(stream)))
    else:
        d3, squeeze = _batch3(_prep_numpy(depth_ig, np.float32, "depth_ig"), "depth_ig")
        l3, _ = _batch3(_prep_numpy(left_gray, np.uint8, "left_gray"), "left_gray")
        r3, _ = _batch3(_prep_numpy(right_gray, np.uint8, "right_gray"), "right_gray")
        if l3.shape != d3.shape or r3.shape != d3.shape:
            raise ValueError("depth_ig, left_gray and right_gray shapes differ")
        n, rows, cols = d3.shape
        out = np.empty_like(d3) if out is None else out.reshape(d3.shape)
        disp = np.empty_like(d3) if return_disparity else None
        lib.check(lib.dcmt_stereo_refine_f32_host(_np_ptr(d3), _np_ptr(l3), _np_ptr(r3), _np_ptr(out),
                                                  _np_ptr(disp) if return_disparity else None, rows, cols, n, C.byref(prm)))
    if squeeze:
        out = out[0]
        disp = disp[0] if return_disparity else None
    return (out, disp) if return_disparity else out


def _device_planes(lib, fn_name, arrays, n_out, extra, stream, out_like=None):
    """Helper for the per-function stereo entry points (device pointers only in the ABI): numpy inputs are
    staged through torch."""
    first = arrays[0]
    host = not _is_torch(first)
    if host:
        if torch is None or not torch.cuda.is_available():
            raise _lib.DcmtError(_lib.DCMT_E_CUDA, "no CUDA device available; depth_completion_mt_b200 has no CPU fallback")
        tens = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]
    else:
        tens = [a.contiguous() for a in arrays]
    t3 = [_batch3(t, "plane")[0] for t in tens]
    squeeze = tens[0].ndim == 2
    n, rows, cols = t3[0].shape
    outs = [torch.empty_like(t3[0]) for _ in range(n_out)]
    with torch.cuda.device(t3[0].device):
        fn = getattr(lib, fn_name)
        lib.check(fn(*[t.data_ptr() for t in t3], *[o.data_ptr() for o in outs], rows, cols, n, *extra, _stream_ptr(stream)))
    outs = [o[0] if squeeze else o for o in outs]
    if host:
        outs = [o.cpu().numpy() for o in outs]
    return outs


def calculateMeasuementDerivatives(value, *, stream=None, lib: _lib.Library | None = None):
    """calculateMeasuementDerivatives (sic), main_sl.cpp:715-745: value plane -> (dx, dy)."""
    lib = lib or _lib.load()
    dx, dy = _device_planes(lib, "dcmt_measurement_derivatives_f32", [value], 2, (), stream)
    return dx, dy


def get_initial_disparity(depth, baseline: float = 0.54, focal: float = 9.597910e02, *, stream=None,
                          lib: _lib.Library | None = None):
    """get_initial_disparity, main_sl.cpp:846-861."""
    lib = lib or _lib.load()
    return _device_planes(lib, "dcmt_get_initial_disparity_f32", [depth], 1, (baseline, focal), stream)[0]


def retrieve_optimized_depth(disp, baseline: float = 0.54, focal: float = 9.597910e02, depth_clip: float = 100.0, *,
                             stream=None, lib: _lib.Library | None = None):
    """retrieve_optimized_depth, main_sl.cpp:863-885."""
    lib = lib or _lib.load()
    return _device_planes(lib, "dcmt_retrieve_optimized_depth_f32", [disp], 1, (baseline, focal, depth_clip), stream)[0]


def optimize_IG(value_left, value_right, disp, num_iterations: int = 4, damp_factor: float = 500.0,
                err_clip: float = 255.0, *, stream=None, lib: _lib.Library | None = None):
    """optimize_IG, main_sl.cpp:804-843.  Returns the refined disparity (the reference updates it in place)."""
    lib = lib or _lib.load()
    host = not _is_torch(disp)
    if host:
        if torch is None or not torch.cuda.is_available():
            raise _lib.DcmtError(_lib.DCMT_E_CUDA, "no CUDA device available; depth_completion_mt_b200 has no CPU fallback")
        vl, vr, d = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (value_left, value_right, disp))
    else:
        vl, vr, d = value_left.contiguous(), value_right.contiguous(), disp.clone()
    d3, squeeze = _batch3(d, "disp")
    vl3, _ = _batch3(vl, "value_left")
    vr3, _ = _batch3(vr, "value_right")
    n, rows, cols = d3.shape
    with torch.cuda.device(d3.device):
        lib.check(lib.dcmt_optimize_ig_f32(vl3.data_ptr(), vr3.data_ptr(), d3.data_ptr(), rows, cols, n, int(num_iterations),
                                           float(damp_factor), float(err_clip), _stream_ptr(stream)))
    out = d3[0] if squeeze else d3
    return out.cpu().numpy() if host else out


# ---------------------------------------------------------------------------------------------- evaluation (8f #3)
EVAL_VARIANTS = {
    # variant: (mode, tolerance)   mode 0: mask gt > tol, mode 1: mask gt > tol and r > tol
    "lidar_only": (0, 0.0),    # src/DC_lidar_only/main.cpp:16-34       `int tolerance = 0`
    "lidar_camera": (1, 0.0),  # src/DC_lidar_camera/main_lc.cpp:85-116 `int tolerance = 0.1` truncates to 0
    "stereo_lidar": (1, 2.0),  # src/DC_stereo_lidar/main_sl.cpp:1031-1061 `int tolerance = 2`
}


def evaluate(gt, dense, variant: str = "lidar_camera", *, stream=None, lib: _lib.Library | None = None):
    """The masked error sums behind the reference's evaluation functions, one record per frame.

    Returns a numpy structured array with fields count, sum_err, sum_abs, sum_sq (float64) and mean_err, mae, rmse
    (float32).  ``gt`` / ``dense`` are float32 (rows, cols) or (n, rows, cols), numpy (host entry point) or torch CUDA
    tensors (device entry point; the records are read back, which synchronises the stream)."""
    lib = lib or _lib.load()
    mode, tol = EVAL_VARIANTS[variant]
    dt = np.dtype([("count", "f8"), ("sum_err", "f8"), ("sum_abs", "f8"), ("sum_sq", "f8"), ("mean_err", "f4"), ("mae", "f4"),
                   ("rmse", "f4"), ("pad", "i4")])
    if _is_torch(gt):
        g3, _ = _batch3(_prep_torch(gt, torch.float32, "gt"), "gt")
        r3, _ = _batch3(_prep_torch(dense, torch.float32, "dense"), "dense")
        if g3.shape != r3.shape:
            raise ValueError("gt and dense shapes differ")
        n, rows, cols = g3.shape
        res = torch.empty((n, dt.itemsize), dtype=torch.uint8, device=g3.device)
        with torch.cuda.device(g3.device):
            lib.check(lib.dcmt_evaluate_f32(g3.data_ptr(), r3.data_ptr(), rows, cols, 0, 0, n, float(tol), mode, res.data_ptr(),
                                            _stream_ptr(stream)))
        return res.cpu().numpy().view(dt).reshape(n)
    g3, _ = _batch3(_prep_numpy(gt, np.float32, "gt"), "gt")
    r3, _ = _batch3(_prep_numpy(dense, np.float32, "dense"), "dense")
    if g3.shape != r3.shape:
        raise ValueError("gt and dense shapes differ")
    n, rows, cols = g3.shape
    res = np.zeros(n, dt)
    lib.check(lib.dcmt_evaluate_f32_host(_np_ptr(g3), _np_ptr(r3), rows, cols, 0, 0, n, float(tol), mode, _np_ptr(res)))
    return res


def evaluate_performance(GT_img, r_img, variant: str = "lidar_camera", **kw):
    """evaluate_performance(GT_img, r_img, mse[, mae]) of the reference, for ONE frame.

    variant "lidar_only"   (main.cpp:16-34)      -> mse            (= mean of gt - r over gt > 0: a signed mean, sic)
    variant "lidar_camera" (main_lc.cpp:85-116)  -> (mse, mae)     (mse = sqrt(sum d^2 / count), sic)"""
    rec = evaluate(GT_img, r_img, variant, **kw)[0]
    if variant == "lidar_only":
        return float(rec["mean_err"])
    return float(rec["rmse"]), float(rec["mae"])


def evaluate_performances(GT_img, r_img, **kw):
    """evaluate_performances(GT_img, r_img, mae, rmse), main_sl.cpp:1031-1061 (tolerance 2) -> (mae, rmse)."""
    rec = evaluate(GT_img, r_img, "stereo_lidar", **kw)[0]
    return float(rec["mae"]), float(rec["rmse"])


# ---------------------------------------------------------------------------------------------- LiDAR projection (8f #2)
def lidar_project(points, T, P, rows: int, cols: int, norm=(0.0, 80.0), *, return_count: bool = False, stream=None,
                  lib: _lib.Library | None = None):
    """main_sl.cpp:478-523: Velodyne points (n, 4) float32 -> (projected_depths, normalized_depths).

    ``T`` is the 4x4 velodyne-to-camera transform, ``P`` the 3x4 projection matrix (numpy, row-major like the maths;
    the reference holds them as Eigen matrices).  Last point in file order wins a pixel (:515);
    ``normalized = cv::normalize(projected, norm[0], norm[1], NORM_MINMAX)`` (:521)."""
    lib = lib or _lib.load()
    Tm = np.ascontiguousarray(np.asarray(T, np.float32).reshape(4, 4))
    Pm = np.ascontiguousarray(np.asarray(P, np.float32).reshape(3, 4))
    if _is_torch(points):
        pts = _prep_torch(points, torch.float32, "points")
        if pts.ndim != 2 or pts.shape[1] != 4:
            raise ValueError("points must be (n, 4)")
        proj = torch.empty((rows, cols), dtype=torch.float32, device=pts.device)
        nrm = torch.empty_like(proj)
        cnt = torch.zeros(1, dtype=torch.int32, device=pts.device)
        with torch.cuda.device(pts.device):
            lib.check(lib.dcmt_lidar_project_f32(pts.data_ptr() if pts.numel() else None, pts.shape[0], _np_ptr(Tm), _np_ptr(Pm), rows, cols,
                                                 proj.data_ptr(), nrm.data_ptr(), float(norm[0]), float(norm[1]), cnt.data_ptr(),
                                                 _stream_ptr(stream)))
        return (proj, nrm, int(cnt.item())) if return_count else (proj, nrm)
    pts = _prep_numpy(points, np.float32, "points")
    if pts.ndim != 2 or pts.shape[1] != 4:
        raise ValueError("points must be (n, 4)")
    proj = np.empty((rows, cols), np.float32)
    nrm = np.empty_like(proj)
    cnt = np.zeros(1, np.int32)
    lib.check(lib.dcmt_lidar_project_f32_host(_np_ptr(pts) if pts.size else None, pts.shape[0], _np_ptr(Tm), _np_ptr(Pm), rows, cols,
                                              _np_ptr(proj), _np_ptr(nrm), float(norm[0]), float(norm[1]), _np_ptr(cnt)))
    return (proj, nrm, int(cnt[0])) if return_count else (proj, nrm)


def bgr2gray(bgr, *, stream=None, lib: _lib.Library | None = None):
    """cv::cvtColor(img, gray, COLOR_BGR2GRAY) (main_sl.cpp:1167,1171): (rows, cols, 3) or (n, rows, cols, 3) uint8 -> gray uint8."""
    lib = lib or _lib.load()
    is_t = _is_torch(bgr)
    x = _prep_torch(bgr, torch.uint8, "bgr") if is_t else _prep_numpy(bgr, np.uint8, "bgr")
    if x.ndim not in (3, 4) or x.shape[-1] != 3:
        raise ValueError("bgr must be (rows, cols, 3) or (n, rows, cols, 3)")
    squeeze = x.ndim == 3
    x4 = x[None] if squeeze else x
    n, rows, cols = int(x4.shape[0]), int(x4.shape[1]), int(x4.shape[2])
    if is_t:
        out = torch.empty((n, rows, cols), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            lib.check(lib.dcmt_bgr2gray_u8(x4.data_ptr(), out.data_ptr(), rows, cols, 0, 0, n, _stream_ptr(stream)))
    else:
        out = np.empty((n, rows, cols), np.uint8)
        lib.check(lib.dcmt_bgr2gray_u8_host(_np_ptr(x4), _np_ptr(out), rows, cols, 0, 0, n))
    return out[0] if squeeze else out


def bgr2lab(bgr, *, stream=None, lib: _lib.Library | None = None):
    """cv::cvtColor(img, lab, COLOR_BGR2Lab) (main_lc.cpp:182-183, main_sl.cpp:438): (rows, cols, 3) or (n, rows, cols, 3)
    uint8 BGR -> uint8 Lab of the same shape, bit-equal to OpenCV's 8-bit conversion."""
    lib = lib or _lib.load()
    is_t = _is_torch(bgr)
    x = _prep_torch(bgr, torch.uint8, "bgr") if is_t else _prep_numpy(bgr, np.uint8, "bgr")
    if x.ndim not in (3, 4) or x.shape[-1] != 3:
        raise ValueError("bgr must be (rows, cols, 3) or (n, rows, cols, 3)")
    squeeze = x.ndim == 3
    x4 = x[None] if squeeze else x
    n, rows, cols = int(x4.shape[0]), int(x4.shape[1]), int(x4.shape[2])
    if is_t:
        out = torch.empty((n, rows, cols, 3), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            lib.check(lib.dcmt_bgr2lab_u8(x4.data_ptr(), out.data_ptr(), rows, cols, 0, 0, n, _stream_ptr(stream)))
    else:
        out = np.empty((n, rows, cols, 3), np.uint8)
        lib.check(lib.dcmt_bgr2lab_u8_host(_np_ptr(x4), _np_ptr(out), rows, cols, 0, 0, n))
    return out[0] if squeeze else out


def lidar_project_batch(points, counts, T, P, rows: int, cols: int, norm=(0.0, 80.0), *, stream=None, lib: _lib.Library | None = None):
    """main_sl.cpp:478-523 for a batch of clouds in four launches.  ``points``: CUDA tensor (n_clouds, max_points, 4) float32;
    ``counts``: CUDA int32 (n_clouds,) points per cloud, or None (max_points each).  Returns (projected, normalized, n_projected):
    (n_clouds, rows, cols) float32 twice and (n_clouds,) int32."""
    lib = lib or _lib.load()
    Tm = np.ascontiguousarray(np.asarray(T, np.float32).reshape(4, 4))
    Pm = np.ascontiguousarray(np.asarray(P, np.float32).reshape(3, 4))
    pts = _prep_torch(points, torch.float32, "points")
    if pts.ndim != 3 or pts.shape[2] != 4:
        raise ValueError("points must be (n_clouds, max_points, 4)")
    nc, mp = int(pts.shape[0]), int(pts.shape[1])
    cn = _prep_torch(counts, torch.int32, "counts") if counts is not None else None
    proj = torch.empty((nc, rows, cols), dtype=torch.float32, device=pts.device)
    nrm = torch.empty_like(proj)
    cnt = torch.zeros(nc, dtype=torch.int32, device=pts.device)
    with torch.cuda.device(pts.device):
        lib.check(lib.dcmt_lidar_project_batch_f32(pts.data_ptr() if pts.numel() else None, cn.data_ptr() if cn is not None else None, mp, mp, nc,
                                                   _np_ptr(Tm), _np_ptr(Pm), rows, cols, proj.data_ptr(), nrm.data_ptr(), float(norm[0]),
                                                   float(norm[1]), cnt.data_ptr(), _stream_ptr(stream)))
    return proj, nrm, cnt


# ---------------------------------------------------------------------------------------------- SLIC (8f #1)
def generate_superpixels(lab_image, step, nc: int, *, iterations: int = 10, return_centers: bool = False, stream=None,
                         lib: _lib.Library | None = None):
    """Slic::generate_superpixels(lab_image, step, nc), slic.cpp:101-182.

    ``lab_image`` is (rows, cols, 3) or a batch (n, rows, cols, 3) uint8 after COLOR_BGR2Lab; ``step`` is truncated to int
    like the reference's int parameter (main_lc.cpp:197-201 passes a double).  Returns the label map ``Slic::clusters`` as
    int32 [row][col] (-1 = never assigned) and, optionally, ``Slic::centers`` (K, 5) float64 (with a leading batch
    dimension for a batch).  ``K = len(centers)`` is the ``n_clusters`` argument of interpolate_with_superpixels."""
    return _superpixels("dcmt_slic_u8c3", lab_image, "lab_image", step, nc, iterations, return_centers, stream, lib)


def generate_superpixels_bgr(bgr_image, step, nc: int, *, iterations: int = 10, return_centers: bool = False, stream=None,
                             lib: _lib.Library | None = None):
    """cv::cvtColor(img, lab, COLOR_BGR2Lab) followed by Slic::generate_superpixels(lab, step, nc) (main_lc.cpp:182-201,
    main_sl.cpp:438-450) in one call: ``bgr_image`` is the uint8 colour image as read, (rows, cols, 3) or
    (n, rows, cols, 3).  The Lab image stays on the device.  Returns what generate_superpixels returns for
    ``bgr2lab(bgr_image)``."""
    return _superpixels("dcmt_slic_bgr_u8c3", bgr_image, "bgr_image", step, nc, iterations, return_centers, stream, lib)


def _superpixels(entry: str, image, what: str, step, nc, iterations, return_centers, stream, lib):
    """SLIC through the C entry point ``entry`` (device) / ``entry + '_host'`` on a CV_8UC3 image or batch."""
    lib = lib or _lib.load()
    step = int(step)
    is_t = _is_torch(image)
    img = _prep_torch(image, torch.uint8, what) if is_t else _prep_numpy(image, np.uint8, what)
    if img.ndim not in (3, 4) or img.shape[-1] != 3:
        raise ValueError(f"{what} must be (rows, cols, 3) or (n, rows, cols, 3)")
    squeeze = img.ndim == 3
    n = 1 if squeeze else int(img.shape[0])
    rows, cols = int(img.shape[-3]), int(img.shape[-2])
    k = lib.dcmt_slic_center_count(rows, cols, step)
    if is_t:
        labels = torch.empty((n, rows, cols), dtype=torch.int32, device=img.device)
        centers = torch.empty((n, max(k, 1), 5), dtype=torch.float64, device=img.device)
        with torch.cuda.device(img.device):
            lib.check(getattr(lib, entry)(img.data_ptr(), rows, cols, n, step, int(nc), int(iterations), labels.data_ptr(),
                                          centers.data_ptr(), _stream_ptr(stream)))
    else:
        labels = np.empty((n, rows, cols), np.int32)
        centers = np.empty((n, max(k, 1), 5), np.float64)
        lib.check(getattr(lib, entry + "_host")(_np_ptr(img), rows, cols, n, step, int(nc), int(iterations), _np_ptr(labels),
                                                _np_ptr(centers)))
    centers = centers[:, :k]
    if squeeze:
        labels, centers = labels[0], centers[0]
    return (labels, centers) if return_centers else labels


# ---------------------------------------------------------------------------------------------- raw Mat files (8f #4)
_CV_DEPTH = {0: np.uint8, 1: np.int8, 2: np.uint16, 3: np.int16, 4: np.int32, 5: np.float32, 6: np.float64}


def read_M(filename):
    """read_M (src/DC_lidar_only/utils.cpp:15-41): the raw cv::Mat dump `int rows, cols, depth, type, channels, nbytes`
    followed by the payload.  Returns a numpy array (rows, cols[, channels]); feed uint16 / float32 depth planes
    straight to img_completion."""
    with open(filename, "rb") as fh:
        rows, cols, depth, mtype, channels, nbytes = np.frombuffer(fh.read(24), np.int32)
        data = fh.read(int(nbytes))
    dt = _CV_DEPTH[int(mtype) & 7]
    ch = (int(mtype) >> 3) + 1
    a = np.frombuffer(data, dt).reshape((int(rows), int(cols), ch) if ch > 1 else (int(rows), int(cols)))
    return a.copy()


def write_M(filename, mat):
    """write_M (utils.cpp:43-58): the inverse of read_M."""
    a = np.ascontiguousarray(mat)
    depth = {v: k for k, v in _CV_DEPTH.items()}[a.dtype.type]
    ch = a.shape[2] if a.ndim == 3 else 1
    hdr = np.array([a.shape[0], a.shape[1], depth, depth + ((ch - 1) << 3), ch, a.nbytes], np.int32)
    with open(filename, "wb") as fh:
        fh.write(hdr.tobytes())
        fh.write(a.tobytes())


# ---------------------------------------------------------------------------------------------- page-locked host buffers
class HostBuffer:
    """A page-locked host array for the host entry points (``dcmt_host_alloc``): ``.array`` is a numpy view.
    ``write_combined=True`` suits input buffers the host only writes (do not read them back on the host)."""

    def __init__(self, shape, dtype, write_combined: bool = False, lib: _lib.Library | None = None):
        self._lib = lib or _lib.load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = C.c_void_p()
        self._lib.check(self._lib.dcmt_host_alloc(self.nbytes, int(write_combined), C.byref(ptr)))
        self._ptr = ptr
        self.array = np.frombuffer((C.c_char * self.nbytes).from_address(ptr.value), dtype=dtype).reshape(shape)

    def close(self):
        if self._ptr is not None:
            self.array = None
            self._lib.dcmt_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
