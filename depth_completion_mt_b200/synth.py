"""Synthetic KITTI-shaped inputs for tests and bench.py (SURVEY.md section 8d).

The reference ships no data (its mains hard-code ``../depth_selection/...`` paths,
src/DC_lidar_only/main.cpp:71-72), so every measurement here runs on seeded synthetic frames
with the KITTI geometry the reference is written for: 352 x 1216, uint16 depth / 256
(main.cpp:75-82), about 5 % valid pixels.
"""
from __future__ import annotations

import numpy as np

KITTI_ROWS = 352
KITTI_COLS = 1216
BASE_SEED = 1234


def sparse_depth_q8(frame: int, rows: int = KITTI_ROWS, cols: int = KITTI_COLS, density: float = 0.05,
                    kitti_like: bool = False) -> np.ndarray:
    """uint16 q8 sparse depth (value / 256 = metres, 0 = empty), 2..80 m."""
    rng = np.random.default_rng(BASE_SEED + frame)
    mask = rng.random((rows, cols)) < density
    d16 = rng.integers(512, 20480, (rows, cols), dtype=np.uint16)
    if kitti_like:
        mask[: int(0.35 * rows)] = False
    d16[~mask] = 0
    return d16


def sparse_depth(frame: int, rows: int = KITTI_ROWS, cols: int = KITTI_COLS, density: float = 0.05,
                 kitti_like: bool = False) -> np.ndarray:
    """float32 metres, exactly what ``convertTo(CV_32F, 1/256)`` yields (main.cpp:79)."""
    return sparse_depth_q8(frame, rows, cols, density, kitti_like).astype(np.float32) / np.float32(256.0)


def sparse_depth_float(frame: int, rows: int, cols: int, density: float = 0.05, hi: float = 90.0) -> np.ndarray:
    """Non-q8 float depths (exercise the generic float path, e.g. cv::normalize'd stereo input)."""
    rng = np.random.default_rng(BASE_SEED + 100003 + frame)
    mask = rng.random((rows, cols)) < density
    d = rng.uniform(0.5, hi, (rows, cols)).astype(np.float32)
    d[~mask] = 0
    return d


def superpixel_labels(frame: int, rows: int = KITTI_ROWS, cols: int = KITTI_COLS, step: int = 18,
                      jitter: int = 2) -> tuple[np.ndarray, int]:
    """Grid superpixels with per-pixel boundary jitter (stand-in for SLIC output,
    main_lc.cpp:187-201: step = sqrt(w*h/1200) -> 18).  Returns (labels int32 [row][col], K)."""
    rng = np.random.default_rng(BASE_SEED + 7919 + frame)
    jy = rng.integers(-jitter, jitter + 1, (rows, cols))
    jx = rng.integers(-jitter, jitter + 1, (rows, cols))
    y = np.clip(np.arange(rows)[:, None] + jy, 0, rows - 1)
    x = np.clip(np.arange(cols)[None, :] + jx, 0, cols - 1)
    gw = (cols + step - 1) // step
    gh = (rows + step - 1) // step
    labels = (y // step) * gw + (x // step)
    return labels.astype(np.int32), int(gw * gh)


def _smooth_noise(rng, rows, cols, passes: int = 6) -> np.ndarray:
    a = rng.random((rows, cols))
    for _ in range(passes):  # cheap separable box smoothing, no cv2/scipy dependency
        a = (np.roll(a, 1, 0) + a + np.roll(a, -1, 0)) / 3.0
        a = (np.roll(a, 1, 1) + a + np.roll(a, -1, 1)) / 3.0
    a -= a.min()
    a /= max(a.max(), 1e-12)
    return a


def stereo_pair(frame: int, rows: int = KITTI_ROWS, cols: int = KITTI_COLS, density: float = 0.05):
    """(depth_ig f32, left u8, right u8): smooth 3..80 m surface, textured left image, right image =
    left warped by the true disparity bf/depth (main_sl.cpp:846-861 geometry)."""
    rng = np.random.default_rng(BASE_SEED + 15485863 + frame)
    depth_true = (3.0 + 77.0 * _smooth_noise(rng, rows, cols, 8)).astype(np.float32)
    tex = _smooth_noise(rng, rows, cols, 2)
    left = np.clip(np.rint(255.0 * tex), 0, 255).astype(np.uint8)
    bf = np.float32(0.54) * np.float32(959.791)
    disp = bf / depth_true
    xs = np.arange(cols)[None, :] + disp  # right(y, x) = left(y, x + d)
    x0 = np.clip(np.floor(xs).astype(np.int64), 0, cols - 1)
    x1 = np.clip(x0 + 1, 0, cols - 1)
    w = (xs - np.floor(xs)).astype(np.float32)
    lf = left.astype(np.float32)
    yy = np.arange(rows)[:, None].repeat(cols, 1)
    right = np.clip(np.rint(lf[yy, x0] * (1 - w) + lf[yy, x1] * w), 0, 255).astype(np.uint8)
    # initial guess: a noisy dense depth (what interpolate_with_superpixels would hand over)
    noise = rng.normal(0.0, 0.5, (rows, cols)).astype(np.float32)
    depth_ig = np.clip(depth_true + noise, 0.5, 100.0).astype(np.float32)
    holes = rng.random((rows, cols)) < 0.01  # a few zero pixels: disparity stays 0 there
    depth_ig[holes] = 0.0
    return depth_ig, left, right


# KITTI raw calibration, drive 2011_09_26 (public calib_velo_to_cam.txt / calib_cam_to_cam.txt values): velodyne -> camera 0,
# rectification, projection of camera 2.  Used for synthetic LiDAR clouds only.
KITTI_T_VELO_TO_CAM = np.array([
    [7.533745e-03, -9.999714e-01, -6.166020e-04, -4.069766e-03],
    [1.480249e-02, 7.280733e-04, -9.998902e-01, -7.631618e-02],
    [9.998621e-01, 7.523790e-03, 1.480755e-02, -2.717806e-01],
    [0.0, 0.0, 0.0, 1.0]], np.float32)
KITTI_P_RECT_02 = np.array([
    [7.215377e+02, 0.0, 6.095593e+02, 4.485728e+01],
    [0.0, 7.215377e+02, 1.728540e+02, 2.163791e-01],
    [0.0, 0.0, 1.0, 2.745884e-03]], np.float32)


def velodyne_cloud(frame: int, n_points: int = 120000) -> np.ndarray:
    """Synthetic Velodyne HDL-64 sweep as the (n, 4) float32 payload of a KITTI .bin: 64 elevation rings over the full
    azimuth, ranges from a random piecewise-smooth scene (3 .. 80 m), intensity in [0, 1)."""
    rng = np.random.default_rng(BASE_SEED + 300007 + frame)
    az = rng.uniform(-np.pi, np.pi, n_points)
    el = np.deg2rad(rng.integers(0, 64, n_points) * (26.8 / 63.0) - 24.8)
    rg = 3.0 + 77.0 * np.abs(np.sin(3.0 * az + rng.uniform(0, 6.28))) * rng.uniform(0.3, 1.0, n_points)
    x, y, z = rg * np.cos(el) * np.cos(az), rg * np.cos(el) * np.sin(az), rg * np.sin(el)
    return np.stack([x, y, z, rng.random(n_points)], axis=1).astype(np.float32)


def lab_image(frame: int, rows: int = KITTI_ROWS, cols: int = KITTI_COLS) -> np.ndarray:
    """Synthetic CV_8UC3 Lab image (what cv::cvtColor(COLOR_BGR2Lab) hands to Slic::generate_superpixels): smooth colour
    regions with edges and noise, so that superpixels have something to follow."""
    rng = np.random.default_rng(BASE_SEED + 500009 + frame)
    yy, xx = np.mgrid[0:rows, 0:cols].astype(np.float64)
    img = np.empty((rows, cols, 3), np.float64)
    for c in range(3):
        f = rng.uniform(0.005, 0.03, 4)
        ph = rng.uniform(0, 6.28, 4)
        base = 128 + 60 * np.sin(f[0] * xx + ph[0]) * np.cos(f[1] * yy + ph[1]) + 30 * np.sign(np.sin(f[2] * xx + f[3] * yy + ph[2]))
        img[:, :, c] = base + rng.normal(0, 4, (rows, cols))
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def bgr_image(frame: int, rows: int = KITTI_ROWS, cols: int = KITTI_COLS) -> np.ndarray:
    """Synthetic CV_8UC3 BGR camera frame (what cv::imread hands to cv::cvtColor(COLOR_BGR2Lab), main_lc.cpp:182-184):
    a few smooth colour regions split by straight edges, with a shading gradient and sensor noise."""
    rng = np.random.default_rng(BASE_SEED + 700001 + frame)
    yy, xx = np.mgrid[0:rows, 0:cols].astype(np.float64)
    img = np.zeros((rows, cols, 3), np.float64)
    region = np.zeros((rows, cols), np.int64)
    for bit in range(3):  # three random half-planes: up to 8 regions with straight edges
        t = rng.uniform(0, np.pi)
        region |= ((np.cos(t) * (xx - rng.uniform(0, cols)) + np.sin(t) * (yy - rng.uniform(0, rows))) > 0).astype(np.int64) << bit
    colours = rng.uniform(20, 235, (8, 3))
    img[:] = colours[region]
    shade = 0.75 + 0.25 * np.sin(rng.uniform(0.002, 0.01) * xx + rng.uniform(0, 6.28)) * np.cos(rng.uniform(0.002, 0.01) * yy)
    img = img * shade[:, :, None] + rng.normal(0, 3, (rows, cols, 3))
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)
