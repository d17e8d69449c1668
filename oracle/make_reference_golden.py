"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/reference.npz: the values tests/test_reference_build.py compares with
the reference build, stored so that tests/test_reference_golden.py checks the same cases where the reference build is
absent.

    python -m oracle.make_reference_golden

Every value is computed by the restatement that tests/test_reference_build.py requires to agree with the reference build
on that input (the plain-C restatement, or the cv2 transliteration where that is the one the module compares bit for
bit).  Where the reference build exists (oracle/ref_oracle.py), each value is checked against the reference's own output
before anything is written, with the tolerance the module uses (0 = bit for bit): the file then holds the reference's
outputs.  Large arrays are stored as the sha256 of their bytes; scalars and small arrays as they are.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

from depth_completion_mt_b200 import api, synth
from oracle import c_oracle as co
from oracle import cv2_oracle as cvo
from oracle import ref_oracle as ro

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference.npz")
T, P = synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02
SMALL = 4096  # elements: arrays up to this size are stored whole, larger ones as a digest

# the inputs of tests/test_reference_build.py
LIDAR_CASES = [((352, 1216), 0.05, False), ((352, 1216), 0.05, True), ((352, 1216), 0.01, False), ((97, 211), 0.03, False),
               ((120, 64), 0.002, False), ((31, 17), 0.2, False), ((4, 300), 0.1, False), ((1, 1), 1.0, False), ((5, 1), 0.5, False)]
GUIDED_CASES = [((64, 96), 18), ((50, 70), 12)]
SLIC_CASES = [((352, 1216), 18, 40), ((120, 200), 18, 40), ((64, 90), 10, 20), ((40, 40), 50, 40)]
STEREO_SHAPES = [(352, 1216), (64, 100), (9, 12), (3, 3)]
EVAL_SHAPES = [(37, 53), (352, 1216)]
PROJ_CASES = [(352, 1216, 120000), (375, 1242, 60000), (64, 200, 20000), (48, 160, 30000)]
GPU_LIDAR_CASES = [(0, 0.05, False), (1, 0.05, True), (2, 0.01, False), (3, 0.2, False)]


def digest(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def lidar_input(shape, density, kitti_like):
    return synth.sparse_depth(40, shape[0], shape[1], density, kitti_like=kitti_like)


def special_values_frame():
    t = np.float32(0.1)
    s = np.zeros((40, 48), np.float32)
    s[3, 5], s[10, 10], s[11, 40], s[20, 7], s[30, 30] = -4.0, 99.95, t, np.nextafter(t, np.float32(0)), 100.0
    s[25, 12] = 12.5
    return s


CONSTANT_FRAMES = {"zeros": np.zeros((33, 35), np.float32), "full": np.full((33, 35), 7.25, np.float32)}


def guided_input(shape, step):
    rows, cols = shape
    s = synth.sparse_depth(7, rows, cols, 0.08)
    lab, k = synth.superpixel_labels(7, rows, cols, step=step)
    lab = lab.copy()
    lab[5:9, 10:14] = -1
    return s, lab, k


def stereo_zero_far_input():
    dig, left, right = synth.stereo_pair(8, 40, 64)
    dig = dig.copy()
    dig[:5] = 0.0
    dig[5:8] = 5000.0
    return dig, left, right


def eval_input(shape):
    rng = np.random.default_rng(11)
    gt = np.where(rng.random(shape) < 0.3, rng.uniform(0.5, 80, shape), 0).astype(np.float32)
    dense = (rng.uniform(0.0, 85, shape) * (rng.random(shape) < 0.9)).astype(np.float32)
    return gt, dense


def proj_input(rows, cols, n):
    pts = synth.velodyne_cloud({1216: 0, 1242: 5, 200: 0, 160: 1}[cols], n)
    if cols == 160:  # many points per pixel: last writer in file order wins
        pts = np.concatenate([pts, pts[::-1] * np.float32(1.0001), pts[: n // 2]])
    return pts


def degenerate_clouds():
    behind = synth.velodyne_cloud(3, 2000)
    behind[:, 0] = -np.abs(behind[:, 0]) - 1.0
    return {"empty": np.zeros((0, 4), np.float32), "behind": behind}


def guided_gpu_input():
    rows, cols = 64, 96
    s = synth.sparse_depth(9, rows, cols, 0.08)
    lab, k = synth.superpixel_labels(9, rows, cols, step=12)
    lab = lab.copy()
    lab[3:6, 40:50] = -1
    return s, lab, k


def raw_mat():
    return synth.sparse_depth(4, 37, 53, 0.3)


class Writer:
    def __init__(self, have_ref):
        self.have_ref = have_ref
        self.values = {}

    def put(self, key, value, ref_fn=None, tol=0.0):
        """value as the restatement computes it; where the reference build exists, checked against ref_fn()."""
        value = np.asarray(value)
        if self.have_ref and ref_fn is not None:
            ref = np.asarray(ref_fn())
            assert ref.shape == value.shape and ref.dtype == value.dtype, f"{key}: {ref.shape}/{ref.dtype} vs {value.shape}/{value.dtype}"
            if tol == 0.0:
                assert ref.tobytes() == value.tobytes(), f"{key}: differs from the reference build"
            else:
                assert np.abs(ref.astype(np.float64) - value).max() <= tol, f"{key}: more than {tol} from the reference build"
        assert key not in self.values, key
        self.values[key] = value if value.size <= SMALL or tol else np.array(digest(value))


def main(out=OUT):
    have_ref = ro.available()
    w = Writer(have_ref)
    put = w.put
    for shape, density, kitti in LIDAR_CASES:
        s = lidar_input(shape, density, kitti)
        for bt in ("none", "gaussian"):
            put(f"lidar_{shape[0]}x{shape[1]}_{density}_{int(kitti)}_{bt}", co.img_completion(s, bt), lambda: ro.img_completion(s, bt))
    s = synth.sparse_depth_float(3, 97, 211, 0.05)
    put("float_none", co.img_completion(s, "none"), lambda: ro.img_completion(s, "none"))
    put("float_gaussian", cvo.img_completion(s, "gaussian"), lambda: ro.img_completion(s, "gaussian"))
    s = special_values_frame()
    put("special_none", co.img_completion(s, "none"), lambda: ro.img_completion(s, "none"))
    put("special_gaussian", cvo.img_completion(s, "gaussian"), lambda: ro.img_completion(s, "gaussian"), tol=1e-4)
    for name, frame in CONSTANT_FRAMES.items():
        for bt in ("none", "gaussian"):
            put(f"constant_{name}_{bt}", co.img_completion(frame, bt), lambda: ro.img_completion(frame, bt))
    for shape, step in GUIDED_CASES:
        s, lab, k = guided_input(shape, step)
        for n in (k, k - 3):
            put(f"guided_{shape[0]}x{shape[1]}_n{n}_sp1", co.interpolate_with_superpixels(s, lab, n, literal=True),
                lambda: ro.interpolate_with_superpixels(lab, s, use_superpixel=1, n_clusters=n))
        put(f"guided_{shape[0]}x{shape[1]}_n{k}_sp0", co.interpolate_with_superpixels(s, lab, k, use_superpixel=0),
            lambda: ro.interpolate_with_superpixels(lab, s, use_superpixel=0, n_clusters=k))
    slic_cases = [(f"slic_{r}x{c}_{step}_{nc}", synth.lab_image(2, r, c), step, nc) for (r, c), step, nc in SLIC_CASES]
    slic_cases.append(("slic_flat", np.full((48, 64, 3), 128, np.uint8), 9, 40))
    for key, img, step, nc in slic_cases:
        lab, cen = co.slic(img, step, nc)
        put(key + "_labels", lab, lambda: ro.generate_superpixels(img, step, nc)[0])
        put(key + "_centers", cen, lambda: ro.generate_superpixels(img, step, nc)[1])
    for shape in STEREO_SHAPES:
        dig, left, right = synth.stereo_pair(5, shape[0], shape[1])
        out_, disp = co.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)
        key = f"stereo_{shape[0]}x{shape[1]}"
        put(key + "_disp", disp, lambda: ro.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)[1])
        put(key + "_depth", out_, lambda: ro.stereo_refine(dig, left, right, final_gauss=False))
        if min(shape) >= 5:  # the module compares the transliteration bit for bit here, the C port within 1e-4
            put(key + "_blurred", np.asarray(cvo.stereo_refine(dig, left, right)), lambda: ro.stereo_refine(dig, left, right))
        else:
            put(key + "_blurred", co.stereo_refine(dig, left, right), lambda: ro.stereo_refine(dig, left, right), tol=1e-4)
    dig, left, right = synth.stereo_pair(6, 48, 80)
    lf, rf = left.astype(np.float32), right.astype(np.float32)
    dx, dy = co.measurement_derivatives(rf)
    put("one_by_one_dx", dx, lambda: ro.measurement_derivatives(rf)[0])
    put("one_by_one_dy", dy, lambda: ro.measurement_derivatives(rf)[1])
    d0 = np.asarray(cvo.get_initial_disparity(dig))
    put("one_by_one_d0", d0, lambda: ro.get_initial_disparity(dig))
    d4 = co.stereo_refine(dig, left, right, final_gauss=False, return_disp=True)[1]
    put("one_by_one_d4", d4, lambda: ro.optimize_IG(lf, rf, d0))
    put("one_by_one_depth", np.asarray(cvo.retrieve_optimized_depth(d4)), lambda: ro.retrieve_optimized_depth(d4))
    dig, left, right = stereo_zero_far_input()
    put("stereo_zero_far", co.stereo_refine(dig, left, right, final_gauss=False), lambda: ro.stereo_refine(dig, left, right, final_gauss=False))
    for shape in EVAL_SHAPES:
        gt, dense = eval_input(shape)
        key = f"eval_{shape[0]}x{shape[1]}"
        if shape[0] < 100:
            put(key + "_lidar_only", np.float32(co.evaluate(gt, dense, 0, 0)["mean_err"]), lambda: ro.evaluate(gt, dense, "lidar_only"))
        o = co.evaluate(gt, dense, 0, 1)
        put(key + "_lidar_camera", np.float32([o["rmse"], o["mae"]]), lambda: np.float32(ro.evaluate(gt, dense, "lidar_camera")))
        o = co.evaluate(gt, dense, 2, 1)
        put(key + "_stereo_lidar", np.float32([o["mae"], o["rmse"]]), lambda: np.float32(ro.evaluate(gt, dense, "stereo_lidar")))
    for rows, cols, n in PROJ_CASES:
        pts = proj_input(rows, cols, n)
        cp, cn, cc = co.lidar_project(pts, T, P, rows, cols)
        key = f"proj_{rows}x{cols}_{n}"
        put(key + "_projected", cp, lambda: ro.lidar_project(pts, T, P, rows, cols)[0])
        put(key + "_normalized", cn, lambda: ro.lidar_project(pts, T, P, rows, cols)[1])
        put(key + "_count", np.int64(cc), lambda: np.int64(ro.lidar_project(pts, T, P, rows, cols)[2]))
    for name, pts in degenerate_clouds().items():
        cp, cn, cc = co.lidar_project(pts, T, P, 40, 60)
        put(f"proj_{name}_projected", cp, lambda: ro.lidar_project(pts, T, P, 40, 60)[0])
        put(f"proj_{name}_normalized", cn, lambda: ro.lidar_project(pts, T, P, 40, 60)[1])
        put(f"proj_{name}_count", np.int64(cc), lambda: np.int64(ro.lidar_project(pts, T, P, 40, 60)[2]))
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:  # utils.cpp:39-58: the bytes write_M puts in the file
        api.write_M(os.path.join(tmp, "pkg.bin"), raw_mat())
        ro_path = os.path.join(tmp, "ref.bin")
        put("raw_mat_bytes", np.frombuffer(open(os.path.join(tmp, "pkg.bin"), "rb").read(), np.uint8),
            lambda: (ro.write_M(ro_path, raw_mat()), np.frombuffer(open(ro_path, "rb").read(), np.uint8))[1])
    # the inputs of the GPU tests against the reference build
    for frame, density, kitti in GPU_LIDAR_CASES:
        s = synth.sparse_depth_q8(frame, density=density, kitti_like=kitti).astype(np.float32) / np.float32(256)
        for bt in ("gaussian", "none"):
            put(f"gpu_lidar_{frame}_{bt}", co.img_completion(s, bt), lambda: ro.img_completion(s, bt))
    s, lab, k = guided_gpu_input()
    for sp in (1, 0):
        put(f"gpu_guided_sp{sp}", co.interpolate_with_superpixels(s, lab, k, use_superpixel=sp),
            lambda: ro.interpolate_with_superpixels(lab, s, use_superpixel=sp, n_clusters=k))
    dig, left, right = synth.stereo_pair(4)
    put("gpu_stereo_nogauss", co.stereo_refine(dig, left, right, final_gauss=False), lambda: ro.stereo_refine(dig, left, right, final_gauss=False))
    put("gpu_stereo_blurred", np.asarray(cvo.stereo_refine(dig, left, right)), lambda: ro.stereo_refine(dig, left, right))
    img = synth.lab_image(1)
    lab, cen = co.slic(img, 18, 40)
    put("gpu_slic_labels", lab, lambda: ro.generate_superpixels(img, 18, 40)[0])
    put("gpu_slic_centers", cen, lambda: ro.generate_superpixels(img, 18, 40)[1])
    np.savez_compressed(out, **w.values)
    print("written", out, "(checked against the reference build)" if have_ref else "(reference build not available: unchecked)")


if __name__ == "__main__":
    main()
