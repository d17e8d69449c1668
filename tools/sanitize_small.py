"""Small fused-path workload for compute-sanitizer (memcheck / racecheck / initcheck): a few shapes incl. border tiles,
a straddling width, uint16 input, a very sparse multi-pass frame, plus SLIC / projection / evaluation."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from depth_completion_mt_b200 import _lib, api, synth  # noqa: E402
from oracle import c_oracle as co  # noqa: E402

lib = _lib.load()
for k, (rows, cols, p) in enumerate(((97, 171, 0.05), (100, 321, 0.004), (64, 96, 0.1), (193, 40, 0.05))):
    s = synth.sparse_depth(k, rows, cols, p)
    out = api.img_completion(torch.from_numpy(s).cuda(), False, "gaussian", lib=lib).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), co.img_completion(s, "gaussian").view(np.uint32)), (rows, cols)
    d16 = synth.sparse_depth_q8(k, rows, cols, p)
    out = api.img_completion(torch.from_numpy(d16).cuda(), False, "none", lib=lib).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), co.img_completion(d16.astype(np.float32) / np.float32(256), "none").view(np.uint32))
# the float32 dictionary path (rank_f32.cu + k_q8_tail<true>), incl. a tile that overhangs the image on both sides
for k, (rows, cols, p) in enumerate(((97, 171, 0.05), (64, 96, 0.1), (193, 40, 0.05))):
    f = synth.sparse_depth_float(40 + k, rows, cols, p)
    for blur in ("none", "gaussian"):
        out = api.img_completion(torch.from_numpy(f).cuda(), False, blur, path="rank", lib=lib).cpu().numpy()
        assert np.array_equal(out.view(np.uint32), co.img_completion(f, blur).view(np.uint32)), (rows, cols, blur)
lab = synth.lab_image(0, 64, 96)
labels = api.generate_superpixels(torch.from_numpy(lab).cuda(), 10, 40, lib=lib)
assert np.array_equal(labels.cpu().numpy(), co.slic(lab, 10, 40)[0])
pts = synth.velodyne_cloud(0, 20000)
proj, nrm = api.lidar_project(torch.from_numpy(pts).cuda(), synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, 64, 200, lib=lib)
assert np.array_equal(proj.cpu().numpy(), co.lidar_project(pts, synth.KITTI_T_VELO_TO_CAM, synth.KITTI_P_RECT_02, 64, 200)[0])
api.evaluate(proj, nrm, "lidar_camera", lib=lib)
torch.cuda.synchronize()
print("SANITIZE_WORKLOAD_OK")
