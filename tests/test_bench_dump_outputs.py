"""bench.py --dump-outputs: the output of the last timed step as float32 .npy, at most 64 MB, the same seeded sample from run to
run, so that two builds can be compared output for output; and --steps is the number of timed steps."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT, assert_bit_equal

DUMP_LIMIT = 64 * 10**6


def _bench(*args, cwd=ROOT):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *map(str, args)], capture_output=True, text=True, timeout=600,
                          cwd=cwd)


def test_dump_samples_whole_frames_in_order(tmp_path):
    import torch

    import bench

    out = torch.arange(64, dtype=torch.float32)[:, None, None].expand(64, 352, 1216).contiguous()  # every pixel holds its frame index
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "depth", out)
    path = tmp_path / "a" / "depth.npy"
    assert os.path.getsize(path) <= DUMP_LIMIT
    a = np.load(path)
    assert a.dtype == np.float32 and a.shape[1:] == (352, 1216) and 1 <= a.shape[0] < 64
    frames = a[:, 0, 0]
    assert (np.diff(frames) > 0).all() and (a == frames[:, None, None]).all()
    assert_bit_equal(np.load(tmp_path / "b" / "depth.npy"), a, "the same sample on every run")


def test_dump_keeps_a_small_batch_whole_and_samples_a_huge_frame(tmp_path):
    import torch

    import bench

    small = torch.rand(3, 40, 50, dtype=torch.float32)
    bench.dump_outputs(str(tmp_path), "small", small)
    assert_bit_equal(np.load(tmp_path / "small.npy"), small.numpy(), "whole batch")
    huge = torch.arange(1 << 24, dtype=torch.float32).reshape(1, 4096, 4096)  # one 67 MB frame; float32 holds these integers exactly
    bench.dump_outputs(str(tmp_path), "huge", huge)
    assert os.path.getsize(tmp_path / "huge.npy") <= DUMP_LIMIT
    h = np.load(tmp_path / "huge.npy")
    assert h.ndim == 1 and h.size > 1 << 23 and (np.diff(h) > 0).all()


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bad_arguments_are_refused_before_any_work(args, tmp_path):
    r = _bench(*args, cwd=tmp_path)
    assert r.returncode == 2 and "error" in r.stderr
    assert not os.path.exists(tmp_path / "x")


@pytest.mark.gpu
def test_dump_holds_the_last_timed_step_and_steps_count(tmp_path, gpu_lib):
    from depth_completion_mt_b200 import synth
    from oracle import c_oracle as co

    rows, cols, frames = 64, 96, 70  # more frames than the 64 unique ones: replicas included
    lines = {}
    for steps in (1, 3):
        r = _bench("--steps", steps, "--warmup", 1, "--frames", frames, "--rows", rows, "--cols", cols, "--no-e2e", "--no-cpu-baseline",
                   "--dump-outputs", tmp_path / str(steps))
        assert r.returncode == 0, r.stderr[-2000:]
        lines[steps] = json.loads(r.stdout.strip().splitlines()[-1])
        assert lines[steps]["steps"] == steps
    assert lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"] > 0
    got = np.load(tmp_path / "3" / "depth.npy")
    assert got.shape == (frames, rows, cols) and got.dtype == np.float32
    assert_bit_equal(np.load(tmp_path / "1" / "depth.npy"), got, "same arguments but --steps: same outputs")
    for f in range(frames):
        assert_bit_equal(got[f], co.img_completion(synth.sparse_depth(f % 64, rows, cols, 0.05), "gaussian"), f"frame {f}")
