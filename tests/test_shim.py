"""The C++ host shim (pl-slam_b200/cpp/stvo_shim.h: StVO::StereoFrameHandler & co. on top of the C ABI), driven by
vo_demo = the VO part of the reference's frame loop (app/plslam_dataset.cpp:111-163)."""
import os
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
DEMO = ROOT / "pl-slam_b200" / "lib" / "vo_demo"


def write_frames(path, cam, frames):
    with open(path, "wb") as f:
        f.write(struct.pack("<3i", len(frames), cam["width"], cam["height"]))
        f.write(struct.pack("<5d", cam["fx"], cam["fy"], cam["cx"], cam["cy"], cam["b"]))
        for L, R in frames:
            f.write(np.ascontiguousarray(L, np.uint8).tobytes())
            f.write(np.ascontiguousarray(R, np.uint8).tobytes())


def test_shim_builds_and_fails_loudly_without_gpu(built, tmp_path):
    """Run with every device hidden (CUDA_VISIBLE_DEVICES=""), so that the failure path is checked on GPU machines too."""
    assert DEMO.exists()
    cam = dict(width=64, height=48, fx=50.0, fy=50.0, cx=32.0, cy=24.0, b=0.1)
    p = tmp_path / "f.bin"
    write_frames(p, cam, [(np.zeros((48, 64), np.uint8),) * 2])
    r = subprocess.run([str(DEMO), str(p)], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 2 and "no CUDA device" in r.stderr      # std::runtime_error from the handler ctor


@pytest.mark.gpu
def test_shim_loop_matches_python_pipeline(built, tmp_path):
    import plslam_b200 as plf
    from oracle import synth
    cam = dict(plf.KITTI_CAMERA, width=640, height=360, cx=320.0, cy=180.0, fx=500.0, fy=500.0)
    world = synth.World(seed=4, length=50.0, n_quads=160, n_segs=80, half_width=8.0, half_height=3.5)
    frames = [(L, R) for L, R, _ in synth.stream(cam, 5, world=world, seed=11, step=0.15)]
    p = tmp_path / "frames.bin"
    write_frames(p, cam, frames)
    r = subprocess.run([str(DEMO), str(p), "700", "150"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rows = [ln.split() for ln in r.stdout.strip().splitlines()]
    assert len(rows) == 5
    lim = plf.default_limits(); lim.max_batch = 1
    T = np.eye(4)
    with plf.Frontend(camera=cam, limits=lim, orb_nfeatures=700, lsd_nfeatures=150) as fe:
        for k, (L, R) in enumerate(frames):
            g = fe.process_batch(L, R)[0]
            T = T @ g["DT"]
            row = rows[k]
            assert int(row[0]) == k and int(row[1]) == g["status"]
            assert int(row[2]) == g["n_stereo_pt"] and int(row[3]) == g["n_stereo_ls"]
            if k > 0:
                assert int(row[4]) == g["n_inliers_pt"] + g["n_inliers_ls"]
            Tfw = np.array([float(v) for v in row[6:22]]).reshape(4, 4)
            assert np.allclose(Tfw, T, rtol=0, atol=1e-12)
    assert int(rows[0][1]) == 2 and all(int(r_[1]) == 0 for r_ in rows[1:])   # first frame = initialize, then tracked
