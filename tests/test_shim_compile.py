"""CPU test (SURVEY §8 a10, VERDICT r1 #5): the reference's own src/keyFrame.cpp - the code that deep-copies a
StVO::StereoFrame (img_l/r, four descriptor blocks, safeCopy() of every feature; :39-53, :63-77) - compiled UNMODIFIED
from the reference source tree (oracle.refbin.reference_dir: PLF_REFERENCE_DIR, else BASELINE.json's reference_path)
against pl-slam_b200/cpp/stvo_shim.h through the forwarding headers INTEGRATION.md describes
(oracle/ref_build/shim_compile: <stereoFrame.h> etc. -> the shim, <eigen3/Eigen/Core> -> the shim's value types,
<opencv/cv.h> -> the OpenCV stand-in), linked with a driver that checks the deep copy.  Skipped where that tree is
absent or cannot be read: its sources cannot be stored in this repository."""
import os
import shutil
import subprocess
from pathlib import Path

import pytest

from oracle.refbin import reference_dir

ROOT = Path(__file__).resolve().parents[1]
REF = reference_dir()
pytestmark = pytest.mark.skipif(REF is None or not os.path.isfile(REF / "src" / "keyFrame.cpp") or shutil.which("g++") is None,
                                reason="needs a readable reference source tree and g++")


def test_reference_keyframe_compiles_and_deep_copies_against_the_shim(tmp_path):
    inc = [ROOT / "oracle", ROOT / "oracle/ref_build/shim_compile", ROOT / "oracle/ref_build/opencv_stub", ROOT / "include",
           ROOT / "pl-slam_b200/cpp", REF / "include", REF / "3rdparty/DBoW2/include", REF / "3rdparty/DBoW2/include/DBoW2"]
    exe = tmp_path / "kftest"
    cmd = ["g++", "-std=c++14", "-O1", "-w"] + [f"-I{p}" for p in inc] + [
        str(REF / "src/keyFrame.cpp"), str(ROOT / "oracle/ref_build/shim_compile/keyframe_test.cpp"),
        str(REF / "3rdparty/DBoW2/src/DBoW2/BowVector.cpp"), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "keyframe-shim ok" in r.stdout, r.stdout + r.stderr
