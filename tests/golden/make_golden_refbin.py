"""Generates tests/golden/refbin_v1.npz: what the reference's OWN vendored code returns, compiled unmodified into
oracle/_ref/liblinedesc_ref.so (oracle/ref_build/Makefile, oracle/refbin.py), on the inputs tests/test_refbin_pin.py
defines (also used by the reference comparisons of tests/test_lbd_gpu.py):
  kl<i>, lbd<i>      LSDDetectorC::detect KeyLines and BinaryDescriptor::compute descriptors of images()[i]
  med_idx, med_dir   PLSLAM::MapPoint's median observation and mean direction for each of median_trials()
  hamming, forb      cv::line_descriptor::match and DBoW2::FORB::distance on the row pairs of hamming_rows();
  hamming_tail       cv::line_descriptor::match on its odd-length pairs
Needs oracle/_ref built (make -C oracle/ref_build REF=<reference tree>): python tests/golden/make_golden_refbin.py"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "pl-slam_b200"))
sys.path.insert(0, str(ROOT / "tests"))
from oracle import clib, refbin  # noqa: E402
from test_refbin_pin import GOLD, hamming_rows, images, median_trials, min_line_length  # noqa: E402


def main():
    if not refbin.available():
        raise SystemExit("oracle/_ref/liblinedesc_ref.so is not built")
    out = {}
    for i, img in enumerate(images()):
        h, w = img.shape
        kl = refbin.keylines(img, min_length=min_line_length(img))
        mine = clib.keylines_from_segments(clib.lsd(img), w, h, min_line_length(img))
        assert kl.tobytes() == mine.tobytes(), "oracle KeyLines differ from the reference binary"
        assert np.array_equal(kl["class_id"], np.arange(len(kl))), "KeyLines are not numbered in detection order"
        out[f"kl{i}"], out[f"lbd{i}"] = kl, refbin.lbd(img, kl)
    med = [refbin.median_descriptor(desc, dirs) for desc, dirs in median_trials()]
    out["med_idx"] = np.array([m[0] for m in med], np.int32)
    out["med_dir"] = np.stack([m[1] for m in med])
    a, b, tail = hamming_rows()
    out["hamming"] = np.array([refbin.hamming(x, y) for x, y in zip(a, b)], np.int32)
    out["forb"] = np.array([refbin.forb_distance(x, y) for x, y in zip(a, b)], np.float64)
    out["hamming_tail"] = np.array([refbin.hamming(x, y) for x, y in tail], np.int32)
    np.savez_compressed(GOLD, **out)
    print(GOLD.name, GOLD.stat().st_size, "bytes; keylines", [len(out[f"kl{i}"]) for i in range(4)])


if __name__ == "__main__":
    main()
