"""CPU tests: oracle/lbd.c pinned against the reference's OWN vendored line_descriptor code, compiled unmodified from
the reference tree into oracle/_ref/liblinedesc_ref.so (oracle/ref_build/Makefile; OpenCV primitives supplied by the
cv2-pinned restatements).  What that library returned on the inputs below is stored in tests/golden/refbin_v1.npz
(tests/golden/make_golden_refbin.py), so the comparison runs without the reference tree."""
import ctypes as C
from pathlib import Path

import numpy as np

import plslam_b200 as plf
from oracle import clib
from plslam_b200 import synth

GOLD = Path(__file__).parent / "golden" / "refbin_v1.npz"


def images():
    """KITTI-size scene pair, EuRoC-size scene, first left frame of the KITTI-shape stream."""
    L, R = synth.scene_pair()
    E = synth.scene_pair(w=752, h=480, seed=9)[0]
    S = next(iter(synth.stream(plf.KITTI_CAMERA, 1, world=synth.World(seed=7), seed=42)))[1]
    return [L, R, E, S]


def min_line_length(img):
    return float(np.float32(0.025)) * min(img.shape)


def median_trials():
    """300 landmarks: (descriptors [n, 32], observation directions [n, 3])."""
    rng = np.random.default_rng(5)
    out = []
    for trial in range(300):
        n = int(rng.integers(2, 40))
        if trial % 3 == 0:      # few distinct descriptors: many equal distances and equal medians
            base = rng.integers(0, 256, (3, 32), dtype=np.uint8)
            desc = base[rng.integers(0, 3, n)]
        else:                   # noisy copies of one descriptor
            proto = rng.integers(0, 256, 32, dtype=np.uint8)
            desc = (proto[None, :] ^ np.packbits(rng.random((n, 256)) < 0.08, axis=1)).astype(np.uint8)
        out.append((desc, rng.normal(0, 1, (n, 3))))
    return out


def hamming_rows():
    """200 pairs of 32-byte rows, then pairs of lengths that exercise the byte-LUT tail."""
    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, (200, 32), dtype=np.uint8); b = rng.integers(0, 256, (200, 32), dtype=np.uint8)
    tail = [(rng.integers(0, 256, n, dtype=np.uint8), rng.integers(0, 256, n, dtype=np.uint8)) for n in (1, 7, 16, 17, 31, 33)]
    return a, b, tail


def test_lbd_descriptor_equals_vendored_binary_descriptor():
    """BinaryDescriptor::compute (binary_descriptor_custom.cpp:524-687, :1026-1372) == orc_lbd_compute, bit for bit."""
    g = np.load(GOLD)
    total = 0
    for i, img in enumerate(images()):
        h, w = img.shape
        kl = clib.keylines_from_segments(clib.lsd(img), w, h, min_line_length(img))
        kl["class_id"] = np.arange(len(kl), dtype=np.int32)
        assert len(kl) > 150
        assert kl.tobytes() == g[f"kl{i}"].tobytes()       # the KeyLines the reference descriptors were computed on
        assert np.array_equal(g[f"lbd{i}"], clib.lbd_compute(img, kl))
        total += len(kl)
    assert total > 1500


def test_keyline_stage_equals_vendored_lsd_detector():
    """LSDDetectorC::detect (LSDDetector_custom.cpp:218-324) == orc_keylines_from_segments on EVERY field, `angle`
    included: the reference build resolves atan2(float, float) at :286 to glibc's atan2f, and so does the restatement
    (round 1 narrowed the f64 atan2 instead: 1 ulp off on ~10 % of the lines)."""
    g = np.load(GOLD)
    libm = C.CDLL("libm.so.6")
    libm.atan2f.restype = C.c_float
    libm.atan2f.argtypes = [C.c_float, C.c_float]
    n_diff_f64 = 0
    for i, img in enumerate(images()):
        h, w = img.shape
        ref = g[f"kl{i}"]
        mine = clib.keylines_from_segments(clib.lsd(img), w, h, min_line_length(img))
        assert len(ref) == len(mine) > 150
        for f in ref.dtype.names:
            assert np.array_equal(ref[f].view(np.int32), mine[f].view(np.int32)), f
        dy = ref["endPointY"] - ref["startPointY"]; dx = ref["endPointX"] - ref["startPointX"]
        assert np.array_equal(ref["angle"], np.array([libm.atan2f(float(y), float(x)) for y, x in zip(dy, dx)], np.float32))
        n_diff_f64 += int((ref["angle"] != np.arctan2(dy.astype(np.float64), dx.astype(np.float64)).astype(np.float32)).sum())
    assert n_diff_f64 > 0   # the inputs do exercise the atan2f-vs-narrowed-atan2 distinction


def test_median_descriptor_equals_reference_mappoint():
    """PLSLAM::MapPoint::updateAverageDescDir (src/mapFeatures.cpp:51-93, compiled unmodified) picks the same
    observation as oracle/mapfeatures.py for every landmark, ties included."""
    from oracle import mapfeatures as mf
    g = np.load(GOLD)
    trials = median_trials()
    assert len(trials) == len(g["med_idx"])
    for trial, ((desc, dirs), ri, rd) in enumerate(zip(trials, g["med_idx"], g["med_dir"])):
        oi, od = mf.median_descriptor(desc, dirs)
        assert ri == oi, (trial, len(desc))
        assert np.array_equal(rd, od)      # (under the stand-in's zero-initialised accumulator, see eigen_stub)


def test_hamming_primitive_equals_reference_bitops():
    """oracle/matching.py's distance == cv::line_descriptor::match (src/bitops_custom.hpp:83-96) on 32-byte rows and
    on lengths that exercise its byte-LUT tail."""
    from oracle import matching as om
    g = np.load(GOLD)
    a, b, tail = hamming_rows()
    d = om.hamming_matrix(a, b) if hasattr(om, "hamming_matrix") else None
    for i in range(200):
        ref = int(g["hamming"][i])
        assert ref == int(np.unpackbits(a[i] ^ b[i]).sum())
        if d is not None:
            assert ref == int(d[i, i])
        assert g["forb"][i] == ref          # DBoW2::FORB::distance agrees as well
    assert len(tail) == len(g["hamming_tail"])
    for (x, y), ref in zip(tail, g["hamming_tail"]):
        assert int(ref) == int(np.unpackbits(x ^ y).sum())
