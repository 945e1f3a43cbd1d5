"""GPU parity tests for the LBD prelude (blur + Sobel) and the LBD descriptor, through the C ABI."""
from pathlib import Path

import numpy as np
import pytest

from oracle import clib, synth
from test_refbin_pin import GOLD as REF_GOLD
from test_refbin_pin import images as refbin_images

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).parent / "golden" / "lines_v1.npz"


def test_gradients_golden(fe):
    g = np.load(GOLD)
    dx, dy = fe.lbd_gradients(g["left"])
    assert np.array_equal(dx, g["dx"]) and np.array_equal(dy, g["dy"])   # cv2 GaussianBlur+Sobel, bit-exact


@pytest.mark.parametrize("shape", [(2, 2), (3, 70), (17, 64), (16, 65), (375, 1242), (480, 752), (33, 129)])
def test_gradients_shapes_vs_oracle(fe, shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    dx, dy = fe.lbd_gradients(img)
    odx, ody = clib.sobel3_i16(clib.gaussian_blur_u8(img, 5, 1.0))
    assert np.array_equal(dx, odx) and np.array_equal(dy, ody)


def test_gradients_strided_input(fe):
    rng = np.random.default_rng(7)
    big = rng.integers(0, 256, (100, 300), dtype=np.uint8)
    view = big[:, 10:210]                      # non-contiguous rows (stride 300, width 200)
    import ctypes as C
    out = np.empty((100, 200, 2), np.int16)
    st = fe.lib.plf_lbd_gradients(fe._ctx, view.ctypes.data_as(C.POINTER(C.c_uint8)), 200, 100, 300,
                                  out.ctypes.data_as(C.POINTER(C.c_int16)))
    assert st == 0
    odx, ody = clib.sobel3_i16(clib.gaussian_blur_u8(np.ascontiguousarray(view), 5, 1.0))
    assert np.array_equal(out[..., 0], odx) and np.array_equal(out[..., 1], ody)


def test_lbd_golden_bit_exact(fe):
    g = np.load(GOLD)
    desc, fl = fe.lbd(g["left"], g["keylines"], want_float=True)
    assert np.array_equal(desc, g["lbd"])
    assert np.array_equal(fl.view(np.uint32), g["lbd_float"].view(np.uint32))   # float descriptor bit-exact too


def test_lbd_full_size_scene(fe):
    """C1 scene at KITTI size: cv2 LSD segments -> KeyLines -> LBD, CUDA vs C restatement."""
    cv2 = pytest.importorskip("cv2")
    L, R = synth.scene_pair()
    lsd = cv2.createLineSegmentDetector(0, 1.2, 0.6, 2.0, 22.5, 1.0, 0.6, 1024)
    for img in (L, R):
        segs = lsd.detect(img)[0].reshape(-1, 4)
        kl = clib.keylines_from_segments(segs, 1242, 375, 0.025 * 375)
        assert len(kl) > 300
        assert np.array_equal(fe.lbd(img, kl), clib.lbd_compute(img, kl))


def test_lbd_edge_cases(fe):
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (120, 160), dtype=np.uint8)
    # empty list: reference prints a message and returns; we return OK with no output
    assert fe.lbd(img, np.zeros(0, clib.KEYLINE_DTYPE)).shape == (0, 32)
    # lines hugging the border / leaving the image (support region is clamped, :1155-1158), 1-pixel line,
    # flat image (all gradients 0 -> NaN descriptor -> all compares false -> zero bytes)
    segs = np.float32([[0, 0, 159, 119], [0, 0, 0, 119], [159, 0, 159, 119], [5, 5, 5.4, 5.2],
                       [0, 60, 159, 60], [150, 110, 159, 119]])
    kl = clib.keylines_from_segments(segs, 160, 120, 0.0)
    assert np.array_equal(fe.lbd(img, kl), clib.lbd_compute(img, kl))
    flat = np.full((120, 160), 77, np.uint8)
    d = fe.lbd(flat, kl)
    assert np.array_equal(d, clib.lbd_compute(flat, kl)) and (d == 0).all()


def test_lbd_equals_vendored_reference_code(fe):
    """CUDA LBD vs the reference's own BinaryDescriptor::compute (vendored sources compiled unmodified into
    oracle/_ref/liblinedesc_ref.so, see oracle/refbin.py; its descriptors are stored in tests/golden/refbin_v1.npz):
    bit-exact descriptors."""
    g = np.load(REF_GOLD)
    L, R = synth.scene_pair()
    for i, img in enumerate((L, R)):
        kl = clib.keylines_from_segments(clib.lsd(img), 1242, 375, 0.025 * 375)
        kl["class_id"] = np.arange(len(kl), dtype=np.int32)
        assert len(kl) > 300
        assert kl.tobytes() == g[f"kl{i}"].tobytes()       # the KeyLines the reference descriptors were computed on
        assert np.array_equal(fe.lbd(img, kl), g[f"lbd{i}"])


def test_cuda_lines_end_to_end_equal_vendored_reference_code(built):
    """The whole CUDA line path (LSD -> KeyLine stage -> LBD, one call: plf_detect_lines) against the reference's own
    LSDDetectorC::detect + BinaryDescriptor::compute compiled unmodified (oracle/_ref, outputs stored in
    tests/golden/refbin_v1.npz): every KeyLine field - `angle` (glibc atan2f, LSDDetector_custom.cpp:286) included - and
    every descriptor bit, end to end, nothing of the oracle's restatement in between."""
    import plslam_b200 as plf
    g = np.load(REF_GOLD)
    n_ulp = 0
    for i, img in enumerate(refbin_images()):
        h, w = img.shape
        cam = dict(plf.KITTI_CAMERA, width=w, height=h)
        with plf.Frontend(camera=cam, lsd_nfeatures=0) as fe:          # keep every line, detection order
            kl, desc = fe.detect_lines(img)
        ref_kl = g[f"kl{i}"]
        assert len(kl) == len(ref_kl) > 150
        for f in ref_kl.dtype.names:
            assert np.array_equal(kl[f].view(np.int32), ref_kl[f].view(np.int32)), f
        assert np.array_equal(desc, g[f"lbd{i}"])
        dy = ref_kl["endPointY"] - ref_kl["startPointY"]; dx = ref_kl["endPointX"] - ref_kl["startPointX"]
        n_ulp += int((ref_kl["angle"] != np.arctan2(dy.astype(np.float64), dx.astype(np.float64)).astype(np.float32)).sum())
    assert n_ulp > 0      # the lines do include cases where atan2f and the narrowed f64 atan2 differ
