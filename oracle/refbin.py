"""TEST INFRASTRUCTURE.  ctypes access to oracle/_ref/liblinedesc_ref.so: the reference's own vendored
3rdparty/line_descriptor (LSDDetectorC::detect, BinaryDescriptor::compute) and src/mapFeatures.cpp (MapPoint), compiled
UNMODIFIED from the reference source tree (reference_dir()) by
oracle/ref_build/Makefile against a stand-in for the OpenCV API whose primitives on this path are the cv2-pinned
restatements of oracle/*.c.  Used only to pin oracle/lbd.c (KeyLine stage + LBD) against the shipped reference code
(tests/golden/make_golden_refbin.py stores what it returns); available() is False where it is not built."""
import ctypes as C
import json
import os
import subprocess
from pathlib import Path

import numpy as np

from oracle.clib import KEYLINE_DTYPE

_DIR = Path(__file__).resolve().parent
_SO = _DIR / "_ref" / "liblinedesc_ref.so"
_lib = None


def reference_dir():
    """The reference source tree: the PLF_REFERENCE_DIR environment variable if set, else BASELINE.json's
    reference_path.  None where that tree is absent or cannot be read (os.path.isfile is False on a permission error,
    where Path.exists raises)."""
    d = os.environ.get("PLF_REFERENCE_DIR") or json.loads((_DIR.parent / "BASELINE.json").read_text()).get("reference_path")
    if d and os.path.isfile(os.path.join(d, "3rdparty", "line_descriptor", "src", "binary_descriptor_custom.cpp")):
        return Path(d)
    return None


def build():
    """Compiles the vendored sources if the reference tree is given (no-op otherwise)."""
    ref = reference_dir()
    if ref is not None:
        subprocess.run(["make", "-C", str(_DIR / "ref_build"), f"REF={ref}"], check=True, capture_output=True)


def available():
    if not _SO.exists():
        try:
            build()
        except Exception:
            return False
    if not _SO.exists():
        return False
    try:
        lib()
    except OSError:
        return False
    return True


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(str(_SO))
        _lib.ref_keylines.restype = C.c_int
        _lib.ref_lbd.restype = C.c_int
    return _lib


def hamming(a, b):
    """cv::line_descriptor::match(P, Q, codelb) of the vendored bitops_custom.hpp:83-96."""
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    return int(lib().ref_hamming(a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), a.size))


def forb_distance(a, b):
    """DBoW2::FORB::distance (3rdparty/DBoW2/src/DBoW2/FORB.cpp:78-101) on two 32-byte rows."""
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    f = lib().ref_forb_distance
    f.restype = C.c_double
    return float(f(a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p)))


def median_descriptor(desc, dirs):
    """PLSLAM::MapPoint (src/mapFeatures.cpp) fed the observations one by one: (index of the observation whose
    descriptor is med_desc, med_obs_dir under the stand-in's zero-initialised accumulator)."""
    desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
    dirs = np.ascontiguousarray(dirs, np.float64).reshape(-1, 3)
    idx = C.c_int(-1)
    md = np.zeros(3, np.float64)
    r = lib().ref_median_descriptor(desc.ctypes.data_as(C.c_void_p), len(desc), dirs.ctypes.data_as(C.c_void_p), C.byref(idx),
                                    md.ctypes.data_as(C.c_void_p))
    if r != 0:
        raise RuntimeError("ref_median_descriptor failed")
    return idx.value, md


def keylines(img, scale_arg=1, num_octaves=1, refine=0, scale=1.2, sigma_scale=0.6, quant=2.0, ang_th=22.5, log_eps=1.0,
             density_th=0.6, n_bins=1024, min_length=0.0, cap=65536):
    """LSDDetectorC::detect(image, keylines, scale_arg, num_octaves, opts) of the vendored code."""
    img = np.ascontiguousarray(img, np.uint8)
    out = np.zeros(cap, KEYLINE_DTYPE)
    n = lib().ref_keylines(img.ctypes.data_as(C.c_void_p), img.shape[1], img.shape[0], int(scale_arg), int(num_octaves), int(refine),
                           C.c_double(scale), C.c_double(sigma_scale), C.c_double(quant), C.c_double(ang_th), C.c_double(log_eps),
                           C.c_double(density_th), int(n_bins), C.c_double(min_length), out.ctypes.data_as(C.c_void_p), cap)
    if n < 0:
        raise RuntimeError(f"ref_keylines failed ({n})")
    return out[:n].copy()


def lbd(img, kls):
    """BinaryDescriptor::compute(image, keylines, descriptors) of the vendored code: uint8 [n, 32]."""
    img = np.ascontiguousarray(img, np.uint8)
    kl = np.ascontiguousarray(kls, KEYLINE_DTYPE)
    desc = np.zeros((len(kl), 32), np.uint8)
    n = lib().ref_lbd(img.ctypes.data_as(C.c_void_p), img.shape[1], img.shape[0], kl.ctypes.data_as(C.c_void_p), len(kl),
                      desc.ctypes.data_as(C.c_void_p))
    if n != len(kl):
        raise RuntimeError(f"ref_lbd failed ({n})")
    return desc
