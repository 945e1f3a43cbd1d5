"""CPU tests: the C-ABI library loads and exports every symbol include/plslam_b200.h declares,
and fails loudly (no fallback) when no CUDA device is present."""
import os
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def declared_symbols():
    txt = (ROOT / "include" / "plslam_b200.h").read_text()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(plf_[a-z0-9_]+)\s*\(", txt)))


def test_header_symbols_exported(built):
    import plslam_b200 as plf
    lib = plf.load_library()
    syms = declared_symbols()
    assert len(syms) >= 8
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, f"declared in header but not exported: {missing}"
    assert lib.plf_abi_version() == 1


def test_struct_sizes_match(built):
    """ctypes mirrors of the POD structs have the same size as the C side assumes (defaults round-trip)."""
    import plslam_b200 as plf
    p = plf.default_params()
    assert p.orb_nlevels == 4 and abs(p.min_ratio_12_p - 0.9) < 1e-6 and p.lsd_n_bins == 1024
    assert p.homog_th == 1e-7 and p.max_iters_ref == 10
    l = plf.default_limits()
    assert l.max_batch > 0 and l.max_keypoints >= 2000


def test_no_cpu_fallback(built):
    """Without a GPU plf_create must fail with PLF_ERR_NO_DEVICE, not silently compute on the CPU.  Checked in a child
    process that sees no device (CUDA_VISIBLE_DEVICES=""), so that it runs on GPU machines as well."""
    code = ("import sys\n"
            "sys.path[:0] = sys.argv[1:]\n"
            "import plslam_b200 as plf\n"
            "try:\n"
            "    plf.Frontend(device=0)\n"
            "except plf.PlfError as e:\n"
            "    print(e)\n"
            "else:\n"
            "    sys.exit('a Frontend was created without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code, str(ROOT), str(ROOT / "pl-slam_b200")], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CUDA device" in r.stdout
