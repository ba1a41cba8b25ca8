"""CPU tests (no GPU): the C-ABI library builds, loads, exports every symbol include/sslpl.h declares, fails loudly
without a CUDA device (no CPU fallback), and the product never references the oracle."""
import ctypes as C
import os
import re
import subprocess
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "sslpl.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(sslpl_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg.lib()
    syms = _declared_symbols()
    assert len(syms) >= 45
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, f"declared in include/sslpl.h but not exported: {missing}"
    assert lib.sslpl_version() == 1


def test_library_is_sm100a_only():
    so = os.path.join(ROOT, "structure-slam-pointline_b200", "libsslpl_b200.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_struct_layouts(pkg):
    assert pkg.KEYPOINT_DTYPE.itemsize == 28 and pkg.KEYLINE_DTYPE.itemsize == 68          # cv::KeyPoint / KeyLine
    assert C.sizeof(pkg.OrbParams) == 36 and C.sizeof(pkg.FeatVec) == 32


def test_no_cpu_fallback_without_gpu(pkg):
    """Without a CUDA device every create call must fail loudly (SSLPL_ERR_CUDA), never compute on the host."""
    import torch
    if torch.cuda.is_available():                       # (a device node such as /dev/nvidia0 need not exist where a GPU does)
        pytest.skip("a GPU is present")
    assert pkg.device_count() == 0
    with pytest.raises(pkg.SslplError, match="no CUDA device|CUDA"):
        pkg.ORBextractor(1000, 1.2, 8, 20, 7)
    with pytest.raises(pkg.SslplError):
        pkg.Matcher()
    with pytest.raises(pkg.SslplError):
        pkg.LineSegment(40)


def test_product_does_not_touch_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may use oracle/."""
    pk = os.path.join(ROOT, "structure-slam-pointline_b200")
    for dp, _, files in os.walk(pk):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")) or f == "Makefile":
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "liboracle" not in txt and "orc_" not in txt and "from oracle" not in txt and "import oracle" not in txt, f
    so = os.path.join(pk, "libsslpl_b200.so")
    ldd = subprocess.run(["ldd", so], capture_output=True, text=True).stdout
    assert "liboracle" not in ldd


def test_feature_vector_csr_matches_oracle_helper(pkg, oracle):
    rng = np.random.default_rng(0)
    node = rng.integers(0, 50, 400).astype(np.int32)
    a = pkg.feature_vector_csr(node); b = oracle.feature_vector_csr(node)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    ids, off, idx = a
    assert np.all(np.diff(ids) > 0) and off[-1] == 400
    for k in range(len(ids)):
        seg = idx[off[k]:off[k + 1]]
        assert np.all(node[seg] == ids[k]) and np.all(np.diff(seg) > 0)       # ascending feature indices (FeatureVector.cpp:31-45)


def test_orbextractor_adapter_keeps_the_reference_signature():
    """host/ORBextractor.h keeps the reference's class surface (include/ORBextractor.h:45-111) and compiles against the OpenCV
    stand-in of oracle/refshim (no OpenCV C++ in this image; the other adapters are compiled against the reference's real headers below)."""
    H = os.path.join(ROOT, "structure-slam-pointline_b200", "host")
    r = subprocess.run(["/usr/bin/g++", "-std=c++14", "-fsyntax-only", "-w", "-I", os.path.join(ROOT, "oracle", "refshim"), "-I", H,
                        "-I", os.path.join(ROOT, "include"), os.path.join(H, "ORBextractor.cc")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    hdr = open(os.path.join(H, "ORBextractor.h")).read()
    for sig in ["ORBextractor(int nfeatures, float scaleFactor, int nlevels, int iniThFAST, int minThFAST)",
                "void operator()( cv::InputArray image, cv::InputArray mask,", "std::vector<cv::Mat> mvImagePyramid;",
                "GetScaleFactors()", "GetInverseScaleSigmaSquares()"]:
        assert sig in hdr, sig


def test_header_is_plain_c99(tmp_path):
    """include/sslpl.h is the C-ABI boundary: it must compile as C (not only C++), and a C program must link against the library."""
    src = tmp_path / "abi.c"
    src.write_text('#include "sslpl.h"\nint main(void) { return (sslpl_version() > 0 && sslpl_device_count() >= 0) ? 0 : 1; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    exe = tmp_path / "abi"
    lib = os.path.join(ROOT, "structure-slam-pointline_b200")
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L", lib, "-lsslpl_b200",
                        "-Wl,-rpath," + lib], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.stdout, r.stderr)


def test_reference_side_adapters_compile_against_the_reference_headers():
    """host/*.cc are compiled against the reference's REAL headers (include/ORBmatcher.h, LSDmatcher.h, Frame.h, KeyFrame.h,
    ExtractLineSegment.h, MapPoint.h, Thirdparty/DBoW2) read in place from /root/reference, with the functional OpenCV / Eigen
    stand-ins of oracle/refshim (OpenCV C++ is not installed) — the same flags tests/integration/build_ref_link.sh uses to LINK them
    with the reference's own objects (run on the GPU by tests/test_integration_gpu.py).  Skipped where the reference is absent."""
    ref = os.environ.get("SSLPL_REFERENCE_DIR", "/root/reference")
    if not os.path.isdir(os.path.join(ref, "src")):
        import pytest
        pytest.skip("reference tree absent")
    H = os.path.join(ROOT, "structure-slam-pointline_b200", "host")
    flags = ["-std=c++14", "-fsyntax-only", "-w", "-include", os.path.join(H, "ORBextractor.h"), "-I", H, "-I", os.path.join(ROOT, "include"),
             "-I", os.path.join(ROOT, "oracle", "refshim"), "-I", os.path.join(ref, "include"), "-I", ref]
    for f in ("ORBextractor.cc", "matcher_b200.cc", "bow_b200.cc", "ExtractLineSegment_b200.cc"):
        r = subprocess.run(["/usr/bin/g++"] + flags + [os.path.join(H, f)], capture_output=True, text=True)
        assert r.returncode == 0, (f, r.stderr[-3000:])
