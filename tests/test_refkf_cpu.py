"""CPU tests of the keyframe-set ABI: every new entry point is declared and exported, and creating a set without a CUDA device
fails with SSLPL_ERR_CUDA (no CPU fallback)."""
import ctypes as C
import os
import re
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["sslpl_kfset_create", "sslpl_kfset_destroy", "sslpl_kfset_store_device", "sslpl_kfset_store", "sslpl_kfset_set_masks",
       "sslpl_kfset_clear", "sslpl_match_ref_kf_batch_device"]


def test_keyframe_set_symbols_are_declared_and_exported(pkg):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "sslpl.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(sslpl_[a-z0-9_]+)\s*\(", hdr))
    assert set(NEW) <= declared
    lib = pkg.lib()
    assert [s for s in NEW if not hasattr(lib, s)] == []


def test_keyframe_set_needs_a_device(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    assert pkg.lib().sslpl_kfset_create(0, 4, 1024, 64, C.byref(h)) == -2          # SSLPL_ERR_CUDA
    assert not h.value
    with pytest.raises(pkg.SslplError, match="no CUDA device"):
        pkg.KeyframeSet(4, 1024, 64)
