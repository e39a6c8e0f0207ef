"""The C-ABI shared library loads on a CPU-only box and exports every symbol include/fdbm_b200.h
declares (no compute calls here).  Product code must fail loudly without the library / a B200."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "fdbm_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fdbm_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_surface():
    names = _declared()
    for must in ("fdbm_stft_compress", "fdbm_decompress_istft", "fdbm_bridge_step", "fdbm_prior_sample",
                 "fdbm_conv_igemm", "fdbm_groupnorm_act", "fdbm_ncsnpp_forward", "fdbm_sampler_run"):
        assert must in names


def test_library_exports_every_declared_symbol():
    from fdbm_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "libfdbm_b200.so has not been built (run __graft_entry__.build())"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/fdbm_b200.h but not exported"
    assert sorted(_lib.EXPORTS) == declared, "fdbm_b200/_lib.py EXPORTS out of sync with the header"
    _lib.load()                                                # argtypes for every symbol resolve
    assert lib.fdbm_version() >= 100


def test_no_silent_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from fdbm_b200 import _lib, SpecsDataModule
    rc = _lib.load().fdbm_check_device()
    assert rc != 0                                             # CUDA / arch error, never "ok"
    with pytest.raises(RuntimeError):
        _lib.check(rc, "fdbm_check_device")
    with pytest.raises(RuntimeError):
        SpecsDataModule(n_fft=512, hop_length=256, window="sqrthann").stft(torch.zeros(1, 4000))


def test_conv_descriptor_size_is_checked_first():
    """fdbm_conv_igemm_ex refuses a descriptor whose struct_bytes is not the library's sizeof(fdbm_conv_desc) before it
    looks at the device, so a stale ctypes layout is an error message here rather than a misread pointer on the GPU."""
    from fdbm_b200 import _lib
    lib = _lib.load()
    d = _lib.ConvDesc()
    d.struct_bytes = ctypes.sizeof(_lib.ConvDesc) - 8
    rc = lib.fdbm_conv_igemm_ex(ctypes.byref(d), None)
    msg = lib.fdbm_last_error().decode()
    assert rc == -1 and "struct_bytes" in msg and "sizeof(fdbm_conv_desc)" in msg, (rc, msg)
    assert lib.fdbm_conv_igemm_ex(None, None) == -1 and "struct_bytes" in lib.fdbm_last_error().decode()
    # the right size gets past that check: without a B200 the device check refuses it; with one, the empty descriptor (no
    # segments) is refused by the launch's own host-side checks, before any launch
    d = _lib.ConvDesc()
    rc = lib.fdbm_conv_igemm_ex(ctypes.byref(d), None)
    msg = lib.fdbm_last_error().decode()
    assert rc != 0 and "struct_bytes" not in msg, (rc, msg)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rethinking-flow-and-diffusion-bridge-models-for-speech-enhancement_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "fdbm_oracle" not in txt and "import oracle" not in txt, f
