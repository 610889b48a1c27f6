"""CPU tests of the drop-in boundary: the C-ABI library builds, loads and exports every symbol include/aae_b200.h
declares; the Python binding covers them all; without a GPU every compute entry point fails loudly."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "aae_b200.h")).read()
    return sorted(set(re.findall(r"AAE_API\s+[\w\s\*]+?\b(aae_\w+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    from augmentedautoencoder_b200 import build_ext, _lib
    build_ext.build()
    return _lib.lib()


def test_header_declares_the_expected_surface():
    syms = header_symbols()
    for s in ["aae_encoder_create", "aae_encoder_forward_u8", "aae_codebook_create", "aae_codebook_match", "aae_topk_merge",
              "aae_decoder_forward", "aae_bootstrap_l2_loss", "aae_train_step", "aae_last_error_string"]:
        assert s in syms
    assert len(syms) >= 28


def test_library_exports_every_declared_symbol(lib):
    for s in header_symbols():
        assert hasattr(lib, s), "libaae_b200.so does not export %s" % s


def test_python_binding_covers_every_declared_symbol(lib):
    from augmentedautoencoder_b200 import _lib
    assert sorted(_lib._SIGS) == header_symbols()


def test_no_torch_types_in_the_abi():
    src = open(os.path.join(ROOT, "include", "aae_b200.h")).read()
    assert "torch" not in src and "at::" not in src and "#include <cuda" not in src


def test_version_and_error_string(lib):
    assert lib.aae_version() >= 100
    assert isinstance(lib.aae_last_error_string(), bytes)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_a_gpu(lib):
    from augmentedautoencoder_b200 import _lib
    cfg = _lib.make_cfg(128, 128, 3, [128, 256, 512, 512], [2, 2, 2, 2], 5, 128, 4, 0)
    h = ctypes.c_void_p()
    st = lib.aae_encoder_create(0, ctypes.byref(cfg), ctypes.byref(h))
    assert st != 0 and h.value is None
    assert b"no CUDA device" in lib.aae_last_error_string()
    with pytest.raises(_lib.AaeError):
        _lib.check(st, "create")
    from augmentedautoencoder_b200.ae.session import Session
    with pytest.raises(RuntimeError):
        Session()


def test_invalid_arguments_are_reported_not_crashed(lib):
    from augmentedautoencoder_b200 import _lib
    h = ctypes.c_void_p()
    assert lib.aae_encoder_create(0, None, ctypes.byref(h)) == -1
    cfg = _lib.make_cfg(128, 128, 3, [128], [3], 5, 128, 4, 0)  # stride 3 unsupported
    assert lib.aae_encoder_create(0, ctypes.byref(cfg), ctypes.byref(h)) == -1
    assert b"stride" in lib.aae_last_error_string()
    assert lib.aae_codebook_match(None, None, 1, 1, 0, None, None, None) == -1
    assert lib.aae_encoder_destroy(None) == 0 and lib.aae_codebook_destroy(None) == 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "augmentedautoencoder_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("# oracle", ""), "%s mentions the oracle" % f


def test_library_reads_only_the_documented_environment_variables():
    # DESIGN §7: one test hook and four diagnostics; none of them selects a kernel variant
    csrc = os.path.join(ROOT, "augmentedautoencoder_b200", "csrc")
    names = set()
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh")):
            txt = open(os.path.join(csrc, f)).read()
            found = re.findall(r'getenv\(\s*"(\w+)"\s*\)', txt)
            assert len(found) == txt.count("getenv("), "%s reads an environment variable whose name is not a literal" % f
            names.update(found)
    assert names == {"AAE_TC_NO_TMA_OUT", "AAE_TC_TRACE", "AAE_C1_TRACE", "AAE_MATCH_TRACE", "AAE_TC_VERBOSE"}
