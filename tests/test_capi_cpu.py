"""CPU: the C-ABI library loads, exports every symbol include/cmbpo_b200.h declares, the ctypes
prototypes cover all of them, and the product path fails loudly without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "cmbpo_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cmbpo_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported_and_bound():
    import cmbpo_b200
    from cmbpo_b200 import _lib
    names = _declared()
    assert len(names) >= 25
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "missing export %s" % n
        assert n in _lib.SIGNATURES, "no ctypes prototype for %s" % n
    assert sorted(_lib.SIGNATURES) == names
    assert _lib.load().cmbpo_abi_version() == 3


def test_struct_layouts_match_header():
    from cmbpo_b200 import _lib
    assert ctypes.sizeof(_lib.EnvCfg) == 5 * 4
    assert ctypes.sizeof(_lib.RolloutBufs) == 25 * 8
    assert _lib.RolloutCfg.env.offset % 4 == 0 and ctypes.sizeof(_lib.RolloutCfg) == 80


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import cmbpo_b200
    with pytest.raises(cmbpo_b200.CmbpoError):
        cmbpo_b200.Engine(0)
    h = ctypes.c_void_p()
    lib = cmbpo_b200._lib.load()
    assert lib.cmbpo_ctx_create(0, ctypes.byref(h)) != 0
    assert b"no CPU fallback" in lib.cmbpo_last_error()


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "constrained-model-based-policy-optimization_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f
