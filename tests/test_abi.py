"""The C-ABI library loads on a CPU-only box and exports every symbol the header declares.
No compute calls are made here (there is no GPU in the authoring container)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "ribotricer_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rt_[a-z_0-9]+)\s*\(", text)))


def test_header_declares_the_expected_surface():
    from ribotricer_b200 import _lib

    assert sorted(_lib.EXPORTS) == header_symbols()


def test_library_exports_every_declared_symbol_and_abi_version(built):
    from ribotricer_b200 import _lib

    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in header_symbols():
        assert hasattr(lib, name), name
    assert _lib.load().rt_abi_version() == 4


def test_no_cpu_fallback(built):
    """Without a GPU the product path must fail loudly, not fall back to the oracle."""
    import torch

    from ribotricer_b200 import _lib
    from ribotricer_b200.engine import Engine

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(_lib.RtError):
        Engine(0)
    ctx = ctypes.c_void_p()
    rc = _lib.load().rt_create(0, ctypes.byref(ctx))
    assert rc != 0 and b"no CPU fallback" in _lib.load().rt_last_error(None)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ribotricer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("oracle/", "").lower() or f == "synth.py" and False, \
                    f"{f} mentions the oracle"


def test_len_table_rules():
    from ribotricer_b200 import _lib
    from ribotricer_b200.engine import make_len_table

    t = make_len_table({28: 12, 29: 13}, None)
    assert t[28] == 12 and t[29] == 13 and t[30] == _lib.RT_LEN_UNUSED
    t = make_len_table({28: 12, 31: 13}, [28, 29])
    assert t[28] == 12 and t[29] == _lib.RT_LEN_UNUSED and t[30] == _lib.RT_LEN_FILTERED
    assert t[31] == _lib.RT_LEN_FILTERED   # an offset for a length split_bam never kept is moot
    # inferred offsets can be negative (metagene.py:319-324): they are offsets, not sentinels
    t = make_len_table({28: -1, 29: -2, 30: -5, 31: 0}, None)
    assert [int(t[k]) for k in (28, 29, 30, 31)] == [-1, -2, -5, 0] and t[32] == _lib.RT_LEN_UNUSED
    assert _lib.RT_LEN_UNUSED < -_lib.RT_MAX_OFFSET and _lib.RT_LEN_FILTERED < -_lib.RT_MAX_OFFSET
