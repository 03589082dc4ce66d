"""The C-ABI library loads on a CPU-only box and exports exactly what include/panacea_b200.h declares."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _declared():
    text = (ROOT / "include" / "panacea_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pn_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_entry_points():
    names = _declared()
    assert "pn_gemm" in names and "pn_attention" in names and len(names) >= 20


def test_library_exports_every_declared_symbol():
    from panacea_b200 import _lib, build
    build.build()
    lib = _lib.load()
    names = _declared()
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(names)
    assert lib.pn_abi_version() == 3


def test_struct_layout_matches_header_field_order():
    from panacea_b200 import _lib
    from panacea_b200.ops import SAMPLER_MODES
    text = (ROOT / "include" / "panacea_b200.h").read_text()
    for cname, cls in (("pn_gemm_args", _lib.GemmArgs), ("pn_attn_args", _lib.AttnArgs),
                       ("pn_sampler_args", _lib.SamplerArgs)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), text, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        fields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(","):
                fields.append(re.sub(r"\[.*?\]", "", part.strip().split()[-1].lstrip("*")))
        assert fields == [f[0] for f in cls._fields_], (cname, fields)
    modes = dict(re.findall(r"PN_SAMPLER_([A-Z0-9_]+) = (\d+)", text))
    assert {k.lower(): int(v) for k, v in modes.items()} == SAMPLER_MODES


def test_compute_entry_points_fail_loudly_without_cuda():
    """No CPU fallback: on a box without a GPU a compute call returns an error status (never a result)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("has a GPU")
    from panacea_b200 import _lib
    lib = _lib.load()
    buf = (ctypes.c_float * 64)()
    rc = lib.pn_add_inplace(ctypes.cast(buf, ctypes.c_void_p), ctypes.cast(buf, ctypes.c_void_p), 64, None)
    assert rc != 0 and lib.pn_last_error()
    a = _lib.GemmArgs()
    assert lib.pn_gemm(ctypes.byref(a), None) != 0
