"""CPU: the ctypes prototypes of vppstereo_b200/_lib.py equal the C ABI of include/vppstereo_b200.h (names, order, arity, return and
argument types, the two parameter structs), and a call that does not fit a prototype is refused before it reaches C."""
import ctypes
import os
import re

import pytest

from conftest import ROOT

# the type rule stated above _lib.PROTOTYPES; a C type missing here fails the test, so a new one has to be mapped on purpose
SCALARS = {"int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double, "size_t": ctypes.c_size_t,
           "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32}
POINTEES = {"void", "uint8_t", "uint16_t", "uint32_t", "int32_t", "int64_t", "float", "double", "int"}   # -> c_void_p


def _header():
    """include/vppstereo_b200.h without comments and preprocessor lines"""
    text = open(os.path.join(ROOT, "include", "vppstereo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    return "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))


def _structs(text):
    """{typedef name: [(field, C declaration without the name)]} of every `typedef struct { ... } name;`"""
    out = {}
    for body, name in re.findall(r"typedef\s+struct\s*\{(.*?)\}\s*(\w+)\s*;", text, flags=re.S):
        fields = []
        for decl in filter(None, (d.strip() for d in body.split(";"))):
            base, first = re.fullmatch(r"((?:const\s+)?\w+)\s+(.*)", decl, flags=re.S).groups()
            for d in first.split(","):
                stars, field = re.fullmatch(r"\s*(\**)\s*(\w+)\s*", d).groups()
                fields.append((field, f"{base} {stars}".strip()))
        out[name] = fields
    return out


def _prototypes(text):
    """[(name, return type, [parameter declarations])] of every vppb200_* function, in the header's order"""
    text = re.sub(r"typedef\s+struct\s*\{.*?\}\s*\w+\s*;", " ", text, flags=re.S)
    out = []
    for m in re.finditer(r"([\w\s\*]+?)\b(vppb200_\w+)\s*\(([^)]*)\)\s*;", text):
        ret = " ".join(m.group(1).split())
        params = [" ".join(p.split()) for p in m.group(3).split(",")]
        out.append((m.group(2), ret, [] if params == ["void"] else params))
    return out


def _ctype(decl, structs):
    """ctypes type of one parameter / field / return type under the rule above; fails on a type the rule does not know"""
    decl = re.sub(r"\bconst\b", " ", decl)
    stars = decl.count("*")
    words = decl.replace("*", " ").split()
    assert stars <= 1 and words, f"unexpected C declaration {decl!r}"
    base = words[0]
    if stars == 0:
        assert base in SCALARS, f"C type {base!r} has no ctypes mapping in the rule"
        return SCALARS[base]
    if base in structs:
        return ctypes.POINTER(structs[base])
    assert base in POINTEES, f"pointer to {base!r} has no ctypes mapping in the rule"
    return ctypes.c_void_p


def _param_type(param, structs):
    """ctypes type of one named parameter (`const uint8_t *src`, `int W`)"""
    m = re.fullmatch(r"(.*[\s\*])\w+", param)
    assert m, f"unnamed or unexpected parameter {param!r}"
    return _ctype(m.group(1), structs)


@pytest.fixture(scope="module")
def abi():
    from vppstereo_b200 import _lib
    text = _header()
    return _lib, _structs(text), _prototypes(text)


def test_struct_fields_match_header(abi):
    _lib, structs, _ = abi
    assert set(structs) == {"vppb200_sgm_params", "vppb200_rsgm_taps"}, set(structs)
    for name, cls in (("vppb200_sgm_params", _lib.VppSgmParams), ("vppb200_rsgm_taps", _lib.RsgmTaps)):
        want = [(field, _ctype(decl, {})) for field, decl in structs[name]]
        assert [(f, t) for f, t in cls._fields_] == want, name


def test_prototypes_match_header(abi):
    _lib, _, protos = abi
    structs = {"vppb200_sgm_params": _lib.VppSgmParams, "vppb200_rsgm_taps": _lib.RsgmTaps}
    assert len(protos) >= 44
    assert [p[0] for p in protos] == list(_lib.PROTOTYPES), "PROTOTYPES: names or order differ from the header"
    assert _lib.SYMBOLS == tuple(_lib.PROTOTYPES)
    for name, ret, params in protos:
        restype, argtypes = _lib.PROTOTYPES[name]
        want_ret = ctypes.c_char_p if re.fullmatch(r"const char ?\*", ret) else _ctype(ret, structs)
        assert restype is want_ret, f"{name}: restype {restype} vs header {ret!r}"
        assert len(argtypes) == len(params), f"{name}: {len(argtypes)} argtypes vs {len(params)} parameters in the header"
        for k, (t, p) in enumerate(zip(argtypes, params)):
            assert t is _param_type(p, structs), f"{name}: argument {k} is {t.__name__}, header says {p!r}"


def test_bind_applies_every_prototype():
    from vppstereo_b200 import _lib
    other = _lib.bind(ctypes.CDLL(_lib.LIB_PATH))
    for name, (restype, argtypes) in _lib.PROTOTYPES.items():
        fn = getattr(other, name)
        assert fn.restype is restype and tuple(fn.argtypes) == argtypes, name


def test_call_refuses_wrong_arity():
    from vppstereo_b200 import _lib
    with pytest.raises(TypeError, match="takes 2 arguments"):
        _lib.call("vppb200_set_tuning", _lib.TUNE_SGM_SWEEP, 1, 0)
    with pytest.raises(TypeError, match="takes 2 arguments"):
        _lib.call("vppb200_set_tuning", _lib.TUNE_SGM_SWEEP)


def test_float_for_int_parameter_is_refused():
    from vppstereo_b200 import _lib
    one = ctypes.c_void_p(16)         # never dereferenced: the call is refused before it reaches C
    with pytest.raises(ctypes.ArgumentError):
        _lib.lib().vppb200_census5x5(one, one, 32.0, 8, 1, None)
