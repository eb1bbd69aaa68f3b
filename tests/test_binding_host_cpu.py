"""CPU-side checks of the ctypes binding: the argument and return types of every entry point follow its prototype in
include/aadff.h, and a C type the binding cannot map fails the import instead of falling back to ctypes' default
(which converts every Python int to a 32-bit int and would truncate a 64-bit pointer or size)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT

SCALARS = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "double": ctypes.c_double}
RETURNS = dict(SCALARS, **{"const char*": ctypes.c_char_p})
HANDLES = ("aadff_psfnet_t", "aadff_trainer_t")


@pytest.fixture(scope="module")
def nat():
    import aadff_b200
    return aadff_b200.native


def header_text():
    """include/aadff.h without comments and preprocessor lines."""
    with open(os.path.join(ROOT, "include", "aadff.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))


def header_prototypes():
    """[(return type, name, [parameter declarations])], read statement by statement from the header."""
    text = header_text()
    protos = []
    for stmt in text.split(";"):
        if "(" not in stmt:
            continue
        head, params = stmt.split("(", 1)
        *ret, name = head.replace("*", "* ").split()
        if not name.startswith("aadff_"):
            continue
        params = [p.strip() for p in params.rsplit(")", 1)[0].split(",")]
        protos.append((" ".join(ret).replace("* ", "*").replace(" *", "*").strip(), name,
                       [] if params == ["void"] else params))
    return protos


def test_argtypes_and_restype_follow_every_header_prototype(nat):
    protos = header_prototypes()
    names = sorted(name for _, name, _ in protos)
    assert names == nat.exported_symbols()
    # every function the header declares, found by a plain scan: neither parse may drop a prototype
    assert names == sorted(set(re.findall(r"\b(aadff_\w+)\s*\(", header_text()))) and "aadff_version" in names
    for ret, name, params in protos:
        fn = getattr(nat.lib, name)
        assert fn.restype is RETURNS[ret], (name, ret, fn.restype)
        assert fn.argtypes is not None and len(fn.argtypes) == len(params), (name, fn.argtypes, params)
        for decl, t in zip(params, fn.argtypes):
            words = decl.split()
            if "*" in decl or "[" in decl or words[0] in HANDLES:
                assert t is ctypes.c_void_p, (name, decl, t)
            else:
                assert t is SCALARS[" ".join(words[:-1])], (name, decl, t)


def test_a_type_outside_the_map_is_refused(nat):
    for proto, bad in [("int aadff_x(size_t n);", "size_t"), ("int aadff_x(int a,\n unsigned int b);", "unsigned int"),
                       ("void* aadff_x(int a);", "void*"), ("float* aadff_x(void);", "float*")]:
        with pytest.raises(TypeError, match=re.escape(f"'{bad}'")):
            nat._prototypes(proto)
    # multi-line parameter lists, arrays, handles and comments
    got = nat._prototypes("/* a (comment); */ int64_t aadff_x(aadff_trainer_t t, const int64_t s[5],\n"
                          "                               const float* const* w, double d, void* stream);\n"
                          "const char* aadff_y(void);")
    assert got == {"aadff_x": (ctypes.c_int64, [ctypes.c_void_p] * 3 + [ctypes.c_double, ctypes.c_void_p]),
                   "aadff_y": (ctypes.c_char_p, [])}
