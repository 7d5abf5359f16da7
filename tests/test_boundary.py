"""CPU: the C-ABI boundary.  The library loads, exports every symbol include/pnp_ovss_b200.h declares, the ctypes
table covers exactly those symbols, argument validation works without a GPU, and nothing in the product imports
the oracle or falls back to the CPU."""
import ast
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pnp_ovss_b200.h")


def _declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pnp_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    from pnp_ovss_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        g.build()
    return _lib.load()


def test_every_declared_symbol_is_exported_and_bound(lib):
    from pnp_ovss_b200 import _lib
    declared = _declared_symbols()
    assert len(declared) >= 20
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), "library does not export %s" % name
    assert sorted(_lib.SIGNATURES) == declared


def test_abi_version_and_arch(lib):
    assert lib.pnp_abi_version() == 1
    assert lib.pnp_compiled_sm() == 100
    assert lib.pnp_error_string(0) == b"ok"
    assert b"workspace" in lib.pnp_error_string(-2)


def test_argument_validation_without_gpu(lib):
    null = ctypes.c_void_p(0)
    assert lib.pnp_xattn_softmax_fwd(null, null, null, 1, 12, 4, 442, 0.125, null) == -1
    assert lib.pnp_argmax_channels(null, null, 1, 3, 16, null) == -1
    assert lib.pnp_gaussian_blur_workspace_bytes(3, 336, 336, 0.0) == 0
    assert lib.pnp_gaussian_blur_workspace_bytes(3, 336, 336, 16.8) > 3 * 336 * 336 * 4
    assert lib.pnp_lattice_storage_bytes(3, 1, 100) == 0          # only d = 2 and d = 5 exist
    assert lib.pnp_lattice_storage_bytes(5, 2, 100) > 0
    assert lib.pnp_threshold_upsample_workspace_bytes(35, 20, 21) >= 35 * 20 * 441 * 4


def test_ops_refuse_cpu_tensors():
    import torch
    from pnp_ovss_b200 import PnpError, ops
    with pytest.raises(PnpError):
        ops.softmax_fwd(torch.zeros(1, 12, 4, 442))
    with pytest.raises(PnpError):
        ops.argmax_channels(torch.zeros(1, 3, 16))
    with pytest.raises(PnpError):
        ops.gaussian_blur(torch.zeros(1, 8, 8), 1.0)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pnp_ovss_b200")
    for fn in os.listdir(pkg):
        if not fn.endswith(".py"):
            continue
        tree = ast.parse(open(os.path.join(pkg, fn)).read())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            for n in names:
                assert not n.split(".")[0] in ("oracle", "scipy"), "%s imports %s" % (fn, n)
    for fn in os.listdir(os.path.join(pkg, "csrc")):
        if fn.endswith((".cu", ".cuh")):
            assert "oracle" not in open(os.path.join(pkg, "csrc", fn)).read().replace("CPU oracle", "")


def test_library_reads_no_environment():
    """Every choice a kernel launch makes is fixed in the source or derived from its arguments: no environment switch, so
    concurrent calls from several host threads cannot see different configurations."""
    csrc = os.path.join(ROOT, "pnp_ovss_b200", "csrc")
    for fn in os.listdir(csrc):
        if fn.endswith((".cu", ".cuh", ".h", ".cpp")):
            assert "getenv" not in open(os.path.join(csrc, fn)).read(), fn
    header = open(HEADER).read()
    for name in ("PNP_ATT_TCGEN05", "PNP_ATT_VARIANT", "PNP_SPLAT_ATOMIC", "PNP_VALUE_PITCH", "PNP_GRID_MULT", "PNP_BLUR_FUSE",
                 "PNP_UPDATE_CPL", "PNP_UPDATE_OCC3_MIN_NCH"):
        assert name not in header, name


def test_header_cites_reference_lines():
    text = open(HEADER).read()
    for cite in ("MED:267-283", "BITM:415-433", "DRV:810-853", "DRV:638-647", "DRV:1149-1153", "DRV:1030-1074", "DRV:1106-1112"):
        assert cite in text


def test_header_is_plain_c():
    """The boundary is a C ABI: the header must compile as C99 (no C++ types, no torch types)."""
    import subprocess
    import tempfile
    with tempfile.NamedTemporaryFile("w", suffix=".c", delete=False) as f:
        f.write('#include "pnp_ovss_b200.h"\nint main(void) { return pnp_abi_version() == PNP_ABI_VERSION ? 0 : 1; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), f.name],
                       capture_output=True, text=True)
    os.unlink(f.name)
    assert r.returncode == 0 and not r.stderr.strip(), r.stderr


def test_ctypes_lattice_struct_matches_the_header_layout(tmp_path):
    """struct pnp_lattice crosses the boundary by pointer: the ctypes mirror in _lib.py must have the field order, offsets
    and size the C compiler gives the header's struct."""
    import subprocess
    from pnp_ovss_b200 import _lib
    names = [n for n, _ in _lib.Lattice._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pnp_ovss_b200.h"\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(struct pnp_lattice));\n' +
                   "".join('  printf("%s %%zu\\n", offsetof(struct pnp_lattice, %s));\n' % (n, n) for n in names) +
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr          # fails to compile if _lib.py names a field the header lacks
    out = subprocess.run([str(exe)], capture_output=True, text=True).stdout.split("\n")
    assert int(out[0]) == ctypes.sizeof(_lib.Lattice)
    for line, name in zip(out[1:], names):
        field, off = line.split()
        assert field == name and int(off) == getattr(_lib.Lattice, name).offset, line
    # and the header has no field the mirror lacks
    body = re.search(r"struct pnp_lattice\s*\{(.*?)\}\s*pnp_lattice\s*;", open(HEADER).read(), re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    declared = re.findall(r"(\w+)\s*;", body)
    assert declared == names, (declared, names)


def test_ctypes_signatures_match_the_header_prototypes():
    """Every prototype of the header, parsed as C: parameter count and the class of each parameter (pointer / integer /
    float / double / size_t) must agree with the argtypes in _lib.SIGNATURES, and so must the return type."""
    from pnp_ovss_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    protos = re.findall(r"^\s*(?:PNP_API\s+)?([A-Za-z_][\w\s\*]*?)\b(pnp_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.M)
    assert len(protos) == len(_lib.SIGNATURES)

    def c_class(decl):
        decl = decl.strip()
        if "*" in decl or "pnp_stream_t" in decl:
            return "ptr"
        base = re.sub(r"\b\w+$", "", decl).strip() if re.search(r"\w+\s+\w+$", decl) else decl   # drop the parameter name
        base = base.replace("const", "").strip()
        return {"int": "int", "int32_t": "int", "unsigned": "int", "unsigned int": "int", "long long": "i64", "int64_t": "i64",
                "size_t": "size", "float": "float", "double": "double", "void": "void"}[base]

    def py_class(t):
        if t is None:
            return "void"
        if t in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(t, "contents") or issubclass(t, ctypes._Pointer):
            return "ptr"
        return {ctypes.c_int: "int", ctypes.c_uint: "int", ctypes.c_longlong: "i64", ctypes.c_size_t: "size",
                ctypes.c_float: "float", ctypes.c_double: "double"}[t]

    for ret, name, params in protos:
        restype, argtypes = _lib.SIGNATURES[name]
        plist = [] if params.strip() in ("", "void") else [p for p in params.split(",")]
        assert len(plist) == len(argtypes), "%s: header has %d parameters, ctypes %d" % (name, len(plist), len(argtypes))
        for i, (p, t) in enumerate(zip(plist, argtypes)):
            assert c_class(p) == py_class(t), "%s parameter %d: header '%s', ctypes %s" % (name, i, p.strip(), t)
        assert c_class(ret + " x") == py_class(restype), "%s return type" % name
