"""CPU-side checks of the drop-in boundary: liba3d.so loads and exports every symbol that
include/a3d.h declares, and the ctypes table in ann3depth_b200/_lib.py covers all of them."""
import ctypes
import os
import re

import pytest


def declared_symbols(root):
    text = open(os.path.join(root, "include", "a3d.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(a3d_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(repo_root):
    import __graft_entry__ as g
    g.build()
    lib = ctypes.CDLL(os.path.join(repo_root, "ann3depth_b200", "liba3d.so"))
    names = declared_symbols(repo_root)
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/a3d.h but not exported"


def test_ctypes_table_matches_header(repo_root):
    from ann3depth_b200 import _lib
    names = set(declared_symbols(repo_root))
    table = {n for n in _lib.SIGNATURES if not n.startswith("a3d_debug_")}
    assert names == table, (names - table, table - names)
    lib = _lib.load()
    assert lib.a3d_version() == 201 == _lib.ABI_VERSION


def test_no_device_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    from ann3depth_b200 import _lib, ops
    with pytest.raises(_lib.A3DError):
        ops.Context(0)
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.a3d_create(0, ctypes.byref(h)) != 0
    assert b"no CUDA device" in lib.a3d_last_error() or b"CPU fallback" in lib.a3d_last_error()


def test_product_never_imports_oracle(repo_root):
    pkg = os.path.join(repo_root, "ann3depth_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_conv_desc_layout_matches_header(repo_root, tmp_path):
    """The ctypes mirror of a3d_conv_desc must have the C struct's size and field offsets (the struct grew in ABI 200), and
    the mirrored constants the header's values: a C program compiled against include/a3d.h prints them."""
    import subprocess
    from ann3depth_b200 import _lib
    fields = [n for n, _ in _lib.ConvDesc._fields_]
    src = tmp_path / "layout.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"a3d.h\"\nint main(void) {\n"
                   "  printf(\"%zu\\n\", sizeof(a3d_conv_desc));\n" +
                   "".join(f"  printf(\"%zu\\n\", offsetof(a3d_conv_desc, {f}));\n" for f in fields) +
                   "  printf(\"%d\\n\", A3D_DENSE_WGRAD_ADAM_MAX_M);\n"
                   "  printf(\"%d\\n\", A3D_VERSION);\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(repo_root, "include"), "-o", str(exe), str(src)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.ConvDesc)
    assert out[1:-2] == [getattr(_lib.ConvDesc, f).offset for f in fields]
    assert out[-2] == _lib.DENSE_WGRAD_ADAM_MAX_M
    assert out[-1] == _lib.ABI_VERSION
