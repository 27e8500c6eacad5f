"""CPU-side checks of the drop-in boundary: the library loads and exports exactly what include/*.h declares."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "upretinex_b200.h")


def declared_prototypes():
    """{entry point: (return type, parameter count)} as include/upretinex_b200.h declares them."""
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"UPR_API\s+([\w\s\*]+?)\b(upr_\w+)\s*\(([^)]*)\)", src):
        protos[name] = (" ".join(ret.split()), 0 if params.strip() == "void" else params.count(",") + 1)
    return protos


def declared_symbols():
    return sorted(declared_prototypes())


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from retinex_image_enhancement_b200 import native
    return native.lib()


def test_header_declares_symbols():
    syms = declared_symbols()
    assert "upr_clahe_lab_f32" in syms and len(syms) >= 7


def test_library_exports_every_declared_symbol(lib):
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    assert not missing, f"declared in include/upretinex_b200.h but not exported: {missing}"


def test_every_entry_point_has_a_prototype(lib):
    """Loading the library declares every entry point: the header's return type, and one argtype per parameter.  An entry
    point called without argtypes would get its 64-bit pointers truncated to a C int."""
    restypes = {"int": ctypes.c_int, "size_t": ctypes.c_size_t, "const char*": ctypes.c_char_p}
    wrong = {name: (ret, nparams) for name, (ret, nparams) in declared_prototypes().items()
             if getattr(lib, name).restype is not restypes[ret] or len(getattr(lib, name).argtypes or ()) != nparams}
    assert not wrong, f"declared differently by native._declare than in include/upretinex_b200.h (return type, parameters): {wrong}"


def test_no_torch_types_in_abi():
    src = open(HEADER).read()
    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    assert "torch" not in code.lower() and "at::" not in code and "extern \"C\"" in code


def test_host_only_calls(lib):
    assert b"sm_100a" in lib.upr_version()
    lib.upr_status_string.restype = ctypes.c_char_p
    assert b"UPR_E_SHAPE" in lib.upr_status_string(-2)
    assert lib.upr_clahe_workspace_bytes(1, 1080, 1920, 8, 8) >= 3 * 1080 * 1920
    assert lib.upr_clahe_workspace_bytes(1, 0, 1920, 8, 8) == 0


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "retinex-image-enhancement_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f"{f} imports the oracle"
                assert "upr_oracle" not in text, f"{f} references the oracle"
