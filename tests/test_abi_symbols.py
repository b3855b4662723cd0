"""CPU tests of the C-ABI library: it builds, loads, exports every symbol include/dsat.h declares,
and fails loudly (no fallback) when there is no GPU."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols(headers=("dsat.h", "dsat_debug.h")):
    found = set()
    for h in headers:
        text = open(os.path.join(ROOT, "include", h)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        found |= set(re.findall(r"\b(dsat_[a-z_0-9]+)\s*\(", text))
    return sorted(found)


def test_product_header_holds_no_debug_hooks():
    product = _declared_symbols(("dsat.h",))
    assert not [s for s in product if "debug" in s or "profile" in s or s.endswith("_test")]
    assert "dsat_hist_reduce" in product and "dsat_sample" in product


def test_library_exports_every_declared_symbol(dsat_lib):
    from diffusionsat_b200 import _lib
    declared = _declared_symbols()
    assert len(declared) >= 20
    raw = ctypes.CDLL(_lib.library_path())
    for name in declared:
        assert hasattr(raw, name), "libdsat.so does not export %s" % name
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared       # the ctypes binding covers the whole header
    assert dsat_lib.dsat_version() >= 1


def test_no_cpu_fallback_without_gpu(dsat_lib):
    """Creating a context without a CUDA device raises; on a machine with GPUs the child process is shown none."""
    import subprocess
    import sys
    code = ("from diffusionsat_b200 import _lib\n"
            "try:\n    _lib.Context(0)\nexcept _lib.DsatError as exc:\n    print(exc)\n")
    proc = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert proc.returncode == 0, proc.stderr[-2000:]
    assert "no CPU fallback" in proc.stdout


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "diffusionsat_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|#include\s+\"[^\"]*oracle", text, flags=re.M), f


def test_ctypes_prototypes_have_the_arity_of_the_header_declarations():
    """Every prototype in include/*.h against the ctypes declaration that binds it: same number of parameters, pointer
    parameters bound as pointers (a drifted binding would pass garbage across the C ABI without any error)."""
    import ctypes as C
    from diffusionsat_b200 import _lib
    text = ""
    for h in ("dsat.h", "dsat_debug.h"):
        text += re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", h)).read(), flags=re.S)
    protos = re.findall(r"\b(dsat_[a-z_0-9]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S)
    assert len(protos) >= 20
    seen = set()
    for name, params in protos:
        params = " ".join(params.split())
        plist = [] if params in ("", "void") else [p.strip() for p in params.split(",")]
        res, argtypes = _lib._SIGNATURES[name]
        assert len(argtypes) == len(plist), "%s: header has %d parameters, ctypes binding %d" % (name, len(plist), len(argtypes))
        for decl, ctype in zip(plist, argtypes):
            is_ptr = "*" in decl
            bound_ptr = ctype in (C.c_void_p, C.c_char_p) or hasattr(ctype, "contents") or issubclass(ctype, C._Pointer)
            assert is_ptr == bound_ptr, "%s: parameter %r bound as %r" % (name, decl, ctype)
        seen.add(name)
    assert seen == set(_lib.EXPORTED_SYMBOLS)
