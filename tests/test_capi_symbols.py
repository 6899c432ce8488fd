"""The C-ABI library loads on a CPU-only host and exports every symbol include/sed_b200.h declares."""
import ctypes
import os
import re

from sed_b200 import capi


def _declared_functions():
    src = open(capi.HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"#ifdef SED_PROFILE.*?#endif", "", src, flags=re.S)  # developer-build entries
    decls = re.findall(r"\b(?:int|long|const char\s*\*)\s+(sed_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", src, flags=re.S)
    out = {}
    for name, args in decls:
        args = args.strip()
        out[name] = 0 if args == "void" else len([a for a in args.split(",") if a.strip()])
    return out


def test_library_is_built():
    assert os.path.isfile(capi.LIB_PATH), "run __graft_entry__.build() first"


def test_every_declared_symbol_is_exported():
    decl = _declared_functions()
    assert len(decl) >= 12
    lib = ctypes.CDLL(capi.LIB_PATH)
    for name in decl:
        assert hasattr(lib, name), "missing export " + name


def test_every_exported_symbol_is_declared():
    """library -> header: the shipped ABI has no undeclared `sed_*` entry point (debug / profiling entries live in
    the -DSED_PROFILE build only) and none of its own code calls getenv."""
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if ln.split()[-1].startswith("sed_")}
    assert exported, "nm found no sed_* exports"
    assert exported == set(_declared_functions()), exported ^ set(_declared_functions())
    csrc = os.path.join(os.path.dirname(capi.LIB_PATH), "csrc")
    for name in os.listdir(csrc):
        if not name.endswith((".cu", ".cuh", ".h")):
            continue
        depth = 0
        for ln in open(os.path.join(csrc, name)):
            t = ln.strip()
            if t.startswith("#if"):
                depth += 1 if (depth or "SED_PROFILE" in t and "ifdef" in t) else 0
            elif t.startswith("#endif") and depth:
                depth -= 1
            elif t.startswith("#else") and depth == 1:
                depth = 0
            assert depth or "getenv(" not in ln, "%s: getenv outside #ifdef SED_PROFILE: %s" % (name, t)


def test_binding_matches_header():
    decl = _declared_functions()
    assert set(decl) == set(capi.SIGNATURES)
    for name, nargs in decl.items():
        assert len(capi.SIGNATURES[name][0]) == nargs, name
    lib = capi.load()
    assert lib.sed_abi_version() == 13
    assert isinstance(lib.sed_last_error_string(), bytes)


def test_null_pointer_is_rejected_without_a_gpu():
    lib = capi.load()
    rc = lib.sed_mha_core(None, 1, 1, 0, 0, None, 0, None)
    assert rc == 4  # SED_ERR_NULL
    assert b"null pointer" in lib.sed_last_error_string()


def test_no_link_time_driver_dependency():
    """libcuda must not be a DT_NEEDED entry: the library has to load for symbol checks on driverless hosts."""
    import subprocess
    out = subprocess.run(["readelf", "-d", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out
