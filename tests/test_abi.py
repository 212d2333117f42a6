"""The C-ABI shared library loads on a CPU-only host and exports exactly the symbols include/rtucker.h and
include/rtucker_debug.h declare, with the ctypes signatures of _lib.PROTOTYPES."""
import ctypes
import glob
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADERS = ("rtucker.h", "rtucker_debug.h")


def header_text(h):
    """One header with its comments stripped."""
    text = open(os.path.join(ROOT, "include", h)).read()
    return re.sub(r"/\*.*?\*/", "", text, flags=re.S)


def declared_symbols(headers=HEADERS):
    """Entry points of the drop-in boundary (rtucker.h) and of the debug / self-test header (rtucker_debug.h)."""
    syms = set()
    for h in headers:
        syms |= set(re.findall(r"\b(rt_[a-z0-9_]+)\s*\(", header_text(h)))
    return sorted(syms)


def declarations():
    """name -> (return type, [parameter declarations]) of every function the two headers declare."""
    decls = {}
    for h in HEADERS:
        text = re.sub(r"^\s*#.*$", "", header_text(h), flags=re.M)
        for ret, name, params in re.findall(r"([^;{}()]*?)\b(rt_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", text):
            params = [" ".join(p.split()) for p in params.split(",")]
            decls[name] = (" ".join(ret.split()), [] if params == ["void"] else params)
    return decls


def test_debug_entry_points_are_not_in_the_public_header():
    public = declared_symbols(("rtucker.h",))
    for s in ("rt_tc_selftest", "rt_mma_probe", "rt_score_v3_set_profile", "rt_score_bce_v3_phases"):
        assert s not in public and s in declared_symbols(("rtucker_debug.h",))


def test_header_declares_the_path():
    syms = declared_symbols()
    for s in ("rt_rank_filtered", "rt_score_bce_fwd_bwd", "rt_query_fwd", "rt_query_bwd", "rt_gram", "rt_apply",
              "rt_small_retract", "rt_small_project", "rt_eigh", "rt_score_rank_fused"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    import rtucker_b200
    if not os.path.isfile(rtucker_b200.LIB_PATH):
        pytest.skip("library not built (run __graft_entry__.build())")
    handle = ctypes.CDLL(rtucker_b200.LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(handle, s)]
    assert not missing, missing
    assert handle.rt_abi_version() == 1


def test_library_exports_only_declared_symbols():
    """Helpers shared between the library's own source files are C++ functions, not exported rt_* symbols."""
    import rtucker_b200
    if not os.path.isfile(rtucker_b200.LIB_PATH):
        pytest.skip("library not built (run __graft_entry__.build())")
    out = subprocess.run(["nm", "-D", "--defined-only", rtucker_b200.LIB_PATH], check=True, capture_output=True,
                         text=True).stdout
    exported = sorted({f[-1] for f in map(str.split, out.splitlines()) if f and f[-1].startswith("rt_")})
    assert exported == declared_symbols(), sorted(set(exported) ^ set(declared_symbols()))


def test_prototypes_cover_the_header():
    from rtucker_b200._lib import PROTOTYPES
    assert sorted(PROTOTYPES) == declared_symbols()


SCALARS = {"int": ctypes.c_int, "int32_t": ctypes.c_int, "int64_t": ctypes.c_int64, "size_t": ctypes.c_size_t,
           "float": ctypes.c_float, "double": ctypes.c_double, "unsigned long long": ctypes.c_ulonglong,
           "uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32}


def test_prototypes_match_the_headers():
    """Argument count, scalar types and pointer-ness of every PROTOTYPES entry agree with its header declaration."""
    from rtucker_b200._lib import PROTOTYPES
    decls = declarations()
    assert sorted(decls) == declared_symbols()
    for name, (ret, params) in decls.items():
        res, args = PROTOTYPES[name]
        want_res = ctypes.c_char_p if ret == "const char*" else SCALARS.get(ret)
        assert want_res is not None, f"{name}: no ctypes mapping for return type {ret!r}"
        assert res is want_res, f"{name}: returns {ret}, PROTOTYPES says {res.__name__}"
        assert len(args) == len(params), f"{name}: {len(params)} parameters, PROTOTYPES lists {len(args)}"
        for i, (p, a) in enumerate(zip(params, args)):
            if "*" in p:
                assert a is ctypes.c_void_p or issubclass(a, ctypes._Pointer), \
                    f"{name} parameter {i} ({p}): pointer, PROTOTYPES says {a.__name__}"
            else:
                ctype = p.rsplit(" ", 1)[0]
                assert ctype in SCALARS, f"{name} parameter {i} ({p}): no ctypes mapping for {ctype!r}"
                assert a is SCALARS[ctype], f"{name} parameter {i} ({p}): PROTOTYPES says {a.__name__}"


def csrc_sources():
    """file name -> text with comments stripped, for every .cu, .cuh and .h under csrc/."""
    sources = {}
    for ext in ("cu", "cuh", "h"):
        for path in sorted(glob.glob(os.path.join(ROOT, "r-tucker_b200", "csrc", "*." + ext))):
            sources[os.path.basename(path)] = re.sub(r"//[^\n]*|/\*.*?\*/", "", open(path).read(), flags=re.S)
    return sources


def test_every_kernel_is_referenced():
    """Every __global__ function in csrc/ is named somewhere besides its own definition: a kernel nothing launches
    still compiles into the library and reads as a live path."""
    text = "\n".join(csrc_sources().values())
    text = re.sub(r"__launch_bounds__\s*\([^()]*\)", "", text)
    definitions = re.findall(r"__global__\s[^;{}()]*?\b(\w+)\s*\(", text)
    unreferenced = sorted(k for k in set(definitions)
                          if len(re.findall(r"\b%s\b" % k, text)) <= definitions.count(k))
    assert not unreferenced, "never referenced: " + " ".join(unreferenced)


def test_exact_score_arithmetic_is_written_once():
    """The element arithmetic that the dense, fused and recheck kernels must share bit for bit (accurate sigmoid,
    clamped BCE logs, guarded BCE gradient, ex2.approx of the softmax) is spelled out only in exact.cuh.  The fp16
    score variant (score_bce_v3.cu) keeps its own approximate ex2."""
    rules = {"log1pf(": r"\blog1pf\(", "fmaxf(.., 1e-12f)": r"\bfmaxf\([^();]*\b1e-12f",
             "expf(-": r"(?<!\w)expf\(\s*-", "ex2.approx": r"ex2\.approx"}
    found = {rule: sorted(f for f, text in csrc_sources().items() if re.search(pattern, text))
             for rule, pattern in rules.items()}
    for rule in ("log1pf(", "fmaxf(.., 1e-12f)", "expf(-"):
        assert found[rule] == ["exact.cuh"], (rule, found[rule])
    assert len([f for f in found["ex2.approx"] if f != "score_bce_v3.cu"]) <= 1, found["ex2.approx"]


def test_no_cpu_fallback():
    """Ops refuse CPU tensors loudly instead of silently computing elsewhere."""
    import torch
    import rtucker_b200
    from rtucker_b200 import ops
    if not os.path.isfile(rtucker_b200.LIB_PATH):
        pytest.skip("library not built")
    with pytest.raises(rtucker_b200.RTuckerError):
        ops.gram(torch.zeros(4, 2), torch.zeros(4, 2))
