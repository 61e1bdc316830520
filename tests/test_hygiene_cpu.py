"""CPU: structural rules of the repo that the parity claims rest on."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _files(sub, exts):
    for d, _, fs in os.walk(os.path.join(ROOT, sub)):
        if os.sep + "build" in d or os.sep + "lib" in d or "__pycache__" in d:
            continue
        for f in fs:
            if f.endswith(exts):
                yield os.path.join(d, f)


def test_product_never_touches_the_oracle_or_the_reference_tree():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may use oracle/; nothing shipped may read
    /root/reference."""
    bad = []
    for path in _files("moonshine_b200", (".py", ".cpp", ".cu", ".h", ".cuh")):
        text = open(path, encoding="utf-8", errors="replace").read()
        if re.search(r"^\s*(from|import)\s+oracle\b", text, re.M) or "oracle/" in text or "/root/reference" in text:
            bad.append(os.path.relpath(path, ROOT))
    assert not bad, bad


def test_no_cpu_fallback_in_the_model_path():
    """The loaders must fail without an sm_100a device instead of computing on the host."""
    src = open(os.path.join(ROOT, "moonshine_b200", "csrc", "model.cu")).read()
    assert "requires an sm_100a GPU" in src
    api = open(os.path.join(ROOT, "moonshine_b200", "api.py")).read()
    assert not re.search(r"^\s*(import|from)\s+torch", api, re.M)  # the binding is ctypes over the C ABI, nothing else


def test_environment_switches_are_the_kept_ones():
    """The native code reads only these variables, each by its literal name: SPEC_VERIFY (the tests' A/B switch of draft
    verification), V4_COOP (Nsight Compute cannot replay a launch that is both clustered and cooperative), PROF,
    HOST_PROF, VERBOSE and DEBUG_SYNC (diagnostics that compute nothing differently) and GEMM=simt (every GEMM on the
    exact fp32 SIMT reference).  A variable that selects between two paths does not belong in the product."""
    names = set()
    for path in _files(os.path.join("moonshine_b200", "csrc"), (".cpp", ".cu", ".h", ".cuh")):
        names.update(a.strip() for a in re.findall(r"getenv\(([^)]*)\)", open(path, encoding="utf-8").read()))
    kept = {"SPEC_VERIFY", "V4_COOP", "PROF", "HOST_PROF", "VERBOSE", "DEBUG_SYNC", "GEMM"}
    assert names == {f'"MOONSHINE_B200_{k}"' for k in kept}, sorted(names)


def test_header_symbols_are_all_exported():
    import ctypes
    from moonshine_b200 import api
    lib = api.load_library()
    hdr = open(os.path.join(ROOT, "include", "moonshine_b200.h")).read()
    names = set(re.findall(r"\b(moonshine_[a-z0-9_]+)\s*\(", hdr))
    assert names, "no declarations found"
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing
    assert set(api.EXPORTED_SYMBOLS) <= names | {"moonshine_get_version"}
