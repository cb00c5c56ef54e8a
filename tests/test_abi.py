"""CPU-only checks of the drop-in boundary: the shared library loads, exports exactly the symbols
include/rpst.h declares, the ctypes table mirrors the header, and argument validation works without
touching a GPU."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rpst.h")


def header_prototypes():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"RPST_API\s+([\w\s\*]+?)\s*\b(rpst_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = [a.strip() for a in m.group(3).split(",") if a.strip() and a.strip() != "void"]
        protos[m.group(2)] = (m.group(1).strip(), args)
    return protos


@pytest.fixture(scope="module")
def lib():
    import rpst
    return rpst._lib.lib()


def test_library_exports_every_declared_symbol(lib):
    import rpst
    protos = header_prototypes()
    assert len(protos) >= 11
    out = subprocess.run(["nm", "-D", "--defined-only", rpst._lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\b(rpst_\w+)\b", out))
    assert set(protos) == exported, (set(protos) ^ exported)
    for name in protos:
        assert getattr(lib, name) is not None


def test_ctypes_table_mirrors_header():
    import rpst
    protos = header_prototypes()
    assert set(protos) == set(rpst._lib.SIGNATURES)
    kind = {ctypes.c_void_p: "ptr", ctypes.c_int64: "int64_t", ctypes.c_size_t: "size_t", ctypes.c_float: "float",
            ctypes.c_int: "int", ctypes.c_char_p: "const char*", ctypes.c_double: "double"}
    for name, (ret, args) in protos.items():
        res, argtypes = rpst._lib.SIGNATURES[name]
        assert len(args) == len(argtypes), name
        for decl, ct in zip(args, argtypes):
            k = kind[ct]
            if k == "ptr":
                assert "*" in decl, (name, decl)
            elif k == "const char*":
                assert "char" in decl and "*" in decl, (name, decl)
            else:
                assert re.match(rf"^{re.escape(k)}\s+\w+$", decl), (name, decl, k)


def test_debug_hooks_are_not_in_the_product_library():
    """VERDICT r1: `rpst_debug_*` must not be exported from librpst.so; they live in librpst_debug.so
    (include/rpst_debug.h), which the schedule tests load."""
    import rpst
    out = subprocess.run(["nm", "-D", "--defined-only", rpst._lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "rpst_debug" not in out
    dbg = subprocess.run(["nm", "-D", "--defined-only", rpst._lib.DEBUG_LIB_PATH], capture_output=True, text=True).stdout
    assert set(rpst._lib.DEBUG_SIGNATURES) <= set(re.findall(r"\b(rpst_\w+)\b", dbg))
    assert rpst._lib.debug_lib().rpst_debug_adain_schedule is not None


def test_watchdog_knob_round_trips_without_gpu():
    import rpst
    assert rpst.get_tuning("watchdog_ms") == 4000
    rpst.set_tuning("watchdog_ms", 0)          # opt out (no device here: only the host-side value changes)
    rpst.set_tuning("watchdog_ms", 4000)


def test_version_and_tuning(lib):
    import rpst
    assert rpst.version() == 100
    old = rpst.get_tuning("adain_lag_bytes")
    rpst.set_tuning("adain_lag_bytes", 1 << 20)
    assert rpst.get_tuning("adain_lag_bytes") == 1 << 20
    rpst.set_tuning("adain_lag_bytes", old)
    with pytest.raises(rpst.RpstError):
        rpst.set_tuning("no_such_knob", 1)


API_SRC = os.path.join(ROOT, "rp-style-transfer_b200", "csrc", "api.cu")
INT64_MAX = 2**63 - 1


def header_knobs():
    """{name: (lo, hi, default)} of every ranged knob in the doc block above rpst_set_tuning in include/rpst.h."""
    src = open(HEADER).read()
    block = re.search(r"/\* Tuning knobs(.*?)\*/\s*RPST_API int rpst_set_tuning", src, flags=re.S).group(1)
    num = r"(-?\d+|INT64_MAX)"
    bound = lambda t: INT64_MAX if t == "INT64_MAX" else int(t)  # noqa: E731
    return {m.group(1): (bound(m.group(2)), bound(m.group(3)), int(m.group(4)))
            for m in re.finditer(rf'^ \*\s+"(\w+)"\s+{num}\.\.{num}\s+(-?\d+)\s', block, flags=re.M)}


def table_knobs():
    """Knob names of api.cu's table, in order."""
    table = re.search(r"kKnobs\[\] = \{(.*?)\n\};", open(API_SRC).read(), flags=re.S).group(1)
    rows = re.findall(r'\{"(\w+)", &Knobs::(\w+), ', table)
    assert all(name == field for name, field in rows), rows
    return [name for name, _ in rows]


def test_knob_docs_match_table():
    documented = header_knobs()
    table = table_knobs()
    assert len(table) == len(set(table)) >= 23
    assert set(documented) == set(table), set(documented) ^ set(table)
    block = re.search(r"/\* Tuning knobs(.*?)\*/", open(HEADER).read(), flags=re.S).group(1)
    named = set(re.findall(r'^ \*\s+"(\w+)"', block, flags=re.M))
    assert named == set(table) | {"watchdog_ms", "wct_ns_flagged"}, named ^ (set(table) | {"watchdog_ms", "wct_ns_flagged"})


def test_knob_defaults_in_fresh_process():
    documented = header_knobs()
    code = ("import json, sys; sys.path.insert(0, sys.argv[1]); import rpst; "
            "print(json.dumps({n: rpst.get_tuning(n) for n in sys.argv[2:]}))")
    out = subprocess.run([sys.executable, "-c", code, ROOT, *documented], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    got = json.loads(out.stdout.strip().splitlines()[-1])
    assert got == {name: d for name, (_, _, d) in documented.items()}


def test_knob_ranges_are_enforced(lib):
    """Both ends of each documented range are accepted; one step outside is rejected, names the knob, the range and
    the value, and leaves the knob as it was."""
    documented = header_knobs()
    assert len(documented) >= 23
    for name, (lo, hi, _) in documented.items():
        key = name.encode()
        old = lib.rpst_get_tuning(key)
        try:
            for v in (lo, hi):
                assert lib.rpst_set_tuning(key, v) == 0, lib.rpst_last_error()
                assert lib.rpst_get_tuning(key) == v, name
            for v in (lo - 1, hi + 1):
                if v > INT64_MAX:
                    continue
                assert lib.rpst_set_tuning(key, v) == -1, (name, v)
                err = lib.rpst_last_error()
                assert all(s.encode() in err for s in (name, f"{lo}..{hi}", str(v))), err
                assert lib.rpst_get_tuning(key) == hi, name
        finally:
            assert lib.rpst_set_tuning(key, old) == 0
        assert lib.rpst_get_tuning(key) == old, name


def test_read_only_knob_is_rejected(lib):
    assert lib.rpst_set_tuning(b"wct_ns_flagged", 0) == -1
    assert b"read-only" in lib.rpst_last_error()


def test_argument_validation_without_gpu(lib):
    # invalid arguments are rejected before any CUDA call, so this runs on a GPU-less box
    assert lib.rpst_adain_fwd(None, None, None, None, 1, 1, 16, 16, 1e-5, None, None, 0, None) == -1
    assert b"null" in lib.rpst_last_error()
    assert lib.rpst_adain_fwd(None, None, None, None, -1, 1, 16, 16, 1e-5, None, None, 0, None) == -1
    assert lib.rpst_stats_workspace_bytes(8192, 262144) >= 8192 * 8
    assert lib.rpst_adain_fwd(None, None, None, None, 0, 4, 16, 64, 1e-5, None, None, 0, None) == 0  # empty batch


def test_product_path_has_no_cpu_fallback():
    import torch
    import rpst
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        rpst.adaptive_instance_normalization(torch.zeros(1, 2, 4, 4), torch.zeros(1, 2, 4, 4))
    with pytest.raises(AssertionError):
        rpst.adaptive_instance_normalization(torch.zeros(1, 2, 4, 4), torch.zeros(1, 2, 4, 2))
    pkg = os.path.join(ROOT, "rp-style-transfer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in re.sub(r'""".*?"""', "", text, flags=re.S), f"{f} references the oracle"


def test_library_is_sm_100a_with_tcgen05_and_tma_sass():
    """The shipped library is built for sm_100a only and its SASS carries the Blackwell instructions the design
    claims: tcgen05.mma (UTCHMMA), tcgen05.ld (LDTM), tcgen05.commit (UTCBAR), cp.async.bulk / TMA (UBLKCP),
    tensor-map TMA (UTMALDG: covariance and pointwise-convolution input boxes), fp64 tensor-core MMAs (DMMA:
    Newton-Schulz roots), 256-bit global stores and mbarriers (SYNCS) — B200_PROFILING.md's mnemonics."""
    import shutil
    import rpst
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    elf = subprocess.run([cuobjdump, "-lelf", rpst._lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"\.(sm_\w+)\.cubin", elf))
    assert archs == {"sm_100a"}, archs
    sass = subprocess.run([cuobjdump, "-sass", rpst._lib.LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTCHMMA.2CTA", "LDTM", "STTM", "UTCBAR", "UBLKCP", "UTMALDG.2D", "DMMA", "STG.E.ENL2.256", "SYNCS"):
        assert mnemonic in sass, mnemonic
