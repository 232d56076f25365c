"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol the header declares, the binding
layout matches, catalog accessors answer, and compute entry points fail loudly without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

import gpud_b200 as g
from gpud_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported():
    hdr = open(os.path.join(ROOT, "include", "gpud_b200.h")).read()
    declared = set(re.findall(r"\b(gpud_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(capi.SYMBOLS), declared ^ set(capi.SYMBOLS)
    L = g.lib()
    for s in declared:
        assert hasattr(L, s), s


def test_every_exported_symbol_is_declared():
    """the reverse: nothing is exported that a header does not declare - the integrator's header, or the test hooks' own header"""
    import subprocess
    decl = set()
    for h in ("gpud_b200.h", "gpud_b200_hooks.h"):
        decl |= set(re.findall(r"\b(gpudh?_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", h)).read()))
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l and re.match(r"gpudh?_", l.split()[-1])}
    internal = {"gpud_ring_range_prepare", "gpud_ring_range_pass", "gpud_ring_range_note", "gpud_ring_quantile", "gpud_scan_state_free", "gpud_comm_state_free",
                "gpud_parallel_memcpy", "gpud_host_tables"}      # C++-mangled internals never match; these are listed for clarity
    assert exported - internal <= decl, sorted(exported - internal - decl)
    assert decl <= exported, sorted(decl - exported)


def test_layout_and_version():
    L = g.lib()
    assert L.gpud_abi_version() == 1
    assert L.gpud_sizeof(2) == 128 == C.sizeof(g.FabricLocal)
    assert L.gpud_sizeof(99) == -1


def test_catalog_accessors():
    L = g.lib()
    assert L.gpud_xid_description(79, 0) == b"GPU has fallen off the bus"
    assert L.gpud_xid_mnemonic(79) == b"ROBUST_CHANNEL_GPU_HAS_FALLEN_OFF_THE_BUS"
    assert L.gpud_xid_description(133, 0) == b"" and L.gpud_xid_description(99999, 0) == b""
    assert b"cartridge" in L.gpud_xid_description(149, 1)
    assert L.gpud_sxid_name(20034) != b"" and L.gpud_sxid_name(11111) == b""


def test_hit_json_host_rendering():
    from oracle import pyoracle as O
    L = g.lib()
    h = g.XidHit()
    h.kind, h.code, h.n_actions = 1, 79, 2
    h.actions[0], h.actions[1] = 2, 3
    h.device = b"PCI:0000:05:00"
    buf = C.create_string_buffer(2048)
    assert L.gpud_hit_detail_json(C.byref(h), 1740327858, buf, 2048) == 0
    x = O.xid_match(b"NVRM: Xid (PCI:0000:05:00): 79, GPU has fallen off the bus.")
    assert buf.value.decode() == O.xid_event_detail_json(x, 1740327858)
    assert L.gpud_hit_detail_json(C.byref(h), 0, buf, 8) == -4


@pytest.mark.skipif(any(re.fullmatch(r"nvidia\d+", d) for d in os.listdir("/dev")), reason="a GPU is present")
def test_no_cpu_fallback():      # a container may expose only some GPU's node (/dev/nvidia6), not /dev/nvidia0
    with pytest.raises(g.GpudError):
        g.Context([0])


def test_header_is_plain_c():
    """what cgo would feed its C compiler: the header alone, as C99 with every warning on, and as C++11"""
    import os
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "gpud_b200.h")
    for cmd in (["gcc", "-x", "c", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", hdr],
                ["g++", "-x", "c++", "-std=c++11", "-Wall", "-Werror", "-fsyntax-only", hdr]):
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr


def test_c_consumer_links_and_runs(tmp_path):
    """a C program including only gpud_b200.h, linked with -lgpud_b200: the boundary as a cgo file uses it"""
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    exe = str(tmp_path / "abi_consumer")
    libdir = os.path.dirname(capi.LIB_PATH)
    libname = os.path.basename(capi.LIB_PATH)
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "abi_consumer.c"),
                        "-o", exe, "-L", libdir, "-l:" + libname, "-Wl,-rpath," + libdir, "-Wl,-rpath,/usr/local/cuda/lib64"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr


def test_product_never_touches_the_oracle():
    """the oracle is the checker only: no Python module of the product imports it, the shared library neither links nor dlopens it"""
    import glob
    import subprocess
    for path in glob.glob(os.path.join(ROOT, "gpud_b200", "*.py")):
        src = open(path).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), path
    for path in glob.glob(os.path.join(ROOT, "gpud_b200", "csrc", "*")):
        if path.endswith((".cu", ".cpp", ".h")):
            src = open(path).read()
            assert "liboracle" not in src and not re.search(r'#include\s+"[^"]*oracle', src), path
    out = subprocess.run(["ldd", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "liboracle" not in out
    blob = open(capi.LIB_PATH, "rb").read()
    assert b"liboracle" not in blob and b"orc_scan_lines" not in blob


def test_scan_one_shot_on_a_cpu_only_host():
    """BASELINE configs[0] (plumbing): the `gpud scan`-shaped driver runs without CUDA and prints one CheckResult per component in the
    api/v1 HealthState shape (pkg/scan/scan.go:20-28,74-102)."""
    import json
    import subprocess
    exe = os.path.join(ROOT, "gpud_b200", "gpud-scan")
    if not os.path.exists(exe):
        pytest.skip("gpud-scan not built")
    assert "cuda" not in subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout
    states = [json.loads(l) for l in out.splitlines() if l.startswith("{")]
    assert [s["component"] for s in states] == ["cpu", "memory", "os"]
    for s in states:
        assert s["name"] == s["component"] and s["health"] in ("Healthy", "Degraded", "Unhealthy") and s["reason"] and s["time"].endswith("Z")
    assert "scanning the host" in out and "scan complete" in out
