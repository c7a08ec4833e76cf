"""Drop-in proof at the source level: the UNMODIFIED reference CLI (dsv_main.c) compiles against include/compat
and links against libdsv1_b200.so; and the library exports every symbol include/exports.txt lists (no compute
calls here: this runs without a GPU)."""
import ctypes
import os
import subprocess

import pytest

import dsvlibs as L
import refdigest

REF_MAIN = "/root/reference/dsv_main.c"


def test_exports_present():
    if not os.path.exists(L.GPU_SO):
        subprocess.run(["make", "-s", "-C", L.PKG], check=True)
    lib = ctypes.CDLL(L.GPU_SO)
    for sym in open(os.path.join(L.ROOT, "include", "exports.txt")).read().split():
        assert hasattr(lib, sym), sym


def test_reference_cli_links(tmp_path):
    if not os.path.exists(REF_MAIN):
        pytest.skip("reference tree not present")
    if not os.path.exists(L.GPU_SO):
        subprocess.run(["make", "-s", "-C", L.PKG], check=True)
    exe = str(tmp_path / "dsv1_b200")
    subprocess.run(["gcc", "-O1", "-w", "-I" + os.path.join(L.ROOT, "include", "compat"), REF_MAIN, "-o", exe,
                    "-L" + L.PKG, "-ldsv1_b200", "-Wl,-rpath," + L.PKG], check=True)
    # usage text only: anything further needs a GPU
    r = subprocess.run([exe], capture_output=True, text=True)
    assert "usage" in (r.stdout + r.stderr).lower() or r.returncode in (0, 1)


def _declared_functions(header):
    """Function names declared at file scope of a C header (comments, preprocessor lines, struct bodies dropped)."""
    import re
    src = open(header).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"\\\n", "", src)
    src = re.sub(r"^\s*#.*?$", "", src, flags=re.M)
    src = src.replace('extern "C" {', "")
    depth, out = 0, []
    for ch in src:
        if ch == "{":
            depth += 1
        elif ch == "}":
            depth = max(0, depth - 1)
        elif depth == 0:
            out.append(ch)
    names = set()
    for stmt in "".join(out).split(";"):
        st = stmt.strip()
        if not st or st.startswith("typedef"):
            continue
        m = re.search(r"\b([a-z_][a-z0-9_]*)\s*\((?:[^()]|\([^()]*\))*\)\s*$", st, flags=re.S)
        if m:
            names.add(m.group(1))
    return names


def test_every_declared_function_is_exported():
    """include/*.h is the contract: each function it declares must be a symbol of the shared library, and
    include/exports.txt must list exactly those (plus data symbols)."""
    if not os.path.exists(L.GPU_SO):
        subprocess.run(["make", "-s", "-C", L.PKG], check=True)
    lib = ctypes.CDLL(L.GPU_SO)
    declared = set()
    for h in ("dsv1_b200.h", "dsv1_b200_batch.h", "dsv1_b200_kernels.h"):
        fns = _declared_functions(os.path.join(L.ROOT, "include", h))
        assert len(fns) >= 9, (h, fns)
        declared |= fns
    for sym in sorted(declared):
        assert hasattr(lib, sym), sym
    listed = set(open(os.path.join(L.ROOT, "include", "exports.txt")).read().split())
    assert declared <= listed, sorted(declared - listed)
    assert listed - declared <= {"dsv_lvlname"}, sorted(listed - declared)  # the only data symbol


def _frame_helpers(lib):
    import numpy as np
    outs = []
    for (w, h, fmt, seed) in FRAME_HELPER_CASES:
        sub = L.SUBSAMP[fmt]
        yuv = L.synth_sequence(w, h, fmt, 1, seed, 0)
        cap = 64 + ((w + 1) // 2 + 128) * ((h + 1) // 2 + 128) + L.frame_bytes(w, h, sub)
        o = np.zeros(cap, dtype=np.uint8)
        f = lib.fn("frame_helpers_probe", api=True)
        f.restype = ctypes.c_long
        n = f(L.ptr(yuv), w, h, sub, L.ptr(o), ctypes.c_long(cap))
        assert n > 0, n
        outs.append(o[:n])
    return outs


FRAME_HELPER_CASES = [(64, 48, "420", 1), (90, 70, "444", 2), (54, 38, "422", 3), (176, 144, "411", 4)]


def test_public_frame_helpers_match_reference(gpu, ref):
    """dsv.h also declares host frame helpers the codec path does not call (dsv_ds2x_frame_luma,
    dsv_extend_frame_luma, dsv_frame_avg_luma, dsv_frame_add, dsv_plane_xy): same caller code
    (tools/api_harness.c: frame_helpers_probe) against both libraries, byte for byte.  Host-only, no GPU."""
    import numpy as np
    got = _frame_helpers(gpu)
    want = refdigest.table(ref, "frame_helpers_probe", _frame_helpers)
    for a, b, case in zip(want, got, FRAME_HELPER_CASES):
        assert np.array_equal(a, b), case


def test_nothing_the_reference_headers_declare_is_missing():
    """Every function the reference's public headers declare (dsv.h, dsv_encoder.h, dsv_decoder.h, util.h) is in
    include/exports.txt -- a caller of any of them links."""
    if not os.path.exists("/root/reference/dsv.h"):
        pytest.skip("reference tree not present")
    declared = set()
    for h in ("dsv.h", "dsv_encoder.h", "dsv_decoder.h", "util.h"):
        declared |= _declared_functions(os.path.join("/root/reference", h))
    assert len(declared) >= 36
    listed = set(open(os.path.join(L.ROOT, "include", "exports.txt")).read().split())
    assert declared <= listed, sorted(declared - listed)
