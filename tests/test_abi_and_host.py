"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol include/pvk.h
declares (no compute calls without a GPU); host-side logic of pypevoc_b200."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import pv_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    from pypevoc_b200 import build
    return build.build()


def header_symbols():
    src = open(os.path.join(ROOT, "include", "pvk.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pvk_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(libpath):
    from pypevoc_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 8
    assert sorted(_lib.SIGNATURES) == syms, "pypevoc_b200/_lib.py and include/pvk.h disagree"
    lib = ctypes.CDLL(libpath)
    for s in syms:
        assert hasattr(lib, s), s
    _lib.declare(lib)
    assert lib.pvk_version() == 5
    assert lib.pvk_last_error() == b""


def test_argument_validation_without_gpu(libpath):
    """Argument checks happen before any CUDA call, so they can be exercised on the CPU box."""
    from pypevoc_b200 import _lib
    lib = _lib.declare(ctypes.CDLL(libpath))
    assert lib.pvk_analyze_tables_bytes(1000) == -1
    assert lib.pvk_analyze_tables_bytes(16384) == -1
    assert lib.pvk_analyze_tables_bytes(2048) > 0
    st = lib.pvk_analyze(None, 1, 0, 10, None, None, None, None, 1000, 1, 1, 0.0, 0.0, 0.0, 0, 1, 1, 0,
                         None, None, None, None, None, None, None, None, None)
    assert st == 1 and b"power of two" in lib.pvk_last_error()
    st = lib.pvk_analyze(None, 1, 0, 10, None, None, None, None, 1024, 0, 1, 0.0, 0.0, 0.0, 0, 1, 1, 0,
                         None, None, None, None, None, None, None, None, None)
    assert st == 1 and b"hop" in lib.pvk_last_error()
    st = lib.pvk_analyze(None, 1, 0, 2000, None, None, None, None, 1024, 512, 20, 0.0, 0.0, 0.0, 0, 5, 1, 0,
                         None, None, None, None, None, None, None, None, None)
    assert st == 1 and b"last frame" in lib.pvk_last_error()
    assert lib.pvk_track_workspace_bytes(1, 100, 50) > 0
    st = lib.pvk_track(None, None, 1, 10, 5000, 0.5, None, None, None, None, 0, None)
    assert st == 1 and b"npks" in lib.pvk_last_error()


def test_analyze_batch_rejects_spectra_with_guard_rows(libpath):
    """spec_out has no guard rows: with out_rows_per_clip > nframes the batch call refuses it before
    any CUDA call; without spec_out the same arguments pass that check."""
    from pypevoc_b200 import _lib
    lib = _lib.declare(ctypes.CDLL(libpath))
    spec = np.zeros((2, 10, 512, 2), dtype=np.float32)
    p = spec.ctypes.data_as(ctypes.c_void_p)
    st = lib.pvk_analyze_batch(None, 2, 20000, 20000, None, None, None, None, 1024, 256, 20, 0.005, 0.0, 0.0, 0, 10,
                               1, 0, None, None, None, None, None, None, None, p, None, None, 13, None)
    assert st == 1 and b"spec_out" in lib.pvk_last_error() and b"out_rows_per_clip=13" in lib.pvk_last_error()
    st = lib.pvk_analyze_batch(None, 2, 20000, 20000, None, None, None, None, 1024, 256, 20, 0.005, 0.0, 0.0, 0, 10,
                               1, 0, None, None, None, None, None, None, None, None, None, None, 13, None)
    assert st == 1 and b"NULL pointer" in lib.pvk_last_error()


def test_product_fails_loudly_without_gpu_or_library(monkeypatch):
    import torch
    import pypevoc_b200
    from pypevoc_b200 import _lib
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            pypevoc_b200.PV(np.zeros(4096), 44100)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libpvk.so")
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(RuntimeError, match="not built"):
        _lib.lib()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pypevoc_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+\.*oracle", src, flags=re.M), fn
                assert "oracle." not in src and "libpvk_emu" not in src, fn


def test_host_tables_match_reference_expressions():
    from pypevoc_b200.pv import host_tables, n_frames, synth_geometry
    for sr, nfft, hop in ((44100, 2048, 512), (16000, 512, 128), (48000, 8192, 1024), (22050, 1024, 300)):
        a, b = host_tables(sr, nfft, hop), orc.pv_tables(sr, nfft, hop)
        for k in ("win", "wfact", "fstep", "dt", "fbin", "wfbin"):
            assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    for nsamp, nfft, hop in ((100, 1024, 512), (1024, 1024, 512), (1025, 1024, 512), (2048 + 3 * 512, 2048, 512),
                             (44100, 2048, 1024)):
        assert n_frames(nsamp, nfft, hop) == orc.n_frames(nsamp, nfft, hop)
    assert n_frames(2048 + 3 * 512, 2048, 512) == 3
    assert synth_geometry(84, 512, 1024, 512) == (86 * 512 + 512, 512)


def test_ctypes_signatures_match_the_header_types():
    """Every prototype of include/pvk.h against the ctypes signature of pypevoc_b200/_lib.py: same
    number of parameters, same classes (pointer / int64_t / int / double) in the same order, same
    return type.  A drifted hand-written binding would corrupt the call frame, not fail cleanly."""
    from pypevoc_b200 import _lib
    src = open(os.path.join(ROOT, "include", "pvk.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = re.findall(r"^\s*((?:const\s+)?[A-Za-z_0-9]+\s*\*?)\s*(pvk_[a-z_0-9]+)\s*\(([^;]*?)\)\s*;", src, flags=re.M | re.S)
    assert len(protos) == len(_lib.SIGNATURES)

    def cls(decl):
        decl = decl.strip()
        if "*" in decl:
            return ctypes.c_char_p if decl.replace(" ", "").startswith("constchar*") else ctypes.c_void_p
        base = decl.split()[-2] if len(decl.split()) > 1 else decl
        base = decl.rsplit(None, 1)[0] if len(decl.split()) > 1 else decl
        base = base.replace("const", "").strip()
        return {"int64_t": ctypes.c_int64, "int": ctypes.c_int, "double": ctypes.c_double}[base]
    for ret, name, params in protos:
        res, args = _lib.SIGNATURES[name]
        plist = [p for p in (q.strip() for q in params.replace("\n", " ").split(",")) if p and p != "void"]
        got = [cls(p) for p in plist]
        assert got == list(args), (name, [g.__name__ for g in got], [a.__name__ for a in args])
        rcls = ctypes.c_char_p if "char" in ret else cls(ret + " x")
        assert rcls == res, name


def test_host_pipeline_helpers():
    """Pure host helpers of the streamed / sharded paths."""
    from pypevoc_b200.pv import _chunk_bounds
    from pypevoc_b200 import dist as D
    for n in (0, 1, 63, 64, 1000, 51676):
        for chunks in (1, 2, 3, 8):
            b = _chunk_bounds(n, chunks)
            assert len(b) == chunks + 1 and b[0] == 0 and b[-1] == n and all(x <= y for x, y in zip(b, b[1:]))
    b = _chunk_bounds(51676, 8)
    assert b[1] - b[0] < b[2] - b[1] and b[-1] - b[-2] < b[-2] - b[-3]          # short first and last piece
    saved = os.environ.pop("PVK_PEER_GATHER", None)
    try:
        assert D._peer_gather_wanted(2) and D._peer_gather_wanted(4) and not D._peer_gather_wanted(8)
        os.environ["PVK_PEER_GATHER"] = "1"
        assert D._peer_gather_wanted(8)
        os.environ["PVK_PEER_GATHER"] = "0"
        assert not D._peer_gather_wanted(2)
    finally:
        os.environ.pop("PVK_PEER_GATHER", None)
        if saved is not None:
            os.environ["PVK_PEER_GATHER"] = saved
    # every rank's block range is known without any count, and trimming it gives render_range()
    nfft, hop = 2048, 512
    for world in (2, 3, 8):
        F = 400
        plans = D.plan_segments(nfft + (F - 1) * hop + 1, nfft, hop, world)
        for max_end in (F - 1, F - 40, 120, 5):
            total = 0
            for p in plans:
                b0, b1, bound = D.render_range_local(p, plans, p["w1"] - 1 if p["nown"] else -1, hop, nfft, hop)
                nrender = max(min(b1 * hop, bound) - b0 * hop, 0)
                n, s0 = D.trim_local(nrender, b0, p, plans, max_end, hop, nfft, hop)
                g0, g1, nout = D.render_range(p, plans, max_end, hop, nfft, hop)
                assert n == max(min(g1 * hop, nout) - g0 * hop, 0)
                total += n
            assert total == D.render_range(plans[0], plans, max_end, hop, nfft, hop)[2]
