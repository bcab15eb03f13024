"""TEST INFRASTRUCTURE ONLY -- builds and drives tests/analyze_block_ref.cu, analyze_kernel<LOGM> (one
CTA per frame) at nfft 1024 / 2048, to compare analyze_warp_kernel with the kernel it was read off.

Two builds of the same source:
  - ``build_emu()``: g++ against the SIMT emulator (the flags of tests/emu/build_emu.sh), next to
    libpvk_emu.so, rebuilt when a source is newer;
  - ``build_gpu(dirpath)``: nvcc for sm_100a with pypevoc_b200.build.NVCC_FLAGS, into ``dirpath``.
Both export ``pvkt_analyze_block`` with the arguments of pvk_analyze_ex (run_frames must be >= 1)."""
import ctypes as C
import os
import subprocess

import numpy as np

from pypevoc_b200 import _lib as binding
from pypevoc_b200 import build as pbuild

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "analyze_block_ref.cu")
EMU = os.path.join(HERE, "emu")
EMU_SO = os.path.join(EMU, "libanalyze_block_ref_emu.so")
INCLUDES = ["-I", os.path.join(ROOT, "include"), "-I", pbuild.CSRC]


def _declare(lib):
    fn = lib.pvkt_analyze_block
    fn.restype, fn.argtypes = binding.SIGNATURES["pvk_analyze_ex"]
    lib.pvk_last_error.restype = C.c_char_p
    return lib


def build_emu(force=False):
    deps = [SRC, __file__, os.path.join(EMU, "cuda_emu.h"), os.path.join(EMU, "cuda_emu.cc"),
            os.path.join(ROOT, "include", "pvk.h")] + [os.path.join(pbuild.CSRC, f) for f in os.listdir(pbuild.CSRC)]
    if force or not os.path.isfile(EMU_SO) or any(os.path.getmtime(d) > os.path.getmtime(EMU_SO) for d in deps):
        tmp = EMU_SO + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-g", "-fPIC", "-shared", "-ffp-contract=off", "-DPVK_EMU",
                               "-Wall", "-Wno-unknown-pragmas", "-Wno-unused-function", "-I", EMU] + INCLUDES +
                              ["-x", "c++", SRC, os.path.join(EMU, "cuda_emu.cc"), "-o", tmp, "-lpthread"])
        os.replace(tmp, EMU_SO)
    return EMU_SO


_emu = None


def emu_lib():
    global _emu
    if _emu is None:
        _emu = _declare(C.CDLL(build_emu()))
    return _emu


def build_gpu(dirpath):
    """nvcc build of the reference for sm_100a into ``dirpath``; returns the loaded library."""
    out = os.path.join(dirpath, "libanalyze_block_ref.so")
    res = subprocess.run([pbuild._nvcc()] + pbuild.NVCC_FLAGS + INCLUDES + [SRC, "-o", out],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building %s:\n%s" % (SRC, res.stdout[-3000:]))
    return _declare(C.CDLL(out))


def analyze_emu(x, sr, nfft, hop, npks, pkthresh=0.005, run_frames=4):
    """analyze_kernel on the emulator: the dict of emu_harness.analyze(..., spectra=True, refine=True)."""
    import emu_harness as eh
    L, B = eh.lib(), emu_lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    if x.ndim == 1:
        x = x[None, :]
    nclips, nsamp = x.shape
    tb = eh.host_tables(sr, nfft, hop)
    nframes = -(-(nsamp - nfft) // hop)
    tables = np.zeros(L.pvk_analyze_tables_bytes(nfft), dtype=np.uint8)
    eh.check(L.pvk_analyze_init(nfft, eh.ptr(tables), None))
    shp = (nclips, nframes, npks)
    out = {k: np.full(shp, np.nan) for k in ("f", "mag", "ph", "realph", "binno", "fine_pos", "fine_val")}
    npk = np.full((nclips, nframes), -7, dtype=np.int32)
    totalmag = np.full((nclips, nframes), np.nan)
    spec = np.zeros((nclips, nframes, nfft // 2, 2), dtype=np.float32)
    p = eh.ptr
    st = B.pvkt_analyze_block(p(x), nclips, x.strides[0] // 4, nsamp, p(tb["win_scaled"]), p(tb["fbin"]), p(tb["wfbin"]),
                              p(tables), nfft, hop, npks, pkthresh, tb["dt"], tb["fstep"], 0, nframes, 1, run_frames,
                              p(out["f"]), p(out["mag"]), p(out["ph"]), p(out["realph"]), p(out["binno"]), p(npk),
                              p(totalmag), p(spec), p(out["fine_pos"]), p(out["fine_val"]), None)
    if st != 0:
        raise RuntimeError("pvkt_analyze_block: %s" % B.pvk_last_error().decode())
    out.update(npk=npk, totalmag=totalmag, nframes=nframes, fx=spec[..., 0] + 1j * spec[..., 1])
    return out
