"""ctypes binding of libpvk.so (include/pvk.h) -- the only way the host side reaches the GPU.

The library is built in-tree by ``pypevoc_b200/build.py`` (nvcc, sm_100a).  There is no CPU
fallback: if the shared object is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PVK_LIB: load an experimental build variant of the same library (tuning runs only)
LIB_PATH = os.environ.get("PVK_LIB") or os.path.join(_HERE, "libpvk.so")

_p = C.c_void_p
_i64 = C.c_int64
_i = C.c_int
_d = C.c_double

# name -> (restype, argtypes); mirrors include/pvk.h one to one
SIGNATURES = {
    "pvk_version": (_i, []),
    "pvk_last_error": (C.c_char_p, []),
    "pvk_launch_count": (_i64, []),
    "pvk_analyze_tables_bytes": (_i64, [_i]),
    "pvk_analyze_init": (_i, [_i, _p, _p]),
    "pvk_analyze": (_i, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _i, _i, _i, _d, _d, _d, _i64, _i64,
                         _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pvk_analyze_ex": (_i, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _i, _i, _i, _d, _d, _d, _i64, _i64,
                            _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pvk_analyze_batch": (_i, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _i, _i, _i, _d, _d, _d, _i64, _i64,
                               _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "pvk_harmonic": (_i, [_p, _i64, _p, _p, _p, _p, _i, _i, _i, _d, _d, _d, _p, _i64, _i, _p, _p, _p, _p, _p, _p]),
    "pvk_stft_bank": (_i, [_p, _i64, _p, _p, _i, _i, _i64, _i, _p, _p, _p, _i, _p, _i, _i, _p, _d, _p, _p]),
    "pvk_frame_stats": (_i, [_p, _p, _i64, _i, _d, _d, _d, _p, _p, _p, _p]),
    "pvk_harmonic_power": (_i, [_p, _p, _i64, _i, _d, _p, _p, _p, _p, _p]),
    "pvk_track_workspace_bytes": (_i64, [_i64, _i64, _i]),
    "pvk_track": (_i, [_p, _p, _i64, _i64, _i, _d, _p, _p, _p, _p, _i64, _p]),
    "pvk_track_spans": (_i, [_p, _i64, _i, _i64, _p, _p, _p]),
    "pvk_track_stats": (_i, [_p, _p, _i64, _i64, _i, _p, _p]),
    "pvk_clip_spans": (_i, [_p, _p, _i64, _i64, _i64, _p, _p, _p]),
    "pvk_track_pack_workspace_bytes": (_i64, [_i64]),
    "pvk_track_pack": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "pvk_track_pack_dev": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "pvk_segment_summary": (_i, [_p, _i, _i64, _i64, _i64, _p, _p]),
    "pvk_segment_resolve": (_i, [_p, _i, _i, _i, _p, _i64, _p, _p, _p]),
    "pvk_segment_rename": (_i, [_p, _i64, _p, _p, _p, _p]),
    "pvk_segment_rename_push": (_i, [_p, _i64, _p, _p, _p, _i, _i64, _p]),
    "pvk_segment_rename_mcast": (_i, [_p, _i64, _p, _p, _p, _i64, _p]),
    "pvk_resynth_workspace_bytes": (_i64, [_i64, _i, _i64, _i64]),
    "pvk_resynth": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _i, _p, _i64, _i64,
                         _i64, _p, _i64, _i, _p]),
    "pvk_resynth_dev": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _i, _p, _i64, _i64,
                             _i64, _p, _i64, _i, _p]),
    "pvk_resynth_ex": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _i, _p, _i64, _i64,
                            _i64, _p, _i64, _i, _i, _d, _p, _i64, _p]),
    "pvk_resynth_render": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _i, _p, _i64,
                                _i64, _i64, _p, _i64, _i, _i, _d, _p, _i64, _p]),
    "pvk_resynth_scan": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _p, _i64, _p, _i64, _i64,
                              _i64, _p, _i64, _p]),
    "pvk_resynth_handover": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _i64, _p, _i64, _i, _i, _i64, _p, _i64, _p]),
    "pvk_nyquist_flags": (_i, [_p, _p, _i64, _d, _d, _p, _i64, _p]),
    "pvk_resynth_import_flags": (_i, [_p, _i64, _i, _i64, _p, _p, _i64, _i64, _p, _i64, _p, _i64, _p]),
    "pvk_resynth_ex_curve": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _i, _p, _i64,
                                  _i64, _i64, _p, _i64, _i, _i, _d, _p, _i64, _p, _i64, _p]),
    "pvk_resynth_render_curve": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _i, _p, _i64,
                                      _i64, _i64, _p, _i64, _i, _i, _d, _p, _i64, _p, _i64, _p]),
    "pvk_resynth_scan_curve": (_i, [_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _d, _i, _i, _i, _d, _p, _i64, _p, _i64, _p,
                                    _i64, _i64, _i64, _p, _i64, _p]),
    "pvk_nyquist_flags_curve": (_i, [_p, _p, _i64, _d, _d, _p, _i64, _i, _p, _i64, _p]),
}


def declare(lib, strict=True):
    """Attach restype/argtypes for every symbol of pvk.h; raise if one is missing."""
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            if strict:
                raise RuntimeError("libpvk: symbol %s declared in include/pvk.h is not exported" % name)
            continue
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "pypevoc_b200: CUDA extension %s is not built (run `python -m pypevoc_b200.build`); "
                "there is no CPU fallback" % LIB_PATH)
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


def check(status, what=""):
    if status != 0:
        msg = lib().pvk_last_error().decode("utf-8", "replace")
        raise RuntimeError("libpvk %s failed (status %d): %s" % (what, status, msg))
