"""ctypes bindings for the in-tree native libraries (see ``draco_b200/build.py``).

``host()`` loads ``libdraco_host.so`` (pure C++, works everywhere).  ``cuda()`` loads ``libdraco_cuda.so`` (every
sm_100a kernel + the symmetric-memory runtime); it raises loudly when CUDA is present but the library is missing,
because silently falling back to PyTorch ops on a GPU box would hide that the product path is not running.

The ``Structure`` classes mirror, field for field, the argument structs in ``csrc/cuda/*.cu``.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

LIB_DIR = Path(__file__).resolve().parent / "_lib"

MAX_R = 8
MAX_DST = 16
MAX_WORKERS = 32
TILE = 1024
THREADS = 256

_host: Optional[C.CDLL] = None
_cuda: Optional[C.CDLL] = None

u64 = C.c_ulonglong
i64 = C.c_longlong
ptr = C.c_void_p


class TensorMeta(C.Structure):
    _fields_ = [("offset", i64), ("numel", i64), ("is_bf16", C.c_int), ("pad", C.c_int)]


class HyperParams(C.Structure):
    _fields_ = [("lr", C.c_float), ("momentum", C.c_float), ("weight_decay", C.c_float), ("dampening", C.c_float),
                ("nesterov", C.c_int), ("optimizer", C.c_int), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("pad", C.c_int * 3)]


class TileView(C.Structure):
    _fields_ = [("tile_tensor", ptr), ("meta", ptr), ("ntiles", C.c_int), ("ntensors", C.c_int)]


class FlagList(C.Structure):
    _fields_ = [("ptr", ptr * MAX_DST), ("n", C.c_int)]


class PushArgs(C.Structure):
    _fields_ = [("g32", ptr * MAX_R), ("g16", ptr * MAX_R), ("coef_re", C.c_float * MAX_R), ("coef_im", C.c_float * MAX_R),
                ("R", C.c_int), ("cyclic", C.c_int), ("dst", ptr), ("tv", TileView), ("adv_bitmap", ptr),
                ("adv_len", C.c_int), ("step_ptr", ptr), ("worker", C.c_int), ("attack", C.c_int),
                ("magnitude", C.c_float), ("seed", u64), ("done_counter", ptr), ("flag", ptr), ("local_copy", ptr),
                ("tile_begin", C.c_int), ("tile_end", C.c_int), ("src_table", ptr)]


class OmniArgs(C.Structure):
    _fields_ = [("grad_in", ptr), ("slot_stride", i64), ("honest_mask", C.c_uint), ("worker", C.c_int),
                ("magnitude", C.c_float), ("total", i64), ("done_counter", ptr), ("flag", ptr), ("step_ptr", ptr)]


class CollusionArgs(C.Structure):
    _fields_ = [("grad_in", ptr), ("slot_stride", i64), ("P", C.c_int), ("tv", TileView), ("tile_begin", C.c_int),
                ("tile_end", C.c_int), ("adv_bitmap", ptr), ("adv_len", C.c_int), ("step_ptr", ptr), ("mode", C.c_int),
                ("param", C.c_float)]


class VoteArgs(C.Structure):
    _fields_ = [("grad_in", ptr), ("slot_stride", i64), ("group_table", ptr), ("G", C.c_int), ("max_r", C.c_int),
                ("tv", TileView), ("neq_mask", ptr), ("tile_begin", C.c_int), ("tile_end", C.c_int)]


class ResolveArgs(C.Structure):
    _fields_ = [("neq_mask", ptr), ("group_table", ptr), ("G", C.c_int), ("max_r", C.c_int), ("T", C.c_int),
                ("winner_slot", ptr), ("winner_member", ptr), ("clear_mask", ptr), ("t_begin", C.c_int), ("t_end", C.c_int)]


class UpdateArgs(C.Structure):
    _fields_ = [("mode", C.c_int), ("grad_in", ptr), ("slot_stride", i64), ("select", ptr), ("K", C.c_int),
                ("scale", C.c_float), ("recomb", ptr), ("tv", TileView), ("params", ptr), ("momentum", ptr),
                ("exp_avg_sq", ptr), ("max_exp_avg_sq", ptr), ("hp", ptr), ("step_ptr", ptr), ("first_step", u64), ("grad_out", ptr), ("mc_params", ptr),
                ("dst", ptr * MAX_DST), ("ndst", C.c_int), ("done_counter", ptr), ("flags", FlagList),
                ("tile_begin", C.c_int), ("tile_end", C.c_int), ("trim", C.c_int)]


class StreamPushArgs(C.Structure):
    _fields_ = [("src", ptr), ("dst", ptr), ("nbytes", ptr), ("nbytes_out", ptr), ("step_ptr", ptr), ("done_counter", ptr),
                ("flag", ptr)]


class CastArgs(C.Structure):
    _fields_ = [("src", ptr), ("dst", ptr), ("tv", TileView)]


class WaitArgs(C.Structure):
    _fields_ = [("flags", ptr * MAX_WORKERS), ("n", C.c_int), ("step_ptr", ptr), ("addend", i64), ("timeout_ns", u64),
                ("error", ptr), ("stamps", ptr)]


class SetFlagArgs(C.Structure):
    _fields_ = [("flags", FlagList), ("step_ptr", ptr), ("addend", i64)]


class ProjectArgs(C.Structure):
    _fields_ = [("R", ptr), ("slot_stride", i64), ("n", C.c_int), ("f", ptr), ("tv", TileView), ("E", ptr), ("Epart", ptr)]


class LocateArgs(C.Structure):
    _fields_ = [("E", ptr), ("T", C.c_int), ("n", C.c_int), ("s", C.c_int), ("rel_tol", C.c_double), ("recomb", ptr),
                ("healthy", ptr), ("flagged", ptr)]


class GeoMedArgs(C.Structure):
    _fields_ = [("grad_in", ptr), ("slot_stride", i64), ("P", C.c_int), ("tv", TileView), ("median", ptr),
                ("weights", ptr), ("done", ptr), ("dist2", ptr), ("move2", ptr)]


class GeoMedPrepArgs(C.Structure):
    _fields_ = [("T", C.c_int), ("P", C.c_int), ("dist2", ptr), ("move2", ptr), ("weights", ptr), ("done", ptr),
                ("iter", C.c_int), ("eps", C.c_double)]


class GeoMedWeightsArgs(C.Structure):
    _fields_ = [("pair_d2", ptr), ("T", C.c_int), ("P", C.c_int), ("max_iter", C.c_int), ("eps", C.c_double), ("weights", ptr),
                ("iters", ptr)]


class PairDistArgs(C.Structure):
    _fields_ = [("grad_in", ptr), ("slot_stride", i64), ("P", C.c_int), ("tv", TileView), ("pair_d2", ptr)]


class KrumSelectArgs(C.Structure):
    _fields_ = [("pair_d2", ptr), ("T", C.c_int), ("P", C.c_int), ("s", C.c_int), ("select", ptr), ("m", C.c_int)]


def _maybe_build() -> None:
    if os.environ.get("DRACO_NO_AUTOBUILD"):
        return
    try:
        from . import build
        build.build_host()
    except Exception:
        pass


def host() -> C.CDLL:
    """The pure-C++ helper library (builds it on first use if a compiler is around)."""
    global _host
    if _host is None:
        path = LIB_DIR / "libdraco_host.so"
        if not path.exists():
            _maybe_build()
        if not path.exists():
            raise RuntimeError(f"{path} missing: run `python -m draco_b200.build`")
        lib = C.CDLL(str(path))
        lib.drc_host_locate.argtypes = [ptr, C.c_int, C.c_int, C.c_int, C.c_double, ptr, ptr, ptr]
        lib.drc_host_solve_poly_a.argtypes = [ptr, C.c_int, C.c_int, ptr]
        lib.drc_codec_bound.restype = u64
        lib.drc_codec_bound.argtypes = [u64, C.c_uint]
        lib.drc_codec_encode.restype = u64
        lib.drc_codec_encode.argtypes = [ptr, u64, C.c_uint, ptr, u64]
        lib.drc_codec_decode.restype = u64
        lib.drc_codec_decode.argtypes = [ptr, u64, ptr, u64]
        lib.drc_codec_raw_size.restype = u64
        lib.drc_codec_raw_size.argtypes = [ptr, u64]
        lib.drc_codec_valid.restype = C.c_int
        lib.drc_codec_valid.argtypes = [ptr, u64]
        lib.drc_codec_itemsize_flags.restype = C.c_uint
        lib.drc_codec_itemsize_flags.argtypes = [ptr, u64]
        lib.drc_host_geomedian.argtypes = [ptr, C.c_int, i64, i64, C.c_double, C.c_int, ptr]
        lib.drc_host_vote.argtypes = [ptr, i64, i64, ptr, C.c_int]
        lib.drc_host_krum.argtypes = [ptr, C.c_int, i64, i64, C.c_int]
        _host = lib
    return _host


def cuda_available() -> bool:
    return (LIB_DIR / "libdraco_cuda.so").exists()


def cuda() -> C.CDLL:
    """The sm_100a kernel library.  Never falls back: a missing library on a GPU box is an error."""
    global _cuda
    if _cuda is None:
        path = LIB_DIR / "libdraco_cuda.so"
        if not path.exists():
            raise RuntimeError(f"{path} missing: run `python -m draco_b200.build` (nvcc cross-compiles without a GPU)")
        lib = C.CDLL(str(path))
        st = ptr  # cudaStream_t
        for name, args in {
            "drc_push_encode": [C.POINTER(PushArgs), C.c_int, st],
            "drc_omniscient": [C.POINTER(OmniArgs), C.c_int, st],
            "drc_collude": [C.POINTER(CollusionArgs), C.c_int, st],
            "drc_vote_compare": [C.POINTER(VoteArgs), C.c_int, st],
            "drc_vote_resolve": [C.POINTER(ResolveArgs), st],
            "drc_aggregate_update": [C.POINTER(UpdateArgs), C.c_int, st],
            "drc_cast_params": [C.POINTER(CastArgs), C.c_int, st],
            "drc_wait_flags": [C.POINTER(WaitArgs), st],
            "drc_step_add": [ptr, i64, st],
            "drc_set_flags": [C.POINTER(SetFlagArgs), st],
            "drc_cyclic_project": [C.POINTER(ProjectArgs), C.c_int, st],
            "drc_cyclic_locate": [C.POINTER(LocateArgs), st],
            "drc_geomed_iter": [C.POINTER(GeoMedArgs), C.c_int, st],
            "drc_geomed_prep": [C.POINTER(GeoMedPrepArgs), st],
            "drc_geomed_weights": [C.POINTER(GeoMedWeightsArgs), st],
            "drc_pair_dist": [C.POINTER(PairDistArgs), C.c_int, st],
            "drc_krum_select": [C.POINTER(KrumSelectArgs), st],
            "drc_gemm_bf16": [ptr, i64, C.c_int, ptr, i64, C.c_int, ptr, i64, C.c_int, C.c_int, C.c_int, C.c_int, ptr, ptr,
                              C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, st],
            "drc_rt_init": [C.c_int],
            "drc_rt_granularity": [C.c_int, C.POINTER(u64)],
            "drc_rt_alloc": [C.c_int, u64, C.POINTER(ptr), C.POINTER(u64), C.POINTER(C.c_int)],
            "drc_rt_import": [C.c_int, C.c_int, u64, C.POINTER(ptr), C.POINTER(u64)],
            "drc_rt_unmap": [ptr, u64, u64],
            "drc_rt_close_fd": [C.c_int],
            "drc_rt_mc_supported": [C.c_int, C.POINTER(C.c_int)],
            "drc_rt_mc_granularity": [C.c_int, u64, C.POINTER(u64)],
            "drc_rt_mc_create": [C.c_int, u64, C.POINTER(u64), C.POINTER(C.c_int)],
            "drc_rt_mc_import": [C.c_int, C.POINTER(u64)],
            "drc_rt_mc_add_device": [u64, C.c_int],
            "drc_rt_mc_bind": [u64, u64, u64, u64, u64],
            "drc_rt_mc_map": [C.c_int, u64, u64, C.POINTER(ptr)],
            "drc_rt_peer_access": [C.c_int, C.c_int, C.POINTER(C.c_int)],
            "drc_rt_memset_async": [ptr, C.c_int, u64, st],
            "drc_rt_memcpy_async": [ptr, ptr, u64, st],
            "drc_rt_sm_count": [C.c_int, C.POINTER(C.c_int)],
        }.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int
        _cuda = lib
    return _cuda


def check(code: int, what: str) -> None:
    if code != 0:
        raise RuntimeError(f"{what} failed with code {code}")
