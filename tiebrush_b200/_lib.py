"""ctypes binding of the C ABI (include/tiebrush_b200.h) exported by libtiebrush_b200.so.

The shared library is built in-tree by __graft_entry__.build() / `make -C tiebrush_b200/csrc`.
There is no fallback: a missing library or a missing CUDA device raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtiebrush_b200.so")

SYMBOLS = ["tb_create", "tb_destroy", "tb_last_error", "tb_set_stream", "tb_get_stream", "tb_sync",
           "tb_collapse_window", "tb_collapse_window_carry", "tc_coverage_window", "tc_sample_window", "tb_launch_count", "tb_set_profiling",
           "tb_last_kernel_ms", "tb_version", "tb_last_path", "tb_last_yd_path", "tb_last_yd_stat", "tb_last_heavy_slots", "tb_last_ord_deep", "tb_last_tile_gen", "tb_last_tile_stat",
           "tc_coverage_stream", "tb_comm_unique_id", "tb_comm_init", "tb_comm_destroy", "tb_comm_rank", "tb_comm_world",
           "tc_shard_coverage", "tc_shard_coverage_gather", "tc_shard_gather", "tc_shard_stat", "tc_stream_windows", "tc_last_exact"]


class SoaIn(C.Structure):
    _fields_ = [("n", C.c_int64), ("n_files", C.c_int32), ("tid", C.c_int32), ("run_off", C.c_void_p),
                ("file_merged", C.c_void_p), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p),
                ("strand", C.c_void_p), ("nh", C.c_void_p), ("cig_off", C.c_void_p), ("cigar", C.c_void_p),
                ("md_off", C.c_void_p), ("md", C.c_void_p), ("qhash", C.c_void_p), ("yc_in", C.c_void_p),
                ("yx_in", C.c_void_p), ("yd_in", C.c_void_p), ("on_device", C.c_int32),
                ("n_cig", C.c_int64), ("n_md", C.c_int64), ("pos_lo", C.c_int32), ("pos_hi", C.c_int32),
                ("n_cigar8", C.c_void_p), ("cigar16", C.c_void_p), ("cigar_ext", C.c_void_p), ("n_ext", C.c_int64),
                ("pos_d8", C.c_void_p), ("pos_ext", C.c_void_p), ("n_pos_ext", C.c_int64), ("meta8", C.c_void_p), ("meta_dict", C.c_void_p),
                ("n_meta_dict", C.c_int32), ("meta_ext", C.c_void_p), ("n_meta_ext", C.c_int64)]


class GroupsOut(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("n_groups", C.c_int64), ("n_kept", C.c_int64), ("rep_index", C.c_void_p),
                ("yc", C.c_void_p), ("yx", C.c_void_p), ("yd", C.c_void_p), ("on_device", C.c_int32)]


class YdCarry(C.Structure):
    _fields_ = [("tid", C.c_int32), ("pos_hi", C.c_int32), ("n_chains", C.c_int32), ("capacity", C.c_int64), ("n_segs", C.c_int64),
                ("chain_off", C.c_void_p), ("seg_start", C.c_void_p), ("seg_end", C.c_void_p)]


class CovIn(C.Structure):
    _fields_ = [("n", C.c_int64), ("tid", C.c_void_p), ("pos", C.c_void_p), ("yc", C.c_void_p), ("strand", C.c_void_p),
                ("cig_off", C.c_void_p), ("cigar", C.c_void_p), ("on_device", C.c_int32), ("n_cig", C.c_int64), ("end", C.c_void_p)]


class RunsOut(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("n_runs", C.c_int64), ("tid", C.c_void_p), ("start0", C.c_void_p),
                ("end0", C.c_void_p), ("value", C.c_void_p), ("on_device", C.c_int32)]


class JuncsOut(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("n_juncs", C.c_int64), ("tid", C.c_void_p), ("start", C.c_void_p),
                ("end", C.c_void_p), ("strand", C.c_void_p), ("value", C.c_void_p), ("on_device", C.c_int32)]


_lib = None


def load():
    """Load libtiebrush_b200.so and declare prototypes. Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the hot path)")
    lib = C.CDLL(LIB_PATH)
    lib.tb_create.restype = C.c_void_p
    lib.tb_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.tb_destroy.argtypes = [C.c_void_p]
    lib.tb_destroy.restype = None
    lib.tb_last_error.restype = C.c_char_p
    lib.tb_last_error.argtypes = [C.c_void_p]
    lib.tb_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.tb_get_stream.argtypes = [C.c_void_p]
    lib.tb_get_stream.restype = C.c_void_p
    lib.tb_sync.argtypes = [C.c_void_p]
    lib.tb_collapse_window.argtypes = [C.c_void_p, C.POINTER(SoaIn), C.POINTER(GroupsOut)]
    lib.tb_collapse_window_carry.argtypes = [C.c_void_p, C.POINTER(SoaIn), C.POINTER(YdCarry), C.POINTER(GroupsOut), C.POINTER(YdCarry)]
    lib.tc_coverage_window.argtypes = [C.c_void_p, C.POINTER(CovIn), C.POINTER(RunsOut), C.POINTER(JuncsOut)]
    lib.tc_sample_window.argtypes = [C.c_void_p, C.POINTER(CovIn), C.c_void_p, C.POINTER(RunsOut)]
    lib.tb_launch_count.argtypes = [C.c_void_p]
    lib.tb_launch_count.restype = C.c_int64
    lib.tb_set_profiling.argtypes = [C.c_void_p, C.c_int]
    lib.tb_last_kernel_ms.argtypes = [C.c_void_p, C.c_int]
    lib.tb_last_kernel_ms.restype = C.c_float
    lib.tb_version.restype = C.c_char_p
    lib.tb_last_path.argtypes = [C.c_void_p]
    lib.tb_last_path.restype = C.c_int
    lib.tb_last_yd_path.argtypes = [C.c_void_p]
    lib.tb_last_yd_path.restype = C.c_int
    lib.tb_last_yd_stat.argtypes = [C.c_void_p, C.c_int]
    lib.tb_last_yd_stat.restype = C.c_int64
    lib.tb_last_heavy_slots.argtypes = [C.c_void_p]
    lib.tb_last_heavy_slots.restype = C.c_int64
    lib.tb_last_ord_deep.argtypes = [C.c_void_p]
    lib.tb_last_ord_deep.restype = C.c_int64
    lib.tb_last_tile_gen.argtypes = [C.c_void_p]
    lib.tb_last_tile_gen.restype = C.c_int
    lib.tb_last_tile_stat.argtypes = [C.c_void_p, C.c_int]
    lib.tb_last_tile_stat.restype = C.c_int64
    lib.tc_coverage_stream.argtypes = [C.c_void_p, C.POINTER(CovIn), C.c_int64, C.c_void_p, C.POINTER(RunsOut), C.POINTER(JuncsOut), C.POINTER(C.c_int64)]
    lib.tb_comm_unique_id.argtypes = [C.c_void_p]
    lib.tb_comm_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.tb_comm_destroy.argtypes = [C.c_void_p]
    lib.tb_comm_rank.argtypes = [C.c_void_p]
    lib.tb_comm_world.argtypes = [C.c_void_p]
    lib.tc_shard_coverage.argtypes = [C.c_void_p, C.POINTER(CovIn), C.c_int, C.c_int64, C.POINTER(RunsOut), C.POINTER(JuncsOut)]
    lib.tc_shard_coverage_gather.argtypes = [C.c_void_p, C.POINTER(CovIn), C.c_int, C.c_int64, C.POINTER(RunsOut), C.POINTER(JuncsOut), C.POINTER(RunsOut), C.POINTER(JuncsOut), C.POINTER(C.c_int64)]
    lib.tc_shard_gather.argtypes = [C.c_void_p, C.POINTER(RunsOut), C.POINTER(JuncsOut), C.POINTER(RunsOut), C.POINTER(JuncsOut), C.POINTER(C.c_int64)]
    lib.tc_shard_stat.argtypes = [C.c_void_p, C.c_int]
    lib.tc_shard_stat.restype = C.c_int64
    lib.tc_stream_windows.argtypes = [C.c_void_p]
    lib.tc_stream_windows.restype = C.c_int64
    lib.tc_last_exact.argtypes = [C.c_void_p]
    _lib = lib
    return lib
