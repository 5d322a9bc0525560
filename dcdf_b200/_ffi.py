"""ctypes binding of include/dcdf_cuda.h (libdcdf_cuda.so).

The library is the product; this module only declares its C-ABI.  There is no CPU fallback: if the
shared object is missing or no CUDA device is present, loading / context creation fails loudly.
"""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdcdf_cuda.so")
CSRC = os.path.join(HERE, "csrc")

OK = 0
ERR_NAMES = {0: "OK", 1: "NONFINITE", 2: "PRECISION_LOSS", 3: "OVERFLOW", 4: "BAD_LEVELS", 5: "OUT_OF_BOUNDS",
             6: "BAD_FORMAT", 7: "CUDA", 8: "BAD_ARG"}
ENC_I32, ENC_I64, ENC_F32, ENC_F64 = 4, 8, 32, 64
MEM_HOST, MEM_DEVICE = 0, 1
REF_ELIDED, REF_LOCAL, REF_EXTERNAL = 0, 1, 2
KT_ENCODE, KT_STATS, KT_GATHER, KT_WINDOW, KT_CELL, KT_SEARCH, KT_REDUCE, KT_TIME_STATS = range(8)


class Array3(C.Structure):
    _fields_ = [("base", C.c_void_p), ("shape", C.c_int64 * 3), ("strides", C.c_int64 * 3),
                ("encoding", C.c_int32), ("mem", C.c_int32)]


class BuildStats(C.Structure):
    _fields_ = [("size", C.c_uint64), ("elided", C.c_uint32), ("local", C.c_uint32), ("external", C.c_uint32),
                ("snapshots", C.c_uint32), ("logs", C.c_uint32)]


class Cube(C.Structure):
    _fields_ = [("start", C.c_int64), ("end", C.c_int64), ("top", C.c_int64), ("bottom", C.c_int64),
                ("left", C.c_int64), ("right", C.c_int64)]


class SuperchunkInfo(C.Structure):
    _fields_ = [("shape", C.c_int64 * 3), ("sidelen", C.c_int64), ("chunks_sidelen", C.c_int64),
                ("subsidelen", C.c_int64), ("levels", C.c_uint32), ("encoding", C.c_int32),
                ("fractional_bits", C.c_int32), ("n_refs", C.c_uint32), ("max_dac_bytes", C.c_uint64),
                ("min_dac_bytes", C.c_uint64), ("chunk_bytes", C.c_uint64), ("stats", BuildStats)]


CID_BYTES = 36
NODE_LINKS, NODE_SUBCHUNK, NODE_SUPERCHUNK = 1, 4, 5
FETCH_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_uint64))


def build_library(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a into libdcdf_cuda.so (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".hpp", ".sh"))]
    srcs.append(os.path.join(os.path.dirname(HERE), "include", "dcdf_cuda.h"))
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    r = subprocess.run(["bash", os.path.join(CSRC, "build.sh")], capture_output=True, text=True, timeout=1800)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libdcdf_cuda.so failed")
    return LIB_PATH


_lib = None

_P = C.POINTER


def _declare(lib):
    vp, i32, i64, u32, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64
    sig = {
        "dcdf_abi_version": (i32, []),
        "dcdf_ctx_create": (i32, [i32, _P(vp)]),
        "dcdf_ctx_destroy": (i32, [vp]),
        "dcdf_ctx_set_stream": (i32, [vp, vp]),
        "dcdf_ctx_set_option": (i32, [vp, C.c_char_p, i64]),
        "dcdf_ctx_get_stat": (i32, [vp, C.c_char_p, _P(i64)]),
        "dcdf_ctx_synchronize": (i32, [vp]),
        "dcdf_last_error": (C.c_char_p, [vp]),
        "dcdf_ctx_launch_count": (u64, [vp]),
        "dcdf_ctx_last_kernel_ms": (i32, [vp, i32, _P(C.c_float)]),
        "dcdf_suggest_fraction": (i32, [vp, _P(Array3), _P(i32), _P(i32)]),
        "dcdf_min_max": (i32, [vp, _P(Array3), i32, i32, vp, vp]),
        "dcdf_to_fixed": (i32, [vp, vp, i32, u64, i32, i32, vp, i32]),
        "dcdf_from_fixed": (i32, [vp, vp, u64, i32, vp, i32, i32]),
        "dcdf_chunk_build": (i32, [vp, _P(Array3), i32, i32, i32, _P(vp), _P(BuildStats)]),
        "dcdf_chunk_open": (i32, [vp, vp, u64, i32, _P(vp)]),
        "dcdf_chunk_free": (i32, [vp]),
        "dcdf_chunk_size": (i32, [vp, _P(u64)]),
        "dcdf_chunk_bytes": (i32, [vp, vp, vp, u64, i32]),
        "dcdf_chunk_info": (i32, [vp, _P(i64 * 3), _P(i32), _P(i32), _P(u32)]),
        "dcdf_chunk_block_instants": (i32, [vp, vp, vp]),
        "dcdf_chunk_get_batch": (i32, [vp, vp, u64, vp, vp, i32, i32]),
        "dcdf_chunk_cell_batch": (i32, [vp, vp, u64, vp, vp, vp, i32, i32]),
        "dcdf_chunk_window": (i32, [vp, vp, _P(Cube), vp, i32, i32]),
        "dcdf_chunk_search": (i32, [vp, vp, _P(Cube), i64, i64, vp, u64, _P(u64), i32]),
        "dcdf_superchunk_build": (i32, [vp, _P(Array3), _P(u32), u32, i32, i32, i32, i32, i64, _P(vp)]),
        "dcdf_superchunk_free": (i32, [vp]),
        "dcdf_superchunk_count": (i32, [vp, _P(u32)]),
        "dcdf_superchunk_get_info": (i32, [vp, u32, _P(SuperchunkInfo)]),
        "dcdf_superchunk_node_count": (i32, [vp, _P(u32)]),
        "dcdf_superchunk_node_info": (i32, [vp, u32, u32, _P(SuperchunkInfo)]),
        "dcdf_superchunk_node_refs": (i32, [vp, vp, u32, u32, vp, vp, vp, vp, vp]),
        "dcdf_superchunk_node_bytes": (i32, [vp, vp, u32, u32, i32, vp, u64, i32]),
        "dcdf_superchunk_refs": (i32, [vp, vp, u32, vp, vp, vp, vp]),
        "dcdf_superchunk_bytes": (i32, [vp, vp, u32, i32, vp, u64, i32]),
        "dcdf_superchunk_total_bytes": (i32, [vp, _P(u64)]),
        "dcdf_superchunk_get_batch": (i32, [vp, vp, u64, vp, vp, i32, i32]),
        "dcdf_superchunk_cell_batch": (i32, [vp, vp, u64, vp, vp, vp, i32, i32]),
        "dcdf_superchunk_window": (i32, [vp, vp, _P(Cube), vp, i32, i32]),
        "dcdf_superchunk_window_batch": (i32, [vp, vp, u64, vp, vp, vp, i32, i32]),
        "dcdf_superchunk_window_stats": (i32, [vp, vp, u64, vp, vp, vp, vp, vp, vp, vp, i32]),
        "dcdf_superchunk_time_stats": (i32, [vp, vp, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32]),
        "dcdf_superchunk_search_batch": (i32, [vp, vp, u64, vp, vp, vp, vp, vp, u64, _P(u64), i32]),
        "dcdf_superchunk_search_values": (i32, [vp, vp, u64, vp, vp, vp, vp, vp, u64, _P(u64), i32]),
        "dcdf_superchunk_save": (i32, [vp, vp, u32, _P(vp)]),
        "dcdf_saved_free": (i32, [vp]),
        "dcdf_saved_count": (i32, [vp, _P(u32)]),
        "dcdf_saved_node": (i32, [vp, u32, vp, _P(i32), _P(u64)]),
        "dcdf_saved_node_bytes": (i32, [vp, vp, u32, vp, u64, i32]),
        "dcdf_saved_all_bytes": (i32, [vp, vp, vp, u64, vp]),
        "dcdf_saved_stats": (i32, [vp, _P(BuildStats)]),
        "dcdf_superchunk_open": (i32, [vp, u32, vp, FETCH_FN, vp, _P(vp)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return sig


DECLARED = None


def lib():
    """Load libdcdf_cuda.so.  Raises if it has not been built -- there is no fallback implementation."""
    global _lib, DECLARED
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run dcdf_b200.build() (nvcc, sm_100a); there is no CPU fallback")
        l = C.CDLL(LIB_PATH)
        DECLARED = _declare(l)
        if l.dcdf_abi_version() != 1:
            raise RuntimeError("libdcdf_cuda.so ABI version mismatch")
        _lib = l
    return _lib
