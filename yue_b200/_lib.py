"""ctypes binding of libyue_b200.so (include/yue_b200.h).  There is no fallback: if the CUDA
library is missing or does not load, importing the product path raises."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libyue_b200.so")
SRC = os.path.join(HERE, "csrc", "yue_b200.cu")
HEADER = os.path.join(ROOT, "include", "yue_b200.h")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
              "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread"]


HASH_PATH = LIB_PATH + ".srchash"


def _sources():
    return sorted(os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc"))) + [HEADER]


def _source_hash():
    import hashlib
    h = hashlib.sha256()
    for s in _sources():
        h.update(os.path.basename(s).encode() + b"\0")
        with open(s, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def is_stale():
    """True when the library was not built from the sources as they are now (compared by content -- a copy of the tree
    to the GPU box does not keep file times in order)."""
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as f:
        return f.read().strip() != _source_hash()


def build(force=False, verbose=False):
    """Compile the CUDA library in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    import fcntl
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:       # ranks of one job may all find it stale at once
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not is_stale():
            return LIB_PATH
        nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
        tmp = LIB_PATH + ".tmp%d" % os.getpid()
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp, SRC, "-ldl"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
        if verbose:
            print(res.stderr)
        os.replace(tmp, LIB_PATH)
        with open(HASH_PATH, "w") as f:
            f.write(_source_hash() + "\n")
    return LIB_PATH


class YueError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("yue_b200 error %d: %s" % (code, msg))
        self.code = code


E_ARG, E_CUDA, E_STATE, E_NUMERIC, E_NCCL, E_UNSUPPORTED = 1, 2, 3, 4, 5, 6
MODE_SERIAL, MODE_HOGWILD, MODE_HOGWILD_STORE = 0, 1, 2
RANK_EXACT, RANK_TC, RANK_AUTO = 0, 1, 2
BUF_P, BUF_Q, BUF_Q_DELTA, BUF_Q_SNAPSHOT = 0, 1, 2, 3

_i64p, _i32p, _f32p, _f64p = (C.POINTER(t) for t in (C.c_int64, C.c_int32, C.c_float, C.c_double))
_H = C.c_void_p

# name -> (restype, argtypes); kept in step with include/yue_b200.h (tests/test_abi.py checks it)
SIGNATURES = {
    "yue_version": (C.c_char_p, []),
    "yue_last_error": (C.c_char_p, [_H]),
    "yue_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "yue_create": (C.c_int, [C.c_int, C.POINTER(_H)]),
    "yue_destroy": (C.c_int, [_H]),
    "yue_sync": (C.c_int, [_H]),
    "yue_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "yue_host_free": (C.c_int, [C.c_void_p]),
    "yue_set_interactions": (C.c_int, [_H, C.c_int64, C.c_int64, _i64p, _i32p, _i64p, _i32p]),
    "yue_set_interactions_shard": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                             _i64p, _i32p, _i64p, _i32p]),
    "yue_set_factors": (C.c_int, [_H, C.c_int, _f32p, _f32p]),
    "yue_get_factors": (C.c_int, [_H, _f32p, _f32p]),
    "yue_sample_negatives": (C.c_int, [_H, C.c_uint64, C.c_uint32, C.c_uint32, _i32p]),
    "yue_bpr_epoch": (C.c_int, [_H, C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_uint32,
                                C.c_int, _f64p]),
    "yue_bpr_epoch_part": (C.c_int, [_H, C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_uint32,
                                     C.c_int, C.c_int, C.c_int, _f64p]),
    "yue_bpr_apply": (C.c_int, [_H, _i32p, _i32p, _i32p, C.c_int64, C.c_double, C.c_double,
                                C.c_double, C.c_int, _f64p]),
    "yue_apr_epoch": (C.c_int, [_H, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_uint64,
                                C.c_uint32, C.c_uint32, C.c_int, _f64p]),
    "yue_apr_apply": (C.c_int, [_H, _i32p, _i32p, _i32p, C.c_int64, C.c_double, C.c_double, C.c_double,
                                C.c_double, C.c_double, C.c_int, _f64p]),
    "yue_cune_set_implicit": (C.c_int, [_H, _i64p, _i32p]),
    "yue_cune_epoch": (C.c_int, [_H, C.c_double, C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_uint32,
                                 C.c_int, _f64p]),
    "yue_gcn_set_events": (C.c_int, [_H, C.c_int64, _i32p, _i32p]),
    "yue_gcn_epoch": (C.c_int, [_H, C.c_int, C.c_int, C.c_double, C.c_double, C.c_uint64, C.c_uint32, C.c_int64, C.c_int64, _f64p]),
    "yue_gcn_apply": (C.c_int, [_H, C.c_int, C.c_int64, _i32p, _i32p, _i32p, C.c_double, C.c_double, _f64p]),
    "yue_gcn_finalize": (C.c_int, [_H, C.c_int]),
    "yue_gcn_moments": (C.c_int, [_H, _f32p, _f32p, _f32p, _f32p, _i64p]),
    "yue_bpr_adam_sample": (C.c_int, [_H, C.c_uint64, C.c_int64, C.c_int, C.c_int, _i32p, _i32p]),
    "yue_bpr_adam_steps": (C.c_int, [_H, C.c_int, C.c_int, C.c_double, C.c_double, C.c_uint64, C.c_int64, C.c_int64, _f64p]),
    "yue_bpr_adam_apply": (C.c_int, [_H, C.c_int64, _i32p, _i32p, _i32p, C.c_double, C.c_double, _f64p]),
    "yue_bpr_adam_moments": (C.c_int, [_H, _f32p, _f32p, _f32p, _f32p, _i64p]),
    "yue_frob2": (C.c_int, [_H, _f64p, _f64p]),
    "yue_predict": (C.c_int, [_H, C.c_int64, _f32p]),
    "yue_rank_topn": (C.c_int, [_H, _i32p, C.c_int64, C.c_int, C.c_int, _i32p, _f32p]),
    "yue_q_snapshot": (C.c_int, [_H]),
    "yue_q_delta_pack": (C.c_int, [_H]),
    "yue_q_delta_apply": (C.c_int, [_H]),
    "yue_set_delta_weights": (C.c_int, [_H, _f32p]),
    "yue_device_buffer": (C.c_int, [_H, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "yue_stream": (C.c_int, [_H, C.POINTER(C.c_void_p)]),
    "yue_comm_unique_id": (C.c_int, [C.c_void_p]),
    "yue_comm_init": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    "yue_allreduce_q_delta": (C.c_int, [_H]),
    "yue_hot_tracks": (C.c_int, [_H, _i32p, C.POINTER(C.c_int)]),
    "yue_set_hot_tracks": (C.c_int, [_H, _i32p, _i64p, C.c_int, C.c_int64]),
    "yue_hot_table_export": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_void_p)]),
    "yue_hot_table_open": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_void_p)]),
    "yue_enable_peer": (C.c_int, [_H, C.c_int]),
    "yue_hot_share": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "yue_hot_pull": (C.c_int, [_H]),
    "yue_hot_unshare": (C.c_int, [_H]),
    "yue_q_exchange_begin": (C.c_int, [_H]),
    "yue_q_exchange_reduce": (C.c_int, [_H]),
    "yue_q_exchange_reduce_peers": (C.c_int, [_H, C.c_int, C.POINTER(C.c_void_p)]),
    "yue_q_exchange_finish": (C.c_int, [_H, C.c_int]),
    "yue_stream2": (C.c_int, [_H, C.POINTER(C.c_void_p)]),
    "yue_set_sgd_concurrency": (C.c_int, [_H, C.c_int, C.c_int]),
    "yue_apr_epoch_part": (C.c_int, [_H, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_uint64,
                                     C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, _f64p]),
    "yue_result_lines": (C.c_int, [C.c_char_p, _i64p, C.c_char_p, _i64p, C.c_int64, _i32p, C.POINTER(C.c_uint8), C.c_int64, C.c_int,
                                   C.c_void_p, C.c_int64, _i64p]),
    "yue_timer_start": (C.c_int, [_H]),
    "yue_timer_stop": (C.c_int, [_H, _f32p]),
    "yue_launch_count": (C.c_int, [_H, _i64p]),
    "yue_rank_stats": (C.c_int, [_H, _i64p, _i64p]),
    "yue_set_event_offsets": (C.c_int, [_H, _i64p]),
    "yue_set_test_set": (C.c_int, [_H, _i64p, _i32p]),
    "yue_ingest_events": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_int64, _i32p, _i32p, C.POINTER(C.c_uint8)]),
    "yue_interaction_sizes": (C.c_int, [_H, _i64p, _i64p, _i64p, _i64p, _i64p]),
    "yue_get_interactions": (C.c_int, [_H, _i64p, _i32p, _i64p, _i32p]),
    "yue_get_test_set": (C.c_int, [_H, _i64p, _i32p]),
    "yue_rank_metrics": (C.c_int, [_H, C.c_int, _i32p, _f64p, _i64p]),
    "yue_flush_l2": (C.c_int, [_H]),
    "yue_wrmf_sweep": (C.c_int, [_H, C.c_int, C.c_double, C.c_double, _f64p]),
    "yue_wrmf_sweep_rows": (C.c_int, [_H, C.c_int, C.c_int64, C.c_int64, C.c_double, C.c_double, _f64p]),
    "yue_wrmf_pair_counts": (C.c_int, [_H, _i32p, _i64p, _i32p, _i32p]),
}

_lib = None


def load():
    """Load the shared library.  A library that was not built from the current sources is rebuilt first when nvcc is
    here; without a compiler it is an error -- tests and benchmarks never run against a stale library."""
    global _lib
    if _lib is not None:
        return _lib
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if os.path.exists(LIB_PATH) and is_stale():
        if os.path.exists(nvcc):
            build()
        else:
            raise ImportError("yue_b200: %s is older than its sources and there is no nvcc to rebuild it" % LIB_PATH)
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "yue_b200: %s is missing.  Build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (needs nvcc); there is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library drift: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
