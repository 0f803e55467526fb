"""ctypes binding of libvbnmf.so (include/vbnmf.h).  This is the same boundary the R `.Call`
shim in r-shim/ binds; nothing here computes anything.  If the CUDA library is missing or no
GPU is usable the calls fail loudly -- there is no CPU fallback."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get("VBNMF_LIB_NAME", "libvbnmf.so"))  # experiments: variants

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)
c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_fp = C.POINTER(C.c_float)
c_u8p = C.POINTER(C.c_uint8)


class VbnmfCfg(C.Structure):
    """vbnmf_cfg of include/vbnmf.h (the fields of `bundle`, R/bayesian.R:252-259, the loop reads)."""
    _fields_ = [("itmax", C.c_int), ("tol", C.c_double), ("hyper_update", C.c_int * 4),
                ("n0", C.c_int), ("dn", C.c_int), ("fudge", C.c_double)]


class VbnmfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libvbnmf error %d: %s" % (code, msg))
        self.code = code


ERR_ARG = 1
ERR_HYPER = 2
ERR_MEMORY = 7

# name -> (restype, argtypes); every symbol declared in include/vbnmf.h
SIGNATURES = {
    "vbnmf_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_int64, c_i32p,
                               c_i64p, c_i32p, c_dp, C.c_int]),
    "vbnmf_create_from_device": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_int64,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "vbnmf_create_from_mtx": (C.c_int, [C.POINTER(C.c_void_p), C.c_char_p, C.c_int, c_i64p]),
    "vbnmf_get_csc": (C.c_int, [C.c_void_p, c_i64p, c_i32p, c_dp]),
    "vbnmf_qc_stats": (C.c_int, [C.c_void_p, c_dp, c_dp, c_dp, c_i64p, c_i64p]),
    "vbnmf_create_subset": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, c_u8p, c_u8p, c_dp]),
    "vbnmf_create_shuffled": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_uint64]),
    "vbnmf_consensus": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int, c_i32p, C.c_int64, c_i64p,
                                  c_i64p, c_i64p, C.c_int64, c_i64p]),
    "vbnmf_destroy": (None, [C.c_void_p]),
    "vbnmf_last_error": (C.c_char_p, [C.c_void_p]),
    "vbnmf_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "vbnmf_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vbnmf_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "vbnmf_comm_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "vbnmf_comm_destroy": (None, [C.c_void_p]),
    "vbnmf_attach_comm": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vbnmf_set_state": (C.c_int, [C.c_void_p, C.c_int, c_dp, c_dp, c_dp, c_dp]),
    "vbnmf_step": (C.c_int, [C.c_void_p, c_dp, C.c_double, c_dp]),
    "vbnmf_run": (C.c_int, [C.c_void_p, C.POINTER(VbnmfCfg), c_dp, c_dp, c_dp, c_ip, c_dp, c_ip]),
    "vbnmf_get_state": (C.c_int, [C.c_void_p, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "vbnmf_get_means": (C.c_int, [C.c_void_p, c_dp]),
    "vbnmf_cluster_id": (C.c_int, [C.c_void_p, c_i32p]),
    "vbnmf_uniform_columns": (C.c_int, [C.c_void_p, C.c_double, c_i32p]),
    "mlnmf_run": (C.c_int, [C.c_void_p, C.c_int, c_dp, c_dp, C.c_int, C.c_double, c_dp, c_dp, c_dp,
                            c_ip]),
    "mlnmf_run2": (C.c_int, [C.c_void_p, C.c_int, c_dp, c_dp, C.c_int, C.c_double, C.c_int, C.c_int,
                             c_dp, c_dp, c_dp, c_dp, c_ip]),
    "vbnmf_bench_iterations": (C.c_int, [C.c_void_p, c_dp, C.c_double, C.c_int, C.c_int, c_dp,
                                         c_i64p, c_dp]),
    "vbnmf_set_host_threads": (C.c_int, [C.c_int]),
    "vbnmf_trim_pool": (C.c_int, [C.c_int]),
    "vbnmf_init_random": (C.c_int, [C.c_void_p, C.c_int, c_dp, C.c_uint64, C.c_int64]),
    "vbnmf_init_svd2": (C.c_int, [C.c_void_p, C.c_int, c_dp, C.c_uint64, C.c_int64]),
    "vbnmf_init_svd": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_int64]),
    "vbnmf_info": (C.c_int, [C.c_void_p, c_i64p]),
    "vbnmf_layout_info": (C.c_int, [C.c_void_p, c_i64p]),
}

_lib = None


def load():
    """Load libvbnmf.so (built in-tree by ccfindr_b200.build).  Raises if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "%s not found: build it with `python -m ccfindr_b200.build` (needs nvcc). "
                "There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, handle=None):
    if rc != 0:
        msg = load().vbnmf_last_error(handle)
        raise VbnmfError(rc, msg.decode() if msg else "unknown")
