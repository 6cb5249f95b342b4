"""ctypes binding of libbpg.so (the C ABI declared in include/bpg.h).

The shared library is built in-tree by `make -C bulletproofs_gadgets_b200/csrc` (nvcc, sm_100a).  There is no
fallback: if the library is missing, or no CUDA device is present when a context is created, the call fails."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbpg.so")
if os.environ.get("BPG_LIB"):  # A/B builds of the same sources (development aid), e.g. BPG_LIB=libbpg_pad.so
    LIB_PATH = os.path.join(os.path.dirname(LIB_PATH), os.environ["BPG_LIB"])

OK, E_CUDA, E_SIZE, E_DECOMPRESS, E_ARG, E_FORMAT, E_NOMEM, E_COMM = 0, -1, -2, -3, -4, -5, -6, -7
FLAG_LEGACY_FRAMING, FLAG_FAST_BLINDING, FLAG_WITNESS_ON_DEVICE = 1, 2, 4
FLAG_NO_LATE_FOLD, FLAG_FORCE_LATE_FOLD = 8, 16

# every symbol include/bpg.h declares: name -> (restype, argtypes)
_u8p, _sz, _i32, _vp = C.c_char_p, C.c_size_t, C.c_int, C.c_void_p
_u32p, _u64p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)
SYMBOLS = {
    "bpg_ctx_create": (_i32, [_i32, C.POINTER(_vp)]),
    "bpg_ctx_destroy": (None, [_vp]),
    "bpg_last_error": (C.c_char_p, [_vp]),
    "bpg_strerror": (C.c_char_p, [_i32]),
    "bpg_launch_count": (C.c_uint64, [_vp]),
    "bpg_sync": (_i32, [_vp]),
    "bpg_set_blocking_sync": (None, [_i32]),
    "bpg_set_sizing_mode": (None, [_i32]),
    "bpg_gens_ensure": (_i32, [_vp, _sz]),
    "bpg_gens_capacity": (_sz, [_vp]),
    "bpg_gens_export": (_i32, [_vp, _sz, _sz, _u8p, _u8p]),
    "bpg_pedersen_gens": (_i32, [_vp, _u8p, _u8p]),
    "bpg_pedersen_commit": (_i32, [_vp, _u8p, _u8p, _sz, _u8p]),
    "bpg_msm": (_i32, [_vp, _u8p, _u8p, _sz, _u8p]),
    "bpg_msm_gens": (_i32, [_vp, _u8p, _u8p, _sz, _sz, _u8p, _u8p, _sz, _u8p]),
    "bpg_msm_gens_dev": (_i32, [_vp, _vp, _vp, _sz, _sz, _u8p]),
    "bpg_msm_gens_partial_dev": (_i32, [_vp, _vp, _vp, _sz, _sz, _u8p]),
    "bpg_points_sum_compress": (_i32, [_vp, _u8p, _sz, _u8p]),
    "bpg_ctx_set_shard": (_i32, [_vp, _i32, _i32, _vp, _vp, _sz, _vp, _vp]),
    "bpg_comm_unique_id": (_i32, [_u8p]),
    "bpg_comm_init": (_i32, [_vp, _i32, _i32, _u8p]),
    "bpg_comm_destroy": (_i32, [_vp]),
    "bpg_msm_gens_sharded_dev": (_i32, [_vp, _vp, _vp, _sz, _sz, _u8p]),
    "bpg_msm_gens_partial_to_dev": (_i32, [_vp, _vp, _vp, _sz, _sz, _vp]),
    "bpg_points_sum_compress_dev": (_i32, [_vp, _vp, _sz, _u8p]),
    "bpg_fold_points": (_i32, [_vp, _u8p, _u8p, _u8p, _u8p, _sz, _u8p]),
    "bpg_mimc_set_constants": (_i32, [_vp, _u8p]),
    "bpg_mimc_hash_batch": (_i32, [_vp, _u8p, _u64p, _sz, _u8p]),
    "bpg_mimc_sponge_batch": (_i32, [_vp, _u8p, _u32p, _sz, _u8p, _u8p]),
    "bpg_circuit_create": (_i32, [_vp, _sz, _sz, _sz, _u32p, _u32p, _u8p, C.POINTER(_vp)]),
    "bpg_circuit_destroy": (None, [_vp]),
    "bpg_circuit_create_batch": (_i32, [_vp, _sz, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_u32p), C.POINTER(_u32p), C.POINTER(C.c_char_p),
                                        C.POINTER(_vp)]),
    "bpg_witness_eval": (_i32, [_vp, _sz, _sz, _u32p, _u32p, _u8p, _u8p, _u8p, _u8p, _u8p]),
    "bpg_witness_eval_batch": (_i32, [_vp, _sz, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_u32p), C.POINTER(_u32p), C.POINTER(C.c_char_p),
                                      C.POINTER(C.c_char_p), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "bpg_r1cs_prove": (C.c_long, [_vp, _vp, _u8p, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, C.c_uint, _u8p, _u8p, _sz]),
    "bpg_r1cs_prove_prefetch": (_i32, [_vp, _vp, _u8p, _sz, _u8p, _u8p, _u8p, C.c_uint]),
    "bpg_r1cs_prove_batch": (_i32, [_vp, _sz, C.POINTER(_vp), C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                    C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), _u8p, C.c_uint, C.POINTER(_vp), C.POINTER(_vp),
                                    C.POINTER(_sz), C.POINTER(_sz)]),
    "bpg_r1cs_verify": (_i32, [_vp, _vp, _u8p, _sz, _u8p, _u8p, _sz, _u8p, C.c_uint, C.POINTER(_i32)]),
    "bpg_r1cs_verify_batch": (_i32, [_vp, _sz, C.POINTER(_vp), C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                     C.POINTER(_sz), _u8p, C.c_uint, C.POINTER(_i32)]),
    "bpg_r1cs_verify_each": (_i32, [_vp, _sz, C.POINTER(_vp), C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                    C.POINTER(_sz), _u8p, C.c_uint, C.POINTER(_i32)]),
    "bpg_transcript_new": (_vp, [_u8p, _sz]),
    "bpg_transcript_free": (None, [_vp]),
    "bpg_transcript_append": (None, [_vp, _u8p, _sz, _u8p, _sz]),
    "bpg_transcript_challenge": (None, [_vp, _u8p, _sz, _u8p, _sz]),
    "bpg_host_rng_lanes": (_i32, []),
    "bpg_host_rng_draw64": (_i32, [_u8p, _sz, _u8p, _sz, _sz, _i32, _u8p]),
    "bpg_dev_alloc": (_i32, [_vp, _sz, C.POINTER(_vp)]),
    "bpg_dev_free": (_i32, [_vp, _vp]),
    "bpg_host_alloc": (_i32, [_vp, _sz, C.POINTER(_vp)]),
    "bpg_host_free": (_i32, [_vp, _vp]),
    "bpg_dev_upload": (_i32, [_vp, _vp, _u8p, _sz]),
    "bpg_dev_download": (_i32, [_vp, _u8p, _vp, _sz]),
    "bpg_event_record": (_i32, [_vp, _i32]),
    "bpg_event_elapsed_ms": (_i32, [_vp, _i32, _i32, C.POINTER(C.c_float)]),
    "bpg_prof_enable": (_i32, [_vp, _i32]),
    "bpg_prof_read": (_i32, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "bpg_prof_read_launches": (C.c_long, [_vp, C.POINTER(C.c_float), _u32p, _sz]),
    "bpg_bench_latency": (_i32, [_vp, _i32, C.POINTER(C.c_double)]),
    "bpg_bench_imad": (_i32, [_vp, _i32, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
}

_lib = None


class BpgError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        super().__init__("libbpg error %d%s" % (code, (": " + detail) if detail else ""))


def load():
    """dlopen libbpg.so and attach prototypes; raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libbpg.so not built: run `make -C bulletproofs_gadgets_b200/csrc` (or __graft_entry__.build())")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib
