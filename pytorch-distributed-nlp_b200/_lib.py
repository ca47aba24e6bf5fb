"""ctypes binding of libb2ddpbert.so (include/b2_ddp_bert.h).

The library is the product: there is no fallback.  If it is missing or a call fails the host raises
``RuntimeError`` with ``b2_last_error()`` — mirroring how the reference surfaces torch errors.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2ddpbert.so")
ABI_VERSION = 18

MAJOR_K, MAJOR_MN = 0, 1
EPI_NONE, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_DROPOUT_RESIDUAL, EPI_RESIDUAL, EPI_GELU_BWD = 0, 1, 2, 3, 4, 5
EPI_RESIDUAL_F32 = 6
EPI_ACCUM_F32 = 7
ACCUM_ADD, ACCUM_FINISH = 0, 1          # b2_grad_accumulate modes
IPC_HANDLE_BYTES = 64
FLAG_SLOTS = 64

vp, i64, i32, u32, u64, f32, f64 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_uint64, C.c_float, C.c_double


class GemmArgs(C.Structure):
    _fields_ = [
        ("M", i64), ("N", i64), ("K", i64),
        ("A", vp), ("lda", i64), ("a_major", i32),
        ("B", vp), ("ldb", i64), ("b_major", i32),
        ("D", vp), ("ldd", i64), ("epilogue", i32),
        ("bias", vp), ("aux_in", vp), ("ld_aux_in", i64), ("aux_out", vp), ("ld_aux_out", i64),
        ("dropout_p", f32), ("rng_state", vp), ("rng_site", u32),
        ("workspace", vp), ("workspace_bytes", i64), ("force_bn", i32), ("force_splits", i32), ("force_kernel", i32), ("debug_timing", vp), ("colsum_out", vp),
    ]


class AdamWHParams(C.Structure):
    _fields_ = [("lr", f64), ("beta1", f64), ("beta2", f64), ("eps", f64), ("weight_decay", f64),
                ("correct_bias", i32), ("grad_scale", vp), ("found_inf", vp), ("skip_flags", vp)]


class FusedAdamWTarget(C.Structure):
    _fields_ = [("master", vp), ("exp_avg", vp), ("exp_avg_sq", vp), ("shadow", vp), ("decay", i32)]


# name -> argtypes; every function returns int32 status unless listed in _SPECIAL
_SIGNATURES = {
    "b2_gemm_bf16": [C.POINTER(GemmArgs), vp],
    "b2_gemm_bf16_grouped": [C.POINTER(GemmArgs), i32, vp],
    "b2_gemm_bf16_grouped_adamw": [C.POINTER(GemmArgs), C.POINTER(FusedAdamWTarget), i32, C.POINTER(AdamWHParams), vp,
                                   vp],
    "b2_gemm_ln_fwd": [C.POINTER(GemmArgs), vp, vp, f32, vp, i64, vp, i64, vp, vp, vp],
    "b2_embed_fwd": [vp, vp, i64, i64, vp, vp, vp, vp, vp, i64, i64, i64, f32, f32, vp, u32, vp, vp, vp, vp, vp, vp,
                     vp, vp],
    "b2_embed_owner_init": [vp, i64, vp],
    "b2_embed_bwd": [vp, i32, vp, vp, vp, vp, vp, vp, i64, i64, i64, i64, i64, i64, f32, vp, u32, vp, vp, vp, vp, vp, vp, vp,
                     i64, vp, vp],
    "b2_layernorm_fwd": [vp, vp, vp, i64, i64, f32, vp, vp, vp, vp],
    "b2_layernorm_bwd": [vp, vp, vp, vp, vp, vp, i64, i64, f32, vp, u32, i32, vp, vp, vp, vp, vp, vp, i64, vp, vp],
    "b2_layernorm_bwd_accum": [vp, vp, vp, vp, vp, i64, i64, f32, vp, u32, vp, vp, vp, vp],
    "b2_colsum_finish": [vp, i32, i32, i64, vp, vp, vp, vp],
    "b2_colsum": [vp, i64, i64, i64, vp, vp, i64, vp],
    "b2_attention_fwd": [vp, vp, i64, i64, i64, i64, f32, vp, u32, vp, vp, vp, vp],
    "b2_attention_bwd": [vp, vp, vp, vp, vp, i64, i64, i64, i64, f32, vp, u32, vp, vp, vp, vp, vp],
    "b2_accum_finish": [vp, vp, vp, i64, i64, vp],
    "b2_head_fwd": [vp, i64, i64, i64, vp, vp, vp, vp, i64, f32, vp, u32, vp, vp, vp],
    "b2_ce_fwd_bwd": [vp, vp, i64, i64, vp, vp, vp],
    "b2_head_bwd": [vp, vp, vp, i64, i64, i64, vp, vp, i64, f32, vp, u32, vp, vp, vp, vp, vp, i32, vp, vp],
    # packed-bin variants (include/b2_ddp_bert.h, "packed bins")
    "b2_embed_fwd_packed": [vp, vp, vp, i64, i64, i64, vp, vp, vp, vp, vp, i64, i64, i64, f32, f32, vp, u32, vp, vp, vp,
                            vp, vp, vp, vp, vp, vp],
    "b2_embed_bwd_packed": [vp, i32, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, i64, i64, i64, f32, vp, u32, vp, vp, vp,
                            vp, vp, vp, vp, i64, vp, vp],
    "b2_attention_fwd_packed": [vp, vp, i64, i64, i64, f32, vp, u32, vp, vp, vp, vp],
    "b2_attention_bwd_packed": [vp, vp, vp, vp, vp, i64, i64, i64, f32, vp, u32, vp, vp, vp, vp],
    "b2_head_fwd_packed": [vp, vp, i64, i64, vp, vp, vp, vp, i64, f32, vp, u32, vp, vp, vp],
    "b2_head_bwd_packed": [vp, vp, vp, vp, i64, i64, i64, vp, vp, i64, f32, vp, u32, vp, vp, vp, vp, vp, i32, vp, vp],
    "b2_head_bwd_split": [vp, vp, vp, vp, i64, i64, i64, i64, vp, vp, i64, f32, vp, u32, vp, vp, vp, vp, vp, i32, vp, vp,
                          vp],
    "b2_bucket_reduce_adamw": [C.POINTER(vp), C.POINTER(vp), i32, i32, vp, vp, vp, vp, i64, i64,
                               C.POINTER(AdamWHParams), vp, vp],
    "b2_adamw_prepare": [C.POINTER(AdamWHParams), vp, vp, vp],
    "b2_adamw_background": [vp, vp, vp, vp, vp, vp, i64, i64, C.POINTER(AdamWHParams), vp, vp],
    "b2_grad_accumulate": [vp, vp, i64, i64, f32, i32, vp],
    "b2_step_advance": [vp, vp, vp, vp],
    "b2_rng_seed": [vp, u64, u64, vp],
    "b2_cast_f32_to_bf16": [vp, vp, i64, vp],
    "b2_cast_bf16_to_f32": [vp, vp, i64, vp],
    "b2_zero": [vp, i64, vp],
    "b2_copy_async": [vp, vp, i64, vp],
    "b2_comm_alloc": [i64, C.POINTER(vp)],
    "b2_comm_free": [vp],
    "b2_comm_export": [vp, C.c_char_p],
    "b2_comm_import": [C.c_char_p, C.POINTER(vp)],
    "b2_comm_unimport": [vp],
    "b2_peer_barrier": [C.POINTER(vp), i32, i32, i32, vp, vp],
    "b2_allgather_rows": [vp, i64, C.POINTER(vp), C.POINTER(vp), i32, i32, i32, vp, vp],
    "b2_scalar_allreduce_mean": [vp, vp, C.POINTER(vp), C.POINTER(vp), i32, i32, i32, vp, vp],
}
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + ["b2_last_error", "b2_abi_version", "b2_launch_count",
                                              "b2_gemm_ln_max_clusters"])

_lib = None


def load():
    """Loads the shared library once.  Raises RuntimeError (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libb2ddpbert.so is not built (%s). Run `python __graft_entry__.py` (nvcc, sm_100a). "
            "There is no CPU or PyTorch fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.b2_last_error.restype = C.c_char_p
    lib.b2_last_error.argtypes = []
    lib.b2_abi_version.restype = i32
    lib.b2_abi_version.argtypes = []
    lib.b2_launch_count.restype = i64
    lib.b2_launch_count.argtypes = []
    lib.b2_gemm_ln_max_clusters.restype = i32     # a count, not a status
    lib.b2_gemm_ln_max_clusters.argtypes = [i64]
    if lib.b2_abi_version() != ABI_VERSION:
        raise RuntimeError("libb2ddpbert.so ABI %d != expected %d: rebuild" % (lib.b2_abi_version(), ABI_VERSION))
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = i32
        fn.argtypes = argtypes
    _lib = lib
    return lib


def launch_count():
    return int(load().b2_launch_count())


def last_error():
    return load().b2_last_error().decode("utf-8", "replace")


def check(status, what=""):
    if status != 0:
        raise RuntimeError("b2 %s failed (%d): %s" % (what, status, last_error()))


def call(name, *args):
    """Calls an entry point and converts a non-zero status into RuntimeError (SURVEY.md §8b error convention)."""
    fn = getattr(load(), name)
    check(fn(*args), name)


def ptr(t):
    """Device (or host) address of a torch tensor, or None."""
    return None if t is None else t.data_ptr()


def ptr_array(addresses):
    arr = (vp * len(addresses))()
    for i, a in enumerate(addresses):
        arr[i] = a
    return arr
