"""ctypes binding of include/kserve_b200.h.  There is NO fallback: if the CUDA library is missing or
fails to load, importing the product path raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200_LIB_PATH") or os.path.join(HERE, "lib", "libkserve_b200.so")   # (override: A/B of two builds on one box)


class ModelConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "vocab_size", "hidden_size", "intermediate_size", "num_layers", "num_heads", "num_kv_heads",
        "head_dim", "max_position")] + [("rms_eps", C.c_float), ("rope_theta", C.c_float)] + [
        (n, C.c_int32) for n in ("max_batch", "max_seq_len", "max_prefill_tokens", "num_kv_pages",
                                 "tp_rank", "tp_size", "device", "num_experts", "num_experts_per_tok")]


class GenParams(C.Structure):
    _fields_ = [("max_new_tokens", C.c_int32), ("pad_token_id", C.c_int64),
                ("eos_token_ids", C.POINTER(C.c_int64)), ("num_eos", C.c_int32),
                ("stop_tokens", C.POINTER(C.c_int64)), ("stop_offsets", C.POINTER(C.c_int32)),
                ("num_stop", C.c_int32), ("forced_tokens", C.POINTER(C.c_int64)),
                ("repetition_penalty", C.c_float), ("do_sample", C.c_int32), ("temperature", C.c_float),
                ("top_p", C.c_float), ("top_k", C.c_int32), ("seed", C.c_uint64)]


class Timing(C.Structure):
    _fields_ = [("prefill_ms", C.c_float), ("decode_ms", C.c_float), ("decode_steps", C.c_int32),
                ("kernel_launches", C.c_int32)]


TOKEN_CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.c_int32)

_lib = None


class B200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(f"{LIB_PATH} is missing: run `python -m kserve_b200.build` "
                        "(kserve_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.b200_last_error.restype = C.c_char_p
    lib.b200_version.restype = C.c_char_p
    lib.b200_engine_create.argtypes = [C.POINTER(ModelConfig), vp, C.POINTER(vp)]
    lib.b200_engine_destroy.argtypes = [vp]
    lib.b200_nccl_unique_id.argtypes = [vp]
    lib.b200_engine_set_weight.argtypes = [vp, C.c_char_p, vp, C.c_int, C.c_int, C.POINTER(i64)]
    lib.b200_engine_finalize_weights.argtypes = [vp]
    lib.b200_engine_set_rope_table.argtypes = [vp, vp, vp, i32]
    lib.b200_generate.argtypes = [vp, vp, vp, i32, i32, C.POINTER(GenParams), vp, C.POINTER(i32),
                                  C.POINTER(i32), vp, TOKEN_CALLBACK, vp]
    lib.b200_engine_last_timing.argtypes = [vp, C.POINTER(Timing)]
    lib.b200_engine_fault.argtypes = [vp, C.POINTER(i32), i32]
    lib.b200_stage_prompt.argtypes = [vp, vp, vp, i32, i32, C.POINTER(GenParams)]
    lib.b200_run_staged.argtypes = [vp, i32, i32]
    lib.b200_run_staged_timed.argtypes = [vp, i32, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.b200_fetch_staged.argtypes = [vp, vp, C.POINTER(i32), C.POINTER(i32)]
    lib.b200_op_gemm.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, i64, vp]
    lib.b200_op_rmsnorm.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_float, vp, C.c_int, vp, vp]
    lib.b200_op_attn_prefill_tc.argtypes = [vp, i64, C.c_int, vp, i64, vp, vp, C.c_int, vp, C.c_int, vp, vp, C.c_int, C.c_int,
                                            C.c_int, C.c_int, vp]
    lib.b200_op_attn_decode.argtypes = [vp, i64, vp, i64, vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int,
                                        C.c_int, C.c_int, vp, vp, vp]
    lib.b200_op_rope_kv.argtypes = [vp, i64, vp, i64, vp, vp, vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int,
                                    C.c_int, vp]
    lib.b200_op_argmax.argtypes = [vp, i64, C.c_int, C.c_int, vp, vp, vp]
    lib.b200_batch_predict.argtypes = [vp, vp, vp, i32, C.POINTER(GenParams), vp, C.POINTER(i32), C.POINTER(i32)]
    lib.b200_batcher_create.argtypes = [i32, i32, C.POINTER(vp)]
    lib.b200_batcher_destroy.argtypes = [vp]
    lib.b200_batcher_config.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    lib.b200_batcher_add.argtypes = [vp, i64, i32, C.POINTER(i64)]
    lib.b200_batcher_tick.argtypes = [vp, i64, i32, vp, vp, vp, C.POINTER(i32), C.POINTER(i32)]
    lib.b200_engine_ipc_export.argtypes = [vp, vp]
    lib.b200_engine_ipc_import.argtypes = [vp, vp, i32]
    lib.b200_kv_swap_out.argtypes = [vp, i32, i32]
    lib.b200_kv_swap_in.argtypes = [vp, i32]
    lib.b200_cb_begin.argtypes = [vp, C.c_int64, C.POINTER(C.c_int64), i32]
    lib.b200_cb_admit.argtypes = [vp, i32, C.POINTER(C.POINTER(C.c_int64)), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32),
                                  C.POINTER(i32), C.POINTER(C.c_int64), C.POINTER(GenParams), C.POINTER(i32)]
    lib.b200_cb_config.argtypes = [vp, i32, i32]
    lib.b200_cb_swap_out.argtypes = [vp, i32]
    lib.b200_cb_swap_in.argtypes = [vp, i32]
    lib.b200_cb_stats.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.b200_cb_step.argtypes = [vp, i32]
    lib.b200_cb_poll.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    lib.b200_cb_read.argtypes = [vp, i32, i32, C.POINTER(C.c_int64), i32, C.POINTER(i32)]
    lib.b200_cb_release.argtypes = [vp, i32]
    lib.b200_cb_end.argtypes = [vp]
    lib.b200_debug_trace.argtypes = [i32]
    lib.b200_debug_trace_read.argtypes = [vp, i32, C.POINTER(i32)]
    _lib = lib
    return lib


class EngineFault(B200Error):
    """rc -8: a device-side wait timed out (tensor-parallel peer lost); the engine must be re-created"""


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().b200_last_error().decode("utf-8", "replace")
        raise (EngineFault if rc == -8 else B200Error)(f"{what} failed (rc={rc}): {msg}")
