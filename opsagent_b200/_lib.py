"""ctypes binding of lib/libopsagent_b200.so (the C ABI in include/opsagent_b200.h).

There is NO fallback: if the CUDA library is missing or does not load, importing callers get an
ImportError/OSError — the product never routes through the CPU oracle."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libopsagent_b200.so")

OA_OK, OA_ERR_BAD_REQUEST, OA_ERR_TIMEOUT, OA_ERR_OVERLOADED, OA_ERR_INTERNAL = 0, 400, 408, 429, 500
OA_FLAG_IGNORE_EOS, OA_FLAG_JSON_TOOLCALL, OA_FLAG_JSON_FINAL, OA_FLAG_JSON_FUNCTION, OA_FLAG_JSON_TEXT = 1, 2, 4, 8, 16


class OaMsg(C.Structure):
    _fields_ = [("role", C.c_char_p), ("content", C.c_char_p)]


class OaChatReq(C.Structure):
    _fields_ = [("model", C.c_char_p), ("msgs", C.POINTER(OaMsg)), ("n_msgs", C.c_int32), ("max_tokens", C.c_int32),
                ("temperature", C.c_float), ("seed", C.c_uint64), ("flags", C.c_uint32), ("functions", C.c_char_p)]


class OaChatResp(C.Structure):
    _fields_ = [("content", C.POINTER(C.c_char)), ("content_len", C.c_int32), ("prompt_tokens", C.c_int32),
                ("completion_tokens", C.c_int32), ("finish_reason", C.c_int32), ("token_ids", C.POINTER(C.c_int32))]


# every symbol include/opsagent_b200.h declares (tests/test_abi.py checks the library exports all of them)
SYMBOLS = [
    "oa_engine_create", "oa_engine_destroy", "oa_chat_complete", "oa_chat_submit", "oa_chat_wait", "oa_free_resp",
    "oa_tokens_submit", "oa_count_tokens", "oa_apply_chat_template", "oa_last_error", "oa_engine_stats", "oa_model_info",
    "oa_debug_prefill_logits", "oa_bench_decode", "oa_bench_decode_ex", "oa_k_rmsnorm", "oa_k_gemm", "oa_k_init_weight", "oa_k_paged_attention",
    "oa_kernel_launches", "oa_version", "oa_host_apply_chat_template", "oa_host_decode_plan", "oa_host_streamk_plan", "oa_host_bpe_encode", "oa_host_bpe_decode", "oa_host_model_info",
    "oa_k_gemm_streamk", "oa_debug_kernel_times", "oa_engine_serve", "oa_host_grammar_step", "oa_host_grammar_step_ex", "oa_host_grammar_token_mask", "oa_http_start", "oa_http_port", "oa_http_stats", "oa_http_stop", "oa_http_last_error", "oa_host_json_roundtrip", "oa_chat_cancel", "oa_chat_submit_ex", "oa_chat_wait_ex",
    "oa_k_paged_attention_ex", "oa_k_sk_resid_rmsnorm", "oa_k_sk_swiglu", "oa_k_qkv_rope", "oa_k_lm_head", "oa_host_clusterk_pick",
]

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing — build it first: python -c 'import __graft_entry__ as g; g.build()' "
                          "(opsagent_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, u64, f32 = C.c_void_p, C.c_int32, C.c_uint64, C.c_float
    L.oa_engine_create.argtypes = [C.c_char_p, C.POINTER(vp)]; L.oa_engine_create.restype = C.c_int
    L.oa_engine_destroy.argtypes = [vp]; L.oa_engine_destroy.restype = None
    L.oa_engine_serve.argtypes = [vp]; L.oa_engine_serve.restype = C.c_int
    L.oa_chat_complete.argtypes = [vp, C.POINTER(OaChatReq), C.POINTER(OaChatResp)]; L.oa_chat_complete.restype = C.c_int
    L.oa_chat_submit.argtypes = [vp, C.POINTER(OaChatReq), C.POINTER(u64)]; L.oa_chat_submit.restype = C.c_int
    L.oa_chat_wait.argtypes = [vp, u64, i32, C.POINTER(OaChatResp)]; L.oa_chat_wait.restype = C.c_int
    L.oa_chat_cancel.argtypes = [vp, u64]; L.oa_chat_cancel.restype = C.c_int
    L.oa_chat_submit_ex.argtypes = [vp, C.POINTER(OaChatReq), C.POINTER(u64), C.c_char_p, C.c_size_t]; L.oa_chat_submit_ex.restype = C.c_int
    L.oa_chat_wait_ex.argtypes = [vp, u64, i32, C.POINTER(OaChatResp), C.c_char_p, C.c_size_t]; L.oa_chat_wait_ex.restype = C.c_int
    L.oa_free_resp.argtypes = [C.POINTER(OaChatResp)]; L.oa_free_resp.restype = None
    L.oa_tokens_submit.argtypes = [vp, vp, i32, i32, C.c_uint32, C.POINTER(u64)]; L.oa_tokens_submit.restype = C.c_int
    L.oa_count_tokens.argtypes = [vp, C.POINTER(OaMsg), i32, C.POINTER(i32)]; L.oa_count_tokens.restype = C.c_int
    L.oa_apply_chat_template.argtypes = [vp, C.POINTER(OaMsg), i32, vp, i32, C.POINTER(i32)]; L.oa_apply_chat_template.restype = C.c_int
    L.oa_last_error.restype = C.c_char_p
    L.oa_engine_stats.argtypes = [vp, C.c_char_p, C.c_size_t]; L.oa_engine_stats.restype = C.c_int
    L.oa_model_info.argtypes = [vp, C.c_char_p, C.c_size_t]; L.oa_model_info.restype = C.c_int
    L.oa_debug_prefill_logits.argtypes = [vp, vp, i32, vp]; L.oa_debug_prefill_logits.restype = C.c_int
    L.oa_bench_decode.argtypes = [vp, i32, i32, i32, i32, C.POINTER(C.c_double), i32]; L.oa_bench_decode.restype = C.c_int
    L.oa_bench_decode_ex.argtypes = [vp, i32, i32, i32, i32, C.POINTER(C.c_double), i32, vp, vp]; L.oa_bench_decode_ex.restype = C.c_int
    L.oa_k_rmsnorm.argtypes = [vp, vp, vp, i32, i32, f32, vp]; L.oa_k_rmsnorm.restype = C.c_int
    L.oa_k_gemm.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]; L.oa_k_gemm.restype = C.c_int
    L.oa_k_gemm_streamk.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp]; L.oa_k_gemm_streamk.restype = C.c_int
    L.oa_debug_kernel_times.argtypes = [vp, C.c_char_p, C.c_size_t, i32]; L.oa_debug_kernel_times.restype = C.c_int
    L.oa_k_init_weight.argtypes = [vp, u64, u64, C.c_int64, C.c_int64, C.c_int64, f32, f32, vp]; L.oa_k_init_weight.restype = C.c_int
    L.oa_k_paged_attention.argtypes = [vp, vp, vp, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, vp]; L.oa_k_paged_attention.restype = C.c_int
    L.oa_k_paged_attention_ex.argtypes = [vp, vp, vp, i32, i32, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    L.oa_k_paged_attention_ex.restype = C.c_int
    L.oa_k_sk_resid_rmsnorm.argtypes = [i32, vp, vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, f32, vp, vp]; L.oa_k_sk_resid_rmsnorm.restype = C.c_int
    L.oa_k_sk_swiglu.argtypes = [i32, vp, vp, i32, i32, i32, i32, vp, vp, vp]; L.oa_k_sk_swiglu.restype = C.c_int
    L.oa_k_qkv_rope.argtypes = [i32, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    L.oa_k_qkv_rope.restype = C.c_int
    L.oa_k_lm_head.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, i32, i32, vp, vp, vp]; L.oa_k_lm_head.restype = C.c_int
    L.oa_host_apply_chat_template.argtypes = [C.c_char_p, C.POINTER(OaMsg), i32, vp, i32, C.POINTER(i32)]; L.oa_host_apply_chat_template.restype = C.c_int
    L.oa_host_bpe_encode.argtypes = [C.c_char_p, C.c_char_p, i32, vp, i32, C.POINTER(i32)]; L.oa_host_bpe_encode.restype = C.c_int
    L.oa_host_bpe_decode.argtypes = [C.c_char_p, vp, i32, vp, i32, C.POINTER(i32)]; L.oa_host_bpe_decode.restype = C.c_int
    L.oa_host_streamk_plan.argtypes = [i32, i32, i32, i32, vp, i32, vp, vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]; L.oa_host_streamk_plan.restype = C.c_int
    L.oa_host_clusterk_pick.argtypes = [i32, i32, i32, i32]; L.oa_host_clusterk_pick.restype = i32
    L.oa_host_decode_plan.argtypes = [vp, i32, i32, i32, i32, vp, i32, vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]; L.oa_host_decode_plan.restype = C.c_int
    L.oa_host_grammar_step.argtypes = [i32, vp, i32, vp, C.POINTER(i32)]; L.oa_host_grammar_step.restype = C.c_int
    L.oa_host_grammar_step_ex.argtypes = [i32, C.c_char_p, vp, i32, vp, C.POINTER(i32)]; L.oa_host_grammar_step_ex.restype = C.c_int
    L.oa_host_grammar_token_mask.argtypes = [C.c_char_p, i32, i32, C.c_char_p, vp, i32, vp, i32, C.c_char_p, i32]; L.oa_host_grammar_token_mask.restype = C.c_int
    L.oa_http_start.argtypes = [C.POINTER(vp), i32, C.c_char_p, C.POINTER(vp)]; L.oa_http_start.restype = C.c_int
    L.oa_http_port.argtypes = [vp]; L.oa_http_port.restype = i32
    L.oa_http_stats.argtypes = [vp, C.c_char_p, C.c_size_t]; L.oa_http_stats.restype = C.c_int
    L.oa_http_stop.argtypes = [vp]; L.oa_http_stop.restype = None
    L.oa_http_last_error.restype = C.c_char_p
    L.oa_host_json_roundtrip.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]; L.oa_host_json_roundtrip.restype = C.c_int
    L.oa_host_model_info.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]; L.oa_host_model_info.restype = C.c_int
    L.oa_kernel_launches.restype = u64
    L.oa_version.restype = C.c_char_p
    _lib = L
    return L


def last_error() -> str:
    return (load().oa_last_error() or b"").decode("utf-8", "replace")
