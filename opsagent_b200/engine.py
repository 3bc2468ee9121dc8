"""Engine — thin object wrapper over the C ABI (one process-global engine per GPU)."""
from __future__ import annotations

import ctypes as C
import json
from typing import Sequence

from . import _lib


class EngineError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[{code}] {message}")
        self.code, self.message = code, message


def _check(rc: int):
    if rc != _lib.OA_OK:
        raise EngineError(rc, _lib.last_error())


def _msgs(messages) -> tuple:
    arr = (_lib.OaMsg * len(messages))()
    keep = []
    for i, (role, content) in enumerate(messages):
        r = role.encode("utf-8") if isinstance(role, str) else role
        c = content.encode("utf-8") if isinstance(content, str) else content
        keep += [r, c]
        arr[i].role, arr[i].content = r, c
    return arr, keep


class Completion:
    __slots__ = ("content", "token_ids", "prompt_tokens", "completion_tokens", "finish_reason")

    def __init__(self, resp: "_lib.OaChatResp"):
        self.content = C.string_at(resp.content, resp.content_len) if resp.content_len > 0 else b""
        self.token_ids = [resp.token_ids[i] for i in range(resp.completion_tokens)]
        self.prompt_tokens, self.completion_tokens = resp.prompt_tokens, resp.completion_tokens
        self.finish_reason = "stop" if resp.finish_reason == 0 else "length"


class Engine:
    def __init__(self, config: dict | str):
        self._L = _lib.load()
        cfg = config if isinstance(config, str) else json.dumps(config)
        h = C.c_void_p()
        _check(self._L.oa_engine_create(cfg.encode(), C.byref(h)))
        self._h = h
        self.info = json.loads(self._json(self._L.oa_model_info))

    def close(self):
        if getattr(self, "_h", None):
            self._L.oa_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _json(self, fn) -> str:
        buf = C.create_string_buffer(4096)
        _check(fn(self._h, buf, 4096))
        return buf.value.decode()

    def serve(self):
        """tensor-parallel follower: replay the leader's steps until it shuts the group down"""
        _check(self._L.oa_engine_serve(self._h))

    def stats(self) -> dict:
        return json.loads(self._json(self._L.oa_engine_stats))

    # ---- chat path (what LocalCUDAClient.Chat uses) ----
    def _req(self, model, messages, max_tokens, flags, functions=None):
        arr, keep = _msgs(messages)
        m = model.encode() if model else None
        f = functions.encode() if functions else None
        req = _lib.OaChatReq(m, arr, len(messages), max_tokens, 1.401298464324817e-45, 0, flags, f)
        return req, (arr, keep, m, f)

    def chat_submit(self, model: str, messages, max_tokens: int, flags: int = 0) -> int:
        req, _keep = self._req(model, messages, max_tokens, flags)
        t = C.c_uint64()
        _check(self._L.oa_chat_submit(self._h, C.byref(req), C.byref(t)))
        return t.value

    def wait(self, ticket: int, timeout_ms: int = -1) -> Completion:
        resp = _lib.OaChatResp()
        _check(self._L.oa_chat_wait(self._h, ticket, timeout_ms, C.byref(resp)))
        try:
            return Completion(resp)
        finally:
            self._L.oa_free_resp(C.byref(resp))

    def cancel(self, ticket: int) -> None:
        """abandon a submitted request (frees its KV pages at the next step boundary); waiting on the ticket afterwards is an error"""
        _check(self._L.oa_chat_cancel(self._h, ticket))

    def chat_complete(self, model: str, messages, max_tokens: int, flags: int = 0, functions: str | None = None) -> Completion:
        req, _keep = self._req(model, messages, max_tokens, flags, functions)
        resp = _lib.OaChatResp()
        _check(self._L.oa_chat_complete(self._h, C.byref(req), C.byref(resp)))
        try:
            return Completion(resp)
        finally:
            self._L.oa_free_resp(C.byref(resp))

    # ---- raw-token path (bench + parity) ----
    def tokens_submit(self, prompt: Sequence[int], max_tokens: int, flags: int = 0) -> int:
        arr = (C.c_int32 * len(prompt))(*prompt)
        t = C.c_uint64()
        _check(self._L.oa_tokens_submit(self._h, arr, len(prompt), max_tokens, flags, C.byref(t)))
        return t.value

    def generate(self, prompt: Sequence[int], max_tokens: int, flags: int = 0) -> Completion:
        return self.wait(self.tokens_submit(prompt, max_tokens, flags))

    def apply_chat_template(self, messages) -> list[int]:
        arr, _keep = _msgs(messages)
        n = C.c_int32()
        _check(self._L.oa_apply_chat_template(self._h, arr, len(messages), None, 0, C.byref(n)))
        out = (C.c_int32 * n.value)()
        _check(self._L.oa_apply_chat_template(self._h, arr, len(messages), out, n.value, C.byref(n)))
        return list(out)

    def count_tokens(self, messages) -> int:
        arr, _keep = _msgs(messages)
        n = C.c_int32()
        _check(self._L.oa_count_tokens(self._h, arr, len(messages), C.byref(n)))
        return n.value

    def debug_prefill_logits(self, tokens: Sequence[int]):
        import numpy as np
        toks = np.ascontiguousarray(tokens, dtype=np.int32)
        out = np.empty((len(toks), self.info["vocab"]), dtype=np.float32)
        _check(self._L.oa_debug_prefill_logits(self._h, toks.ctypes.data, len(toks), out.ctypes.data))
        return out

    def kernel_times(self, reset: bool = True) -> dict:
        buf = C.create_string_buffer(4096)
        _check(self._L.oa_debug_kernel_times(self._h, buf, 4096, int(reset)))
        return json.loads(buf.value.decode())

    def bench_decode(self, batch: int, ctx_len: int, steps: int, warmup: int, last_outputs: bool = False) -> dict:
        """last_outputs: also return what the last timed step computed, "last_ids" (int32 [batch]) and "last_logits" (fp32 [batch, vocab])"""
        import numpy as np
        out = (C.c_double * 8)()
        ids = np.zeros(batch, np.int32) if last_outputs else None
        logits = np.zeros((batch, self.info["vocab"]), np.float32) if last_outputs else None
        _check(self._L.oa_bench_decode_ex(self._h, batch, ctx_len, steps, warmup, out, 8, None if ids is None else ids.ctypes.data,
                                          None if logits is None else logits.ctypes.data))
        r = {"ms_per_step": out[0], "prefill_ms": out[1], "launches_per_step": out[2], "mean_ctx": out[3],
             "attn_ms_per_step": out[4], "algorithmic_bytes_per_step": out[5], "device_ms_per_step": out[6]}
        if last_outputs:
            r["last_ids"], r["last_logits"] = ids, logits
        return r
