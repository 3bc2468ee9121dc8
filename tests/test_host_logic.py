"""Host-side logic on the CPU: chat template/tokenizer (C++ vs the oracle's Python restatement), decode work plan
invariants, model presets, Chat() retry semantics of the Python mirror (reference pkg/llms/openai.go:69-104)."""
import ctypes as C
import json

import numpy as np
import pytest

from opsagent_b200 import _lib
from opsagent_b200.llms import LocalCUDAClient, APIError, ChatCompletionMessage, new_client
from opsagent_b200.dp import shard_requests, replica_of
from oracle import oracle as O


def host_template(spec, msgs):
    L = _lib.load()
    arr = (_lib.OaMsg * len(msgs))()
    keep = []
    for i, (r, c) in enumerate(msgs):
        rb, cb = r.encode(), c.encode(); keep += [rb, cb]
        arr[i].role, arr[i].content = rb, cb
    n = C.c_int32()
    cfg = json.dumps(spec.engine_json()).encode()
    assert L.oa_host_apply_chat_template(cfg, arr, len(msgs), None, 0, C.byref(n)) == 0
    out = (C.c_int32 * n.value)()
    assert L.oa_host_apply_chat_template(cfg, arr, len(msgs), out, n.value, C.byref(n)) == 0
    return list(out)


# the ReAct loop's message shapes: system+user seeds (pkg/handlers/execute.go:190-199), then assistant JSON +
# user observation JSON per iteration (pkg/assistants/simple.go:358,496-501)
CONVS = [
    [("system", "你是Kubernetes和云原生网络的技术专家"), ("user", "how many namespace in the cluster?")],
    [("system", "sys"), ("user", "q"), ("assistant", '{"question":"q","thought":"t","action":{"name":"kubectl","input":"get ns"}}'),
     ("user", '{"question":"q","observation":"default\\nkube-system"}')],
    [("user", "")],
]


@pytest.mark.parametrize("name", ["llama-3-8b", "llama-3.2-1b", "qwen2.5-32b", "llama-3-70b", "tiny-llama", "tiny-qwen"])
@pytest.mark.parametrize("conv", CONVS)
def test_chat_template_matches_restatement(name, conv):
    spec = O.PRESETS[name]
    ids = host_template(spec, conv)
    assert ids == O.apply_chat_template(spec, conv)
    assert all(0 <= t < spec.vocab for t in ids)


def test_real_special_token_ids():
    ids = host_template(O.PRESETS["llama-3-8b"], [("user", "hi")])
    assert ids[0] == 128000 and ids[1] == 128006 and 128007 in ids and 128009 in ids
    ids = host_template(O.PRESETS["qwen2.5-32b"], [("user", "hi")])
    assert ids[0] == 151644 and 151645 in ids


@pytest.mark.parametrize("name", ["llama-3.2-1b", "llama-3-8b", "qwen2.5-32b", "llama-3-70b"])
def test_presets_agree_with_survey_table(name):
    """SURVEY.md §8d model constants: W_dec GB and KV bytes/token"""
    L = _lib.load()
    buf = C.create_string_buffer(2048)
    assert L.oa_host_model_info(json.dumps({"model": name}).encode(), buf, 2048) == 0
    info = json.loads(buf.value)
    spec = O.PRESETS[name]
    for k in ("hidden", "n_layers", "n_heads", "n_kv_heads", "head_dim", "ffn", "vocab", "tie_embeddings", "qkv_bias", "rope_scaling"):
        assert info[k] == getattr(spec, k), k
    expect = {"llama-3.2-1b": (2.472, 32768), "llama-3-8b": (15.010, 131072), "qwen2.5-32b": (63.971, 262144), "llama-3-70b": (139.006, 327680)}[name]
    assert abs(info["decode_weight_bytes"] / 1e9 - expect[0]) < 0.02
    assert info["kv_bytes_per_token"] == expect[1]


def test_bad_configs_are_rejected():
    L = _lib.load()
    buf = C.create_string_buffer(512)
    assert L.oa_host_model_info(b'{"model": "gpt-4"}', buf, 512) == 400
    assert L.oa_host_model_info(b'{"model": "x", "hidden": 256, "n_layers": 1, "n_heads": 4, "n_kv_heads": 4, "head_dim": 32, "ffn": 512, "vocab": 1024}', buf, 512) == 400
    assert L.oa_host_model_info(b'not json', buf, 512) == 400


def plan(ctx, n_kv, n_ctas, force=0):
    L = _lib.load()
    ctx = np.ascontiguousarray(ctx, np.int32)
    cap = len(ctx) * n_kv * 64 + n_ctas + 64
    segs = np.zeros((cap, 5), np.int32); ptr = np.zeros(cap + 1, np.int32)
    nc, ns, nsl = C.c_int32(), C.c_int32(), C.c_int32()
    assert L.oa_host_decode_plan(ctx.ctypes.data, len(ctx), n_kv, n_ctas, force, segs.ctypes.data, cap, ptr.ctypes.data, cap,
                                 C.byref(nc), C.byref(ns), C.byref(nsl)) == 0
    return segs[:ns.value], ptr[:nc.value + 1], nsl.value


@pytest.mark.parametrize("ctx,n_kv,n_ctas,force", [
    ([1664] * 128, 8, 296, 0), ([1, 63, 64, 65, 200, 1000, 129, 517], 2, 296, 0), ([5], 1, 296, 0), ([16896] * 64, 1, 296, 0),
    ([100, 3000, 7, 64 * 40], 8, 7, 0), ([1, 63, 64, 65, 200, 1000], 2, 296, 3), (list(range(1, 300, 7)), 4, 296, 0)])
def test_decode_plan_covers_every_page_exactly_once_and_is_balanced(ctx, n_kv, n_ctas, force):
    segs, ptr, n_slots = plan(ctx, n_kv, n_ctas, force)
    assert ptr[0] == 0 and ptr[-1] == len(segs) and (np.diff(ptr) >= 0).all()
    cover = {}
    for s, h, b, e, slot in segs:
        assert 0 <= b < e
        for c in range(b, e):
            assert (s, h, c) not in cover
            cover[(s, h, c)] = slot
    for s, c in enumerate(ctx):
        for h in range(n_kv):
            for ch in range((c + 63) // 64):
                assert (s, h, ch) in cover
    assert len(cover) == sum((c + 63) // 64 for c in ctx) * n_kv
    # partial slots: unique, dense, and only for items cut into several pieces
    slots = [x for x in segs[:, 4] if x >= 0]
    assert sorted(slots) == list(range(n_slots))
    pieces = {}
    for s, h, b, e, slot in segs:
        pieces.setdefault((s, h), []).append(slot)
    for k, v in pieces.items():
        assert (len(v) == 1 and v[0] == -1) or (len(v) > 1 and all(x >= 0 for x in v) and sorted(v) == list(range(min(v), min(v) + len(v))))
    if not force:
        load = [sum(segs[i][3] - segs[i][2] for i in range(ptr[c], ptr[c + 1])) for c in range(len(ptr) - 1)]
        assert max(load) - min(load[:-1] or load) <= 1 or max(load) <= -(-len(cover) // len(load))


def test_empty_and_zero_length_plans():
    segs, ptr, n_slots = plan([0, 0], 4, 296)
    assert len(segs) == 0 and n_slots == 0


# ---- Chat() retry semantics of the Python mirror (reference pkg/llms/openai.go:77-103) ----
class FakeEngine:
    def __init__(self, codes):
        self.codes, self.calls = list(codes), 0

    def chat_complete(self, model, msgs, max_tokens, flags=0):
        from opsagent_b200.engine import EngineError
        self.calls += 1
        c = self.codes.pop(0)
        if c:
            raise EngineError(c, f"status {c}")

        class R:
            content = b'{"question":"q","thought":"t","action":{"name":"kubectl","input":"get ns"},"observation":"","final_answer":""}'
        return R()


def test_chat_retries_429_and_500_with_doubling_backoff():
    sleeps = []
    eng = FakeEngine([429, 500, 429, 0])
    cli = LocalCUDAClient(eng, sleep=sleeps.append)
    out = cli.Chat("m", 8192, [ChatCompletionMessage("user", "x")])
    assert json.loads(out)["action"]["name"] == "kubectl"
    assert sleeps == [1.0, 2.0, 4.0] and eng.calls == 4


def test_chat_gives_up_after_five_tries():
    sleeps = []
    cli = LocalCUDAClient(FakeEngine([500] * 5), sleep=sleeps.append)
    with pytest.raises(RuntimeError, match="OpenAI request throttled after retrying 5 times"):
        cli.Chat("m", 10, [ChatCompletionMessage("user", "x")])
    assert sleeps == [1.0, 2.0, 4.0, 8.0, 16.0]


@pytest.mark.parametrize("code", [401, 400, 404])
def test_chat_fails_fast_on_other_statuses(code):
    sleeps = []
    eng = FakeEngine([code])
    with pytest.raises(APIError) as e:
        LocalCUDAClient(eng, sleep=sleeps.append).Chat("m", 10, [ChatCompletionMessage("user", "x")])
    assert e.value.HTTPStatusCode == code and sleeps == [] and eng.calls == 1


def test_new_client_requires_api_key_like_the_reference():
    with pytest.raises(ValueError, match="OPENAI_API_KEY is not set"):
        new_client("", "cuda://llama-3-8b")
    with pytest.raises(ValueError):
        new_client("sk-x", "https://api.openai.com/v1")


def test_request_sharding_is_a_partition():
    for n, w in [(1024, 8), (10, 3), (5, 8), (128, 1)]:
        seen = []
        for r in range(w):
            sh = shard_requests(n, r, w)
            seen += list(sh)
            for i in sh:
                assert replica_of(i, n, w) == r
        assert seen == list(range(n))


# ---- ToolPrompt grammar: C++ automaton (csrc/grammar.hpp) vs the oracle-side restatement ----
def _cpp_mask(kind, prefix: bytes):
    L = _lib.load()
    buf = (C.c_uint8 * max(1, len(prefix)))(*prefix)
    mask = (C.c_uint32 * 8)(); done = C.c_int32()
    rc = L.oa_host_grammar_step(kind, buf, len(prefix), mask, C.byref(done))
    return rc, list(mask), done.value


@pytest.mark.parametrize("kind", [O.GRAMMAR_TOOLCALL, O.GRAMMAR_FINAL])
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_grammar_random_walks_agree_and_yield_toolprompt_json(kind, seed):
    rng = np.random.default_rng(seed)
    g = O.ToolPromptGrammar(kind)
    out = bytearray()
    while not g.done():
        rc, mask, done = _cpp_mask(kind, bytes(out))
        assert rc == 0 and not done and mask == g.mask_words()
        allowed = sorted(g.allowed())
        # bias towards closing strings now and then so walks terminate at varied lengths
        b = 0x22 if (0x22 in allowed and rng.random() < 0.15) else int(rng.choice(allowed))
        out.append(b); assert g.advance(b)
    rc, mask, done = _cpp_mask(kind, bytes(out))
    assert rc == 0 and done == 1 and mask == [0] * 8
    doc = json.loads(out.decode("ascii"))
    # exactly the ToolPrompt fields (reference pkg/tools/tool.go:29-38)
    assert list(doc.keys()) == ["question", "thought", "action", "observation", "final_answer"]
    assert list(doc["action"].keys()) == ["name", "input"] and doc["observation"] == ""
    if kind == O.GRAMMAR_TOOLCALL:
        assert doc["action"]["name"] in O.TOOLS and doc["action"]["input"] and doc["final_answer"] == ""
    else:
        assert doc["action"] == {"name": "", "input": ""} and len(doc["final_answer"]) >= 10   # not a placeholder (simple.go:640-654)


def test_function_call_and_text_grammars():
    L = _lib.load()
    fns = "kubectl:command,trivy:image,python:code"
    rng = np.random.default_rng(5)
    for kind in (O.GRAMMAR_FUNCTION, O.GRAMMAR_TEXT):
        g = O.ToolPromptGrammar(kind, fns)
        out = bytearray()
        while not g.done():
            buf = (C.c_uint8 * max(1, len(out)))(*out); mask = (C.c_uint32 * 8)(); done = C.c_int32()
            assert L.oa_host_grammar_step_ex(kind, fns.encode(), buf, len(out), mask, C.byref(done)) == 0 and list(mask) == g.mask_words()
            allowed = sorted(g.allowed())
            b = g.close if (g.close in allowed and rng.random() < 0.2) else int(rng.choice(allowed))
            out.append(b); assert g.advance(b)
        if kind == O.GRAMMAR_FUNCTION:
            doc = json.loads(out.decode("ascii"))
            assert doc["name"] in ("kubectl", "trivy", "python")
            assert list(doc["arguments"].keys()) == [{"kubectl": "command", "trivy": "image", "python": "code"}[doc["name"]]]
        else:
            assert out.endswith(b"\n") and 10 <= len(out) - 1 <= 200
    mask = (C.c_uint32 * 8)(); done = C.c_int32()
    assert L.oa_host_grammar_step_ex(O.GRAMMAR_FUNCTION, b"", (C.c_uint8 * 1)(), 0, mask, C.byref(done)) == 400     # no functions offered


def test_grammar_rejects_bytes_outside_the_schema():
    assert _cpp_mask(1, b"[")[0] == 400
    assert _cpp_mask(1, b'{"question":"a","thought":"b","action":{"name":"rm')[0] == 400        # not in the tool registry
    assert _cpp_mask(2, b'{"question":"')[0] == 0
    assert _cpp_mask(7, b"")[0] == 400


# ---- ConstrictPrompt / ReAct loop / HTTP front (host mirrors of the callers either side of the seam) ----
from opsagent_b200.llms import ConstrictPrompt                       # noqa: E402
from opsagent_b200.assistants import AssistantWithConfig, ToolPrompt, isTemplateValue   # noqa: E402


def _cl100k_like(messages):
    """Token counts cl100k_base gives for the reference's own test strings (tokens_test.go:64-90): one token per word /
    punctuation mark / newline, plus 3 per message and 3 for the reply priming (tokens.go:96-106)."""
    import re
    n = 3
    for _role, content in messages:
        n += 3 + len(re.findall(r"\w+|[^\w\s]|\n", content))
    return n


@pytest.mark.parametrize("prompt,limit,want", [
    ("This is a test prompt.", 512, "This is a test prompt."),                       # tokens_test.go:64-72
    ("This is a test prompt.", 1, ""),                                               # tokens_test.go:73-81
    ("This is a test prompt.\nhere is another.", 15, "here is another."),            # tokens_test.go:82-90
])
def test_constrict_prompt_reproduces_the_reference_golden_cases(prompt, limit, want):
    assert ConstrictPrompt(prompt, "gpt-3.5-turbo-0613", limit, _cl100k_like) == want


def test_constrict_prompt_is_a_noop_without_a_tokenizer_like_the_reference():
    # tokens.go:61-66: unknown model -> count 0 -> nothing is ever dropped
    long = "\n".join(f"line {i}" for i in range(5000))
    assert ConstrictPrompt(long, "llama-3-8b", 1024, None) == long


class ScriptedClient:
    def __init__(self, replies):
        self.replies, self.calls = list(replies), []

    def Chat(self, model, maxTokens, prompts):
        self.calls.append([(m.Role, m.Content) for m in prompts])
        return self.replies.pop(0)


def test_react_loop_runs_tools_and_returns_final_answer():
    step = ToolPrompt("q", "need pods", {"name": "kubectl", "input": "get pods"}, "", "").marshal()
    final = ToolPrompt("q", "done", {"name": "", "input": ""}, "", "There are 3 crashing pods in ns-1").marshal()
    cli = ScriptedClient([step, step, final])
    seen = []
    res, hist = AssistantWithConfig("m", [ChatCompletionMessage("system", "s"), ChatCompletionMessage("user", "q")], 2048, True, False, 5, cli,
                                    {"kubectl": lambda i: seen.append(i) or " pod-a Running \n"})
    assert res == "There are 3 crashing pods in ns-1" and seen == ["get pods", "get pods"] and len(cli.calls) == 3
    # the observation goes back as a USER message holding the whole ToolPrompt (simple.go:496-501)
    assert hist[3].Role == "user" and json.loads(hist[3].Content)["observation"] == "pod-a Running"
    assert [m.Role for m in hist] == ["system", "user", "assistant", "user", "assistant", "user", "assistant"]


def test_react_loop_edge_cases_follow_the_reference():
    msgs = [ChatCompletionMessage("user", "q")]
    # non-JSON first reply is returned verbatim (simple.go:367-382)
    assert AssistantWithConfig("m", msgs, 10, False, False, 5, ScriptedClient(["plain text"]), {})[0] == "plain text"
    # unknown tool / failing tool become observation text (simple.go:455,481)
    bad = ToolPrompt("q", "t", {"name": "helm", "input": "x"}).marshal()
    fin = ToolPrompt("q", "t", {"name": "", "input": ""}, "", "a final answer long enough").marshal()
    cli = ScriptedClient([bad, fin])
    AssistantWithConfig("m", msgs, 10, False, False, 5, cli, {})
    assert "Tool helm is not available. Considering switch to other supported tools." in cli.calls[1][-1][1]

    def boom(_):
        raise RuntimeError("exit status 1")
    cli = ScriptedClient([ToolPrompt("q", "t", {"name": "kubectl", "input": "x"}).marshal(), fin])
    AssistantWithConfig("m", msgs, 10, False, False, 5, cli, {"kubectl": boom})
    assert "Tool kubectl failed with error" in cli.calls[1][-1][1]
    # unparsable intermediate reply -> one more "Summarize…" Chat (simple.go:558-566)
    cli = ScriptedClient([ToolPrompt("q", "t", {"name": "kubectl", "input": "x"}).marshal(), "oops", "summary"])
    res, hist = AssistantWithConfig("m", msgs, 10, False, False, 5, cli, {"kubectl": lambda i: "ok"})
    assert res == "summary" and hist[-1].Content.startswith("Summarize all the chat history")
    # iteration cap returns whatever final_answer holds, even empty (simple.go:407-412)
    loop = ToolPrompt("q", "t", {"name": "kubectl", "input": "x"}).marshal()
    res, _ = AssistantWithConfig("m", msgs, 10, False, False, 2, ScriptedClient([loop] * 5), {"kubectl": lambda i: "ok"})
    assert res == ""
    assert isTemplateValue("short") and isTemplateValue("<final_answer goes here>") and not isTemplateValue("3 namespaces are present")
    with pytest.raises(ValueError, match="prompts cannot be empty"):
        AssistantWithConfig("m", [], 10, False, False, 5, ScriptedClient([]), {})


def test_http_front_speaks_the_wire_format_go_openai_expects():
    import urllib.error
    import urllib.request
    from opsagent_b200.engine import EngineError
    from opsagent_b200.http_front import serve

    class Eng:
        info = {"model": "tiny"}

        def chat_complete(self, model, msgs, max_tokens, flags=0, functions=None):
            if flags == 8:          # function call forced by the grammar
                assert functions == "kubectl:command,trivy:image"

                class F:
                    content = b'{"name":"kubectl","arguments":{"command":"get pods -A"}}'; prompt_tokens = 9; completion_tokens = 5; finish_reason = "stop"
                return F()
            if model == "nope":
                raise EngineError(400, "model 'nope' is not loaded")
            if model == "busy":
                raise EngineError(429, "request queue full")

            class R:
                content = ("echo:" + msgs[-1][1]).encode(); prompt_tokens = 7; completion_tokens = 3; finish_reason = "stop"
            return R()

    srv, _ = serve(Eng(), port=0)
    base = f"http://127.0.0.1:{srv.server_address[1]}/v1"

    def post(body, key="sk-x"):
        req = urllib.request.Request(base + "/chat/completions", data=json.dumps(body).encode(),
                                     headers={"Content-Type": "application/json", **({"Authorization": f"Bearer {key}"} if key else {})})
        return json.loads(urllib.request.urlopen(req, timeout=10).read())

    r = post({"model": "tiny", "max_tokens": 8192, "temperature": 1.401298464324817e-45, "messages": [{"role": "system", "content": "s"}, {"role": "user", "content": "hi"}]})
    assert r["choices"][0]["message"] == {"role": "assistant", "content": "echo:hi"} and r["choices"][0]["index"] == 0
    assert r["usage"]["total_tokens"] == 10 and r["object"] == "chat.completion"
    for model, status in (("nope", 400), ("busy", 429)):
        with pytest.raises(urllib.error.HTTPError) as e:
            post({"model": model, "messages": [{"role": "user", "content": "x"}]})
        assert e.value.code == status and json.loads(e.value.read())["error"]["code"] == status
    with pytest.raises(urllib.error.HTTPError) as e:
        post({"model": "tiny", "messages": [{"role": "user", "content": "x"}]}, key=None)
    assert e.value.code == 401
    # function calling as the swarm-go flows use it (reference pkg/workflows/swarm.go:14-78)
    tools = [{"type": "function", "function": {"name": "kubectl", "description": "Run kubectl command", "parameters": {"type": "object", "properties": {"command": {"type": "string"}}, "required": ["command"]}}},
             {"type": "function", "function": {"name": "trivy", "parameters": {"type": "object", "properties": {"image": {"type": "string"}}}}}]
    r = post({"model": "tiny", "tools": tools, "messages": [{"role": "user", "content": "analyze"}]})
    tc = r["choices"][0]["message"]["tool_calls"][0]
    assert r["choices"][0]["finish_reason"] == "tool_calls" and tc["type"] == "function" and tc["function"]["name"] == "kubectl"
    assert json.loads(tc["function"]["arguments"]) == {"command": "get pods -A"} and r["choices"][0]["message"]["content"] is None
    # after `tool_steps` tool results the reply is text again
    hist = [{"role": "user", "content": "analyze"}] + [{"role": "assistant", "tool_calls": [tc]}, {"role": "tool", "tool_call_id": tc["id"], "content": "ok"}] * 3
    r = post({"model": "tiny", "tools": tools, "messages": hist})
    assert r["choices"][0]["finish_reason"] == "stop" and r["choices"][0]["message"]["content"].startswith("echo:")
    srv.shutdown()


# ---- PerfStats mirror + /api/perf/stats bridge (reference pkg/utils/perf.go, pkg/handlers/perf.go; SURVEY.md §8f-4) ----
def test_perf_stats_mirror_accumulates_counts_and_is_request_safe():
    import threading
    from opsagent_b200.perf import PerfStats
    t = [0]
    ps = PerfStats(clock=lambda: t[0])
    ps.StartTimer("op"); t[0] = 1500; assert ps.StopTimer("op") == 1500
    ps.StartTimer("op"); t[0] = 2000; ps.StopTimer("op")
    assert ps.StopTimer("never_started") == 0                       # perf.go:87-93: unknown timer -> zero duration, not counted
    done = ps.TraceFunc("traced"); t[0] = 2600; done()
    ps.RecordMetric("execute_model_llama-3-8b", 42)
    st = ps.GetStats()
    assert st["timers"] == {"op": 2000, "traced": 600, "execute_model_llama-3-8b": 42}
    assert st["callCounts"] == {"op": 2, "traced": 1, "execute_model_llama-3-8b": 1} and st["lastResetTime"].endswith("Z")
    # two requests timing the SAME operation concurrently must not clobber each other's start time (the reference's do: perf.go:64-80)
    real = PerfStats()
    def worker():
        real.StartTimer("assistant_first_chat"); real.StopTimer("assistant_first_chat")
    th = [threading.Thread(target=worker) for _ in range(8)]
    [x.start() for x in th]; [x.join() for x in th]
    assert real.GetStats()["callCounts"] == {"assistant_first_chat": 8}
    ps.Reset()
    assert ps.GetStats()["timers"] == {} and ps.GetStats()["callCounts"] == {}


def test_assistant_loop_records_the_reference_operation_names():
    from opsagent_b200.perf import GetPerfStats
    GetPerfStats().Reset()
    step = '{"question":"q","thought":"t","action":{"name":"kubectl","input":"get ns"},"observation":"","final_answer":""}'
    final = '{"question":"q","thought":"t","action":{"name":"","input":""},"observation":"5 namespaces","final_answer":"there are 5 namespaces"}'
    res, _ = AssistantWithConfig("m", [ChatCompletionMessage("system", "s"), ChatCompletionMessage("user", "u")], 64, False, False, 5,
                                 ScriptedClient([step, final]), {"kubectl": lambda s: "default\nkube-system"})
    assert res == "there are 5 namespaces"
    cc = GetPerfStats().GetStats()["callCounts"]
    assert cc == {"assistant_first_chat": 1, "assistant_parse_tool_prompt": 1, "assistant_tool_kubectl": 1, "assistant_construct_message": 1,
                  "assistant_intermediate_chat": 1, "assistant_parse_intermediate": 1, "assistant_total": 1}   # simple.go:296,341,364,440,491,513,541


def test_http_front_serves_the_perf_stats_endpoints():
    import urllib.error
    import urllib.request
    from opsagent_b200.http_front import serve
    from opsagent_b200.perf import GetPerfStats

    class Eng:
        info = {"model": "tiny"}

        def stats(self):
            return {"decode_steps": 7, "requests_completed": 1}

        def chat_complete(self, model, msgs, max_tokens, flags=0, functions=None):
            class R:
                content = b"ok"; prompt_tokens = 2; completion_tokens = 1; finish_reason = "stop"
            return R()

    GetPerfStats().Reset()
    srv, _ = serve(Eng(), port=0)
    root = f"http://127.0.0.1:{srv.server_address[1]}"
    req = urllib.request.Request(root + "/v1/chat/completions", data=json.dumps({"model": "tiny", "messages": [{"role": "user", "content": "x"}]}).encode(),
                                 headers={"Content-Type": "application/json", "Authorization": "Bearer k"})
    urllib.request.urlopen(req, timeout=10).read()
    hdr = {"Authorization": "Bearer k"}
    with pytest.raises(urllib.error.HTTPError) as e:                                                # served from the authenticated group
        urllib.request.urlopen(root + "/api/perf/stats", timeout=10)
    assert e.value.code == 401
    r = json.loads(urllib.request.urlopen(urllib.request.Request(root + "/api/perf/stats", headers=hdr), timeout=10).read())          # pkg/api/router.go:104
    assert r["status"] == "success" and r["stats"]["callCounts"] == {"chat_completion": 1} and r["stats"]["timers"]["chat_completion"] > 0
    assert r["stats"]["engine"] == {"decode_steps": 7, "requests_completed": 1} and "lastResetTime" in r["stats"]
    r = json.loads(urllib.request.urlopen(urllib.request.Request(root + "/api/perf/reset", data=b"", method="POST", headers=hdr), timeout=10).read())   # router.go:105
    assert r["status"] == "success"
    assert json.loads(urllib.request.urlopen(urllib.request.Request(root + "/api/perf/stats", headers=hdr), timeout=10).read())["stats"]["callCounts"] == {}
    srv.shutdown()


# ---- stream-K unit plan: the invariants the fused SwiGLU epilogue and the consumers rely on (host only) ----
@pytest.mark.parametrize("N,K,G", [(28672, 4096, 148), (6144, 4096, 148), (4096, 4096, 148), (4096, 14336, 148),     # Llama-3-8B decode projections
                                   (7168, 8192, 148), (1280, 8192, 148), (8192, 1024, 148), (8192, 3584, 148),     # Llama-3-70B TP=8 shards
                                   (13824, 5120, 148), (352, 128, 148), (128, 64, 148), (640, 256, 7)])           # Qwen-32B TP=4 gate/up, tiny shapes
def test_streamk_plan_invariants(N, K, G):
    import ctypes as C
    from opsagent_b200 import _lib
    L = _lib.load()
    cap = 4096
    u0 = np.zeros(cap + 1, np.int64); tf = np.zeros(cap, np.int32); tl = np.zeros(cap, np.int32)
    g, nt, kb = C.c_int32(), C.c_int32(), C.c_int32()
    assert L.oa_host_streamk_plan(N, K, 128, G, u0.ctypes.data, cap, tf.ctypes.data, tl.ctypes.data, cap, C.byref(g), C.byref(nt), C.byref(kb)) == 0
    g, nt, kb = g.value, nt.value, kb.value
    total = nt * kb
    assert nt == -(-N // 128) and kb == -(-K // 64) and g == min(G, total)
    u0 = u0[: g + 1]
    assert u0[0] == 0 and u0[-1] == total and (np.diff(u0) >= 1).all()                 # the CTAs' ranges partition the units; nobody is idle
    assert np.diff(u0).max() - np.diff(u0).min() <= 1                                  # balanced: every SM streams the same weight bytes (+-1 k-block)
    for t in range(nt):
        touching = [c for c in range(g) if u0[c] < (t + 1) * kb and u0[c + 1] > t * kb]          # brute force
        assert touching == list(range(tf[t], tl[t] + 1)), (t, touching, tf[t], tl[t])            # the closed form the kernels use
        if len(touching) > 1:
            first = touching[0]
            assert u0[first + 1] == min((t + 1) * kb, u0[first + 1]) and u0[first + 1] <= (t + 1) * kb      # the finisher's piece is the TAIL of its range
            for c in touching[1:]:
                assert u0[c] >= t * kb and u0[c] < (t + 1) * kb                            # ... every other piece is the HEAD of its CTA's range
                assert u0[c] == max(u0[c], t * kb)
            # so a finishing CTA only waits on pieces that their CTAs compute FIRST: the wait-for graph has no cycle


# ---- reference prompts (verbatim fixtures), Go-faithful marshalling, seeded synthetic tools ---------------------------------------
import hashlib    # noqa: E402
import os         # noqa: E402
import subprocess  # noqa: E402
import sys        # noqa: E402

PROMPTS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "prompts")


def test_prompt_fixtures_are_the_reference_constants_verbatim():
    """byte lengths are the ones SURVEY.md §8a measured (3,233 / 3,109 / 1,965 / 2,164 B); index.json holds the byte length and sha256
    of every constant as extract_prompts.py read it from the reference's sources, so every fixture byte is pinned to that extraction"""
    idx = json.load(open(os.path.join(PROMPTS_DIR, "index.json")))
    sys.path.insert(0, PROMPTS_DIR)
    import extract_prompts
    assert set(idx) == set(extract_prompts.SOURCES) | set(extract_prompts.SYSTEM_LINES)
    for name, (rel, *_rest) in {**extract_prompts.SOURCES, **extract_prompts.SYSTEM_LINES}.items():
        assert idx[name]["source"].split(":")[0] == rel, name
    want = {"executeSystemPrompt_cn": 3233, "diagnoseSystemPrompt": 3109, "analysisPrompt": 1965, "auditPrompt": 2164}
    for name, meta in idx.items():
        raw = open(os.path.join(PROMPTS_DIR, name + ".txt"), "rb").read()
        assert len(raw) == meta["bytes"] and hashlib.sha256(raw).hexdigest() == meta["sha256"], name
        if name in want:
            assert len(raw) == want[name]


def test_toolprompt_marshal_is_go_json_marshal_byte_for_byte():
    from opsagent_b200.assistants import go_json_string
    """json.Marshal escapes <, >, & and U+2028/9 (simple.go:497 sends this string as the next user message)"""
    tp = ToolPrompt("q", "t", {"name": "kubectl", "input": "get pods | grep <none> && echo 'a&b'"}, "NODE  <none>\t中 \x01\"\\", "")
    want = ('{"question":"q","thought":"t","action":{"name":"kubectl","input":"get pods | grep \\u003cnone\\u003e \\u0026\\u0026 echo \'a\\u0026b\'"},'
            '"observation":"NODE  \\u003cnone\\u003e\\t中\\u2028\\u0001\\"\\\\","final_answer":""}')
    assert tp.marshal() == want
    assert ToolPrompt.unmarshal(tp.marshal()) == tp
    assert go_json_string("a\b\f\x0b\x7f") == '"a\\b\\f\\u000b\x7f"'          # go 1.22+: \b \f short forms, other controls \u00XX, DEL raw
    # Unmarshal: wrong types are errors (Go: UnmarshalTypeError), null / missing / unknown keys are not, keys match case-insensitively
    for bad in ('{"question": 5}', '{"action": "kubectl"}', '{"action": {"name": 1}}', '[1]', '"x"'):
        with pytest.raises(ValueError):
            ToolPrompt.unmarshal(bad)
    # keys are visited in document order (encoding/json): folded duplicates overwrite each other, null keeps the value, a wrong type anywhere is an error
    got = ToolPrompt.unmarshal('{"que\u017ftion":"a","THOUGHT":"t","thought":null,"action":{"Name":"x"},"ACTION":{"input":"y"}}')
    assert (got.question, got.thought, got.action) == ("a", "t", {"name": "x", "input": "y"})
    assert ToolPrompt.unmarshal('{"thought":"b","Thought":"a"}').thought == "a"
    with pytest.raises(ValueError):
        ToolPrompt.unmarshal('{"Thought": 7, "Thought": "ok"}')
    got = ToolPrompt.unmarshal('{"Question": "Q", "thought": null, "action": {"NAME": "jq"}, "extra": [1]}')
    assert (got.question, got.thought, got.action) == ("Q", "", {"name": "jq", "input": ""})


def test_synthetic_tools_are_seeded_across_processes():
    code = ("from opsagent_b200.synthetic import copilot_tools; import hashlib; t = copilot_tools(7); "
            "print(hashlib.sha256((t['kubectl']('get pods -A') + t['trivy']('nginx:1.25')).encode()).hexdigest())")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = {subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root, env={**os.environ, "PYTHONHASHSEED": str(s)}).stdout.strip()
            for s in (1, 2, 3)}
    assert len(outs) == 1 and len(next(iter(outs))) == 64


def test_http_front_survives_bad_clients():
    """early 401/404 replies drain the request body (HTTP/1.1 keep-alive stays in sync), a truncated grammar-forced call is an
    OpenAI-style error instead of a dropped connection, Content-Length is bounded, and a configured key is compared"""
    import http.client
    from opsagent_b200.http_front import serve

    class Eng:
        info = {"model": "tiny"}

        def chat_complete(self, model, msgs, max_tokens, flags=0, functions=None):
            class R:
                content = (b'{"name":"kubectl","argum' if flags == 8 else b"ok"); prompt_tokens = 3; completion_tokens = 6; finish_reason = "length" if flags == 8 else "stop"
            return R()

    srv, _ = serve(Eng(), port=0, api_key="sk-right")
    conn = http.client.HTTPConnection("127.0.0.1", srv.server_address[1], timeout=10)
    body = json.dumps({"model": "tiny", "messages": [{"role": "user", "content": "x" * 5000}]})

    def post(path, key, b=body, extra=None):
        h = {"Content-Type": "application/json", "Authorization": f"Bearer {key}"}
        h.update(extra or {})
        conn.request("POST", path, body=b, headers=h)
        r = conn.getresponse()
        return r.status, json.loads(r.read() or b"{}")

    # three requests on ONE connection: 401 (wrong key, body unread by the handler logic), 404, then a good one must still parse
    assert post("/v1/chat/completions", "sk-wrong")[0] == 401
    assert post("/v1/nothing", "sk-right")[0] == 404
    st, r = post("/v1/chat/completions", "sk-right")
    assert st == 200 and r["choices"][0]["message"]["content"] == "ok"
    tools = [{"type": "function", "function": {"name": "kubectl", "parameters": {"type": "object", "properties": {"command": {"type": "string"}}}}}]
    st, r = post("/v1/chat/completions", "sk-right", json.dumps({"model": "tiny", "tools": tools, "max_tokens": 6, "messages": [{"role": "user", "content": "x"}]}))
    assert st == 400 and "truncated" in r["error"]["message"]
    st, r = post("/v1/chat/completions", "sk-right")          # and the connection is still usable afterwards
    assert st == 200
    conn.close()
    conn = http.client.HTTPConnection("127.0.0.1", srv.server_address[1], timeout=10)
    conn.putrequest("POST", "/v1/chat/completions"); conn.putheader("Content-Length", "-5"); conn.putheader("Authorization", "Bearer sk-right"); conn.endheaders()
    assert conn.getresponse().status == 400
    conn.close(); srv.shutdown()


def test_follower_side_tiny_presets_equal_the_oracle_presets():
    from opsagent_b200.presets_tiny import TINY_TP
    for name, cfg in TINY_TP.items():
        assert cfg == O.PRESETS[name].engine_json(), name


# ---- grammar masks over a TOKEN vocabulary (csrc/token_mask.hpp) vs the oracle-side brute force ----
@pytest.mark.parametrize("tok", ["", "bpe_llama3_tiny.json", "bpe_qwen2_tiny.json"])
@pytest.mark.parametrize("kind", [O.GRAMMAR_TOOLCALL, O.GRAMMAR_FINAL, O.GRAMMAR_FUNCTION, O.GRAMMAR_TEXT])
def test_token_masks_equal_brute_force_along_random_token_walks(tok, kind):
    """the C++ trie walk must allow exactly the tokens whose bytes all walk the automaton; states sharing a canonical cache key must share a mask"""
    L = _lib.load()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", tok) if tok else ""
    if tok:
        token_bytes = O.bpe_token_bytes(path)
        vocab = len(token_bytes)
    else:
        vocab, token_bytes = 704, O.byte_level_token_bytes()
    fns = "kubectl:command,trivy:image" if kind == O.GRAMMAR_FUNCTION else ""
    words = (vocab + 31) // 32
    rng = np.random.default_rng(5 + kind)
    by_key = {}
    for walk in range(3):
        g = O.ToolPromptGrammar(kind, fns)
        prefix = bytearray()
        for _step in range(400):
            if g.done():
                break
            ref = O.allowed_tokens(g, token_bytes)
            mask = (C.c_uint32 * words)(); key = C.create_string_buffer(256)
            buf = (C.c_uint8 * max(1, len(prefix))).from_buffer_copy(bytes(prefix) or b"\0")
            assert L.oa_host_grammar_token_mask(path.encode() if path else None, vocab, kind, fns.encode(), buf, len(prefix), mask, words, key, 256) == 0
            got = [i for i in range(vocab) if (mask[i >> 5] >> (i & 31)) & 1]
            assert got == ref, (walk, bytes(prefix), set(got) ^ set(ref))
            assert ref, "a grammar state must always allow at least one token"
            by_key.setdefault(key.value, set()).add(tuple(ref))
            tid = int(rng.choice(ref))
            for b in token_bytes[tid]:
                prefix.append(b); assert g.advance(b)
        assert g.done()
    assert all(len(v) == 1 for v in by_key.values())


# ---- data-parallel router: one front, N engines (opsagent_b200/router.py; reference pkg/api/router.go:95 is one process) ----
def test_router_is_sticky_balanced_and_rejects_overload():
    import threading
    import time
    from opsagent_b200.engine import EngineError
    from opsagent_b200.router import Router, conversation_key

    class FakeEngine:
        def __init__(self, i):
            self.i, self.info, self.seen, self.gate = i, {"model": "m"}, [], threading.Event()

        def chat_complete(self, model, msgs, max_tokens, flags=0, functions=None):
            self.seen.append(conversation_key(msgs))
            self.gate.wait(5)
            return self.i

        def stats(self):
            return {"decode_tokens": len(self.seen), "pages_free": 1}

        def close(self):
            pass

    engines = [FakeEngine(i) for i in range(4)]
    rt = Router(engines, max_inflight=2)
    conv = lambda c, steps: [("system", "sys"), ("user", f"question {c}")] + [("assistant", "a"), ("user", "obs")] * steps      # noqa: E731
    results = {}

    def call(c, steps):
        try:
            results[(c, steps)] = rt.chat_complete("m", conv(c, steps), 8)
        except EngineError as e:
            results[(c, steps)] = e.code
    # 8 new conversations arrive together: least-loaded placement puts exactly 2 on each replica
    th = [threading.Thread(target=call, args=(c, 0)) for c in range(8)]
    [t.start() for t in th]
    t_end = time.time() + 5
    while sum(rt.stats()["inflight"]) < 8 and time.time() < t_end:
        time.sleep(0.002)
    assert rt.stats()["inflight"] == [2, 2, 2, 2]
    # a 9th conversation finds every replica at its limit -> 429 for the caller's backoff loop (openai.go:91-94)
    call(99, 0)
    assert results[(99, 0)] == 429 and rt.stats()["rejected_429"] == 1
    [e.gate.set() for e in engines]; [t.join() for t in th]
    home = {c: results[(c, 0)] for c in range(8)}
    # later steps of a conversation (longer history, same first two messages) go back to the replica that holds its prefix pages
    for steps in (1, 2, 3):
        for c in range(8):
            call(c, steps)
            assert results[(c, steps)] == home[c]
    st = rt.stats()
    assert st["sticky_hits"] == 24 and st["routed"] == [8, 8, 8, 8] and st["decode_tokens"] == 32 and st["replicas"] == 4
    assert rt.replica_of(conv(3, 7)) == home[3] and rt.replica_of(conv(12345, 0)) is None


def test_trimspace_is_gos_unicode_isspace_set_not_pythons():
    """strings.TrimSpace (simple.go:444, tokens.go:140) strips unicode.IsSpace; Python's str.strip() would also strip \x1c-\x1f, which Go keeps"""
    from opsagent_b200.llms import TrimSpace
    assert TrimSpace(" \t\n\u2028\u3000\xa0\x85 x y \u200a\r") == "x y"
    assert TrimSpace("\x1c x \x1f") == "\x1c x \x1f"
    assert TrimSpace("\u200b x") == "\u200b x"          # ZERO WIDTH SPACE is not white space in Go


def test_get_token_limits_and_constrict_messages_follow_the_reference():
    """pkg/llms/tokens_test.go:20-51 holds two GetTokenLimits cases; ConstrictMessages (tokens.go:110-125) keeps the first message and drops the oldest after it"""
    from opsagent_b200.llms import ChatCompletionMessage as M, ConstrictMessages, GetTokenLimits
    assert GetTokenLimits("gpt-3.5-turbo-0613") == 4096 and GetTokenLimits("gpt-4") == 8192            # the reference's own golden cases
    assert GetTokenLimits("GPT-4-32K") == 32768 and GetTokenLimits("llama-3-8b") == 4096 and GetTokenLimits("gpt-4", engine_limit=16384) == 16384
    count = lambda ms: sum(3 + len(c) for _, c in ms) + 3          # noqa: E731
    msgs = [M("system", "s" * 100), M("user", "a" * 300), M("assistant", "b" * 300), M("user", "c" * 300)]
    assert ConstrictMessages(msgs, "m", 5000, count) is None                                               # maxTokens >= the 4096 window
    assert ConstrictMessages(msgs, "m", 100, count, engine_limit=2000) == msgs                             # fits: untouched
    got = ConstrictMessages(msgs, "m", 100, count, engine_limit=600)
    assert [m.Content[0] for m in got] == ["s", "c"]                                                       # system prompt + the newest that fit
    with pytest.raises(IndexError):
        ConstrictMessages([M("system", "s" * 1000)], "m", 100, count, engine_limit=600)                   # the reference panics here
