#!/usr/bin/env python
"""bench.py — the reference's headline metric on BASELINE.json configs[1]:
Llama-3-8B bf16, 1xB200, batch=128 concurrent `analyze` ReAct steps over synthetic Pod YAML
(P=1536 prompt tokens, G=256 generated tokens, mean decode context 1664; SURVEY.md §8d config 2).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one decode forward of the whole batch (128 sequences, one new token each) through the hot path.
  value  : decode tokens/s, whole job (all N GPUs), inputs resident in HBM, K steps inside one CUDA-event bracket
           on the engine's stream, max over ranks.
  e2e    : the same metric through the public chat API (LocalCUDAClient / C ABI) with HOST buffers: 128 concurrent
           chat completions per GPU (prompt bytes in, text out), tokenisation, H2D of ids/metadata, prefill, every
           decode step's D2H of sampled ids and detokenisation inside the timed region.
  roofline: dominant kernel = paged decode attention; achieved = algorithmic KV bytes per launch / mean launch time
           (CUDA events on the engine stream) against the measured HBM copy bandwidth.
  cpu_baseline: the CPU oracle (a port — the reference has no model arithmetic of its own) on the host cores.
N>1 = data-parallel replicas (BASELINE configs[2]): one engine per GPU, no data-path collective, weak scaling.
N>=2 additionally runs, AFTER the headline (metric/value unchanged), the tensor-parallel path at t = N over the same N ranks:
  tp.parity : tests/tp_worker.py at t=N against the CPU oracle (t=4: Qwen2.5-32B TP=4's per-rank head layout, t=8: Llama-3-70B TP=8's)
  tp.*      : BASELINE configs[3] (Qwen2.5-32B TP=4, B=256, ctx 2048) at N=4, configs[4] (Llama-3-70B TP=8, B=64, ctx 16.9k incl. its
              1.08M-token prefill) at N=8, Llama-3-8B TP=2 at N=2 — decode ms/step, tokens/s per group and per GPU, fraction of the per-GPU
              HBM roofline, the all-reduce chain (in-situ us per all-reduce x count per step).
`--impl reference` times the CPU port alone (rank 0 only), same JSON line shape.
`--dump-outputs DIR` writes what the last timed decode step computed (rank 0) as DIR/<name>.npy, see dump_outputs().
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "llama-3-8b"
BATCH, PROMPT, GEN, MEAN_CTX = 128, 1536, 256, 1664


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpus="0", period_ms=200):
        self.gpu, self.period, self.rows, self.proc = gpus, period_ms, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.period),
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) > 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


TOKENIZER = os.path.join(ROOT, "tests", "golden", "bpe_k8s_8k.json")     # Llama-3-format byte-level BPE trained on OpsAgent's own kind of text
REACT_TOOL_STEPS = 3


TP_CONFIGS = {2: ("llama-3-8b", 128, 1664, "Llama-3-8B TP=2 (fits one GPU; exercises the collective path at N=2)"),
              4: ("qwen2.5-32b", 256, 2048, "BASELINE configs[3]: Qwen2.5-32B TP=4 over NVLink, B=256, ctx 2048"),
              8: ("llama-3-70b", 64, 16896, "BASELINE configs[4]: Llama-3-70B TP=8, B=64, 16k-token trivy observations (ctx 16.9k)")}
KVB = {"qwen2.5-32b": 262144, "llama-3-70b": 327680, "llama-3-8b": 131072}


def run_tp_block(args, rank, world, nonce, log):
    """Tensor parallelism at t = world over the same ranks: parity first (checker: the CPU oracle on rank 0), then the BASELINE TP
    config for this N.  Rank 0 returns the "tp" block, followers return None.  Own NVLink peer-memory all-reduce, no NCCL on the data path."""
    import importlib.util
    from opsagent_b200 import Engine
    spec = importlib.util.spec_from_file_location("oa_tp_worker", os.path.join(ROOT, "tests", "tp_worker.py"))
    tpw = importlib.util.module_from_spec(spec); spec.loader.exec_module(tpw)
    block = {}
    if not args.no_tp_parity:
        par = tpw.run_cases(rank, world, cases=(args.tp_cases.split(",") if args.tp_cases else None), tag=str(nonce), log=log)
        if rank == 0:
            block["parity"] = {k: par[k] for k in ("t", "cases", "max_dlogit", "tokens_identical", "tokens_compared", "near_tie_flips", "ok")}
            block["parity"]["tolerance"] = {"max_dlogit": tpw.LOGIT_TOL, "tokens": "identical wherever the oracle's top1-top2 margin > 2*tol"}
    model, batch, ctx, what = TP_CONFIGS[world]
    if args.tp_model:
        model, batch, ctx, what = args.tp_model, args.tp_batch, args.tp_ctx, f"override: {args.tp_model} TP={world} B={args.tp_batch} ctx {args.tp_ctx}"
    K, W = min(args.steps, 16), 4
    max_seq = (ctx + K + W + 64 + 63) // 64 * 64
    pages = batch * ((max_seq + 63) // 64) + 64
    eng = Engine({"model": model, "device": rank, "tp": world, "tp_rank": rank, "tp_shm": f"/oa_tp_bench_{nonce}", "tp_nonce": nonce,
                  "num_pages": pages, "max_batch": batch, "max_seq_len": max_seq, "max_step_tokens": 8192, "seed": 1234, "prefix_cache": 0,
                  **json.loads(args.engine_extra)})
    if rank > 0:
        eng.serve(); eng.close()
        return None
    ctx0 = ctx - K // 2 - W
    r = eng.bench_decode(batch, ctx0, K, W)
    peak, peak_src = measured_peaks()
    os.environ["OA_PROFILE_ALL"] = "1"          # in-situ per-class kernel times on the leader (events between launches)
    eng.kernel_times(True)
    eng.bench_decode(batch, min(ctx0, 256), 4, 2)   # the all-reduce does not depend on the context length: a short prefill is enough
    kt = eng.kernel_times(True)
    os.environ["OA_PROFILE_ALL"] = "0"
    info = eng.info
    ar_ms, ar_n = kt.get("resid_rmsnorm", [0.0, 0])
    gb = r["algorithmic_bytes_per_step"]
    block.update({"config": what, "model": model, "t": world, "batch": batch, "mean_ctx": round(r["mean_ctx"], 1), "steps": K, "warmup": W,
                  "ms_per_step": round(r["ms_per_step"], 3), "tok_s_group": round(batch / r["ms_per_step"] * 1e3, 1),
                  "tok_s_per_gpu": round(batch / r["ms_per_step"] * 1e3 / world, 1),
                  "algorithmic_bytes_per_gpu_per_step": gb, "hbm_GBps_per_gpu": round(gb / r["ms_per_step"] / 1e6, 1),
                  "roofline_frac_per_gpu": round(gb / r["ms_per_step"] / 1e6 / peak, 4), "peak_source": peak_src,
                  "allreduce_us": (round(ar_ms / ar_n * 1e3, 2) if ar_n else None), "allreduce_count_per_step": 2 * info["n_layers"],
                  "allreduce_note": "partial -> symmetric buffer + all-reduce + residual + RMSNorm, in-situ CUDA events on the leader (serialised: upper bound)",
                  "prefill_tokens": batch * (ctx0 - 1), "prefill_ms": round(r["prefill_ms"], 1),
                  "prefill_tok_s": round(batch * (ctx0 - 1) / r["prefill_ms"] * 1e3, 1), "launches_per_step": r["launches_per_step"],
                  "collective": ("decode: in-switch reduction (multimem.ld_reduce / multimem.st on an NVLS multicast buffer, tp_nvls.cpp) fused with residual + RMSNorm; "
                                 if info.get("tp_nvls") else "decode: own one-shot all-reduce over NVLink peer memory (bf16 partials, rank-ordered sum) fused with residual + RMSNorm; ") +
                                "prefill chunks: two-shot reduce-scatter + all-gather over peer memory; no NCCL on the data path", "nvls": bool(info.get("tp_nvls"))})
    eng.close()
    return block


def router_block(args, rank, world, barrier, dist=None, cpu_group=None):
    """BASELINE configs[2] as it would be SERVED: one front process (rank 0) owning one engine per GPU behind the OpenAI-compatible HTTP
    endpoint (the reference is one process too, pkg/api/router.go:95) — csrc/http_server.cpp, native, routing inside the server (or, with
    --router-front python, router.py + http_front.py).  world*128 concurrent HTTP clients POST the 40/30/30 mix in the reference's wire
    format; the clients are spread over ALL ranks' processes (the ranks other than 0 have closed their engines and have nothing else to do),
    so the load generator's interpreter is not what is measured.  Sticky least-loaded routing, no data-path collective."""
    import http.client
    import resource
    import torch
    barrier()
    try:
        soft, hard = resource.getrlimit(resource.RLIMIT_NOFILE)
        resource.setrlimit(resource.RLIMIT_NOFILE, (min(hard, 65536) if hard > 0 else 65536, hard))
    except Exception:
        pass
    sys.setswitchinterval(2e-4)
    n_req = world * BATCH
    setup = [None]
    front = rt = srv = None
    if rank == 0:
        try:
            from opsagent_b200 import workloads as WL
            from opsagent_b200.router import Router
            cfg = {"model": MODEL, "kv_gb": args.kv_gb, "max_batch": BATCH, "max_seq_len": 2048, "max_step_tokens": 8192, "seed": 1234, "tokenizer": TOKENIZER,
                   "prefix_cache": 0, "max_queue": 4096, **json.loads(args.engine_extra)}
            rt = Router.create(cfg, list(range(world)), max_inflight=2 * BATCH)          # engine creation in parallel; the Router object itself only routes in python mode
            if args.router_front == "native":
                from opsagent_b200.native_front import NativeFront
                front = NativeFront(rt.engines, max_inflight=2 * BATCH)
                port = front.port
            else:
                from opsagent_b200.http_front import serve
                srv, _th = serve(rt, port=0)
                port = srv.server_address[1]
            bodies, kinds = [], {}
            for gi in range(n_req):
                k, m = WL.mixed_request(gi, rt.count_tokens, p_analyze=PROMPT)
                kinds[k] = kinds.get(k, 0) + 1
                bodies.append(json.dumps({"model": MODEL, "max_tokens": GEN, "temperature": 1.401298464324817e-45,
                                          "messages": [{"role": x.Role, "content": x.Content} for x in m]}).encode("utf-8"))
            setup = [{"port": port, "bodies": bodies, "kinds": kinds}]
        except Exception as e:      # noqa: BLE001
            setup = [{"error": f"{type(e).__name__}: {e}"}]
    if dist is not None:
        dist.broadcast_object_list(setup, src=0, group=cpu_group)
    cfgd = setup[0]
    if "error" in cfgd:
        barrier()
        return cfgd if rank == 0 else None
    port, bodies = cfgd["port"], cfgd["bodies"]
    mine = [i for i in range(n_req) if i % world == rank]
    usage = {}

    def post(i):
        try:
            c = http.client.HTTPConnection("127.0.0.1", port, timeout=600)
            c.request("POST", "/v1/chat/completions", body=bodies[i], headers={"Content-Type": "application/json", "Authorization": "Bearer sk-local"})
            r = c.getresponse(); d = json.loads(r.read()); c.close()
            usage[i] = d["usage"] if r.status == 200 else {"error": r.status}
        except Exception as e:      # noqa: BLE001
            usage[i] = {"error": f"{type(e).__name__}: {e}"}

    def stats():
        if front is not None:
            st = front.stats()
            return {"routed": st["routed"], "rejected_429": st["rejected_429"], "per_replica": st["engines"]}
        return rt.stats()

    def round_(idx):
        idx = list(idx)
        go = threading.Barrier(len(idx) + 1)

        def client(i):
            go.wait()
            post(i)
        th = [threading.Thread(target=client, args=(i,)) for i in idx]
        [t.start() for t in th]
        barrier()                                                  # every rank's client threads exist
        go.wait()                                                  # they all connect now
        t0 = time.perf_counter()
        [t.join() for t in th]
        dt = time.perf_counter() - t0
        if dist is not None:                                       # the round ends when the slowest rank's last response is in
            t = torch.tensor([dt], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=cpu_group)
            dt = float(t.item())
        return dt
    def safe_stats():          # rank-0-only code must not raise between collectives: the other ranks would wait at the next one forever
        try:
            return stats() if rank == 0 else None
        except Exception as e:      # noqa: BLE001
            return {"error": f"{type(e).__name__}: {e}"}
    round_(mine[::16])                                             # warm-up: a few requests on every replica
    s0 = safe_stats()
    usage.clear()
    dt = round_(mine)
    s1 = safe_stats()
    gathered = [None] * world
    if dist is not None:
        dist.all_gather_object(gathered, usage, group=cpu_group)
    else:
        gathered = [usage]
    out = None
    if rank == 0:
        try:
            allu = {}
            for g in gathered:
                allu.update(g)
            ok = [u for u in allu.values() if u and "error" not in u]
            errs = sorted({str(u["error"]) for u in allu.values() if u and "error" in u})
            comp = sum(u["completion_tokens"] for u in ok)
            fw = lambda st: sum(p["prefill_steps"] + p["decode_steps"] for p in st["per_replica"])      # noqa: E731
            out = {"workload": f"BASELINE configs[2] served: {n_req} concurrent HTTP clients (spread over the {world} rank processes) -> one front process ({args.router_front}: "
                               f"OpenAI-compatible endpoint + sticky least-loaded routing) -> {world} engines; mix 40% analyze (P=1536) / 30% diagnose / 30% execute, "
                               "verbatim reference prompts, max_tokens 256",
                   "front": args.router_front, "requests": n_req, "completed": len(ok), "errors": errs, "by_kind": cfgd["kinds"], "seconds": round(dt, 3),
                   "e2e_tokens_per_sec": round(comp / dt, 1), "react_steps_per_sec": round(len(ok) / dt, 2), "completion_tokens": comp,
                   "prompt_tokens_mean": round(sum(u["prompt_tokens"] for u in ok) / max(1, len(ok)), 1),
                   "routed_per_replica": [b - a for a, b in zip(s0["routed"], s1["routed"])], "rejected_429": s1["rejected_429"] - s0["rejected_429"],
                   "engine_forwards": fw(s1) - fw(s0),
                   "engine_busy_ms_max": round(max(b["busy_ms"] - a["busy_ms"] for a, b in zip(s0["per_replica"], s1["per_replica"])), 1)}
        except Exception as e:      # noqa: BLE001
            out = {"error": f"{type(e).__name__}: {e}"}
        for closer in ((front.shutdown if front is not None else None), (srv.shutdown if srv is not None else None), rt.close):
            try:
                if closer:
                    closer()
            except Exception:      # noqa: BLE001
                pass
    barrier()
    return out


def react_block(args, rank, world, local_rank, barrier, allmax):
    """Multi-step ReAct loops inside the measurement contract: per GPU, 128 concurrent conversations driven by the mirror of the
    reference's loop (assistants.AssistantWithConfig <-> pkg/assistants/simple.go:292-616) through LocalCUDAClient.Chat — POST /execute's
    message shape (verbatim executeSystemPrompt_cn + a question), REACT_TOOL_STEPS grammar-forced kubectl tool calls answered by a seeded
    synthetic kubectl, then a final answer.  The history is resent on every step (simple.go:498-501), so the prefix cache is ON here and
    its hit rate is reported.  A ReAct step = one completed Chat call."""
    from opsagent_b200 import Engine, LocalCUDAClient
    from opsagent_b200 import workloads as WL
    from opsagent_b200.assistants import AssistantWithConfig
    from opsagent_b200.synthetic import copilot_tools
    n_agents = args.react_agents
    eng = Engine({"model": MODEL, "device": local_rank, "kv_gb": args.kv_gb, "max_batch": n_agents, "max_seq_len": 8192, "max_step_tokens": 8192,
                  "seed": 1234, "tokenizer": TOKENIZER, "json_mode": 1, "react_tool_steps": REACT_TOOL_STEPS, "prefix_cache": 1,
                  **json.loads(args.engine_extra)})
    calls = [0] * n_agents
    results = [None] * n_agents

    class CountingClient(LocalCUDAClient):
        def __init__(self, engine, slot):
            super().__init__(engine); self.slot = slot

        def Chat(self, model, maxTokens, prompts):
            calls[self.slot] += 1
            return super().Chat(model, maxTokens, prompts)

    def agent(i, salt):
        q = WL.EXECUTE_QUESTIONS[(rank * n_agents + i) % len(WL.EXECUTE_QUESTIONS)]
        msgs = WL.execute_messages("execute " + q, f"(cluster c{salt}-{rank}-{i})")
        tools = copilot_tools(1000 * salt + i)
        if args.react_tool_ms > 0:                # the reference's tools fork/exec kubectl (~100 ms class): agents drift apart, arrivals stagger
            import random
            rr = random.Random(salt * 7919 + i)
            tools = {k: (lambda inp, f=f: (time.sleep(args.react_tool_ms * (0.5 + rr.random()) / 1e3), f(inp))[1]) for k, f in tools.items()}
        results[i] = AssistantWithConfig(MODEL, msgs, 2048, True, False, REACT_TOOL_STEPS + 2, CountingClient(eng, i), tools,
                                         count_tokens=eng.count_tokens)

    def round_(n, salt):
        for i in range(n):
            calls[i] = 0; results[i] = None
        th = [threading.Thread(target=agent, args=(i, salt)) for i in range(n)]
        t0 = time.perf_counter()
        [t.start() for t in th]; [t.join() for t in th]
        return time.perf_counter() - t0

    round_(min(8, n_agents), 1)                  # warm-up: every kernel shape and grammar state seen once
    s0 = eng.stats()
    barrier()
    dt = round_(n_agents, 2)
    barrier()
    s1 = eng.stats()
    n_calls = sum(calls)
    ok = sum(1 for r in results if r and len(r[0]) >= 10)
    dt = allmax(dt)
    hit = s1["prefix_hit_tokens"] - s0["prefix_hit_tokens"]; pre = s1["prefill_tokens"] - s0["prefill_tokens"]
    eng.close()
    return {"workload": f"{n_agents} concurrent ReAct conversations per GPU: verbatim executeSystemPrompt_cn + question, {REACT_TOOL_STEPS} grammar-forced kubectl "
                        "tool steps (seeded synthetic kubectl tables) + final answer; json_mode, prefix cache on",
            "react_steps_per_sec": round(world * n_calls / dt, 2), "chat_calls_per_gpu": n_calls, "seconds": round(dt, 2),
            "conversations_with_final_answer": ok, "conversations": n_agents, "tool_latency_ms": args.react_tool_ms,
            "completion_tokens_per_sec": round(world * (s1["decode_tokens"] - s0["decode_tokens"]) / dt, 1),
            "prefill_tokens": pre, "prefix_hit_tokens": hit, "prefix_hit_rate": round(hit / max(1, hit + pre), 4),
            "decode_steps": s1["decode_steps"] - s0["decode_steps"], "prefill_steps": s1["prefill_steps"] - s0["prefill_steps"],
            "mixed_steps": s1.get("mixed_steps", 0) - s0.get("mixed_steps", 0), "preemptions": s1["preemptions"] - s0["preemptions"],
            "grammar_states_computed": s1.get("grammar_states_computed", 0)}


def run_ours(args, rank, world, local_rank):
    import torch
    import numpy as np
    from opsagent_b200 import Engine, LocalCUDAClient, ChatCompletionMessage
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # A rank that merely WAITS (while rank 0 drives every GPU in the router block) must wait on the host: an NCCL barrier is a kernel
    # spinning on that rank's GPU, taking SMs away from the engine rank 0 runs there (measured: the served round took 8.4 s instead of 3.7 s).
    cpu_group = dist.new_group(backend="gloo") if dist is not None else None

    def host_barrier():
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier(group=cpu_group)

    from opsagent_b200 import dp as DP       # host side of the replica mode: request sharding + max-over-ranks timing (tests/test_dp_gloo.py)

    def allmax(x):
        return DP.allreduce_max(x, dist, device="cuda")

    def tp_block():
        """-> the "tp" block on rank 0 (None on followers); never raises, never hangs the headline: rank 0 gives the leg a deadline"""
        nt = torch.tensor([int(time.time() * 1e3) % (1 << 40) + int(os.environ.get("MASTER_PORT", "0"))], dtype=torch.int64, device="cuda")
        dist.broadcast(nt, 0)                     # same launch id on every rank (shm name + nonce of the TP group)
        res = {}

        def work():
            try:
                res["tp"] = run_tp_block(args, rank, world, int(nt.item()), (lambda m: print(m, file=sys.stderr, flush=True)))
            except Exception as e:                  # the failure is reported, not hidden
                res["tp"] = {"error": f"{type(e).__name__}: {e}"}
        th = threading.Thread(target=work, daemon=True)
        th.start(); th.join(args.tp_deadline)
        if th.is_alive():
            return {"error": f"tensor-parallel leg did not finish within {args.tp_deadline} s"}, True
        return res.get("tp"), False

    if args.tp_only:
        tp, hung = tp_block()
        if rank == 0:
            print(json.dumps({"tp": tp}), flush=True)
        if hung:
            os._exit(3)
        dist.barrier(); dist.destroy_process_group()
        return
    if args.react_only:
        rb = react_block(args, rank, world, local_rank, barrier, allmax)
        if rank == 0:
            print(json.dumps({"react": rb}), flush=True)
        return
    K, W = args.steps, max(args.warmup, 3)
    # context chosen so that the mean over the K timed steps is MEAN_CTX (=P+G/2); a long run gets the sequence length it needs
    ctx0 = max(64, MEAN_CTX - W - K // 2)
    eng = Engine({"model": MODEL, "device": local_rank, "kv_gb": args.kv_gb, "max_batch": BATCH, "max_seq_len": max(2048, (ctx0 + K + W + 64) // 64 * 64),
                  "max_step_tokens": 8192, "seed": 1234, "tokenizer": TOKENIZER,
                  "prefix_cache": 0,       # every timed prompt token is really prefilled: no cached outputs inside the timed region
                  **json.loads(args.engine_extra)})
    info = eng.info
    # ------------------------------------------------------------------ value: device-resident decode steps
    # ONE sampler for the whole job (rank 0, all N GPUs): NVML queries take driver-wide locks; N polling processes are the
    # suspected source of the host gaps seen at N=4 (0.5 ms per 8.5 ms step against 0.02 ms at N=1) and one is enough anyway
    clocks = ClockSampler(",".join(str(i) for i in range(world)), 200 if world == 1 else 500) if rank == 0 else None
    if clocks:
        clocks.start()
    barrier()
    r = eng.bench_decode(BATCH, ctx0, K, W, last_outputs=bool(args.dump_outputs))
    barrier()
    clk = clocks.stop() if clocks else None
    ms_step = allmax(r["ms_per_step"])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r)
    value = world * BATCH / (ms_step / 1e3)
    # ------------------------------------------------------------------ roofline: dominant kernel (decode attention)
    os.environ["OA_PROFILE_ATTN"] = "1"
    rp = eng.bench_decode(BATCH, ctx0, max(4, min(K, 16)), 3)
    os.environ["OA_PROFILE_ATTN"] = "0"
    L = info["n_layers"]
    kv_tok = info["kv_bytes_per_token"]
    attn_launch_ms = rp["attn_ms_per_step"] / L                           # one decode_attention (+ split merge) per layer
    attn_bytes = BATCH * rp["mean_ctx"] * kv_tok / L                      # K and V of every cached token, once
    peak, peak_src = measured_peaks()
    achieved = attn_bytes / (attn_launch_ms * 1e-3) / 1e9 if attn_launch_ms > 0 else 0.0
    traffic = None
    try:      # DRAM bytes of the same kernel from the committed `ncu --set full` capture (per launch)
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["decode_attention_kernel<128>"]
        traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "decode_attention_kernel<128>", "achieved": round(achieved, 1), "peak": peak,
                "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": attn_bytes, "launch_ms": round(attn_launch_ms, 4),
                "kernel_share_of_step": round(rp["attn_ms_per_step"] / rp["device_ms_per_step"], 3) if rp["device_ms_per_step"] else None,
                "step": {"algorithmic_bytes": r["algorithmic_bytes_per_step"],
                         "achieved": round(r["algorithmic_bytes_per_step"] / (ms_step * 1e-3) / 1e9, 1),
                         "frac": round(r["algorithmic_bytes_per_step"] / (ms_step * 1e-3) / 1e9 / peak, 4)}}
    # ------------------------------------------------------------------ e2e: public chat API, host buffers
    # The reference's own request shapes with its system prompts VERBATIM (opsagent_b200/workloads.py <- tests/golden/prompts/), tokenised
    # by the engine's byte-level BPE.  N=1: BASELINE configs[1], 128 analyze requests padded with synthetic Pod YAML to P=1536 tokens.
    # N>=2: configs[2]'s mix per replica: 40 % analyze (P=1536) / 30 % diagnose / 30 % execute (zh prompt); diagnose and execute carry no
    # bulk payload in the reference, so their prompt length is what the verbatim prompt + question tokenise to.
    from opsagent_b200 import workloads as WL
    cli = LocalCUDAClient(eng)
    reqs = []
    for gi in DP.shard_requests(world * BATCH, rank, world):      # this replica's contiguous shard of the job's request ids
        if world == 1:
            reqs.append(("analyze", WL.fit_to_tokens(WL.analyze_messages, WL.synthetic_pod_yaml(gi, 12 * PROMPT), PROMPT, eng.count_tokens)))
        else:
            reqs.append(WL.mixed_request(gi, eng.count_tokens, p_analyze=PROMPT))
    prompts = [m for _k, m in reqs]
    msgs_all = [[(m.Role, m.Content) for m in p] for p in prompts]
    p_tokens = [eng.count_tokens(m) for m in msgs_all]
    by_kind = {}
    for (k, _m), n in zip(reqs, p_tokens):
        by_kind.setdefault(k, []).append(n)

    def one_round():
        t0 = time.perf_counter()
        tickets = [eng.chat_submit(MODEL, m, GEN, flags=1) for m in msgs_all]   # non-blocking submit, as Go would
        outs = [eng.wait(t) for t in tickets]
        dt = time.perf_counter() - t0
        assert all(o.completion_tokens == GEN and o.prompt_tokens == n for o, n in zip(outs, p_tokens))
        return dt, outs

    # one blocking Chat() through the Go-mirror client proves the seam itself (untimed)
    txt = cli.Chat(MODEL, 4, prompts[0])
    assert isinstance(txt, str)
    one_round()                                                                  # warm-up round
    s0 = eng.stats()
    barrier()
    dt, _ = one_round()
    barrier()
    s1 = eng.stats()
    dt = allmax(dt)
    n_fwd = (s1["prefill_steps"] - s0["prefill_steps"]) + (s1["decode_steps"] - s0["decode_steps"])
    e2e = {"value": round(world * BATCH * GEN / dt, 1), "unit": "tokens/s", "react_steps_per_sec": round(world * BATCH / dt, 2),
           "seconds_per_round": round(dt, 3), "requests": world * BATCH, "prompt_tokens": round(sum(p_tokens) / len(p_tokens), 1), "completion_tokens": GEN,
           "prompt_tokens_by_kind": {k: {"n": len(v), "mean": round(sum(v) / len(v), 1)} for k, v in by_kind.items()},
           "prompts": "reference system prompts verbatim (tests/golden/prompts), byte-level BPE tests/golden/bpe_k8s_8k.json",
           "h2d_bytes_per_step": int((s1["h2d_bytes"] - s0["h2d_bytes"]) / max(1, n_fwd)),
           "d2h_bytes_per_step": int((s1["d2h_bytes"] - s0["d2h_bytes"]) / max(1, n_fwd)), "forwards": n_fwd}
    launches = int(round(r["launches_per_step"] * K))
    line = {"metric": "decode_tokens_per_sec", "value": round(value, 1), "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (seeded random-init weights seed=1234; the reference's verbatim system prompts + seeded synthetic Pod YAML; "
                    "byte-level BPE tokenizer trained offline on OpsAgent-domain text)",
            "config": {"workload": ("BASELINE configs[1]: Llama-3-8B bf16, batch=128 concurrent analyze ReAct steps per GPU, " if world == 1 else
                                    f"BASELINE configs[2]: Llama-3-8B replicated data-parallel on {world} GPUs, batch={world * BATCH}, e2e mix 40% analyze / 30% diagnose / 30% execute; value: ") +
                                   f"P={PROMPT} G={GEN}, mean decode ctx {r['mean_ctx']:.0f}",
                       "batch_per_gpu": BATCH, "parallelism": f"dp{world}", "l2": "inputs (15 GB weights + 28 GB KV) exceed L2",
                       "kv_page_tokens": 64, "device_ms_per_step_excl_host_gaps": round(r["device_ms_per_step"], 4)},
            "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
            "prefill": {"tokens": BATCH * (ctx0 - 1), "ms": round(r["prefill_ms"], 1),
                        "tokens_per_sec": round(BATCH * (ctx0 - 1) / (r["prefill_ms"] / 1e3), 1)}}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # the CPU leg runs on rank 0 at N=1 only
        line["cpu_baseline"] = cpu_baseline(args.cpu_tokens)
    eng.close()
    if not args.no_react:
        rb = react_block(args, rank, world, local_rank, barrier, allmax)
        if rank == 0:
            line["react"] = rb
    if world >= 2 and not args.no_router:
        try:
            rb = router_block(args, rank, world, host_barrier, dist, cpu_group)
        except Exception as e:
            rb = {"error": f"{type(e).__name__}: {e}"}
            host_barrier()
        if rank == 0:
            line["router"] = rb
        torch.cuda.set_device(local_rank)          # rank 0 drove engines on every GPU from worker threads; make sure NCCL's device is current again
    hung = False
    if world >= 2 and not args.no_tp:
        tp, hung = tp_block()
        if rank == 0:
            line["tp"] = tp
    if rank == 0:
        print(json.dumps(line), flush=True)      # before any teardown: a hard exit in NCCL/driver teardown must not eat the line
        sys.stdout.flush()
    if hung:
        os._exit(3)                               # a wedged TP leg: the line is out; let torchrun tear the other ranks down
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


DUMP_LOGIT_COLUMNS = 32768


def dump_outputs(out_dir, r):
    """What the last timed decode step computed, so that two builds can be compared output for output on identical inputs (seeded
    weights, seeded prompt ids): every sequence's next-token id, the logit it won with, and the fp32 logits at a fixed seeded sample
    of vocabulary columns (all 128 x 128,256 of them would be 66 MB)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    ids, logits = r["last_ids"], r["last_logits"]
    cols = np.sort(np.random.default_rng(0).choice(logits.shape[1], size=min(DUMP_LOGIT_COLUMNS, logits.shape[1]), replace=False))
    arrays = {"decode_next_token_ids": ids.astype(np.float64), "decode_next_token_logit": logits[np.arange(len(ids)), ids],
              "decode_logits_sample": logits[:, cols], "decode_logits_sample_columns": cols.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_baseline(n_decode=24, n_prompt=32, ctx=MEAN_CTX, repeats=3):
    """The oracle (CPU port of the same decoder, same seeded 8B weights) on the host cores: B=1 (a single-slot local server), decode steps
    at the BENCHMARK's context length — the cache positions [0, ctx) are filled with seeded values (oracle fill_kv: a timing aid, a CPU
    prefill of 1,664 tokens alone would take a minute) — median of `repeats` runs of n_decode tokens; plus a short real prefill for the
    prefill rate.  A bounded sample (about 15 s of CPU work), not the target: the roofline fraction is."""
    from oracle import oracle as O
    import numpy as np
    spec = O.PRESETS[MODEL]
    t0 = time.perf_counter()
    orc = O.Oracle(spec, max_pos=ctx + n_decode * repeats + n_prompt + 16, n_slots=1, mode=1)
    t_init = time.perf_counter() - t0
    prompt = (np.arange(n_prompt) * 7919 % 256).astype(np.int32)
    t0 = time.perf_counter(); orc.forward(prompt); t_pre = time.perf_counter() - t0
    orc.fill_kv(ctx)
    rates, pos = [], ctx
    tok = np.array([1], np.int32)
    for _rep in range(repeats):
        t0 = time.perf_counter()
        for _i in range(n_decode):
            lg = orc.forward(tok, pos0=pos)
            tok = np.array([int(lg[0].argmax())], np.int32); pos += 1
        rates.append(n_decode / (time.perf_counter() - t0))
    cores = O.lib().oa_ref_num_threads()
    orc.close()
    rates.sort()
    return {"value": round(rates[len(rates) // 2], 3), "unit": "tokens/s", "cores": int(cores), "kind": "port", "runs": [round(r, 3) for r in rates],
            "sample": f"oracle/llama_ref.c bf16-faithful mode, Llama-3-8B seed=1234, B=1, median of {repeats} x {n_decode} decode steps at ctx {ctx}-{pos} "
                      f"(cache pre-filled with seeded values, not prefilled on the CPU) + a {n_prompt}-token prefill ({t_pre:.1f}s); weight generation {t_init:.0f}s not timed",
            "prefill_tokens_per_sec": round(n_prompt / t_pre, 2)}


def run_reference(args, rank, world):
    """Reference arm: the reference's own path is an HTTP client with no arithmetic (pkg/llms/openai.go:69); its
    'CPU implementation' is whatever server it points at.  oracle/_ref cannot exist (pure Go, no Go toolchain), so
    this times the CPU port with all host threads on a bounded sample of the same workload."""
    if rank != 0:
        return
    K = max(1, min(args.steps, 64))             # ~0.13 s per token on 16 cores: the whole arm stays well under a few minutes
    cb = cpu_baseline(n_decode=max(8, K // 3 + min(args.warmup, 2)))
    v = cb["value"]
    line = {"impl": "reference", "metric": "decode_tokens_per_sec", "value": v, "unit": "tokens/s", "n_gpus": world, "steps": K,
            "warmup": min(args.warmup, 2), "ms_per_step": round(1e3 / v, 2) if v else None, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 weights, fp32 accumulate", "data": "synthetic (same seeded weights)",
            "config": {"workload": f"BASELINE configs[1] model (Llama-3-8B) on host cores, B=1 sequential (single-slot local server), decode ctx {MEAN_CTX}",
                       "parallelism": "cpu"},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64, help="timed decode steps of the headline")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kv-gb", type=float, default=60.0, dest="kv_gb")
    ap.add_argument("--cpu-tokens", type=int, default=24, dest="cpu_tokens")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--router-front", choices=["native", "python"], default="native", help="the serving block's front: csrc/http_server.cpp (default) or router.py + http_front.py")
    ap.add_argument("--no-router", action="store_true", help="N>=2: skip the one-front / N-engines serving block")
    ap.add_argument("--no-react", action="store_true", help="skip the multi-step ReAct block")
    ap.add_argument("--react-agents", type=int, default=128, dest="react_agents")
    ap.add_argument("--react-tool-ms", type=float, default=0.0, dest="react_tool_ms", help="synthetic tool latency (mean, ms; uniform 0.5x-1.5x): staggers the agents like a real kubectl would")
    ap.add_argument("--react-only", action="store_true", help="dev: only the react block")
    ap.add_argument("--no-tp", action="store_true", help="N>=2: skip the tensor-parallel block")
    ap.add_argument("--no-tp-parity", action="store_true")
    ap.add_argument("--tp-cases", default="", help="comma-separated tiny presets for the TP parity check (default: by degree)")
    ap.add_argument("--tp-model", default="", help="override the TP bench config (dev): model, with --tp-batch/--tp-ctx")
    ap.add_argument("--tp-batch", type=int, default=64)
    ap.add_argument("--tp-ctx", type=int, default=1024)
    ap.add_argument("--engine-extra", default="{}", dest="engine_extra", help="dev: JSON of engine options merged into the config (A/B runs)")
    ap.add_argument("--tp-deadline", type=float, default=900.0, dest="tp_deadline")
    ap.add_argument("--tp-only", action="store_true", help="dev: only the tensor-parallel block (prints {\"tp\": ...}; NOT a bench line)")
    ap.add_argument("--dump-outputs", default="", dest="dump_outputs", metavar="DIR",
                    help="write what the last timed decode step computed as DIR/<name>.npy (float32/float64; that one step also stores its logits)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: spawn torchrun ourselves
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
