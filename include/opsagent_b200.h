/*
 * opsagent_b200.h — C ABI of the B200-native local chat-completion engine.
 *
 * This is the drop-in boundary behind OpsAgent's LLM seam.  The reference has no FFI for this path;
 * its seam is the Go method
 *     func (c *OpenAIClient) Chat(model string, maxTokens int, prompts []openai.ChatCompletionMessage) (string, error)
 * (reference pkg/llms/openai.go:69-104), which today POSTs {model, messages, max_tokens, temperature}
 * to a remote /chat/completions server.  The entry points below are what a `local-cuda` provider binds
 * through cgo instead (INTEGRATION.md shows the Go side).  Plain C types only; no exceptions cross the
 * boundary; every function is safe to call from any thread.
 *
 * Return codes mirror the HTTP statuses the reference's retry loop already understands
 * (pkg/llms/openai.go:85-101): 0 ok; 400 bad request (fails fast); 429 queue/KV full (caller backs
 * off 1,2,4,8,16 s and retries); 500 device or internal fault (retried likewise).
 */
#ifndef OPSAGENT_B200_H
#define OPSAGENT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define OA_API __attribute__((visibility("default")))
#else
#define OA_API
#endif

#define OA_OK 0
#define OA_ERR_BAD_REQUEST 400
#define OA_ERR_TIMEOUT 408
#define OA_ERR_OVERLOADED 429
#define OA_ERR_INTERNAL 500

typedef struct oa_engine oa_engine; /* opaque, process-global, thread-safe */

/* replaces openai.ChatCompletionMessage{Role, Content} (go-openai v1.38.0; used at pkg/llms/openai.go:69) */
typedef struct {
    const char* role;    /* "system" | "user" | "assistant"; UTF-8, NUL-terminated, caller-owned */
    const char* content; /* UTF-8, NUL-terminated, caller-owned */
} oa_msg;

/* replaces openai.ChatCompletionRequest as built at pkg/llms/openai.go:70-75 */
typedef struct {
    const char* model;     /* must name the loaded model (or be empty/NULL) — else 400 */
    const oa_msg* msgs;
    int32_t n_msgs;
    int32_t max_tokens;    /* completion budget (8192 from pkg/handlers/execute.go:205) */
    float temperature;     /* the reference always sends SmallestNonzeroFloat32: greedy. Values > 1e-3 -> 400 */
    uint64_t seed;         /* unused under greedy decoding; kept for ABI stability */
    uint32_t flags;        /* OA_FLAG_* */
    const char* functions; /* OA_FLAG_JSON_FUNCTION: "name:param,name:param" — the functions the request's `tools` array offers */
} oa_chat_req;

#define OA_FLAG_IGNORE_EOS 1u /* throughput runs: always generate exactly max_tokens tokens */
#define OA_FLAG_JSON_TOOLCALL 2u /* force the completion to parse as tools.ToolPrompt (pkg/tools/tool.go:29-38) with an action from the
                                  * tool registry (tool.go:20-26) and an empty final_answer: one ReAct tool-call step */
#define OA_FLAG_JSON_FUNCTION 8u /* OpenAI function calling (swarm-go flows, pkg/workflows/swarm.go:14-78): the completion is
                                  * {"name":"<offered function>","arguments":{"<its parameter>":"..."}} */
#define OA_FLAG_JSON_TEXT 16u    /* one bounded line of printable text (10..200 bytes), newline-terminated */
#define OA_FLAG_JSON_FINAL 4u    /* same schema, empty action, final_answer of >= 10 bytes (not a placeholder per simple.go:640-654) */

/* replaces resp.Choices[0].Message.Content (+ usage) at pkg/llms/openai.go:82 */
typedef struct {
    char* content;         /* engine-owned, NUL-terminated, may contain embedded NULs: use content_len */
    int32_t content_len;
    int32_t prompt_tokens, completion_tokens;
    int32_t finish_reason; /* 0 stop (EOS), 1 length */
    int32_t* token_ids;    /* completion token ids (engine-owned), length completion_tokens */
} oa_chat_resp;

/* config_json: {"model":"llama-3-8b"|"llama-3.2-1b"|"qwen2.5-32b"|"llama-3-70b"|custom dims..., "seed":1234,
 *  "device":0, "kv_gb":100, "max_batch":128, "max_seq_len":4096, "max_step_tokens":8192, ...} — see DESIGN.md */
OA_API int oa_engine_create(const char* config_json, oa_engine** out);
OA_API void oa_engine_destroy(oa_engine*);
/* tensor-parallel groups (config "tp": t, "tp_rank": r, "tp_shm": name; one process per GPU): rank 0 is the engine callers talk
 * to; every other rank calls oa_engine_serve(), which replays the leader's steps and returns when the leader is destroyed */
OA_API int oa_engine_serve(oa_engine*);

/* blocking completion — what (*LocalCUDAClient).Chat calls; replaces CreateChatCompletion (openai.go:79) */
OA_API int oa_chat_complete(oa_engine*, const oa_chat_req*, oa_chat_resp* out);
/* non-blocking pair for callers that must not pin an OS thread per request (Go: submit, then wait) */
OA_API int oa_chat_submit(oa_engine*, const oa_chat_req*, uint64_t* ticket);
OA_API int oa_chat_wait(oa_engine*, uint64_t ticket, int32_t timeout_ms, oa_chat_resp* out);
/* abandon a submitted request (wait timed out, caller's context cancelled): frees its queue slot / KV pages; the ticket dies */
OA_API int oa_chat_cancel(oa_engine*, uint64_t ticket);
/* the same pair with the error text copied into a caller buffer instead of the thread-local oa_last_error(): what the cgo binding
 * uses, so that goroutines need not be pinned to an OS thread with runtime.LockOSThread for the duration of a Chat */
OA_API int oa_chat_submit_ex(oa_engine*, const oa_chat_req*, uint64_t* ticket, char* errbuf, size_t errcap);
OA_API int oa_chat_wait_ex(oa_engine*, uint64_t ticket, int32_t timeout_ms, oa_chat_resp* out, char* errbuf, size_t errcap);
OA_API void oa_free_resp(oa_chat_resp*);

/* same pair on raw token ids (bench + parity tests; bypasses the chat template) */
OA_API int oa_tokens_submit(oa_engine*, const int32_t* prompt, int32_t n_prompt, int32_t max_tokens, uint32_t flags, uint64_t* ticket);

/* tokenizer-accurate counting for pkg/llms/tokens.go:60 NumTokensFromMessages / :128 ConstrictPrompt */
OA_API int oa_count_tokens(oa_engine*, const oa_msg* msgs, int32_t n_msgs, int32_t* out_tokens);
/* chat template + tokenizer only: writes up to cap ids, returns total count in *n_out */
OA_API int oa_apply_chat_template(oa_engine*, const oa_msg* msgs, int32_t n_msgs, int32_t* out_ids, int32_t cap, int32_t* n_out);

OA_API const char* oa_last_error(void);                      /* thread-local message of the last failing call */
OA_API int oa_engine_stats(oa_engine*, char* buf, size_t n); /* JSON: steps, tokens, pages, launches, timings */
OA_API int oa_model_info(oa_engine*, char* buf, size_t n);   /* JSON: resolved architecture */

/* ---- native OpenAI-compatible HTTP front (csrc/http_server.cpp): what the UNMODIFIED reference binary is pointed at (`baseUrl` of POST /api/execute,
 * pkg/handlers/execute.go:21,205; OPENAI_API_BASE for the swarm flows, pkg/workflows/swarm.go:83).  POST /v1/chat/completions in go-openai's wire
 * format (openai.go:70-82) incl. `tools` -> grammar-forced `tool_calls`, GET /v1/models, GET /api/perf/stats.  One OS thread per connection; with
 * n_engines > 1 (data-parallel replicas, BASELINE configs[2]) conversations stick to the replica holding their prefix pages, new ones go to the
 * least-loaded replica, a replica over `max_inflight` answers 429 (openai.go:91-94 backs off).
 * options_json (flat): {"host":"127.0.0.1","port":0,"require_key":1,"api_key":"","tool_steps":3,"max_inflight":256,"max_connections":8192,"max_body_bytes":67108864,"idle_timeout_s":120} */
typedef struct oa_http oa_http;
OA_API int oa_http_start(oa_engine* const* engines, int32_t n_engines, const char* options_json, oa_http** out);
OA_API int32_t oa_http_port(oa_http*);                        /* the bound port (options "port": 0 picks a free one) */
OA_API int oa_http_stats(oa_http*, char* buf, size_t n);      /* JSON: requests, routed / in flight per replica, 429s, sticky hits, engine stats */
OA_API void oa_http_stop(oa_http*);                           /* stops accepting, waits for the connection threads; the engines stay alive */
OA_API const char* oa_http_last_error(void);

/* ---- measurement + parity hooks (used by bench.py and tests/; not part of the Go seam) ---- */
/* fresh single-sequence prefill of `tokens`; fp32 logits of every position -> logits_out[n, vocab] */
OA_API int oa_debug_prefill_logits(oa_engine*, const int32_t* tokens, int32_t n, float* logits_out);
/* Device-resident decode benchmark: builds `batch` sequences of `ctx_len` cached tokens (real chunked prefill of
 * seeded synthetic ids), then runs warmup+steps decode forwards of the whole batch, timed with CUDA events on the
 * engine stream.  out[0]=ms/step over ONE event bracket around all timed steps (host gaps included), out[1]=prefill ms, out[2]=kernel launches per step, out[3]=mean ctx over the
 * timed steps, out[4]=attention-kernel ms/step (avg), out[5]=algorithmic bytes/step,
 * out[6]=sum of per-step device durations / steps (host gaps excluded) */
OA_API int oa_bench_decode(oa_engine*, int32_t batch, int32_t ctx_len, int32_t steps, int32_t warmup, double* out, int32_t n_out);
/* the same, plus what the last timed step computed: next-token ids -> last_ids[batch] and, when last_logits is not NULL, its fp32
 * logits -> last_logits[batch, vocab] (that one step then also stores them; its ids are unchanged).  Either pointer may be NULL. */
OA_API int oa_bench_decode_ex(oa_engine*, int32_t batch, int32_t ctx_len, int32_t steps, int32_t warmup, double* out, int32_t n_out,
                              int32_t* last_ids, float* last_logits);

/* in-situ per-kernel-class timings accumulated while OA_PROFILE_ALL=1 (JSON name -> [total ms, launches]) */
OA_API int oa_debug_kernel_times(oa_engine*, char* buf, size_t n, int32_t reset);

/* kernel-level entry points on raw device pointers (tests call these with torch-allocated memory) */
OA_API int oa_k_rmsnorm(const void* x, const void* gain, void* y, int32_t T, int32_t H, float eps, void* stream);
OA_API int oa_k_gemm(const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t block_n, void* out,
              const void* bias, const void* resid, float* logits, int32_t* argmax_out, void* stream);
/* persistent stream-K GEMM (M <= 128) followed by the fixed-order partial sum: out_f32[M,N] */
OA_API int oa_k_gemm_streamk(const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t block_n, int32_t n_ctas, float* out_f32, void* stream);
OA_API int oa_k_init_weight(void* dst, uint64_t seed, uint64_t tensor_id, int64_t tensor_id_b, int64_t rows, int64_t cols, float std,
                     float mean, void* stream);
/* paged attention on a caller-provided cache [2(K,V)][num_pages][n_kv][64][D] (one layer): decode when q has one
 * row per sequence (n_q_rows == n_seqs), otherwise causal prefill of `q_lens[i]` new rows per sequence */
OA_API int oa_k_paged_attention(const void* q, void* out, const void* kv_cache, int32_t num_pages, const int32_t* block_tables,
                         int32_t max_pages_per_seq, const int32_t* ctx_lens, const int32_t* q_lens, int32_t n_seqs,
                         int32_t n_heads, int32_t n_kv, int32_t head_dim, int32_t force_splits, void* stream);
/* the same on one layer of a cache [n_layers][2][num_pages][n_kv][64][D], with the decode plan's CTA target (<= 0: two per SM, the
 * engine's default) and, for decode, the merge: merge_counters NULL = separate merge kernel, else a device int32 array with one counter
 * per cut (sequence, kv head) item, zeroed once by the caller — the kernel merges in place and each call advances an item's counter by its
 * piece count (the engine's per-layer use within one step) */
OA_API int oa_k_paged_attention_ex(const void* q, void* out, const void* kv_cache, int32_t num_pages, int32_t n_layers, int32_t layer,
                                   const int32_t* block_tables, int32_t max_pages_per_seq, const int32_t* ctx_lens, const int32_t* q_lens,
                                   int32_t n_seqs, int32_t n_heads, int32_t n_kv, int32_t head_dim, int32_t force_splits, int32_t n_ctas_target,
                                   int32_t* merge_counters, void* stream);
/* Decode projections (M <= 128) with their fused epilogues, launched as the engine launches them.  All pointers are device pointers;
 * B is the [N, K] weight; tile_flags = caller-owned zeroed uint32 counters (>= N/128), which the fused kernels leave zeroed again.
 * o / down: x[M, ldx] += A.B^T (bf16, in place), then xn[M, N] = rmsnorm(x) * gain.
 *   path 0: stream-K GEMM + sum/residual/norm consumer (default); 1: stream-K GEMM finishing the residual + norm kernel;
 *   2: cluster split-K GEMM with `cluster` CTAs per tile + norm kernel.  xn NULL (paths 1, 2) skips the norm; with a norm, ldx == N. */
OA_API int oa_k_sk_resid_rmsnorm(int32_t path, const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t n_ctas, int32_t cluster,
                                 void* x, int32_t ldx, const void* gain, void* xn, float eps, uint32_t* tile_flags, void* stream);
/* gate/up: B = [2F, K] with rows interleaved 16 gate / 16 up; act[M, F] = silu(gate) * up.
 *   path 0: stream-K GEMM + SwiGLU consumer; 1: stream-K GEMM finishing the SwiGLU (default). */
OA_API int oa_k_sk_swiglu(int32_t path, const void* A, const void* B, int32_t M, int32_t F, int32_t K, int32_t n_ctas, void* act,
                          uint32_t* tile_flags, void* stream);
/* qkv: B = [(nh + 2 nkv) D, K], optional bias; rows -> (+ bias) -> bf16 -> RoPE at positions[M] -> q_out[M, nh*D] and the K/V rows of
 * slots[M] in layer `layer` of kv_cache [n_layers][2][num_pages][nkv][64][D].  rope_cos/sin: [max_pos, D/2] fp32.
 *   path 0: stream-K GEMM + RoPE/KV consumer (default); 1: stream-K GEMM finishing RoPE + KV write; 2: cluster split-K GEMM with
 *   `cluster` CTAs per tile; 3: tile GEMM (bf16 qkv + bias) + RoPE/KV kernel (the prefill path). */
OA_API int oa_k_qkv_rope(int32_t path, const void* A, const void* B, int32_t M, int32_t K, int32_t n_ctas, int32_t cluster, const void* bias,
                         const int32_t* positions, const int32_t* slots, const float* rope_cos, const float* rope_sin, void* q_out,
                         void* kv_cache, int32_t num_pages, int32_t n_layers, int32_t layer, int32_t nh, int32_t nkv, int32_t D,
                         uint32_t* tile_flags, void* stream);
/* LM head: logits[M, N] fp32 (optional) and ids[M] = per-row arg-max (ties -> lowest column).  Rows with mask_slot[r] >= 0 take the
 * arg-max only over columns c whose bit col_offset + c is set in mask_table[mask_slot[r] * mask_words ...]; ids are shard-local columns. */
OA_API int oa_k_lm_head(const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t block_n, const uint32_t* mask_table,
                        const int32_t* mask_slot, int32_t mask_words, int32_t col_offset, float* logits, int32_t* ids, void* stream);
/* ---- host-only logic, callable without a GPU (CPU tests) ---- */
/* chat template + tokenizer of the model described by config_json */
OA_API int oa_host_apply_chat_template(const char* config_json, const oa_msg* msgs, int32_t n_msgs, int32_t* out_ids, int32_t cap, int32_t* n_out);
/* decode-attention work plan: segs_out[cap_segs*5] = {seq, kvh, chunk_begin, chunk_end, partial_slot}, cta_ptr_out[n_ctas+1];
 * returns the number of CTAs in *n_ctas_out and of segments in *n_segs_out */
OA_API int oa_host_decode_plan(const int32_t* ctx_lens, int32_t n_seqs, int32_t n_kv, int32_t n_ctas_target, int32_t force_splits,
                        int32_t* segs_out, int32_t cap_segs, int32_t* cta_ptr_out, int32_t cap_ctas, int32_t* n_ctas_out,
                        int32_t* n_segs_out, int32_t* n_slots_out);
/* stream-K unit plan of the decode projections (host only, no GPU): CTA c owns k-block units [cta_unit0[c], cta_unit0[c+1]) of
 * n_tiles x kb units (tile-major); tile_first/tile_last = the CTAs holding a tile's first and last k-block, computed with the
 * closed form the kernels use (floor(((u+1)*G-1)/total)).  The fused SwiGLU epilogue relies on: pieces of a tile are exactly
 * CTAs tile_first..tile_last, the first CTA's piece is the LAST segment of that CTA and every other piece is the FIRST segment
 * of its CTA (so the finishing CTA never waits on a CTA that is itself waiting). */
OA_API int oa_host_streamk_plan(int32_t N, int32_t K, int32_t block_n, int32_t n_ctas, int64_t* cta_unit0_out, int32_t cap_ctas,
                         int32_t* tile_first_out, int32_t* tile_last_out, int32_t cap_tiles, int32_t* n_ctas_out, int32_t* n_tiles_out,
                         int32_t* kb_out);
/* cluster size (8, 4, 3, 2) the decode path would give the cluster split-K GEMM of an N x K projection on `sms` SMs, or 0 (keep stream-K) */
OA_API int32_t oa_host_clusterk_pick(int32_t N, int32_t K, int32_t sms, int32_t min_fill_pct);
/* byte-level BPE tokenizer read from a Hugging Face tokenizer.json (Llama-3 / Qwen2.5 format), host only: what the engine uses
 * for text when its config names one ("tokenizer": path) instead of the synthetic byte-level vocabulary.  Loaded files are cached
 * by path.  encode: *n_out = number of ids (written up to cap; OA_ERR_BAD_REQUEST if cap is too small or the file is unsupported);
 * decode: bytes of the ids (control tokens render as their literal content). */
OA_API int oa_host_bpe_encode(const char* tokenizer_json_path, const char* text, int32_t text_len, int32_t* ids_out, int32_t cap, int32_t* n_out);
OA_API int oa_host_bpe_decode(const char* tokenizer_json_path, const int32_t* ids, int32_t n_ids, char* buf, int32_t cap, int32_t* n_out);
/* grammar automaton, host only: feeds `prefix` (n bytes) to the schema `kind` (1 tool call, 2 final) and returns the allowed-byte
 * bitset for the next position in mask_out[8], *done_out = 1 when the JSON is complete; 400 if the prefix is not derivable */
OA_API int oa_host_grammar_step(int32_t kind, const uint8_t* prefix, int32_t n, uint32_t* mask_out, int32_t* done_out);
OA_API int oa_host_grammar_step_ex(int32_t kind, const char* functions, const uint8_t* prefix, int32_t n, uint32_t* mask_out, int32_t* done_out);
/* token-level grammar mask, host only: the bitset (ceil(vocab/32) words) of token ids allowed after `prefix` under schema `kind`, for the
 * byte-level BPE vocabulary of tokenizer_json_path (NULL/"": the synthetic byte-level ids 0..255) — a token is allowed iff all of its bytes
 * walk the automaton.  key_out receives the canonical cache key of the state (states with equal keys have equal masks). */
OA_API int oa_host_grammar_token_mask(const char* tokenizer_json_path, int32_t vocab, int32_t kind, const char* functions, const uint8_t* prefix,
                               int32_t n, uint32_t* mask_out, int32_t cap_words, char* key_out, int32_t key_cap);
OA_API int oa_host_json_roundtrip(const uint8_t* in, size_t n_in, char* out, size_t n_out);   /* the HTTP front's JSON reader + writer, for the CPU tests */
/* resolved architecture + derived byte counts of a config, no device needed */
OA_API int oa_host_model_info(const char* config_json, char* buf, size_t n);
OA_API uint64_t oa_kernel_launches(void);
OA_API const char* oa_version(void);

#ifdef __cplusplus
}
#endif
#endif
