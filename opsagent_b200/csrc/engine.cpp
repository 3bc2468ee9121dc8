// engine.cpp — request scheduler (continuous batching over a paged KV pool) and the C ABI of
// include/opsagent_b200.h.
//
// Concurrency shape preserved from the reference: every in-flight agent request blocks in one Chat call on
// its own goroutine (reference pkg/handlers/execute.go:205 -> pkg/assistants/simple.go:343,515 ->
// pkg/llms/openai.go:69).  Here those callers block in oa_chat_complete / oa_chat_wait while ONE scheduler
// thread batches all of them data-parallel into shared prefill / decode forwards.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <list>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>

#include <cuda_profiler_api.h>

#include "../../include/opsagent_b200.h"
#include "grammar.hpp"
#include "token_mask.hpp"
#include "model.hpp"
#include "tokenizer.hpp"

namespace oa {

static thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) { g_last_error = msg; return code; }

// selects `dev` on the calling thread for a scope and restores what was current before (the CUDA current device is per thread)
struct CallerDevice {
    int prev = -1;
    explicit CallerDevice(int dev) { cudaGetDevice(&prev); cudaSetDevice(dev); }
    ~CallerDevice() { if (prev >= 0) cudaSetDevice(prev); }
};

enum class SeqState { WAITING, PREFILL, DECODE, DONE };

struct Seq {
    uint64_t ticket = 0;
    std::vector<int32_t> tokens;     // prompt + generated so far
    int n_prompt = 0, n_cached = 0, n_generated = 0, max_new = 0;
    uint32_t flags = 0;
    std::vector<int32_t> pages;
    SeqState state = SeqState::WAITING;
    int finish_reason = 1;
    int error = 0; std::string error_msg;
    bool done = false;
    ToolPromptGrammar grammar;       // inactive unless the request asked for schema-constrained JSON
    int n_registered = 0; uint64_t hash_prev = 0;   // prefix cache: full pages already published / hash of that chain
    std::chrono::steady_clock::time_point t_enqueue{};   // arrival (admission batching)
    bool preempted = false;                              // pushed back by the scheduler: re-admit without waiting
    bool cancelled = false;                              // oa_chat_cancel: dropped at the next step boundary
    int est_uncached = -1;                               // prompt tokens a prefill would have to compute (prefix-cache walk, made once)
};

class Engine {
public:
    Engine(const ModelConfig& mc, const EngineOptions& eo) : model_(mc, eo), tok_(mc, eo.tokenizer), opt_(eo) {
        free_pages_.reserve(model_.num_pages);
        for (int p = model_.num_pages - 1; p >= 0; --p) free_pages_.push_back(p);
        page_ref_.assign(model_.num_pages, 0); page_hash_.assign(model_.num_pages, 0); page_parent_.assign(model_.num_pages, 0);
        page_tokens_.assign((size_t)model_.num_pages * 64, 0); lru_pos_.assign(model_.num_pages, lru_.end());
        token_bytes_ = tok_.text_token_bytes();
        trie_.build(token_bytes_, model_.cfg.vocab);
        mask_key_of_.assign((size_t)model_.mask_slots, std::string()); mask_last_use_.assign((size_t)model_.mask_slots, 0);
        if (eo.tp > 1 && eo.tp_rank > 0) follower_ = std::thread([this] { follow(); });   // tensor-parallel follower: replays the leader's steps
        else if (eo.start_thread) worker_ = std::thread([this] { loop(); });
    }
    ~Engine() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
        cv_work_.notify_all();
        if (worker_.joinable()) worker_.join();
        if (model_.comm && opt_.tp_rank == 0) { std::lock_guard<std::mutex> step(step_mu_); CallerDevice on_engine_device(opt_.device); model_.sync(); model_.comm->shutdown(); }
        if (follower_.joinable()) follower_.join();
    }
    bool is_follower() const { return opt_.tp > 1 && opt_.tp_rank > 0; }
    // blocks a follower process until the leader shuts the group down (returns at once on a leader / single-GPU engine)
    int serve() {
        if (!is_follower()) return OA_OK;
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, [&] { return follower_done_; });
        return fatal_ ? fail(OA_ERR_INTERNAL, fatal_msg_) : OA_OK;
    }

    int submit_tokens(std::vector<int32_t>&& prompt, int max_new, uint32_t flags, uint64_t* ticket, const char* functions = nullptr) {
        if (is_follower()) return fail(OA_ERR_BAD_REQUEST, "tensor-parallel followers take no requests: submit to the leader (tp_rank 0)");
        if (prompt.empty()) return fail(OA_ERR_BAD_REQUEST, "empty prompt");
        if (max_new <= 0) return fail(OA_ERR_BAD_REQUEST, "max_tokens must be positive");
        if ((int)prompt.size() + 1 > opt_.max_seq_len)
            return fail(OA_ERR_BAD_REQUEST, "prompt of " + std::to_string(prompt.size()) + " tokens exceeds max_seq_len " + std::to_string(opt_.max_seq_len));
        for (int32_t t : prompt) if (t < 0 || t >= model_.cfg.vocab) return fail(OA_ERR_BAD_REQUEST, "token id out of range");
        auto s = std::make_shared<Seq>();
        s->n_prompt = (int)prompt.size(); s->tokens = std::move(prompt);
        s->max_new = std::min(max_new, opt_.max_seq_len - s->n_prompt); s->flags = flags;
        if (flags & OA_FLAG_JSON_TOOLCALL) s->grammar = ToolPromptGrammar(GRAMMAR_TOOLCALL);
        else if (flags & OA_FLAG_JSON_FINAL) s->grammar = ToolPromptGrammar(GRAMMAR_FINAL);
        else if (flags & OA_FLAG_JSON_FUNCTION) {
            s->grammar = ToolPromptGrammar(GRAMMAR_FUNCTION, functions ? functions : "");
            if (!s->grammar.active()) return fail(OA_ERR_BAD_REQUEST, "OA_FLAG_JSON_FUNCTION needs functions=\"name:param,...\"");
        } else if (flags & OA_FLAG_JSON_TEXT) s->grammar = ToolPromptGrammar(GRAMMAR_TEXT);
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (fatal_) return fail(OA_ERR_INTERNAL, "engine is in a failed state: " + fatal_msg_);
            if ((int)waiting_.size() >= opt_.max_queue) return fail(OA_ERR_OVERLOADED, "request queue full");
            s->ticket = next_ticket_++;
            s->t_enqueue = std::chrono::steady_clock::now();
            waiting_.push_back(s); by_ticket_[s->ticket] = s;
            *ticket = s->ticket;
        }
        cv_work_.notify_one();
        return OA_OK;
    }

    int wait(uint64_t ticket, int timeout_ms, oa_chat_resp* out) {
        std::shared_ptr<Seq> s;
        {
            std::unique_lock<std::mutex> lk(mu_);
            auto it = by_ticket_.find(ticket);
            if (it == by_ticket_.end()) return fail(OA_ERR_BAD_REQUEST, "unknown ticket");
            s = it->second;
            auto pred = [&] { return s->done; };
            if (timeout_ms < 0) cv_done_.wait(lk, pred);
            else if (!cv_done_.wait_for(lk, std::chrono::milliseconds(timeout_ms), pred)) return fail(OA_ERR_TIMEOUT, "timeout");
            by_ticket_.erase(ticket);
        }
        if (s->error) return fail(s->error, s->error_msg);
        std::vector<int32_t> gen(s->tokens.begin() + s->n_prompt, s->tokens.end());
        std::string text = tok_.detokenize(gen);
        out->content = (char*)std::malloc(text.size() + 1);
        std::memcpy(out->content, text.data(), text.size()); out->content[text.size()] = 0;
        out->content_len = (int32_t)text.size();
        out->prompt_tokens = s->n_prompt; out->completion_tokens = (int32_t)gen.size(); out->finish_reason = s->finish_reason;
        out->token_ids = (int32_t*)std::malloc(std::max<size_t>(1, gen.size()) * 4);
        std::memcpy(out->token_ids, gen.data(), gen.size() * 4);
        return OA_OK;
    }

    // Abandon a request (a caller whose oa_chat_wait timed out, a Go context that was cancelled): a waiting sequence is removed at once, a
    // running one is dropped by the scheduler at its next step boundary; either way its KV pages go back to the pool and the ticket dies.
    int cancel(uint64_t ticket) {
        std::lock_guard<std::mutex> lk(mu_);
        auto it = by_ticket_.find(ticket);
        if (it == by_ticket_.end()) return fail(OA_ERR_BAD_REQUEST, "unknown ticket");
        std::shared_ptr<Seq> s = it->second;
        by_ticket_.erase(it);
        if (s->done) return OA_OK;
        s->cancelled = true; ++n_cancelled_;
        for (auto w = waiting_.begin(); w != waiting_.end(); ++w)
            if (*w == s) { waiting_.erase(w); for (int p : s->pages) release_page_locked(p); s->pages.clear(); s->state = SeqState::DONE; s->done = true; break; }
        return OA_OK;
    }

    // ---- exclusive-use helpers (bench / parity); they hold step_mu_ so the scheduler is parked ----
    int debug_prefill_logits(const int32_t* toks, int n, float* logits_out) {
        if (n <= 0 || n > std::min(2048, opt_.max_step_tokens) || n + 1 > opt_.max_seq_len) return fail(OA_ERR_BAD_REQUEST, "debug prefill: 1..min(2048,max_step_tokens) tokens");
        std::lock_guard<std::mutex> step(step_mu_);
        CallerDevice on_engine_device(opt_.device);      // this helper launches from the CALLER's thread
        try {
            const int V = model_.cfg.vocab;
            std::vector<int32_t> pages;
            { std::lock_guard<std::mutex> lk(mu_); if (!alloc_pages_locked(pages, (n + 63) / 64)) return fail(OA_ERR_OVERLOADED, "no free KV pages"); }
            float* d_logits = nullptr;
            cuda_check(cudaMalloc(&d_logits, (size_t)n * V * 4), "cudaMalloc logits");
            StepInput in; in.decode = false; in.n_seqs = 1; in.want_logits = true;
            in.block_tables.assign(model_.max_pages_per_seq, 0);
            for (size_t i = 0; i < pages.size(); ++i) in.block_tables[i] = pages[i];
            in.ctx_lens = {n};
            for (int i = 0; i < n; ++i) { in.tokens.push_back(toks[i]); in.positions.push_back(i); in.slots.push_back(pages[i / 64] * 64 + i % 64); in.sample_rows.push_back(i); }
            for (int r = 0; r < n; r += PREFILL_TILE_ROWS) in.tiles.push_back(PrefillTile{0, r, r, std::min(PREFILL_TILE_ROWS, n - r)});
            run_forward(in, d_logits); model_.sync();
            cudaError_t e = cudaMemcpy(logits_out, d_logits, (size_t)n * V * 4, cudaMemcpyDeviceToHost);
            cudaFree(d_logits);
            { std::lock_guard<std::mutex> lk(mu_); for (int p : pages) release_page_locked(p); }
            cuda_check(e, "logits D2H");
        } catch (const std::exception& ex) { return fail(OA_ERR_INTERNAL, ex.what()); }
        return OA_OK;
    }

    // last_ids [batch] / last_logits [batch, vocab] (host, optional): what the last timed step computed; asking for the logits makes
    // that one step also store them (the arg-max it returns is unchanged)
    int bench_decode(int batch, int ctx_len, int steps, int warmup, double* out, int n_out, int32_t* last_ids = nullptr, float* last_logits = nullptr) {
        if (batch <= 0 || batch > opt_.max_batch || ctx_len <= 0 || ctx_len + steps + warmup + 1 > opt_.max_seq_len || n_out < 6)
            return fail(OA_ERR_BAD_REQUEST, "bench_decode: batch <= max_batch, ctx_len+steps+warmup < max_seq_len, n_out >= 6");
        std::lock_guard<std::mutex> step(step_mu_);
        CallerDevice on_engine_device(opt_.device);
        try {
            const int V = model_.cfg.vocab;
            const int total_len = ctx_len + steps + warmup;
            const int pages_per = (total_len + 63) / 64;
            std::vector<std::vector<int32_t>> pages(batch);
            {
                std::lock_guard<std::mutex> lk(mu_);
                if ((long long)pages_per * batch > (long long)available_pages_locked()) return fail(OA_ERR_OVERLOADED, "bench_decode: not enough KV pages");
                for (int b = 0; b < batch; ++b) alloc_pages_locked(pages[b], pages_per);
            }
            auto synth = [&](int b, int i) { uint64_t h = (uint64_t)(b + 1) * 0x9E3779B97F4A7C15ull + (uint64_t)i * 0xBF58476D1CE4E5B9ull; h ^= h >> 29; return (int32_t)(h % (uint64_t)V); };
            cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
            const bool prof_all = model_.profile_all; model_.profile_all = false;      // in-situ kernel timing covers the decode steps only
            // ---- prefill: ctx_len-1 tokens per sequence, chunked by the step token budget ----
            const int P = ctx_len - 1;
            cudaEventRecord(e0, model_.stream);
            {
                int b = 0, off = 0, n_fwd = 0;
                const bool prof_prefill = std::getenv("OA_CUDA_PROFILER_PREFILL") != nullptr;
                const bool skip_prefill = std::getenv("OA_BENCH_SKIP_PREFILL") != nullptr;   // dev profiling only: decode over whatever the (zero-initialised) pages hold
                while (b < batch && P > 0 && !skip_prefill) {
                    StepInput in; in.decode = false;
                    int budget = opt_.max_step_tokens;
                    while (b < batch && budget > 0 && in.n_seqs < opt_.max_batch) {
                        const int take = std::min(budget, P - off);
                        const int sidx = in.n_seqs++;
                        in.block_tables.resize((size_t)in.n_seqs * model_.max_pages_per_seq, 0);
                        for (size_t i = 0; i < pages[b].size(); ++i) in.block_tables[(size_t)sidx * model_.max_pages_per_seq + i] = pages[b][i];
                        in.ctx_lens.push_back(off + take);
                        const int row0 = (int)in.tokens.size();
                        for (int i = off; i < off + take; ++i) { in.tokens.push_back(synth(b, i)); in.positions.push_back(i); in.slots.push_back(pages[b][i / 64] * 64 + i % 64); }
                        for (int r = 0; r < take; r += PREFILL_TILE_ROWS) in.tiles.push_back(PrefillTile{sidx, row0 + r, off + r, std::min(PREFILL_TILE_ROWS, take - r)});
                        budget -= take; off += take;
                        if (off >= P) { off = 0; ++b; }
                    }
                    if (prof_prefill && n_fwd == 1) { model_.sync(); cudaProfilerStart(); }     // the 2nd prefill chunk (warm)
                    run_forward(in, nullptr);
                    if (prof_prefill && n_fwd == 1) { model_.sync(); cudaProfilerStop(); }
                    ++n_fwd;
                }
            }
            cudaEventRecord(e1, model_.stream); model_.sync();
            float prefill_ms = 0; cudaEventElapsedTime(&prefill_ms, e0, e1);
            // ---- decode steps ----
            model_.profile_all = prof_all;
            std::vector<int32_t> last(batch);
            for (int b = 0; b < batch; ++b) last[b] = synth(b, P);
            float* d_logits = nullptr;
            if (last_logits) cuda_check(cudaMalloc(&d_logits, (size_t)batch * V * 4), "cudaMalloc logits");
            double ctx_sum = 0; float total_ms = 0; uint64_t launches0 = 0;
            cudaEvent_t eb0, eb1; cudaEventCreate(&eb0); cudaEventCreate(&eb1);
            model_.attn_ms_accum = 0;
            for (int it = 0; it < warmup + steps; ++it) {
                const int pos = P + it;
                StepInput in; in.decode = true; in.n_seqs = batch;
                in.block_tables.assign((size_t)batch * model_.max_pages_per_seq, 0);
                for (int b = 0; b < batch; ++b) {
                    for (size_t i = 0; i < pages[b].size(); ++i) in.block_tables[(size_t)b * model_.max_pages_per_seq + i] = pages[b][i];
                    in.tokens.push_back(last[b]); in.positions.push_back(pos); in.slots.push_back(pages[b][pos / 64] * 64 + pos % 64);
                    in.ctx_lens.push_back(pos + 1); in.sample_rows.push_back(b);
                }
                if (it == warmup) {
                    if (std::getenv("OA_CUDA_PROFILER")) { model_.sync(); cudaProfilerStart(); }   // ncu --profile-from-start off
                    launches0 = launches_total(); model_.attn_ms_accum = 0; cudaEventRecord(eb0, model_.stream);
                }
                const bool timed = it >= warmup;
                float* step_logits = it == warmup + steps - 1 ? d_logits : nullptr;
                in.want_logits = step_logits != nullptr;
                if (timed) { cudaEventRecord(e0, model_.stream); ctx_sum += pos + 1; }
                run_forward(in, step_logits);
                if (timed) cudaEventRecord(e1, model_.stream);
                model_.sync();
                if (timed) { float ms = 0; cudaEventElapsedTime(&ms, e0, e1); total_ms += ms; }
                for (int b = 0; b < batch; ++b) last[b] = model_.h_out_ids[b];
            }
            cudaEventRecord(eb1, model_.stream); model_.sync();
            if (std::getenv("OA_CUDA_PROFILER")) cudaProfilerStop();
            float bracket_ms = 0; cudaEventElapsedTime(&bracket_ms, eb0, eb1);
            const uint64_t launches1 = launches_total();
            cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(eb0); cudaEventDestroy(eb1);
            if (last_ids) std::copy(last.begin(), last.end(), last_ids);
            cudaError_t le = cudaSuccess;
            if (d_logits) { le = cudaMemcpy(last_logits, d_logits, (size_t)batch * V * 4, cudaMemcpyDeviceToHost); cudaFree(d_logits); }
            { std::lock_guard<std::mutex> lk(mu_); for (auto& pv : pages) for (int p : pv) release_page_locked(p); }
            cuda_check(le, "logits D2H");
            const double mean_ctx = ctx_sum / steps;
            out[0] = bracket_ms / steps; if (n_out > 6) out[6] = total_ms / steps; out[1] = prefill_ms; out[2] = (double)(launches1 - launches0) / steps; out[3] = mean_ctx;
            out[4] = model_.profile_attn ? model_.attn_ms_accum / steps : 0.0;
            // SURVEY.md §8d: W_dec + sum ctx*KVB + B*KVB (the new token's KV write)
            out[5] = (model_.cfg.decode_weight_bytes() + (double)batch * mean_ctx * (double)model_.cfg.kv_bytes_per_token() +
                      (double)batch * (double)model_.cfg.kv_bytes_per_token()) / opt_.tp;      // per GPU (SURVEY §8d: W_dec/t + ctx*KVB/t)
        } catch (const std::exception& ex) { return fail(OA_ERR_INTERNAL, ex.what()); }
        return OA_OK;
    }

    std::string stats_json() {
        std::lock_guard<std::mutex> lk(mu_);
        char b[1024];
        std::snprintf(b, sizeof b,
                      "{\"requests_completed\": %llu, \"prefill_tokens\": %llu, \"decode_tokens\": %llu, \"prefill_steps\": %llu, "
                      "\"decode_steps\": %llu, \"preemptions\": %llu, \"pages_total\": %d, \"pages_free\": %zu, \"running\": %zu, "
                      "\"waiting\": %zu, \"kernel_launches\": %llu, \"h2d_bytes\": %llu, \"d2h_bytes\": %llu, \"weight_bytes\": %zu, "
                      "\"kv_pool_bytes\": %zu, \"busy_ms\": %.3f, \"prefix_hit_tokens\": %llu, \"pages_cached\": %zu, \"admissions_deferred\": %llu, \"mixed_steps\": %llu, \"cancelled\": %llu, \"grammar_states_computed\": %llu}",
                      (unsigned long long)n_completed_, (unsigned long long)n_prefill_tokens_, (unsigned long long)n_decode_tokens_,
                      (unsigned long long)n_prefill_steps_, (unsigned long long)n_decode_steps_, (unsigned long long)n_preempt_,
                      model_.num_pages, available_pages_locked(), running_.size(), waiting_.size(), (unsigned long long)launches_total(),
                      (unsigned long long)model_.h2d_bytes, (unsigned long long)model_.d2h_bytes, model_.weight_bytes, model_.kv_pool_bytes, busy_ms_, (unsigned long long)n_prefix_hit_tokens_, cached_.size(),
                      (unsigned long long)n_admit_deferred_, (unsigned long long)n_mixed_steps_, (unsigned long long)n_cancelled_, (unsigned long long)n_mask_states_);
        return b;
    }
    std::string info_json() {
        const ModelConfig& c = model_.cfg; char b[1024];
        std::snprintf(b, sizeof b,
                      "{\"model\": \"%s\", \"hidden\": %d, \"n_layers\": %d, \"n_heads\": %d, \"n_kv_heads\": %d, \"head_dim\": %d, \"ffn\": %d, "
                      "\"vocab\": %d, \"tie_embeddings\": %d, \"qkv_bias\": %d, \"rope_scaling\": %d, \"rope_theta\": %.1f, \"rms_eps\": %g, "
                      "\"template\": \"%s\", \"seed\": %llu, \"num_pages\": %d, \"page_size\": 64, \"max_seq_len\": %d, \"max_batch\": %d, "
                      "\"sm_count\": %d, \"decode_weight_bytes\": %.0f, \"kv_bytes_per_token\": %zu, \"tp\": %d, \"tp_nvls\": %d}",
                      c.name.c_str(), c.hidden, c.n_layers, c.n_heads, c.n_kv_heads, c.head_dim, c.ffn, c.vocab, c.tie_embeddings, c.qkv_bias,
                      c.rope_scaling, c.rope_theta, c.rms_eps, c.chat_template.c_str(), (unsigned long long)c.seed, model_.num_pages,
                      opt_.max_seq_len, opt_.max_batch, model_.sm_count, c.decode_weight_bytes(), c.kv_bytes_per_token(), opt_.tp, (model_.comm && model_.comm->nvls()) ? 1 : 0);
        return b;
    }
    bool serves_model(const std::string& name) const {
        if (name == model_.cfg.name) return true;
        const std::string& a = opt_.model_aliases;       // "gpt-4,gpt-4o" or "*": names the unmodified reference sends (execute.go:168-171 defaults to "gpt-4")
        size_t b = 0;
        while (b <= a.size()) {
            size_t e = a.find(',', b); if (e == std::string::npos) e = a.size();
            const std::string item = a.substr(b, e - b);
            if (item == "*" || (!item.empty() && item == name)) return true;
            b = e + 1;
        }
        return false;
    }
    const Tokenizer& tokenizer() const { return tok_; }
    const EngineOptions& options() const { return opt_; }
    const ModelConfig& config() const { return model_.cfg; }
    DeviceModel& model() { return model_; }

private:
    // every forward goes through here: the leader of a tensor-parallel group publishes the step for its followers first
    void run_forward(const StepInput& in, float* logits_out) {
        if (model_.comm && opt_.tp_rank == 0) model_.comm->publish(in);
        model_.forward(in, logits_out);
    }
    void follow() {
        cudaSetDevice(opt_.device);
        try {
            StepInput in;
            while (model_.comm->receive(in)) { model_.forward(in, nullptr); model_.sync(); }
        } catch (const std::exception& ex) {
            std::lock_guard<std::mutex> lk(mu_); fatal_ = true; fatal_msg_ = ex.what();
            std::fprintf(stderr, "opsagent_b200 follower %d failed: %s\n", opt_.tp_rank, ex.what());
        }
        { std::lock_guard<std::mutex> lk(mu_); follower_done_ = true; }
        cv_done_.notify_all();
    }
    // ---- paged-KV allocator with a prefix cache -------------------------------------------------------------------
    // The ReAct loop resends the whole history on every step (reference pkg/assistants/simple.go:498-501), so step k's
    // prompt is step k-1's prompt + reply + observation: full 64-token pages are published under a hash chain
    // (parent hash, 64 token ids) once their KV is complete and are reused, reference-counted, by any later request with
    // the same prefix.  Unreferenced cached pages sit in an LRU list and are evicted only when no free page is left.
    size_t available_pages_locked() const { return free_pages_.size() + lru_.size(); }
    bool alloc_pages_locked(std::vector<int32_t>& dst, int n) {
        if ((int)available_pages_locked() < n) return false;
        for (int i = 0; i < n; ++i) {
            int p;
            if (!free_pages_.empty()) { p = free_pages_.back(); free_pages_.pop_back(); }
            else {                                              // evict the least recently used cached page
                p = lru_.front(); lru_.pop_front(); lru_pos_[p] = lru_.end();
                auto it = cached_.find(page_hash_[p]); if (it != cached_.end() && it->second == p) cached_.erase(it);
                page_hash_[p] = 0;
            }
            page_ref_[p] = 1; dst.push_back(p);
        }
        return true;
    }
    void release_page_locked(int p) {
        if (--page_ref_[p] > 0) return;
        page_ref_[p] = 0;
        if (page_hash_[p] != 0) { lru_.push_back(p); lru_pos_[p] = std::prev(lru_.end()); }
        else free_pages_.push_back(p);
    }
    static uint64_t chain_hash(uint64_t parent, const int32_t* toks) {
        uint64_t h = parent * 0x9E3779B97F4A7C15ull + 0xD6E8FEB86659FD93ull;
        for (int i = 0; i < 64; ++i) { h ^= (uint64_t)(uint32_t)toks[i] + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2); h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 29; }
        return h ? h : 1;
    }
    // reuse cached pages for the longest cached prefix of s->tokens (always leaving >= 1 token to compute)
    void match_prefix_locked(const std::shared_ptr<Seq>& s) {
        s->n_registered = 0; s->hash_prev = 0; s->n_cached = 0;
        if (!opt_.prefix_cache) return;
        const int max_pages = ((int)s->tokens.size() - 1) / 64;
        uint64_t h = 0;
        for (int i = 0; i < max_pages; ++i) {
            const uint64_t hi = chain_hash(h, s->tokens.data() + (size_t)i * 64);
            auto it = cached_.find(hi);
            if (it == cached_.end()) break;
            const int p = it->second;
            if (page_parent_[p] != h || std::memcmp(&page_tokens_[(size_t)p * 64], s->tokens.data() + (size_t)i * 64, 256) != 0) break;   // hash collision guard
            if (page_ref_[p] == 0) { lru_.erase(lru_pos_[p]); lru_pos_[p] = lru_.end(); }
            ++page_ref_[p]; s->pages.push_back(p);
            h = hi; s->n_registered = i + 1; s->hash_prev = h; s->n_cached = (i + 1) * 64;
        }
        n_prefix_hit_tokens_ += s->n_cached;
    }
    // prompt tokens of a waiting sequence that a prefill would really have to compute (read-only walk of the prefix cache)
    int uncached_tokens_locked(const Seq& s) const {
        int hit = 0;
        if (opt_.prefix_cache) {
            const int max_pages = ((int)s.tokens.size() - 1) / 64;
            uint64_t h = 0;
            for (int i = 0; i < max_pages; ++i) {
                const uint64_t hi = chain_hash(h, s.tokens.data() + (size_t)i * 64);
                auto it = cached_.find(hi);
                if (it == cached_.end() || page_parent_[it->second] != h) break;
                h = hi; hit = (i + 1) * 64;
            }
        }
        return (int)s.tokens.size() - hit;
    }
    // publish the pages of s whose KV became complete (n_cached advanced past their last token)
    void register_pages_locked(const std::shared_ptr<Seq>& s) {
        if (!opt_.prefix_cache) return;
        const int full = std::min(s->n_cached, (int)s->tokens.size()) / 64;
        for (int i = s->n_registered; i < full; ++i) {
            const int p = s->pages[i];
            const uint64_t hi = chain_hash(s->hash_prev, s->tokens.data() + (size_t)i * 64);
            if (page_hash_[p] == 0 && cached_.find(hi) == cached_.end()) {
                cached_[hi] = p; page_hash_[p] = hi; page_parent_[p] = s->hash_prev;
                std::memcpy(&page_tokens_[(size_t)p * 64], s->tokens.data() + (size_t)i * 64, 256);
            }
            s->hash_prev = hi; s->n_registered = i + 1;
        }
    }
    void finish_locked(const std::shared_ptr<Seq>& s, int reason) {
        s->finish_reason = reason; s->state = SeqState::DONE; s->done = true;
        for (int p : s->pages) release_page_locked(p);
        s->pages.clear(); ++n_completed_;
    }
    // Accept a sampled token for s (called with mu_ held). Returns true if the sequence finished.
    bool accept_token_locked(const std::shared_ptr<Seq>& s, int32_t t) {
        if (s->grammar.active()) {
            // the masked arg-max can only have produced an allowed token (all of its bytes walk the automaton); a mismatch means the device path is broken
            bool ok = t >= 0 && (size_t)t < token_bytes_.size() && !token_bytes_[(size_t)t].empty();
            if (ok) for (unsigned char ch : token_bytes_[(size_t)t]) if (!s->grammar.advance(ch)) { ok = false; break; }
            if (!ok) { s->error = OA_ERR_INTERNAL; s->error_msg = "grammar-constrained decode produced a disallowed token"; finish_locked(s, 1); return true; }
            s->tokens.push_back(t); ++s->n_generated;
            if (s->grammar.done()) { finish_locked(s, 0); return true; }
            if (s->n_generated >= s->max_new || (int)s->tokens.size() >= opt_.max_seq_len) { finish_locked(s, 1); return true; }
            return false;
        }
        const bool eos = tok_.is_eos(t) && !(s->flags & OA_FLAG_IGNORE_EOS);
        if (eos) { finish_locked(s, 0); return true; }
        s->tokens.push_back(t); ++s->n_generated;
        if (s->n_generated >= s->max_new || (int)s->tokens.size() >= opt_.max_seq_len) { finish_locked(s, 1); return true; }
        return false;
    }

    // device-table row holding the allowed-token bitset of s's grammar state; computes + schedules the upload on a miss (LRU over rows
    // not used by the step being built)
    int32_t mask_slot_locked(const Seq& s, std::vector<uint32_t>& updates) {
        const std::string key = grammar_mask_key(s.grammar, s.grammar.cursor());
        auto it = mask_slot_of_.find(key);
        if (it != mask_slot_of_.end()) { mask_last_use_[(size_t)it->second] = mask_tick_; return it->second; }
        int victim = -1; uint64_t oldest = UINT64_MAX;
        for (int i = 0; i < model_.mask_slots; ++i) {
            if (mask_key_of_[(size_t)i].empty()) { victim = i; break; }
            if (mask_last_use_[(size_t)i] < mask_tick_ && mask_last_use_[(size_t)i] < oldest) { oldest = mask_last_use_[(size_t)i]; victim = i; }
        }
        if (victim < 0) throw std::runtime_error("token-mask table exhausted within one step");      // cannot happen: rows >= 2 * max_batch
        if (!mask_key_of_[(size_t)victim].empty()) mask_slot_of_.erase(mask_key_of_[(size_t)victim]);
        mask_key_of_[(size_t)victim] = key; mask_slot_of_[key] = victim; mask_last_use_[(size_t)victim] = mask_tick_;
        const size_t at = updates.size(), words = (size_t)model_.mask_words;
        updates.resize(at + 1 + words);
        updates[at] = (uint32_t)victim;
        trie_.allowed_tokens(s.grammar, s.grammar.cursor(), &updates[at + 1]);
        ++n_mask_states_;
        return victim;
    }

    void loop() {
        cudaSetDevice(opt_.device);
        while (true) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_work_.wait(lk, [&] { return stop_ || !waiting_.empty() || !running_.empty(); });
                if (stop_) break;
            }
            std::lock_guard<std::mutex> step(step_mu_);
            const auto t0 = std::chrono::steady_clock::now();
            try { step_once(); }
            catch (const std::exception& ex) {
                std::lock_guard<std::mutex> lk(mu_);
                fatal_ = true; fatal_msg_ = ex.what();
                for (auto& s : running_) { s->error = OA_ERR_INTERNAL; s->error_msg = fatal_msg_; s->done = true; }
                for (auto& s : waiting_) { s->error = OA_ERR_INTERNAL; s->error_msg = fatal_msg_; s->done = true; }
                running_.clear(); waiting_.clear();
                cv_done_.notify_all();
            }
            busy_ms_ += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        }
    }

    void step_once() {
        std::vector<std::shared_ptr<Seq>> batch;      // sequences taking part in this forward
        StepInput in;
        std::vector<int> take_of;                       // prefill: tokens consumed per batch entry
        std::vector<std::shared_ptr<Seq>> sampled;      // sequences owning this step's sample rows, in row order
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (n_cancelled_ != n_cancel_seen_) {       // requests abandoned by their callers: free their pages before planning this step
                n_cancel_seen_ = n_cancelled_;
                for (auto& s : running_) if (s->cancelled && !s->done) { finish_locked(s, 1); --n_completed_; }
                running_.erase(std::remove_if(running_.begin(), running_.end(), [](const std::shared_ptr<Seq>& s) { return s->done; }), running_.end());
            }
            // ---- admission batching: a prefill step streams all the weights once, whether it carries one arrival or ten, and the decoding
            // sequences stall for its duration.  While sequences are decoding, arrivals therefore wait (bounded) until enough uncached prompt
            // tokens are queued to be worth that pass.  Nothing running, a preempted sequence, or the time limit admit at once. ----
            bool defer = false;
            if (opt_.prefill_batch_tokens > 0 && !waiting_.empty() && !running_.empty() && !waiting_.front()->preempted) {
                bool all_decoding = true;
                for (auto& s : running_) if (s->state != SeqState::DECODE) { all_decoding = false; break; }
                if (all_decoding) {
                    const auto now = std::chrono::steady_clock::now();
                    long long pending = 0; double oldest_ms = 0;
                    size_t seen = 0;
                    for (auto& s : waiting_) {
                        if (s->est_uncached < 0) s->est_uncached = uncached_tokens_locked(*s);
                        pending += s->est_uncached;
                        oldest_ms = std::max(oldest_ms, std::chrono::duration<double, std::milli>(now - s->t_enqueue).count());
                        if (++seen >= 64 || pending >= opt_.prefill_batch_tokens) break;
                    }
                    defer = pending < opt_.prefill_batch_tokens && oldest_ms < (double)opt_.prefill_max_wait_ms && seen == waiting_.size();
                    if (defer) ++n_admit_deferred_;
                }
            }
            // ---- admission: FIFO while pages for the whole current token list (+1) are free ----
            while (!defer && !waiting_.empty() && (int)running_.size() < opt_.max_batch) {
                auto& s = waiting_.front();
                const int need = ((int)s->tokens.size() + 1 + 63) / 64;
                if (need > model_.num_pages) { s->error = OA_ERR_BAD_REQUEST; s->error_msg = "request larger than the KV pool"; s->done = true; waiting_.pop_front(); cv_done_.notify_all(); continue; }
                match_prefix_locked(s);                                   // cached prefix pages (ref-counted), s->n_cached set
                if (!alloc_pages_locked(s->pages, need - (int)s->pages.size())) {
                    for (int p : s->pages) release_page_locked(p);
                    s->pages.clear(); s->n_cached = 0; s->n_registered = 0; s->hash_prev = 0;
                    break;
                }
                s->state = SeqState::PREFILL; s->preempted = false;
                running_.push_back(s); waiting_.pop_front();
            }
            if (running_.empty()) return;
            bool any_prefill = false;
            for (auto& s : running_) if (s->state == SeqState::PREFILL) { any_prefill = true; break; }
            if (any_prefill) {
                in.decode = false;
                int budget = opt_.max_step_tokens;
                if (opt_.mixed_steps) {
                    // mixed step: the decoding sequences take rows / sequence slots 0..n_decode-1 (one token each, decode attention) and
                    // advance with this forward instead of stalling behind the prefill.  A sequence that cannot get the page for its
                    // newest token sits this step out (preemption stays with the pure decode step).
                    for (auto& s : running_) {
                        if (s->state != SeqState::DECODE || budget <= 1) continue;
                        const int pos = (int)s->tokens.size() - 1;
                        if (pos / 64 >= (int)s->pages.size() && !alloc_pages_locked(s->pages, 1)) continue;
                        const int sidx = in.n_seqs++;
                        in.block_tables.resize((size_t)in.n_seqs * model_.max_pages_per_seq, 0);
                        for (size_t i = 0; i < s->pages.size(); ++i) in.block_tables[(size_t)sidx * model_.max_pages_per_seq + i] = s->pages[i];
                        in.ctx_lens.push_back(pos + 1);
                        in.sample_rows.push_back((int)in.tokens.size());
                        in.tokens.push_back(s->tokens[pos]); in.positions.push_back(pos); in.slots.push_back(s->pages[pos / 64] * 64 + pos % 64);
                        batch.push_back(s); take_of.push_back(0); sampled.push_back(s); --budget;
                    }
                    in.n_decode = in.n_seqs;
                }
                for (auto& s : running_) {
                    if (s->state != SeqState::PREFILL || budget <= 0) continue;
                    const int remaining = (int)s->tokens.size() - s->n_cached;
                    const int take = std::min(remaining, budget);
                    const int sidx = in.n_seqs++;
                    in.block_tables.resize((size_t)in.n_seqs * model_.max_pages_per_seq, 0);
                    for (size_t i = 0; i < s->pages.size(); ++i) in.block_tables[(size_t)sidx * model_.max_pages_per_seq + i] = s->pages[i];
                    in.ctx_lens.push_back(s->n_cached + take);
                    const int row0 = (int)in.tokens.size();
                    for (int i = s->n_cached; i < s->n_cached + take; ++i) {
                        in.tokens.push_back(s->tokens[i]); in.positions.push_back(i); in.slots.push_back(s->pages[i / 64] * 64 + i % 64);
                    }
                    for (int r = 0; r < take; r += PREFILL_TILE_ROWS) in.tiles.push_back(PrefillTile{sidx, row0 + r, s->n_cached + r, std::min(PREFILL_TILE_ROWS, take - r)});
                    if (take == remaining) { in.sample_rows.push_back(row0 + take - 1); sampled.push_back(s); }
                    batch.push_back(s); take_of.push_back(take); budget -= take;
                }
            } else {
                in.decode = true;
                // every decoding sequence needs a slot for its newest token; preempt (recompute later) if the pool is dry
                auto preempt = [&](const std::shared_ptr<Seq>& v) {
                    for (int p : v->pages) release_page_locked(p);
                    v->pages.clear(); v->n_cached = 0; v->state = SeqState::WAITING; v->preempted = true;
                    waiting_.push_front(v); ++n_preempt_;
                };
                for (size_t i = 0; i < running_.size();) {
                    auto s = running_[i];
                    const int pos = (int)s->tokens.size() - 1;
                    if (pos / 64 >= (int)s->pages.size() && !alloc_pages_locked(s->pages, 1)) {
                        auto victim = running_.back();          // most recently admitted
                        running_.pop_back(); preempt(victim);
                        continue;                                // retry slot i (or fall out if s itself was the victim)
                    }
                    ++i;
                }
                if (running_.empty()) return;
                in.n_seqs = (int)running_.size();
                in.block_tables.assign((size_t)in.n_seqs * model_.max_pages_per_seq, 0);
                for (size_t b = 0; b < running_.size(); ++b) {
                    auto& s = running_[b];
                    const int pos = (int)s->tokens.size() - 1;
                    for (size_t i = 0; i < s->pages.size(); ++i) in.block_tables[b * model_.max_pages_per_seq + i] = s->pages[i];
                    in.tokens.push_back(s->tokens[pos]); in.positions.push_back(pos); in.slots.push_back(s->pages[pos / 64] * 64 + pos % 64);
                    in.ctx_lens.push_back(pos + 1); in.sample_rows.push_back((int)b);
                    batch.push_back(s); sampled.push_back(s);
                }
            }
            // grammar-constrained rows: each samples under the token mask of its automaton state.  Masks live in a device table, one row
            // per cached (grammar, canonical state); a state seen for the first time is computed here (trie walk) and shipped with this step.
            bool any = false;
            for (auto& s : sampled) any |= s->grammar.active();
            if (any) {
                ++mask_tick_;
                in.mask_slots.assign(sampled.size(), -1);
                for (size_t i = 0; i < sampled.size(); ++i)
                    if (sampled[i]->grammar.active()) in.mask_slots[i] = mask_slot_locked(*sampled[i], in.mask_updates);
            }
        }
        run_forward(in, nullptr);
        model_.sync();
        {
            std::lock_guard<std::mutex> lk(mu_);
            bool any_done = false;
            if (in.decode) {
                ++n_decode_steps_; n_decode_tokens_ += batch.size();
                for (size_t b = 0; b < batch.size(); ++b) {
                    batch[b]->n_cached = (int)batch[b]->tokens.size(); register_pages_locked(batch[b]);
                    any_done |= accept_token_locked(batch[b], model_.h_out_ids[b]);
                }
            } else {
                ++n_prefill_steps_; n_prefill_tokens_ += in.tokens.size() - (size_t)in.n_decode;
                if (in.n_decode > 0) { ++n_mixed_steps_; n_decode_tokens_ += (uint64_t)in.n_decode; }
                int si = 0;
                for (size_t b = 0; b < batch.size(); ++b) {
                    auto& s = batch[b];
                    if ((int)b < in.n_decode) {          // a decoding sequence that rode along: exactly what a decode step does with it
                        s->n_cached = (int)s->tokens.size(); register_pages_locked(s);
                        any_done |= accept_token_locked(s, model_.h_out_ids[si++]);
                        continue;
                    }
                    s->n_cached += take_of[b]; register_pages_locked(s);
                    if (s->n_cached == (int)s->tokens.size()) { s->state = SeqState::DECODE; any_done |= accept_token_locked(s, model_.h_out_ids[si++]); }
                }
            }
            if (any_done) {
                running_.erase(std::remove_if(running_.begin(), running_.end(), [](const std::shared_ptr<Seq>& s) { return s->done; }), running_.end());
                cv_done_.notify_all();
            }
        }
    }

    DeviceModel model_; Tokenizer tok_; EngineOptions opt_;
    std::mutex mu_, step_mu_;
    std::condition_variable cv_work_, cv_done_;
    std::deque<std::shared_ptr<Seq>> waiting_;
    std::vector<std::shared_ptr<Seq>> running_;
    std::unordered_map<uint64_t, std::shared_ptr<Seq>> by_ticket_;
    std::vector<int32_t> free_pages_;
    std::vector<int32_t> page_ref_; std::vector<uint64_t> page_hash_, page_parent_; std::vector<int32_t> page_tokens_;
    std::unordered_map<uint64_t, int> cached_; std::list<int> lru_; std::vector<std::list<int>::iterator> lru_pos_;
    uint64_t n_prefix_hit_tokens_ = 0;
    uint64_t next_ticket_ = 1;
    bool stop_ = false, fatal_ = false; std::string fatal_msg_;
    std::thread worker_, follower_; bool follower_done_ = false;
    uint64_t n_cancelled_ = 0, n_cancel_seen_ = 0;
    std::vector<std::string> token_bytes_; TokenTrie trie_;
    std::unordered_map<std::string, int> mask_slot_of_; std::vector<std::string> mask_key_of_; std::vector<uint64_t> mask_last_use_; uint64_t mask_tick_ = 0, n_mask_states_ = 0;
    uint64_t n_mixed_steps_ = 0, n_admit_deferred_ = 0, n_completed_ = 0, n_prefill_tokens_ = 0, n_decode_tokens_ = 0, n_prefill_steps_ = 0, n_decode_steps_ = 0, n_preempt_ = 0;
    double busy_ms_ = 0;
};

}  // namespace oa

// =============================================================================================
// C ABI
// =============================================================================================
using namespace oa;
struct oa_engine { std::unique_ptr<Engine> e; };

static int build_messages(const oa_msg* msgs, int32_t n, std::vector<ChatMessage>& out) {
    if (!msgs || n <= 0) return fail(OA_ERR_BAD_REQUEST, "prompts cannot be empty");   // simple.go:312 rejects empty prompts too
    for (int i = 0; i < n; ++i) {
        if (!msgs[i].role || !msgs[i].content) return fail(OA_ERR_BAD_REQUEST, "message role/content must be non-null");
        out.push_back(ChatMessage{msgs[i].role, msgs[i].content});
    }
    return OA_OK;
}

extern "C" {

int oa_engine_create(const char* config_json, oa_engine** out) {
    if (!out) return fail(OA_ERR_BAD_REQUEST, "null out pointer");
    *out = nullptr;
    try {
        ModelConfig mc; EngineOptions eo;
        parse_config(config_json ? config_json : "{}", mc, eo);
        int n_dev = 0;
        if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0)
            return fail(OA_ERR_INTERNAL, "no CUDA device: opsagent_b200 has no CPU fallback (the oracle under oracle/ is test-only)");
        auto h = new oa_engine; h->e.reset(new Engine(mc, eo)); *out = h;
    } catch (const std::exception& ex) { return fail(std::string(ex.what()).find("config json") == 0 || std::string(ex.what()).find("unknown model") == 0 ? OA_ERR_BAD_REQUEST : OA_ERR_INTERNAL, ex.what()); }
    return OA_OK;
}
void oa_engine_destroy(oa_engine* h) { delete h; }

// chat template -> ids; a BPE tokenizer may refuse text (e.g. not NFC): that is the caller's bad request, never an exception across the C ABI
static int template_ids(oa_engine* h, const std::vector<ChatMessage>& msgs, std::vector<int32_t>& ids) {
    try { ids = h->e->tokenizer().apply_chat_template(msgs); }
    catch (const std::exception& ex) { return fail(OA_ERR_BAD_REQUEST, ex.what()); }
    return OA_OK;
}

static int submit_chat(oa_engine* h, const oa_chat_req* r, uint64_t* ticket) {
    if (!h || !r || !ticket) return fail(OA_ERR_BAD_REQUEST, "null argument");
    if (r->model && r->model[0] && !h->e->serves_model(r->model))
        return fail(OA_ERR_BAD_REQUEST, std::string("model '") + r->model + "' is not loaded (engine serves '" + h->e->config().name + "'; config \"model_aliases\" lists other names it answers to, \"*\" = any)");
    if (r->temperature > 1e-3f) return fail(OA_ERR_BAD_REQUEST, "only greedy decoding is implemented (the reference sends temperature=SmallestNonzeroFloat32)");
    std::vector<ChatMessage> msgs;
    int rc = build_messages(r->msgs, r->n_msgs, msgs); if (rc) return rc;
    {   // refuse absurd inputs BEFORE tokenising them on the caller's thread: no tokenizer yields fewer than one token per 16 bytes of text
        size_t bytes = 0; for (auto& m : msgs) bytes += m.content.size() + m.role.size();
        if (bytes > (size_t)h->e->options().max_seq_len * 16)
            return fail(OA_ERR_BAD_REQUEST, "prompt of " + std::to_string(bytes) + " bytes cannot fit max_seq_len " + std::to_string(h->e->options().max_seq_len) + " tokens");
    }
    uint32_t flags = r->flags;
    if (flags == 0 && h->e->options().json_mode) {        // explicit per-request flags always win
        // stateless ReAct policy: the history is resent on every step (simple.go:498-501), so the number of assistant turns
        // tells which step this is — tool calls first, then the final answer
        int turns = 0; for (auto& m : msgs) if (m.role == "assistant") ++turns;
        flags |= (turns < h->e->options().react_tool_steps) ? OA_FLAG_JSON_TOOLCALL : OA_FLAG_JSON_FINAL;
    }
    std::vector<int32_t> ids;
    rc = template_ids(h, msgs, ids); if (rc) return rc;
    return h->e->submit_tokens(std::move(ids), r->max_tokens, flags, ticket, r->functions);
}
int oa_chat_submit(oa_engine* h, const oa_chat_req* r, uint64_t* ticket) { return submit_chat(h, r, ticket); }
int oa_chat_wait(oa_engine* h, uint64_t ticket, int32_t timeout_ms, oa_chat_resp* out) {
    if (!h || !out) return fail(OA_ERR_BAD_REQUEST, "null argument");
    std::memset(out, 0, sizeof *out);
    return h->e->wait(ticket, timeout_ms, out);
}
int oa_chat_complete(oa_engine* h, const oa_chat_req* r, oa_chat_resp* out) {
    uint64_t t = 0; int rc = submit_chat(h, r, &t); if (rc) return rc;
    return oa_chat_wait(h, t, -1, out);
}
int oa_chat_cancel(oa_engine* h, uint64_t ticket) { if (!h) return fail(OA_ERR_BAD_REQUEST, "null engine"); return h->e->cancel(ticket); }
// variants that hand the error text back in a caller buffer: a goroutine may migrate between OS threads around a cgo call, so the
// thread-local oa_last_error() is only safe under runtime.LockOSThread — these need no pinning
static int with_err(int rc, char* errbuf, size_t errcap) { if (errbuf && errcap) std::snprintf(errbuf, errcap, "%s", rc ? g_last_error.c_str() : ""); return rc; }
int oa_chat_submit_ex(oa_engine* h, const oa_chat_req* r, uint64_t* ticket, char* errbuf, size_t errcap) { return with_err(submit_chat(h, r, ticket), errbuf, errcap); }
int oa_chat_wait_ex(oa_engine* h, uint64_t ticket, int32_t timeout_ms, oa_chat_resp* out, char* errbuf, size_t errcap) { return with_err(oa_chat_wait(h, ticket, timeout_ms, out), errbuf, errcap); }
void oa_free_resp(oa_chat_resp* r) { if (!r) return; std::free(r->content); std::free(r->token_ids); std::memset(r, 0, sizeof *r); }

int oa_tokens_submit(oa_engine* h, const int32_t* prompt, int32_t n, int32_t max_tokens, uint32_t flags, uint64_t* ticket) {
    if (!h || !prompt || !ticket || n <= 0) return fail(OA_ERR_BAD_REQUEST, "null or empty prompt");
    return h->e->submit_tokens(std::vector<int32_t>(prompt, prompt + n), max_tokens, flags, ticket);
}
int oa_count_tokens(oa_engine* h, const oa_msg* msgs, int32_t n, int32_t* out_tokens) {
    if (!h || !out_tokens) return fail(OA_ERR_BAD_REQUEST, "null argument");
    std::vector<ChatMessage> m; int rc = build_messages(msgs, n, m); if (rc) return rc;
    std::vector<int32_t> ids;
    rc = template_ids(h, m, ids); if (rc) return rc;
    *out_tokens = (int32_t)ids.size();
    return OA_OK;
}
int oa_apply_chat_template(oa_engine* h, const oa_msg* msgs, int32_t n, int32_t* out_ids, int32_t cap, int32_t* n_out) {
    if (!h || !n_out) return fail(OA_ERR_BAD_REQUEST, "null argument");
    std::vector<ChatMessage> m; int rc = build_messages(msgs, n, m); if (rc) return rc;
    std::vector<int32_t> ids;
    rc = template_ids(h, m, ids); if (rc) return rc;
    *n_out = (int32_t)ids.size();
    if (out_ids) std::memcpy(out_ids, ids.data(), (size_t)std::min<int32_t>(cap, (int32_t)ids.size()) * 4);
    return OA_OK;
}
const char* oa_last_error(void) { return g_last_error.c_str(); }
static int copy_out(const std::string& s, char* buf, size_t n) {
    if (!buf || n == 0) return fail(OA_ERR_BAD_REQUEST, "null buffer");
    std::snprintf(buf, n, "%s", s.c_str()); return OA_OK;
}
int oa_engine_stats(oa_engine* h, char* buf, size_t n) { if (!h) return fail(OA_ERR_BAD_REQUEST, "null engine"); return copy_out(h->e->stats_json(), buf, n); }
int oa_model_info(oa_engine* h, char* buf, size_t n) { if (!h) return fail(OA_ERR_BAD_REQUEST, "null engine"); return copy_out(h->e->info_json(), buf, n); }
int oa_debug_prefill_logits(oa_engine* h, const int32_t* tokens, int32_t n, float* logits_out) {
    if (!h || !tokens || !logits_out) return fail(OA_ERR_BAD_REQUEST, "null argument");
    return h->e->debug_prefill_logits(tokens, n, logits_out);
}
int oa_bench_decode_ex(oa_engine* h, int32_t batch, int32_t ctx_len, int32_t steps, int32_t warmup, double* out, int32_t n_out,
                       int32_t* last_ids, float* last_logits) {
    if (!h || !out) return fail(OA_ERR_BAD_REQUEST, "null argument");
    const char* pa = std::getenv("OA_PROFILE_ATTN");
    h->e->model().profile_attn = pa && pa[0] == '1';
    const char* pall = std::getenv("OA_PROFILE_ALL");
    h->e->model().profile_all = pall && pall[0] == '1';
    int rc = h->e->bench_decode(batch, ctx_len, steps, warmup, out, n_out, last_ids, last_logits);
    h->e->model().profile_attn = false; h->e->model().profile_all = false;
    return rc;
}
int oa_bench_decode(oa_engine* h, int32_t batch, int32_t ctx_len, int32_t steps, int32_t warmup, double* out, int32_t n_out) {
    return oa_bench_decode_ex(h, batch, ctx_len, steps, warmup, out, n_out, nullptr, nullptr);
}
int oa_debug_kernel_times(oa_engine* h, char* buf, size_t n, int32_t reset) {
    if (!h || !buf) return fail(OA_ERR_BAD_REQUEST, "null argument");
    DeviceModel& m = h->e->model();
    std::string s = "{";
    for (int i = 0; i < 14; ++i) {
        char t[128]; std::snprintf(t, sizeof t, "%s\"%s\": [%.4f, %ld]", i ? ", " : "", DeviceModel::kt_name(i), m.kt_ms[i], m.kt_n[i]); s += t;
        if (reset) { m.kt_ms[i] = 0; m.kt_n[i] = 0; }
    }
    s += "}";
    return copy_out(s, buf, n);
}
static std::shared_ptr<BpeTokenizer> cached_bpe(const char* path) {
    static std::mutex mu; static std::map<std::string, std::shared_ptr<BpeTokenizer>> cache;
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(path);
    if (it != cache.end()) return it->second;
    auto t = BpeTokenizer::load(path);
    cache[path] = t;
    return t;
}
int oa_host_bpe_encode(const char* tokenizer_json_path, const char* text, int32_t text_len, int32_t* ids_out, int32_t cap, int32_t* n_out) {
    if (!tokenizer_json_path || (!text && text_len > 0) || text_len < 0 || !n_out) return fail(OA_ERR_BAD_REQUEST, "null argument");
    try {
        std::vector<int32_t> ids;
        cached_bpe(tokenizer_json_path)->encode(std::string(text ? text : "", (size_t)text_len), ids);
        *n_out = (int32_t)ids.size();
        if ((int32_t)ids.size() > cap) return fail(OA_ERR_BAD_REQUEST, "ids buffer too small");
        if (!ids.empty()) std::memcpy(ids_out, ids.data(), ids.size() * 4);
    } catch (const std::exception& e) { return fail(OA_ERR_BAD_REQUEST, e.what()); }
    return OA_OK;
}
int oa_host_bpe_decode(const char* tokenizer_json_path, const int32_t* ids, int32_t n_ids, char* buf, int32_t cap, int32_t* n_out) {
    if (!tokenizer_json_path || (!ids && n_ids > 0) || n_ids < 0 || !n_out) return fail(OA_ERR_BAD_REQUEST, "null argument");
    try {
        const std::string s = cached_bpe(tokenizer_json_path)->decode(ids, (size_t)n_ids);
        *n_out = (int32_t)s.size();
        if ((int32_t)s.size() > cap) return fail(OA_ERR_BAD_REQUEST, "text buffer too small");
        if (!s.empty()) std::memcpy(buf, s.data(), s.size());
    } catch (const std::exception& e) { return fail(OA_ERR_BAD_REQUEST, e.what()); }
    return OA_OK;
}

int oa_engine_serve(oa_engine* h) { if (!h) return fail(OA_ERR_BAD_REQUEST, "null engine"); return h->e->serve(); }
uint64_t oa_kernel_launches(void) { return launches_total(); }
const char* oa_version(void) { return "opsagent_b200 0.1 (sm_100a)"; }

}  // extern "C"
