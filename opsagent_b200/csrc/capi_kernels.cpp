// capi_kernels.cpp — kernel-level C entry points on raw device pointers (parity tests drive these with
// torch-allocated memory; nothing here is on the serving path).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/opsagent_b200.h"
#include <map>
#include <memory>
#include <mutex>
#include "grammar.hpp"
#include "token_mask.hpp"
#include "tokenizer.hpp"
#include "model.hpp"
#include "tokenizer.hpp"

using namespace oa;

namespace {
struct DevBuf {
    void* p = nullptr;
    explicit DevBuf(size_t n) { if (cudaMalloc(&p, n ? n : 16) != cudaSuccess) p = nullptr; }
    ~DevBuf() { if (p) cudaFree(p); }
};
int rc_of(cudaError_t e) { return e == cudaSuccess ? OA_OK : OA_ERR_INTERNAL; }
int device_sm_count() {
    int dev = 0, n = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
}
// A [M,K] and B [N,K] as the decode projections map them: A in 128-row boxes, B in 128-column tiles (BN = 128, the engine's stream-K tile)
bool proj_maps(const void* A, const void* B, int M, int N, int K, CUtensorMap& tmA, CUtensorMap& tmB) {
    return make_tmap_bf16_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 64) == 0 &&
           make_tmap_bf16_2d(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)K, 128, 64) == 0;
}
}  // namespace

// test-only: materialise the deterministic fixed-order sum of stream-K partials as fp32 [M,N]
__global__ void sk_reduce_f32_kernel(const StreamK sk, float* __restrict__ out, int M, int N) {
    const int row = blockIdx.x;
    for (int col = threadIdx.x; col < N; col += blockDim.x) {
        const uint32_t tile = (uint32_t)col / (uint32_t)sk.bn, cc = (uint32_t)col - tile * (uint32_t)sk.bn;
        uint32_t c_first, c_last;
        sk_tile_ctas(sk, tile, c_first, c_last);
        float acc = 0.f;
        for (uint32_t c = c_first; c <= c_last; ++c) acc += sk.ws[((size_t)(c + tile) * sk.rows + row) * sk.bn + cc];
        out[(size_t)row * N + col] = acc;
    }
}

extern "C" {

int oa_k_gemm_streamk(const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t block_n, int32_t n_ctas, float* out_f32, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CUtensorMap tmA, tmB;
    if (make_tmap_bf16_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 64) != 0) return OA_ERR_INTERNAL;
    if (make_tmap_bf16_2d(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)K, (uint32_t)block_n, 64) != 0) return OA_ERR_INTERNAL;
    DevBuf ws(streamk_ws_bytes(N, block_n, n_ctas, M));
    if (!ws.p) return OA_ERR_INTERNAL;
    StreamK sk = make_streamk((float*)ws.p, N, K, block_n, n_ctas, M);
    cudaError_t e = launch_gemm_streamk(&tmA, &tmB, M, N, K, sk, s);
    if (e == cudaSuccess) { sk_reduce_f32_kernel<<<M, 256, 0, s>>>(sk, out_f32, M, N); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return rc_of(e);
}

int oa_k_rmsnorm(const void* x, const void* gain, void* y, int32_t T, int32_t H, float eps, void* stream) {
    return rc_of(launch_rmsnorm(x, gain, y, T, H, eps, (cudaStream_t)stream));
}

int oa_k_init_weight(void* dst, uint64_t seed, uint64_t tensor_id, int64_t tensor_id_b, int64_t rows, int64_t cols, float std,
                     float mean, void* stream) {
    return rc_of(launch_init_weight(dst, seed, tensor_id, tensor_id_b, rows, cols, std, mean, (cudaStream_t)stream));
}

int oa_k_gemm(const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t block_n, void* out,
              const void* bias, const void* resid, float* logits, int32_t* argmax_out, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    CUtensorMap tmA, tmB;
    if (make_tmap_bf16_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 64) != 0) return OA_ERR_INTERNAL;
    if (make_tmap_bf16_2d(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)K, (uint32_t)block_n, 64) != 0) return OA_ERR_INTERNAL;
    GemmParams p{}; p.M = M; p.N = N; p.K = K; p.out = out; p.ldo = epilogue == EPI_SWIGLU ? N / 2 : N;
    p.bias = bias; p.resid = resid; p.ldr = N; p.logits = logits; p.ldl = N;
    if (epilogue == EPI_LOGITS) {
        const int nt = gemm_n_tiles(N, block_n);
        DevBuf av((size_t)M * nt * 4), ai((size_t)M * nt * 4);
        if (!av.p || !ai.p) return OA_ERR_INTERNAL;
        p.amax_val = (float*)av.p; p.amax_idx = (int*)ai.p;
        cudaError_t e = launch_gemm(&tmA, &tmB, p, epilogue, block_n, s);
        if (e == cudaSuccess) e = launch_argmax_reduce(p.amax_val, p.amax_idx, M, nt, argmax_out, nullptr, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        return rc_of(e);
    }
    return rc_of(launch_gemm(&tmA, &tmB, p, epilogue, block_n, s));
}

// ---- the decode step's projections with their epilogues, each through the launcher pairing DeviceModel::forward uses ----
int oa_k_sk_resid_rmsnorm(int32_t path, const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t n_ctas, int32_t cluster,
                          void* x, int32_t ldx, const void* gain, void* xn, float eps, uint32_t* tile_flags, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (M <= 0 || M > 128 || N <= 0 || K <= 0 || n_ctas <= 0 || path < 0 || path > 2) return OA_ERR_BAD_REQUEST;
    if ((path == 0 || xn) && ldx != N) return OA_ERR_BAD_REQUEST;          // the norm kernels read x with row stride N
    if (path == 0 && !xn) return OA_ERR_BAD_REQUEST;
    if (path == 2 && (K + 63) / 64 < cluster) return OA_ERR_BAD_REQUEST;     // every cluster rank needs at least one k-block
    CUtensorMap tmA, tmB;
    if (!proj_maps(A, B, M, N, K, tmA, tmB)) return OA_ERR_INTERNAL;
    DevBuf ws(path == 2 ? 16 : streamk_ws_bytes(N, 128, n_ctas, 128));
    if (!ws.p) return OA_ERR_INTERNAL;
    const StreamK sk = make_streamk((float*)ws.p, N, K, 128, n_ctas, 128);
    cudaError_t e;
    if (path == 0) {
        e = launch_gemm_streamk(&tmA, &tmB, M, N, K, sk, s);
        if (e == cudaSuccess) e = launch_sk_resid_rmsnorm(sk, x, gain, xn, M, N, eps, s);
    } else {
        e = path == 1 ? launch_gemm_streamk_resid(&tmA, &tmB, M, N, K, sk, x, ldx, tile_flags, s)
                      : launch_gemm_clusterk_resid(&tmA, &tmB, M, N, K, cluster, x, ldx, s);
        if (e == cudaSuccess && xn) e = launch_rmsnorm_wide(x, gain, xn, M, N, eps, s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return rc_of(e);
}

int oa_k_sk_swiglu(int32_t path, const void* A, const void* B, int32_t M, int32_t F, int32_t K, int32_t n_ctas, void* act,
                   uint32_t* tile_flags, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (M <= 0 || M > 128 || F <= 0 || K <= 0 || n_ctas <= 0 || path < 0 || path > 1) return OA_ERR_BAD_REQUEST;
    CUtensorMap tmA, tmB;
    if (!proj_maps(A, B, M, 2 * F, K, tmA, tmB)) return OA_ERR_INTERNAL;
    DevBuf ws(streamk_ws_bytes(2 * F, 128, n_ctas, 128));
    if (!ws.p) return OA_ERR_INTERNAL;
    const StreamK sk = make_streamk((float*)ws.p, 2 * F, K, 128, n_ctas, 128);
    cudaError_t e;
    if (path == 0) {
        e = launch_gemm_streamk(&tmA, &tmB, M, 2 * F, K, sk, s);
        if (e == cudaSuccess) e = launch_sk_swiglu(sk, act, M, F, s);
    } else {
        e = launch_gemm_streamk_swiglu(&tmA, &tmB, M, F, K, sk, act, tile_flags, s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return rc_of(e);
}

int oa_k_qkv_rope(int32_t path, const void* A, const void* B, int32_t M, int32_t K, int32_t n_ctas, int32_t cluster, const void* bias,
                  const int32_t* positions, const int32_t* slots, const float* rope_cos, const float* rope_sin, void* q_out, void* kv_cache,
                  int32_t num_pages, int32_t n_layers, int32_t layer, int32_t nh, int32_t nkv, int32_t D, uint32_t* tile_flags, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    const int N = (nh + 2 * nkv) * D;
    if (M <= 0 || M > 128 || K <= 0 || n_ctas <= 0 || path < 0 || path > 3 || nh <= 0 || nkv <= 0 || (D != 64 && D != 128)) return OA_ERR_BAD_REQUEST;
    if (n_layers < 1 || layer < 0 || layer >= n_layers) return OA_ERR_BAD_REQUEST;
    if (path == 2 && (K + 63) / 64 < cluster) return OA_ERR_BAD_REQUEST;
    KvLayout kv{}; kv.base = kv_cache; kv.page_size = 64; kv.n_kv = nkv; kv.head_dim = D; kv.num_pages = num_pages;
    kv.kv_stride_rows = (int64_t)num_pages * nkv * 64; kv.layer_stride_rows = 2 * kv.kv_stride_rows;
    CUtensorMap tmA, tmB;
    if (!proj_maps(A, B, M, N, K, tmA, tmB)) return OA_ERR_INTERNAL;
    cudaError_t e;
    if (path == 3) {          // the tile GEMM's bf16 qkv tensor (+ bias), then RoPE + KV write from it
        DevBuf qkv((size_t)M * N * 2);
        if (!qkv.p) return OA_ERR_INTERNAL;
        GemmParams g{}; g.M = M; g.N = N; g.K = K; g.out = qkv.p; g.ldo = N; g.bias = bias;
        e = launch_gemm(&tmA, &tmB, g, EPI_STORE, 128, s);
        if (e == cudaSuccess) e = launch_rope_kv_write(qkv.p, positions, slots, rope_cos, rope_sin, q_out, kv, layer, M, nh, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        return rc_of(e);
    }
    DevBuf ws(path == 2 ? 16 : streamk_ws_bytes(N, 128, n_ctas, 128));
    if (!ws.p) return OA_ERR_INTERNAL;
    const StreamK sk = make_streamk((float*)ws.p, N, K, 128, n_ctas, 128);
    const SkRopeArgs ra = make_sk_rope_args(bias, positions, slots, rope_cos, rope_sin, q_out, kv, layer, nh);
    if (path == 0) {
        e = launch_gemm_streamk(&tmA, &tmB, M, N, K, sk, s);
        if (e == cudaSuccess) e = launch_sk_rope_kv_write(sk, bias, positions, slots, rope_cos, rope_sin, q_out, kv, layer, M, nh, s);
    } else if (path == 1) {
        e = launch_gemm_streamk_rope(&tmA, &tmB, M, N, K, sk, ra, tile_flags, s);
    } else {
        e = launch_gemm_clusterk_rope(&tmA, &tmB, M, N, K, cluster, ra, s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return rc_of(e);
}

int oa_k_lm_head(const void* A, const void* B, int32_t M, int32_t N, int32_t K, int32_t block_n, const uint32_t* mask_table,
                 const int32_t* mask_slot, int32_t mask_words, int32_t col_offset, float* logits, int32_t* ids, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (M <= 0 || N <= 0 || K <= 0 || !ids) return OA_ERR_BAD_REQUEST;
    CUtensorMap tmA, tmB;
    if (make_tmap_bf16_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 64) != 0) return OA_ERR_INTERNAL;
    if (make_tmap_bf16_2d(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)K, (uint32_t)block_n, 64) != 0) return OA_ERR_INTERNAL;
    const int nt = gemm_n_tiles(N, block_n);
    DevBuf av((size_t)M * nt * 4), ai((size_t)M * nt * 4);
    if (!av.p || !ai.p) return OA_ERR_INTERNAL;
    GemmParams p{}; p.M = M; p.N = N; p.K = K; p.logits = logits; p.ldl = N; p.amax_val = (float*)av.p; p.amax_idx = (int*)ai.p;
    p.mask_table = mask_table; p.mask_slot = mask_slot; p.mask_words = mask_words; p.col_offset = col_offset;
    cudaError_t e = launch_gemm(&tmA, &tmB, p, EPI_LOGITS, block_n, s);
    if (e == cudaSuccess) e = launch_argmax_reduce(p.amax_val, p.amax_idx, M, nt, ids, nullptr, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return rc_of(e);
}

int oa_k_paged_attention(const void* q, void* out, const void* kv_cache, int32_t num_pages, const int32_t* block_tables,
                         int32_t max_pages_per_seq, const int32_t* ctx_lens, const int32_t* q_lens, int32_t n_seqs,
                         int32_t n_heads, int32_t n_kv, int32_t head_dim, int32_t force_splits, void* stream) {
    return oa_k_paged_attention_ex(q, out, kv_cache, num_pages, 1, 0, block_tables, max_pages_per_seq, ctx_lens, q_lens, n_seqs, n_heads, n_kv,
                                   head_dim, force_splits, 2 * 148, nullptr, stream);
}

int oa_k_paged_attention_ex(const void* q, void* out, const void* kv_cache, int32_t num_pages, int32_t n_layers, int32_t layer,
                            const int32_t* block_tables, int32_t max_pages_per_seq, const int32_t* ctx_lens, const int32_t* q_lens, int32_t n_seqs,
                            int32_t n_heads, int32_t n_kv, int32_t head_dim, int32_t force_splits, int32_t n_ctas_target, int32_t* merge_counters,
                            void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (n_layers < 1 || layer < 0 || layer >= n_layers) return OA_ERR_BAD_REQUEST;
    KvLayout kv{}; kv.base = const_cast<void*>(kv_cache); kv.page_size = 64; kv.n_kv = n_kv; kv.head_dim = head_dim; kv.num_pages = num_pages;
    kv.kv_stride_rows = (int64_t)num_pages * n_kv * 64; kv.layer_stride_rows = 2 * kv.kv_stride_rows;
    CUtensorMap tm;      // one map over every layer, as the engine builds it
    if (make_tmap_bf16_2d(&tm, kv_cache, (uint64_t)kv.layer_stride_rows * n_layers, (uint64_t)head_dim, (uint64_t)head_dim, 64, 64) != 0) return OA_ERR_INTERNAL;
    const float scale_log2e = (1.0f / std::sqrt((float)head_dim)) * 1.4426950408889634f;
    const int grp = n_heads / n_kv;
    bool decode = true; int total_q = 0;
    for (int i = 0; i < n_seqs; ++i) { if (q_lens && q_lens[i] != 1) decode = false; total_q += q_lens ? q_lens[i] : 1; }
    DevBuf d_bt((size_t)n_seqs * max_pages_per_seq * 4), d_ctx((size_t)n_seqs * 4);
    if (!d_bt.p || !d_ctx.p) return OA_ERR_INTERNAL;
    cudaMemcpyAsync(d_bt.p, block_tables, (size_t)n_seqs * max_pages_per_seq * 4, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(d_ctx.p, ctx_lens, (size_t)n_seqs * 4, cudaMemcpyHostToDevice, s);
    cudaError_t e;
    if (decode) {
        if (n_ctas_target <= 0) n_ctas_target = 2 * device_sm_count();       // the engine's default: two CTAs per SM
        DecodePlan plan;
        build_decode_plan(ctx_lens, n_seqs, n_kv, n_ctas_target, force_splits, plan);
        DevBuf d_segs(plan.segs.size() * sizeof(DecodeSeg)), d_ptr(plan.cta_ptr.size() * 4), d_merge(plan.merges.size() * sizeof(MergeItem));
        DevBuf d_po((size_t)(plan.n_slots + 1) * grp * head_dim * 4), d_pml((size_t)(plan.n_slots + 1) * grp * 2 * 4);
        if (!d_segs.p || !d_ptr.p || !d_merge.p || !d_po.p || !d_pml.p) return OA_ERR_INTERNAL;
        cudaMemcpyAsync(d_segs.p, plan.segs.data(), plan.segs.size() * sizeof(DecodeSeg), cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(d_ptr.p, plan.cta_ptr.data(), plan.cta_ptr.size() * 4, cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(d_merge.p, plan.merges.data(), plan.merges.size() * sizeof(MergeItem), cudaMemcpyHostToDevice, s);
        DecodeAttnParams a{}; a.q = q; a.out = out; a.block_tables = (const int32_t*)d_bt.p; a.ctx_lens = (const int32_t*)d_ctx.p;
        a.max_pages_per_seq = max_pages_per_seq; a.segs = (const DecodeSeg*)d_segs.p; a.cta_seg_ptr = (const int32_t*)d_ptr.p;
        a.n_ctas = (int)plan.cta_ptr.size() - 1; a.part_o = (float*)d_po.p; a.part_ml = (float*)d_pml.p; a.layer = layer;
        a.n_heads = n_heads; a.n_kv = n_kv; a.scale_log2e = scale_log2e; a.merge_counters = merge_counters;
        e = launch_decode_attention(&tm, kv, a, s);
        if (e == cudaSuccess && !merge_counters)
            e = launch_decode_merge((const MergeItem*)d_merge.p, (int)plan.merges.size(), a.part_o, a.part_ml, out, n_heads, n_kv, head_dim, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        return rc_of(e);
    }
    std::vector<PrefillTile> tiles; int row = 0;
    for (int i = 0; i < n_seqs; ++i) {
        const int ql = q_lens[i], p0 = ctx_lens[i] - ql;
        for (int r = 0; r < ql; r += PREFILL_TILE_ROWS) tiles.push_back(PrefillTile{i, row + r, p0 + r, std::min(PREFILL_TILE_ROWS, ql - r)});
        row += ql;
    }
    DevBuf d_tiles(tiles.size() * sizeof(PrefillTile));
    if (!d_tiles.p) return OA_ERR_INTERNAL;
    cudaMemcpyAsync(d_tiles.p, tiles.data(), tiles.size() * sizeof(PrefillTile), cudaMemcpyHostToDevice, s);
    PrefillAttnParams a{}; a.q = q; a.out = out; a.block_tables = (const int32_t*)d_bt.p; a.max_pages_per_seq = max_pages_per_seq;
    a.tiles = (const PrefillTile*)d_tiles.p; a.n_tiles = (int)tiles.size(); a.layer = layer; a.n_heads = n_heads; a.n_kv = n_kv; a.scale_log2e = scale_log2e;
    const char* leg = std::getenv("OA_PREFILL_ATTN");
    if (leg && std::string(leg) == "legacy") e = launch_prefill_attention(&tm, kv, a, s);
    else {
        CUtensorMap tmq;
        if (make_tmap_bf16_2d(&tmq, q, (uint64_t)total_q, (uint64_t)n_heads * head_dim, (uint64_t)n_heads * head_dim, 128, 64) != 0) return OA_ERR_INTERNAL;
        e = launch_prefill_attention_tc(&tmq, &tm, kv, a, s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return rc_of(e);
}


int oa_host_apply_chat_template(const char* config_json, const oa_msg* msgs, int32_t n_msgs, int32_t* out_ids, int32_t cap, int32_t* n_out) {
    try {
        ModelConfig mc; EngineOptions eo; parse_config(config_json ? config_json : "{}", mc, eo);
        Tokenizer tok(mc, eo.tokenizer);
        std::vector<ChatMessage> m;
        for (int i = 0; i < n_msgs; ++i) m.push_back(ChatMessage{msgs[i].role, msgs[i].content});
        auto ids = tok.apply_chat_template(m);
        *n_out = (int32_t)ids.size();
        if (out_ids) std::memcpy(out_ids, ids.data(), (size_t)std::min<int32_t>(cap, (int32_t)ids.size()) * 4);
    } catch (const std::exception&) { return OA_ERR_BAD_REQUEST; }
    return OA_OK;
}

int oa_host_decode_plan(const int32_t* ctx_lens, int32_t n_seqs, int32_t n_kv, int32_t n_ctas_target, int32_t force_splits,
                        int32_t* segs_out, int32_t cap_segs, int32_t* cta_ptr_out, int32_t cap_ctas, int32_t* n_ctas_out,
                        int32_t* n_segs_out, int32_t* n_slots_out) {
    DecodePlan plan;
    build_decode_plan(ctx_lens, n_seqs, n_kv, n_ctas_target, force_splits, plan);
    if ((int)plan.segs.size() > cap_segs || (int)plan.cta_ptr.size() > cap_ctas + 1) return OA_ERR_BAD_REQUEST;
    for (size_t i = 0; i < plan.segs.size(); ++i) {
        const DecodeSeg& g = plan.segs[i];
        int32_t* o = segs_out + i * 5; o[0] = g.seq; o[1] = g.kvh; o[2] = g.chunk_begin; o[3] = g.chunk_end; o[4] = g.partial_slot;
    }
    std::memcpy(cta_ptr_out, plan.cta_ptr.data(), plan.cta_ptr.size() * 4);
    *n_ctas_out = (int32_t)plan.cta_ptr.size() - 1; *n_segs_out = (int32_t)plan.segs.size(); *n_slots_out = plan.n_slots;
    return OA_OK;
}

int oa_host_streamk_plan(int32_t N, int32_t K, int32_t block_n, int32_t n_ctas, int64_t* cta_unit0_out, int32_t cap_ctas,
                         int32_t* tile_first_out, int32_t* tile_last_out, int32_t cap_tiles, int32_t* n_ctas_out, int32_t* n_tiles_out,
                         int32_t* kb_out) {
    if (N <= 0 || K <= 0 || n_ctas <= 0 || (block_n != 128 && block_n != 256)) return OA_ERR_BAD_REQUEST;
    const StreamK sk = make_streamk(nullptr, N, K, block_n, n_ctas);
    if (sk.G > cap_ctas || sk.n_tiles > cap_tiles) return OA_ERR_BAD_REQUEST;
    for (int c = 0; c <= sk.G; ++c) cta_unit0_out[c] = (long long)c * sk.total / sk.G;            // the kernels' u0/u1
    for (int t = 0; t < sk.n_tiles; ++t) {                                                        // the very function the kernels call
        uint32_t cf, cl;
        sk_tile_ctas(sk, (uint32_t)t, cf, cl);
        tile_first_out[t] = (int32_t)cf; tile_last_out[t] = (int32_t)cl;
    }
    *n_ctas_out = sk.G; *n_tiles_out = sk.n_tiles; *kb_out = sk.kb;
    return OA_OK;
}

int32_t oa_host_clusterk_pick(int32_t N, int32_t K, int32_t sms, int32_t min_fill_pct) { return clusterk_pick(N, K, sms, min_fill_pct); }

int oa_host_grammar_step(int32_t kind, const uint8_t* prefix, int32_t n, uint32_t* mask_out, int32_t* done_out) {
    return oa_host_grammar_step_ex(kind, "", prefix, n, mask_out, done_out);
}
int oa_host_grammar_step_ex(int32_t kind, const char* functions, const uint8_t* prefix, int32_t n, uint32_t* mask_out, int32_t* done_out) {
    if (kind < GRAMMAR_TOOLCALL || kind > GRAMMAR_TEXT) return OA_ERR_BAD_REQUEST;
    ToolPromptGrammar g(kind, functions ? functions : "");
    if (!g.active()) return OA_ERR_BAD_REQUEST;
    for (int i = 0; i < n; ++i) if (!g.advance(prefix[i])) return OA_ERR_BAD_REQUEST;
    g.allowed(mask_out); *done_out = g.done() ? 1 : 0;
    return OA_OK;
}

int oa_host_grammar_token_mask(const char* tokenizer_json_path, int32_t vocab, int32_t kind, const char* functions, const uint8_t* prefix, int32_t n,
                               uint32_t* mask_out, int32_t cap_words, char* key_out, int32_t key_cap) {
    if (kind < GRAMMAR_TOOLCALL || kind > GRAMMAR_TEXT || vocab <= 0 || !mask_out) return OA_ERR_BAD_REQUEST;
    try {
        // one trie per (tokenizer, vocab), built once: the same structure the engine builds at start-up
        static std::mutex mu; static std::map<std::string, std::shared_ptr<TokenTrie>> tries;
        const std::string tk = std::string(tokenizer_json_path ? tokenizer_json_path : "") + "#" + std::to_string(vocab);
        std::shared_ptr<TokenTrie> trie;
        {
            std::lock_guard<std::mutex> lk(mu);
            auto it = tries.find(tk);
            if (it == tries.end()) {
                ModelConfig mc; mc.vocab = vocab; mc.chat_template = "llama3";
                std::vector<std::string> bytes;
                if (tokenizer_json_path && tokenizer_json_path[0]) bytes = BpeTokenizer::load(tokenizer_json_path)->text_token_bytes();
                else { bytes.resize(256); for (int b = 0; b < 256; ++b) bytes[b] = std::string(1, (char)b); }
                trie = std::make_shared<TokenTrie>(); trie->build(bytes, vocab); tries[tk] = trie;
            } else trie = it->second;
        }
        if (trie->words() > cap_words) return OA_ERR_BAD_REQUEST;
        ToolPromptGrammar g(kind, functions ? functions : "");
        if (!g.active()) return OA_ERR_BAD_REQUEST;
        for (int i = 0; i < n; ++i) if (!g.advance(prefix[i])) return OA_ERR_BAD_REQUEST;
        trie->allowed_tokens(g, g.cursor(), mask_out);
        if (key_out && key_cap > 0) std::snprintf(key_out, (size_t)key_cap, "%s", grammar_mask_key(g, g.cursor()).c_str());
    } catch (const std::exception&) { return OA_ERR_BAD_REQUEST; }
    return OA_OK;
}

int oa_host_model_info(const char* config_json, char* buf, size_t n) {
    try {
        ModelConfig c; EngineOptions eo; parse_config(config_json ? config_json : "{}", c, eo);
        std::snprintf(buf, n, "{\"model\": \"%s\", \"hidden\": %d, \"n_layers\": %d, \"n_heads\": %d, \"n_kv_heads\": %d, \"head_dim\": %d, "
                      "\"ffn\": %d, \"vocab\": %d, \"tie_embeddings\": %d, \"qkv_bias\": %d, \"rope_scaling\": %d, \"rope_theta\": %.1f, "
                      "\"rms_eps\": %g, \"template\": \"%s\", \"decode_weight_bytes\": %.0f, \"kv_bytes_per_token\": %zu}",
                      c.name.c_str(), c.hidden, c.n_layers, c.n_heads, c.n_kv_heads, c.head_dim, c.ffn, c.vocab, c.tie_embeddings, c.qkv_bias,
                      c.rope_scaling, c.rope_theta, c.rms_eps, c.chat_template.c_str(), c.decode_weight_bytes(), c.kv_bytes_per_token());
    } catch (const std::exception&) { return OA_ERR_BAD_REQUEST; }
    return OA_OK;
}

}  // extern "C"
