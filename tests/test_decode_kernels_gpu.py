"""The decode step's fused kernels at full model widths against fp32 / fp64 references (pytest -m gpu).

Each projection runs through the launcher pairing DeviceModel::forward uses (oa_k_sk_resid_rmsnorm, oa_k_sk_swiglu, oa_k_qkv_rope) at
the per-rank shapes of the supported models, where the stream-K tiles are cut into many CTA pieces.  The references round where the
kernels round (sum + bias -> bf16 -> RoPE -> bf16; x + acc -> bf16 -> norm; silu(gate) * up -> bf16), so one bf16 ulp plus an fp32
accumulation floor separates them.  Attention inputs (oracle/attention_cases.py) hold one high-scoring key in every split piece of
the decode plan and in every 64-token chunk of a prefill, each with its own large V component, and every test proves on its reference
that dropping or mis-weighting any one of those pieces would move an output far beyond the tolerance."""
import ctypes as C
import math
import zlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from opsagent_b200 import _lib  # noqa: E402
from oracle.attention_cases import (AttnCase, assert_close, assert_sensitive, attn_tol, bf16_ulp, decode_pieces, dev, gen,  # noqa: E402
                                    ptr)

# fp32 references must be fp32: no TF32 tensor-core shortcuts in torch matmuls
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False


@pytest.fixture(scope="module")
def L():
    return _lib.load()


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------------
# per-rank decode shapes (csrc/config.hpp presets; TP ranks shard heads, ffn and vocab)
SHAPES = {
    "llama-3.2-1b": dict(H=2048, nh=32, nkv=8, D=64, F=8192, bias=False, theta=5e5, eps=1e-5, llama3=True),
    "llama-3-8b": dict(H=4096, nh=32, nkv=8, D=128, F=14336, bias=False, theta=5e5, eps=1e-5, llama3=False),
    "qwen2.5-32b": dict(H=5120, nh=40, nkv=8, D=128, F=27648, bias=True, theta=1e6, eps=1e-6, llama3=False),
    "qwen2.5-32b-tp4": dict(H=5120, nh=10, nkv=2, D=128, F=6912, bias=True, theta=1e6, eps=1e-6, llama3=False),
    "llama-3-70b": dict(H=8192, nh=64, nkv=8, D=128, F=28672, bias=False, theta=5e5, eps=1e-5, llama3=False),
    "llama-3-70b-tp8": dict(H=8192, nh=8, nkv=1, D=128, F=3584, bias=False, theta=5e5, eps=1e-5, llama3=False),
}
MS = (1, 5, 37, 128)
MAX_POS = 4096


def proj_dims(s, proj):
    qd = s["nh"] * s["D"]
    return {"qkv": ((s["nh"] + 2 * s["nkv"]) * s["D"], s["H"]), "o": (s["H"], qd), "gu": (2 * s["F"], s["H"]), "down": (s["H"], s["F"])}[proj]


# (shape, n_ctas): 0 = one CTA per SM (the engine's default); small counts give CTAs that own several whole tiles and pieces
CTA_CASES = [(name, 0) for name in SHAPES] + [("llama-3.2-1b", 3), ("llama-3.2-1b", 7), ("llama-3-70b-tp8", 7), ("qwen2.5-32b-tp4", 3)]


def ms_for(n_ctas):
    return MS if n_ctas == 0 else (5, 128)


def weights(N, K, seed):
    g = gen(seed)
    A = torch.randn(128, K, generator=g, device=dev()).to(torch.bfloat16)
    B = (torch.randn(N, K, generator=g, device=dev()) / math.sqrt(K)).to(torch.bfloat16)
    return A, B


def acc_floor(K):
    return 1e-6 * math.sqrt(K)          # fp32 accumulation-order difference of a K-long dot product of O(1) outputs


def drop_kblock(acc, A, B, M):
    """acc with the first 64-wide k-block of tile 0 (columns 0..127) missing: one lost stream-K piece"""
    alt = acc.clone()
    alt[:, :128] -= A[:M, :64].float() @ B[:128, :64].float().T
    return alt


def streamk_pieces(L, N, K, G):
    """max number of CTA pieces a 128-column tile is cut into (the plan the kernels use)"""
    n_tiles = (N + 127) // 128
    u0 = np.zeros(G + 1, np.int64); tf = np.zeros(n_tiles, np.int32); tl = np.zeros(n_tiles, np.int32)
    nc, nt, kb = C.c_int32(), C.c_int32(), C.c_int32()
    assert L.oa_host_streamk_plan(N, K, 128, G, u0.ctypes.data, G, tf.ctypes.data, tl.ctypes.data, n_tiles, C.byref(nc), C.byref(nt), C.byref(kb)) == 0
    return int((tl - tf).max()) + 1


def cluster_sizes(L, N, K, sms):
    kb = (K + 63) // 64
    picked = L.oa_host_clusterk_pick(N, K, sms, 0)
    return sorted({s for s in (2, 3, 4, 8) if kb >= 2 * s} | ({picked} if picked else set()))


# ---------------------------------------------------------------------------------------------------------------------------
def resid_ref(x, acc):
    return (x.float() + acc).to(torch.bfloat16)


def norm_ref(x, gain, eps):
    xf = x.float()
    r = torch.rsqrt(xf.pow(2).mean(1, keepdim=True) + eps)
    return xf * r * gain.float()


@pytest.mark.parametrize("proj", ["o", "down"])
@pytest.mark.parametrize("shape,n_ctas", CTA_CASES)
def test_resid_rmsnorm_projection(L, sms, shape, n_ctas, proj):
    s = SHAPES[shape]
    N, K = proj_dims(s, proj)
    G = n_ctas or sms
    eps = s["eps"]
    A, B = weights(N, K, zlib.crc32(f"{shape}/{proj}".encode()))
    g = gen(7)
    gain = (1 + 0.1 * torch.randn(N, generator=g, device=dev())).to(torch.bfloat16)
    flags = torch.zeros(1024, dtype=torch.int32, device=dev())
    if n_ctas == 0 and N >= 4096:
        assert streamk_pieces(L, N, K, G) >= 3, "full-width shapes cut tiles into three or more CTA pieces"
    ks = cluster_sizes(L, N, K, sms) if n_ctas == 0 else []
    for M in ms_for(n_ctas):
        x0 = torch.randn(M + 3, N, generator=g, device=dev()).to(torch.bfloat16)
        acc = A[:M].float() @ B.float().T
        ref_x = resid_ref(x0[:M], acc)
        tol_x = bf16_ulp(ref_x) + acc_floor(K)

        def run(path, cluster=0, ldx=N, with_norm=True):
            xw = torch.randn(M + 3, ldx, generator=g, device=dev()).to(torch.bfloat16)
            xw[:, :N] = x0
            before = xw.clone()
            xn = torch.full((M + 3, N), float("nan"), dtype=torch.bfloat16, device=dev()) if with_norm else None
            rc = L.oa_k_sk_resid_rmsnorm(path, ptr(A), ptr(B), M, N, K, G, cluster, ptr(xw), ldx, ptr(gain), ptr(xn), eps, ptr(flags), None)
            assert rc == 0, (path, cluster)
            assert int(flags.abs().sum()) == 0, "tile flags are re-armed to zero"
            assert torch.equal(xw[M:], before[M:]), "rows at and beyond M untouched"
            assert torch.equal(xw[:, N:], before[:, N:]), "columns beyond N untouched"
            if with_norm:
                assert torch.isnan(xn[M:].float()).all(), "xn rows at and beyond M untouched"
            return xw[:, :N].contiguous(), xn

        x_p0, xn_p0 = run(0)
        assert_close(x_p0[:M], ref_x, tol_x, f"x (path 0, M={M})")
        xn_ref = norm_ref(x_p0[:M], gain, eps)          # the norm of what the kernel stored: isolates the norm from x's rounding
        assert_close(xn_p0[:M], xn_ref, bf16_ulp(xn_ref) + 1e-6, f"xn (path 0, M={M})")
        assert_sensitive(ref_x, resid_ref(x0[:M], drop_kblock(acc, A, B, M)), tol_x, "dropped stream-K piece")
        if G <= sms:
            x_p1, xn_p1 = run(1)
            assert torch.equal(x_p1, x_p0) and torch.equal(xn_p1[:M], xn_p0[:M]), "fused residual == stream-K + consumer, bit for bit"
            x_again, _ = run(1)
            assert torch.equal(x_again, x_p1), "second launch on the same tile flags"
            x_wide, _ = run(1, ldx=N + 64, with_norm=False)
            assert torch.equal(x_wide, x_p0)
        for S in ks:
            x_c, xn_c = run(2, cluster=S)
            assert_close(x_c[:M], ref_x, tol_x, f"x (cluster S={S}, M={M})")
            assert_close(xn_c[:M], norm_ref(x_c[:M], gain, eps), bf16_ulp(norm_ref(x_c[:M], gain, eps)) + 1e-6, f"xn (cluster S={S})")
            if M * N >= 1 << 20:          # ~1e-4 of the elements flip a bf16 rounding: a million make equality impossible
                assert not torch.equal(x_c, x_p0), "cluster split-K sums in another order: it must not be the stream-K result"
            x_cw, _ = run(2, cluster=S, ldx=N + 64, with_norm=False)
            assert torch.equal(x_cw, x_c)


# ---------------------------------------------------------------------------------------------------------------------------
def swiglu_ref(acc):
    M, N = acc.shape
    a = acc.view(M, N // 32, 2, 16)
    return (torch.nn.functional.silu(a[:, :, 0]) * a[:, :, 1]).reshape(M, N // 2), a[:, :, 0].reshape(M, -1), a[:, :, 1].reshape(M, -1)


@pytest.mark.parametrize("shape,n_ctas", CTA_CASES)
def test_swiglu_projection(L, sms, shape, n_ctas):
    s = SHAPES[shape]
    N, K = proj_dims(s, "gu")
    F, G = N // 2, n_ctas or sms
    A, B = weights(N, K, zlib.crc32(f"{shape}/gu".encode()))
    flags = torch.zeros(1024, dtype=torch.int32, device=dev())
    for M in ms_for(n_ctas):
        acc = A[:M].float() @ B.float().T
        f, gt, up = swiglu_ref(acc)
        ref = f.to(torch.bfloat16)
        tol = bf16_ulp(ref) + acc_floor(K) * (gt.abs() + up.abs() + 1)

        def run(path):
            act = torch.full((M + 3, F), float("nan"), dtype=torch.bfloat16, device=dev())
            assert L.oa_k_sk_swiglu(path, ptr(A), ptr(B), M, F, K, G, ptr(act), ptr(flags), None) == 0, path
            assert int(flags.abs().sum()) == 0, "tile flags are re-armed to zero"
            assert torch.isnan(act[M:].float()).all(), "rows at and beyond M untouched"
            return act

        a0 = run(0)
        assert_close(a0[:M], ref, tol, f"act (path 0, M={M})")
        assert_sensitive(ref, swiglu_ref(drop_kblock(acc, A, B, M))[0].to(torch.bfloat16), tol, "dropped stream-K piece")
        if G <= sms:
            a1 = run(1)
            assert torch.equal(a1[:M], a0[:M]), "fused SwiGLU == stream-K + consumer, bit for bit"
            assert torch.equal(run(1)[:M], a1[:M]), "second launch on the same tile flags"


# ---------------------------------------------------------------------------------------------------------------------------
def rope_tables(s, max_pos=MAX_POS):
    """float64 math then fp32, as csrc/model.cpp rope_table (llama3 scaling: factor 32, low 1, high 4, original context 8192)"""
    D = s["D"]; half = D // 2
    inv = np.array([s["theta"] ** (-2.0 * i / D) for i in range(half)], np.float64)
    if s["llama3"]:
        factor, lo, hi, orig = 32.0, 1.0, 4.0, 8192
        for i in range(half):
            wavelen = 2.0 * math.pi / inv[i]
            if wavelen > orig / lo:
                inv[i] = inv[i] / factor
            elif wavelen >= orig / hi:
                smooth = (orig / wavelen - lo) / (hi - lo)
                inv[i] = (1.0 - smooth) * inv[i] / factor + smooth * inv[i]
    ang = np.arange(max_pos, dtype=np.float64)[:, None] * inv[None, :]
    return (torch.from_numpy(np.cos(ang).astype(np.float32)).to(dev()), torch.from_numpy(np.sin(ang).astype(np.float32)).to(dev()))


def rope_ref(acc, bias, pos, cos, sin, nh, nkv, D, K):
    """-> q [M, nh, D], k [M, nkv, D], v [M, nkv, D] (bf16) and the per-element tolerance of each"""
    M = acc.shape[0]
    pre = acc + (bias.float() if bias is not None else 0)
    pre = pre.to(torch.bfloat16).float().view(M, nh + 2 * nkv, D)
    half = D // 2
    c, s_ = cos[pos][:, None, :], sin[pos][:, None, :]
    a, b = pre[:, : nh + nkv, :half], pre[:, : nh + nkv, half:]
    rot = torch.cat([a * c - b * s_, b * c + a * s_], dim=2)
    # one bf16 ulp of the output, plus the output's response to one ulp of the bf16-rounded inputs
    prop = torch.cat([(a * c).abs() + (b * s_).abs(), (b * c).abs() + (a * s_).abs()], dim=2) * 2.0 ** -7
    rot_b = rot.to(torch.bfloat16)
    tol_rot = bf16_ulp(rot_b) + prop + 2 * acc_floor(K)       # |cos| + |sin| <= sqrt(2) times the sums' floor
    v = pre[:, nh + nkv:].to(torch.bfloat16)
    tol_v = bf16_ulp(v) + acc_floor(K)
    return rot_b[:, :nh], rot_b[:, nh:], v, tol_rot[:, :nh], tol_rot[:, nh:], tol_v


@pytest.mark.parametrize("shape,n_ctas", CTA_CASES)
def test_qkv_rope_kv_write(L, sms, shape, n_ctas):
    s = SHAPES[shape]
    nh, nkv, D = s["nh"], s["nkv"], s["D"]
    N, K = proj_dims(s, "qkv")
    G = n_ctas or sms
    A, B = weights(N, K, zlib.crc32(f"{shape}/qkv".encode()))
    g = gen(11)
    bias = (0.5 * torch.randn(N, generator=g, device=dev())).to(torch.bfloat16) if s["bias"] else None
    cos, sin = rope_tables(s)
    n_layers, layer, num_pages = 3, 1, 160
    cache0 = torch.randn(n_layers, 2, num_pages, nkv, 64, D, generator=g, device=dev()).to(torch.bfloat16)
    flags = torch.zeros(1024, dtype=torch.int32, device=dev())
    ks = cluster_sizes(L, N, K, sms) if n_ctas == 0 else []
    for M in ms_for(n_ctas):
        special = [0, 1, 63, 64, MAX_POS - 2, MAX_POS - 1]
        rest = torch.randint(0, MAX_POS, (M,), generator=g, device=dev()).tolist()
        pos = torch.tensor((special + rest)[:M], dtype=torch.int32, device=dev())
        pages = torch.randperm(num_pages, generator=g, device=dev())[:M]
        offs = torch.randint(0, 64, (M,), generator=g, device=dev())
        offs[0::2] = 0; offs[1::4] = 63                     # both ends of a page
        slots = (pages * 64 + offs).to(torch.int32)
        acc = A[:M].float() @ B.float().T
        q_ref, k_ref, v_ref, tq, tk, tv = rope_ref(acc, bias, pos.long(), cos, sin, nh, nkv, D, K)

        def run(path, cluster=0):
            cache = cache0.clone()
            q = torch.randn(M + 3, nh * D, generator=g, device=dev()).to(torch.bfloat16)
            q_before = q.clone()
            rc = L.oa_k_qkv_rope(path, ptr(A), ptr(B), M, K, G, cluster, ptr(bias), ptr(pos), ptr(slots), ptr(cos), ptr(sin), ptr(q),
                                 ptr(cache), num_pages, n_layers, layer, nh, nkv, D, ptr(flags), None)
            assert rc == 0, (path, cluster)
            assert int(flags.abs().sum()) == 0, "tile flags are re-armed to zero"
            assert torch.equal(q[M:], q_before[M:]), "q rows at and beyond M untouched"
            kk = cache[layer, 0, pages, :, offs].clone()     # [M, nkv, D]
            vv = cache[layer, 1, pages, :, offs].clone()
            written = torch.zeros_like(cache, dtype=torch.bool)
            written[layer, :, pages, :, offs] = True
            assert torch.equal(cache[~written], cache0[~written]), "only the M written K/V rows of the chosen layer change"
            return q[:M].view(M, nh, D), kk, vv

        q0, k0, v0 = run(0)
        assert_close(q0, q_ref, tq, f"q (path 0, M={M})")
        assert_close(k0, k_ref, tk, f"k (path 0, M={M})")
        assert_close(v0, v_ref, tv, f"v (path 0, M={M})")
        q_drop = rope_ref(drop_kblock(acc, A, B, M), bias, pos.long(), cos, sin, nh, nkv, D, K)[0]
        assert_sensitive(q_ref, q_drop, tq, "dropped stream-K piece")
        if G <= sms:
            q1, k1, v1 = run(1)
            assert torch.equal(q1, q0) and torch.equal(k1, k0) and torch.equal(v1, v0), "fused RoPE == stream-K + consumer, bit for bit"
            q1b, k1b, v1b = run(1)
            assert torch.equal(q1b, q1) and torch.equal(k1b, k1) and torch.equal(v1b, v1), "second launch on the same tile flags"
        q3, k3, v3 = run(3)
        assert_close(q3, q_ref, tq, f"q (tile GEMM, M={M})"); assert_close(k3, k_ref, tk, "k (tile GEMM)"); assert_close(v3, v_ref, tv, "v (tile GEMM)")
        for S in ks:
            qc, kc, vc = run(2, cluster=S)
            assert_close(qc, q_ref, tq, f"q (cluster S={S}, M={M})"); assert_close(kc, k_ref, tk, f"k (cluster S={S})")
            assert_close(vc, v_ref, tv, f"v (cluster S={S})")


# ---------------------------------------------------------------------------------------------------------------------------
# attention (inputs: oracle/attention_cases.py — one high-scoring key in every split piece / every 64-token chunk)
DECODE_CASES = {
    "bench-b128": dict(ctx=[1600 + (37 * i) % 191 for i in range(128)], nh=32, nkv=8, D=128, min_pieces=2),
    "ctx32768": dict(ctx=[32768], nh=32, nkv=8, D=128, min_pieces=3),
    "b4-ctx16384-grp8": dict(ctx=[16384] * 4, nh=8, nkv=1, D=128, min_pieces=3),
    "b4-ctx16384-grp5": dict(ctx=[16384, 16000, 16384, 15000], nh=10, nkv=2, D=128, min_pieces=3),
    "d64": dict(ctx=[3000, 2048, 777, 4095, 129, 64, 1, 2500], nh=32, nkv=8, D=64, min_pieces=2),
    "tiny-ctx": dict(ctx=[1, 64, 65, 1, 64, 65, 1000], nh=8, nkv=2, D=128, min_pieces=2),
}


@pytest.mark.parametrize("case", list(DECODE_CASES))
def test_decode_attention_in_kernel_merge(L, sms, case):
    cfg = DECODE_CASES[case]
    ctx, nh, nkv, D = cfg["ctx"], cfg["nh"], cfg["nkv"], cfg["D"]
    target = 2 * sms                                   # the engine's plan: two CTAs per SM
    pieces, cut = decode_pieces(L, ctx, nkv, target)
    assert cut and max(len(pieces[k]) for k in cut) >= cfg["min_pieces"], "the plan must cut items into several pieces"
    ac = AttnCase(ctx, [1] * len(ctx), nh, nkv, D, n_layers=3, seed=len(ctx) * 31 + D + nh, pieces=pieces)
    counters = torch.zeros(len(cut) + 8, dtype=torch.int32, device=dev())     # zeroed once, never reset between layers
    for layer in range(3):
        ref, ref_abs = ac.ref(layer)
        tol = attn_tol(ref, ref_abs)
        sep = ac.run(L, layer=layer, counters=None, n_ctas_target=target)
        fused = ac.run(L, layer=layer, counters=counters, n_ctas_target=target)
        assert_close(sep, ref, tol, f"separate merge, layer {layer}", max_frac=None)
        assert_close(fused, ref, tol, f"in-kernel merge, layer {layer}", max_frac=None)
        assert ((fused.float() - sep.float()).abs() <= bf16_ulp(sep.float())).all(), "the two merges agree to one bf16 ulp"
        if layer == 0:
            # power: dropping, or doubling the weight of, ANY piece of any cut item moves an output by more than 5x the tolerance
            ac.piece_power(0, ref, tol, items=cut)
    got = counters.cpu().tolist()
    for j, key in enumerate(cut):
        assert got[j] == 3 * len(pieces[key]), f"item {j}: counter {got[j]} after 3 layers of {len(pieces[key])} pieces"
    assert all(v == 0 for v in got[len(cut):]), "counters of no item stay zero"


PREFILL_CASES = {
    "chunk-after-14k-grp8": dict(ctx=[16384], q=[2048], nh=8, nkv=1, D=128),
    "chunk-after-14k-grp5": dict(ctx=[16384], q=[2048], nh=10, nkv=2, D=128),
    "fresh-4096-d64": dict(ctx=[4096], q=[4096], nh=8, nkv=2, D=64),
}


@pytest.mark.parametrize("impl", ["tcgen05", "legacy"])
@pytest.mark.parametrize("case", list(PREFILL_CASES))
def test_prefill_attention_long_context(L, case, impl, monkeypatch):
    if impl == "legacy":
        monkeypatch.setenv("OA_PREFILL_ATTN", "legacy")
    else:
        monkeypatch.delenv("OA_PREFILL_ATTN", raising=False)
    cfg = PREFILL_CASES[case]
    ac = AttnCase(cfg["ctx"], cfg["q"], cfg["nh"], cfg["nkv"], cfg["D"], n_layers=2, seed=cfg["ctx"][0] + cfg["nh"])
    out = ac.run(L, layer=1)
    ref, ref_abs = ac.ref(1)
    tol = attn_tol(ref, ref_abs)
    assert_close(out, ref, tol, f"prefill ({impl})", max_frac=None)
    ac.piece_power(1, ref, tol)                        # every 64-token KV chunk matters to the rows that see it


# ---------------------------------------------------------------------------------------------------------------------------
def pack_mask(allowed):
    """bool [S, V] -> uint32 words [S, ceil(V/32)] (bit j of word w = id 32w + j)"""
    S, V = allowed.shape
    W = (V + 31) // 32
    a = np.zeros((S, W * 32), np.uint8); a[:, :V] = allowed
    return np.packbits(a, axis=1, bitorder="little").view(np.uint32).reshape(S, W)


LM_CASES = [  # (vocab of the shard, global vocab, col_offset, K)
    (128256, 128256, 0, 2048),
    (152064, 152064, 0, 1024),
    (38016, 152064, 2 * 38016, 1024),      # Qwen2.5 vocab-parallel rank 2 of 4
    (32008, 32008, 0, 512),                # not a multiple of any block_n
]


@pytest.mark.parametrize("bn", [64, 128, 256])
@pytest.mark.parametrize("N,V,off,K", LM_CASES)
def test_lm_head_grammar_mask(L, N, V, off, K, bn):
    g = gen(N + bn)
    A = torch.randn(128, K, generator=g, device=dev()).to(torch.bfloat16)
    B = (0.1 * torch.randn(N, K, generator=g, device=dev())).to(torch.bfloat16)
    ref = A.float() @ B.float().T
    ids_full = torch.empty(128, dtype=torch.int32, device=dev())
    assert L.oa_k_lm_head(ptr(A), ptr(B), 128, N, K, bn, None, None, 0, off, None, ptr(ids_full), None) == 0
    top = ids_full.cpu().numpy()                   # the kernel's own free arg-max of each row
    rng = np.random.default_rng(N + bn)
    # mask states (global ids): a single id at 0, at the shard's last column, on both sides of a tile boundary; a sparse 1 % set;
    # nothing; all but the row's free arg-max
    def one(local):
        a = np.zeros(V, bool); a[off + local] = True
        if off:
            a[:off] = True               # decoys in another shard: found only if col_offset were ignored
        return a
    singles = [0, N - 1, bn, bn - 1]
    states = [one(c) for c in singles] + [rng.random(V) < 0.01, np.zeros(V, bool)]
    NONE, first_excl = len(singles) + 1, len(states)
    for r in range(8):
        a = np.ones(V, bool); a[off + top[r]] = False; states.append(a)
    table = torch.from_numpy(pack_mask(np.stack(states)).view(np.int32)).to(dev())
    allowed = torch.from_numpy(np.stack(states)[:, off:off + N]).to(dev())
    for M in (1, 37, 128):                   # a partial and a full 128-row A box
        slot = np.full(M, -1, np.int32)
        for r in range(M):
            if r < 8:
                slot[r] = first_excl + r
            elif r % 3 == 0:
                slot[r] = (r // 3) % first_excl
        slot_d = torch.from_numpy(slot).to(dev())
        logits0 = torch.empty(M, N, dtype=torch.float32, device=dev()); ids0 = torch.empty(M, dtype=torch.int32, device=dev())
        assert L.oa_k_lm_head(ptr(A), ptr(B), M, N, K, bn, None, None, 0, off, ptr(logits0), ptr(ids0), None) == 0
        assert ((logits0 - ref[:M]).abs() <= 1e-4 * (K ** 0.5) + 1e-5 * ref[:M].abs()).all(), f"fp32 logits (M={M})"
        logits = torch.empty(M, N, dtype=torch.float32, device=dev()); ids = torch.full((M,), -7, dtype=torch.int32, device=dev())
        assert L.oa_k_lm_head(ptr(A), ptr(B), M, N, K, bn, ptr(table), ptr(slot_d), table.shape[1], off, ptr(logits), ptr(ids), None) == 0
        assert torch.equal(logits, logits0), "stored logits stay unmasked"
        row_allowed = torch.ones(M, N, dtype=torch.bool, device=dev())
        masked_rows = slot_d >= 0
        row_allowed[masked_rows] = allowed[slot_d[masked_rows].long()]
        lg = logits.masked_fill(~row_allowed, float("-inf"))
        mx = lg.max(dim=1, keepdim=True).values
        exp_ids = torch.where((lg == mx) & row_allowed, torch.arange(N, device=dev())[None, :], N).min(dim=1).values
        exp_ids = torch.where(row_allowed.any(1), exp_ids, torch.zeros_like(exp_ids))       # nothing allowed: id 0 (argmax_reduce_kernel)
        assert torch.equal(ids.long(), exp_ids), f"M={M}: rows {torch.nonzero(ids.long() != exp_ids).flatten().tolist()[:8]}"
        # unmasked rows: the free arg-max; excluding it changes the answer; single ids and the empty set are pinned
        free = slot < 0
        assert torch.equal(ids[torch.from_numpy(free).to(dev())], ids0[torch.from_numpy(free).to(dev())])
        nx = min(M, 8)
        assert (ids[:nx].long().cpu().numpy() != ids0[:nx].long().cpu().numpy()).all(), "the mask changed the answer where it excludes the free arg-max"
        for r in range(M):
            if 0 <= slot[r] < len(singles):
                assert int(ids[r]) == singles[slot[r]]
            if slot[r] == NONE:
                assert int(ids[r]) == 0
