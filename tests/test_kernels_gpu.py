"""Kernel-level parity on the B200 (pytest -m gpu): every hand-written sm_100a kernel through its C-ABI entry
point against (a) the CPU oracle where it has the same function and (b) a plain torch fp32 reference of the op."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from opsagent_b200 import _lib  # noqa: E402
from oracle import oracle as O  # noqa: E402  (checker only)
from oracle.attention_cases import AttnCase, assert_close, attn_tol  # noqa: E402

EPI_STORE, EPI_RESID, EPI_SWIGLU, EPI_LOGITS = 0, 1, 2, 3


@pytest.fixture(scope="module")
def L():
    return _lib.load()


def dev():
    return torch.device("cuda:0")


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def bf16_bits(t):
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


# ------------------------------------------------------------------------------------------------
def test_weight_init_bit_exact_vs_oracle(L):
    rows, cols = 96, 320
    dst = torch.empty(rows, cols, dtype=torch.bfloat16, device=dev())
    assert L.oa_k_init_weight(ptr(dst), 1234, 37, -1, rows, cols, 0.02, 0.0, None) == 0
    torch.cuda.synchronize()
    got = bf16_bits(dst)
    lib = O.lib()
    exp = np.array([lib.oa_ref_gen_bf16(1234, 37, i, 0.02, 0.0) for i in range(rows * cols)], dtype=np.uint16).reshape(rows, cols)
    assert (got == exp).all()
    # norm-gain style (mean 1) and the interleaved gate/up layout
    dst2 = torch.empty(1, cols, dtype=torch.bfloat16, device=dev())
    assert L.oa_k_init_weight(ptr(dst2), 99, 7, -1, 1, cols, 0.1, 1.0, None) == 0
    exp2 = np.array([lib.oa_ref_gen_bf16(99, 7, i, 0.1, 1.0) for i in range(cols)], dtype=np.uint16)
    torch.cuda.synchronize()
    assert (bf16_bits(dst2)[0] == exp2).all()
    F, H = 64, 64
    gu = torch.empty(2 * F, H, dtype=torch.bfloat16, device=dev())
    assert L.oa_k_init_weight(ptr(gu), 5, 4, 5, 2 * F, H, 0.02, 0.0, None) == 0
    torch.cuda.synchronize()
    g = np.array([lib.oa_ref_gen_bf16(5, 4, i, 0.02, 0.0) for i in range(F * H)], dtype=np.uint16).reshape(F, H)
    u = np.array([lib.oa_ref_gen_bf16(5, 5, i, 0.02, 0.0) for i in range(F * H)], dtype=np.uint16).reshape(F, H)
    got = bf16_bits(gu)
    for r in range(2 * F):
        blk, w = divmod(r, 32)
        src = g if w < 16 else u
        assert (got[r] == src[blk * 16 + (w & 15)]).all()


@pytest.mark.parametrize("T,H", [(1, 256), (7, 320), (128, 4096), (33, 8192), (5, 2048)])
def test_rmsnorm_vs_oracle(L, T, H):
    g = torch.Generator(device="cpu").manual_seed(T * 1000 + H)
    x = (torch.randn(T, H, generator=g) * 1.7).to(torch.bfloat16)
    gain = (1 + 0.1 * torch.randn(H, generator=g)).to(torch.bfloat16)
    xd, gd = x.to(dev()), gain.to(dev())
    y = torch.empty_like(xd)
    assert L.oa_k_rmsnorm(ptr(xd), ptr(gd), ptr(y), T, H, 1e-5, None) == 0
    torch.cuda.synchronize()
    xf = np.ascontiguousarray(x.float().numpy()); ref = np.empty_like(xf)
    gb = np.ascontiguousarray(bf16_bits(gain))
    O.lib().oa_ref_rmsnorm(xf.ctypes.data, gb.ctypes.data, ref.ctypes.data, T, H, 1e-5, 1)
    got = y.float().cpu().numpy()
    # identical up to the fp32-vs-double sum of squares: at most one bf16 ulp on a handful of elements
    ulp = np.maximum(np.abs(ref), 1e-3) * 2.0 ** -7
    assert (np.abs(got - ref) <= ulp).all()
    assert (got != ref).mean() < 0.02


GEMM_CASES = [  # M, N, K
    (128, 512, 256), (77, 256, 320), (300, 1024, 512), (1, 2304, 256), (128, 4096, 4096), (130, 1000, 192),
]


@pytest.mark.parametrize("bn", [32, 64, 128, 256])
@pytest.mark.parametrize("M,N,K", GEMM_CASES)
def test_gemm_store_and_bias(L, M, N, K, bn):
    g = torch.Generator(device="cpu").manual_seed(M + N + K + bn)
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    B = (torch.randn(N, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    bias = torch.randn(N, generator=g).to(torch.bfloat16).to(dev())
    ref = A.float() @ B.float().T
    for use_bias in (False, True):
        out = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=dev())
        assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_STORE, bn, ptr(out), ptr(bias) if use_bias else None, None, None, None, None) == 0
        torch.cuda.synchronize()
        r = ref + bias.float() if use_bias else ref
        err = (out.float() - r).abs()
        tol = r.abs() * 2.0 ** -8 + 2e-3 * (K ** 0.5) * 0.25 * 2.0 ** -8 + 1e-4
        assert torch.isfinite(out.float()).all()
        assert (err <= tol * 1.01 + 1e-3).all(), float((err - tol).max())


@pytest.mark.parametrize("bn", [32, 128, 256])
def test_gemm_residual_in_place(L, bn):
    M, N, K = 200, 768, 512
    g = torch.Generator(device="cpu").manual_seed(bn)
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    B = (torch.randn(N, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    x = torch.randn(M, N, generator=g).to(torch.bfloat16).to(dev())
    ref = (A.float() @ B.float().T + x.float()).to(torch.bfloat16)
    assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_RESID, bn, ptr(x), None, ptr(x), None, None, None) == 0
    torch.cuda.synchronize()
    diff = (x.float() - ref.float()).abs()
    assert (diff <= ref.float().abs() * 2.0 ** -7 + 1e-3).all()
    assert (x != ref).float().mean() < 0.01      # only accumulation-order rounding flips


@pytest.mark.parametrize("bn", [32, 64, 128, 256])
def test_gemm_swiglu(L, bn):
    M, F, K = 150, 512, 256
    g = torch.Generator(device="cpu").manual_seed(bn + 1)
    A = torch.randn(M, K, generator=g).to(torch.bfloat16).to(dev())
    Wg = (torch.randn(F, K, generator=g) * 0.1).to(torch.bfloat16)
    Wu = (torch.randn(F, K, generator=g) * 0.1).to(torch.bfloat16)
    # physical layout: 16 gate rows then 16 up rows per 32-row block
    W = torch.stack([Wg.view(F // 16, 16, K), Wu.view(F // 16, 16, K)], dim=1).reshape(2 * F, K).contiguous().to(dev())
    out = torch.empty(M, F, dtype=torch.bfloat16, device=dev())
    assert L.oa_k_gemm(ptr(A), ptr(W), M, 2 * F, K, EPI_SWIGLU, bn, ptr(out), None, None, None, None, None) == 0
    torch.cuda.synchronize()
    gt = A.float() @ Wg.to(dev()).float().T
    up = A.float() @ Wu.to(dev()).float().T
    ref = torch.nn.functional.silu(gt) * up
    assert ((out.float() - ref).abs() <= ref.abs() * 2.0 ** -7 + 2e-3).all()


@pytest.mark.parametrize("bn", [64, 256])
@pytest.mark.parametrize("M,N,K", [(128, 2304, 256), (3, 1280, 320), (200, 128256, 256)])
def test_gemm_logits_argmax(L, M, N, K, bn):
    g = torch.Generator(device="cpu").manual_seed(N + bn)
    A = torch.randn(M, K, generator=g).to(torch.bfloat16).to(dev())
    B = (torch.randn(N, K, generator=g) * 0.1).to(torch.bfloat16).to(dev())
    logits = torch.empty(M, N, dtype=torch.float32, device=dev())
    ids = torch.empty(M, dtype=torch.int32, device=dev())
    assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_LOGITS, bn, None, None, None, ptr(logits), ptr(ids), None) == 0
    torch.cuda.synchronize()
    ref = A.float() @ B.float().T
    assert ((logits - ref).abs() <= 1e-4 * (K ** 0.5) + 1e-5 * ref.abs()).all()
    # fused arg-max is exact on the kernel's own logits, ties -> lowest index
    mx = logits.max(dim=1, keepdim=True).values
    first = torch.where(logits == mx, torch.arange(N, device=dev())[None, :], N).min(dim=1).values
    assert (ids.long() == first).all()
    # ... and without materialising logits
    ids2 = torch.empty(M, dtype=torch.int32, device=dev())
    assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_LOGITS, bn, None, None, None, None, ptr(ids2), None) == 0
    assert (ids2 == ids).all()


@pytest.mark.parametrize("M,N,K", [(5000, 2304, 320), (300, 1024, 512), (8192, 6144, 256)])
def test_gemm_persistent_kernel_all_epilogues(L, M, N, K, monkeypatch):
    """prefill path: persistent 128x256 tiles, double-buffered TMEM, transposed coalesced epilogue (forced for small shapes)"""
    monkeypatch.setenv("OA_GEMM_PERSISTENT_MIN_TILES", "1")
    g = torch.Generator(device="cpu").manual_seed(M + N)
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    B = (torch.randn(N, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    bias = torch.randn(N, generator=g).to(torch.bfloat16).to(dev())
    ref = A.float() @ B.float().T
    out = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=dev())
    assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_STORE, 256, ptr(out), ptr(bias), None, None, None, None) == 0
    torch.cuda.synchronize()
    r = ref + bias.float()
    assert torch.isfinite(out.float()).all()
    assert ((out.float() - r).abs() <= r.abs() * 2.0 ** -8 * 1.01 + 2e-3).all()
    x = torch.randn(M, N, generator=g).to(torch.bfloat16).to(dev())
    refx = (ref + x.float()).to(torch.bfloat16)
    assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_RESID, 256, ptr(x), None, ptr(x), None, None, None) == 0
    torch.cuda.synchronize()
    assert ((x.float() - refx.float()).abs() <= refx.float().abs() * 2.0 ** -7 + 1e-3).all()
    F = N // 2
    out2 = torch.full((M, F), float("nan"), dtype=torch.bfloat16, device=dev())
    assert L.oa_k_gemm(ptr(A), ptr(B), M, N, K, EPI_SWIGLU, 256, ptr(out2), None, None, None, None, None) == 0
    torch.cuda.synchronize()
    acc = ref.view(M, N // 32, 2, 16)
    rs = (torch.nn.functional.silu(acc[:, :, 0]) * acc[:, :, 1]).reshape(M, F)
    assert torch.isfinite(out2.float()).all()
    assert ((out2.float() - rs).abs() <= rs.abs() * 2.0 ** -7 + 3e-3).all()


@pytest.mark.parametrize("bn", [128, 256])
@pytest.mark.parametrize("M,N,K,G", [(128, 4096, 4096, 148), (128, 6144, 4096, 148), (77, 1024, 14336, 148), (1, 320, 320, 148),
                                      (128, 28672, 4096, 148), (16, 2304, 256, 5), (128, 512, 512, 3), (100, 1000, 192, 148),
                                      (256, 4096, 4096, 148), (200, 1792, 5120, 148), (129, 320, 320, 7)])
def test_gemm_streamk_partials_sum_to_the_product(L, M, N, K, G, bn):
    if M > 128 and bn != 128:
        pytest.skip("two 128-row tiles need BN=128 (TMEM columns)")
    g = torch.Generator(device="cpu").manual_seed(N + K + bn + G)
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    B = (torch.randn(N, K, generator=g) * 0.5).to(torch.bfloat16).to(dev())
    out = torch.full((M, N), float("nan"), dtype=torch.float32, device=dev())
    assert L.oa_k_gemm_streamk(ptr(A), ptr(B), M, N, K, bn, G, ptr(out), None) == 0, _lib.last_error()
    ref = A.float() @ B.float().T
    assert torch.isfinite(out).all()
    assert ((out - ref).abs() <= 2e-4 * (K ** 0.5) + 1e-5 * ref.abs()).all(), float((out - ref).abs().max())
    # fixed summation order => bitwise reproducible run to run
    out2 = torch.empty_like(out)
    assert L.oa_k_gemm_streamk(ptr(A), ptr(B), M, N, K, bn, G, ptr(out2), None) == 0
    assert torch.equal(out, out2)


# ------------------------------------------------------------------------------------------------
# attention inputs whose output depends on every 64-token chunk (oracle/attention_cases.py); fp64 reference, one bf16 ulp plus the
# bound of the kernels' bf16 probabilities
def _run_paged(L, ac, splits):
    T = ac.q.shape[0]
    out = torch.full((T, ac.nh, ac.D), float("nan"), dtype=torch.bfloat16, device=dev())
    ctx_a = np.array(ac.ctx, np.int32); ql = np.array(ac.q_lens, np.int32); bt_np = np.ascontiguousarray(ac.bt.numpy())
    rc = L.oa_k_paged_attention(ptr(ac.q), ptr(out), ptr(ac.kv[0]), ac.num_pages, bt_np.ctypes.data, ac.maxp, ctx_a.ctypes.data, ql.ctypes.data,
                                len(ac.ctx), ac.nh, ac.nkv, ac.D, splits, None)
    assert rc == 0, _lib.last_error()
    return out


@pytest.mark.parametrize("splits", [0, 3])
@pytest.mark.parametrize("nh,nkv,D", [(32, 8, 128), (8, 2, 64), (5, 1, 64), (8, 1, 128), (40, 8, 128)])
def test_paged_decode_attention(L, nh, nkv, D, splits):
    ctx = [1, 63, 64, 65, 200, 1000, 129, 517]
    ac = AttnCase(ctx, [1] * len(ctx), nh, nkv, D, n_layers=1, seed=11)
    out = _run_paged(L, ac, splits)
    ref, ref_abs = ac.ref(0)
    tol = attn_tol(ref, ref_abs)
    assert_close(out, ref, tol, "decode attention", max_frac=None)
    ac.piece_power(0, ref, tol)


@pytest.mark.parametrize("splits", [0, 3])
@pytest.mark.parametrize("nh,nkv,D", [(32, 8, 128), (5, 1, 64)])
def test_paged_decode_attention_flat(L, nh, nkv, D, splits):
    """random q: the mass spreads over many keys and the running max keeps moving from chunk to chunk"""
    ctx = [1, 65, 1000, 3000, 517]
    ac = AttnCase(ctx, [1] * len(ctx), nh, nkv, D, n_layers=1, seed=13, flat=True)
    out = _run_paged(L, ac, splits)
    ref, ref_abs = ac.ref(0)
    assert_close(out, ref, attn_tol(ref, ref_abs), "flat decode attention", max_frac=None)


@pytest.mark.parametrize("nh,nkv,D", [(8, 2, 128), (4, 2, 64), (5, 1, 64)])
def test_paged_prefill_attention(L, nh, nkv, D):
    # (ctx after the chunk, new rows): fresh prompts, a chunk continuing a cached prefix, ragged tile tails
    cases = [(64, 64), (130, 130), (200, 37), (1, 1), (333, 100), (128, 128)]
    for flat in (False, True):
        ac = AttnCase([c for c, _ in cases], [q for _, q in cases], nh, nkv, D, n_layers=1, seed=3, flat=flat)
        out = _run_paged(L, ac, 0)
        ref, ref_abs = ac.ref(0)
        tol = attn_tol(ref, ref_abs)
        assert_close(out, ref, tol, f"prefill attention (flat={flat})", max_frac=None)
        if not flat:
            ac.piece_power(0, ref, tol)
