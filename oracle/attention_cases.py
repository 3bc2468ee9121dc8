"""Paged-attention test inputs and their fp64 reference (torch, on cuda:0).

TEST INFRASTRUCTURE ONLY, like oracle.py: tests/ import it, the product never does.

AttnCase builds a paged KV cache [n_layers][2][num_pages][n_kv][64][D] whose attention output depends on every piece of KV the kernels
handle separately:
  * every (sequence, kv head) gets one high-scoring key in each of its `pieces` (chunk ranges: the split pieces of the decode plan, or
    every 64-token chunk by default) and in its first, a middle and its last chunk.  q is aligned with those keys, so they share
    almost all of the softmax mass equally;
  * the V row of the key planted in piece k carries +-AMP on dimension k mod D, so losing, repeating or mis-weighting any one piece moves
    that output dimension by about AMP / (number of planted keys), far beyond the tolerance;
  * the other V rows have a per-dimension mean of magnitude 1..2, so every output is of order 1 and a one-ulp tolerance means something.
`piece_power` proves the second point on the reference for every piece, instead of assuming it.
flat=True instead draws q at random (many keys share the mass and the running max keeps moving)."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

AMP = 64.0


def dev():
    return torch.device("cuda:0")


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def gen(seed):
    return torch.Generator(device=dev()).manual_seed(seed)


def bf16_ulp(x):
    """one bf16 ulp at |x| (fp32 tensor); 0 at 0"""
    _, e = torch.frexp(x.float())
    u = torch.ldexp(torch.ones_like(x, dtype=torch.float32), e - 8)
    return torch.where(x == 0, torch.zeros_like(u), u)


def assert_close(got, ref, tol, what, max_frac=0.02):
    """|got - ref| <= tol everywhere and, unless max_frac is None, fewer than max_frac of the elements differ at all from the
    reference rounded to got's type (a systematic error that stays within the tolerance still shows up there)"""
    rounded = ref.to(got.dtype).float()
    got, ref = got.float(), ref.float()
    assert torch.isfinite(got).all(), what
    err = (got - ref).abs()
    bad = err > tol
    assert not bad.any(), f"{what}: {int(bad.sum())} elements off, worst excess {float((err - tol).max()):.3e}"
    if max_frac is not None:
        frac = float((got != rounded).float().mean())
        assert frac < max_frac, f"{what}: {frac:.3%} of elements differ from the reference"


def assert_sensitive(ref, alt, tol, what):
    """the test's own power: a perturbed reference (a dropped k-block / chunk / piece) must fail it by a wide margin"""
    assert ((alt.float() - ref.float()).abs() > 5 * tol).any(), f"{what}: the perturbation stays within the tolerance"


def attn_tol(ref, ref_abs):
    """one bf16 ulp of the output plus the bf16 rounding of the probabilities the P.V product consumes (2^-9 relative each)"""
    return bf16_ulp(ref.float()) + 2.0 ** -8 * ref_abs.float() + 1e-5


def every_chunk(ctx, nkv):
    return {(i, h): [(c, c + 1) for c in range((n + 63) // 64)] for i, n in enumerate(ctx) for h in range(nkv)}


def decode_pieces(L, ctx, nkv, n_ctas_target):
    """the decode plan the kernels run (oa_host_decode_plan): ({(seq, kvh): [(chunk_begin, chunk_end), ...]} of every item,
    [(seq, kvh) of the cut items in merge-counter order])"""
    n = len(ctx)
    ctx_a = np.array(ctx, np.int32)
    cap = sum((c + 63) // 64 for c in ctx) * nkv + n_ctas_target + 16
    segs = np.zeros((cap, 5), np.int32); cta_ptr = np.zeros(n_ctas_target + 2, np.int32)
    nc, ns, nsl = C.c_int32(), C.c_int32(), C.c_int32()
    assert L.oa_host_decode_plan(ctx_a.ctypes.data, n, nkv, n_ctas_target, 0, segs.ctypes.data, cap, cta_ptr.ctypes.data, n_ctas_target + 1,
                                 C.byref(nc), C.byref(ns), C.byref(nsl)) == 0
    pieces, cut = {}, []
    for sq, kvh, cb, ce, slot in segs[: ns.value].tolist():
        pieces.setdefault((sq, kvh), []).append((cb, ce))
        if slot >= 0 and (not cut or cut[-1] != (sq, kvh)):
            cut.append((sq, kvh))
    return pieces, cut


class AttnCase:
    def __init__(self, ctx, q_lens, nh, nkv, D, n_layers, seed, pieces=None, flat=False):
        g = gen(seed)
        rng = np.random.default_rng(seed)
        self.ctx, self.q_lens, self.nh, self.nkv, self.D, self.n_layers = list(ctx), list(q_lens), nh, nkv, D, n_layers
        self.pieces = pieces if pieces is not None else every_chunk(ctx, nkv)
        n = len(ctx)
        npg = [(c + 63) // 64 for c in ctx]
        self.maxp = max(npg)
        self.num_pages = sum(npg) + 5
        perm = torch.randperm(self.num_pages, generator=g, device=dev()).cpu()
        self.bt = torch.zeros(n, self.maxp, dtype=torch.int32); k = 0
        for i in range(n):
            self.bt[i, :npg[i]] = perm[k:k + npg[i]].to(torch.int32); k += npg[i]
        cache = torch.randn(n_layers, 2, self.num_pages, nkv, 64, D, generator=g, device=dev())
        mu = 2 * torch.rand(n_layers, 1, 1, nkv, 1, D, generator=g, device=dev()) - 1
        cache[:, 1] = mu[:, 0] + torch.sign(mu[:, 0]) + 0.5 * cache[:, 1]        # V: per-dimension mean of magnitude 1..2
        u = torch.randn(n, nkv, D, generator=g, device=dev())
        u = u / u.norm(dim=-1, keepdim=True) * math.sqrt(D)
        # planted keys: (seq, kvh, token, V dimension that carries +-AMP or -1)
        rows = []
        for i, c in enumerate(ctx):
            for h in range(nkv):
                used = set()
                for kk, (cb, ce) in enumerate(self.pieces[(i, h)]):
                    t = int(rng.integers(cb * 64, min(ce * 64, c)))
                    used.add(t)
                    rows.append((i, h, t, kk % D, 1.0 if (kk // D) % 2 == 0 else -1.0))
                for t in {int(rng.integers(0, min(64, c))), c // 2, c - 1} - used:
                    rows.append((i, h, t, -1, 0.0))
        pl = np.array(rows, np.float64)
        seq_, kvh_, tok_ = pl[:, 0].astype(np.int64), pl[:, 1].astype(np.int64), pl[:, 2].astype(np.int64)
        page = torch.from_numpy(self.bt.numpy()[seq_, tok_ // 64].astype(np.int64)).to(dev())
        off = torch.from_numpy(tok_ % 64).to(dev())
        kv_h = torch.from_numpy(kvh_).to(dev())
        cache[:, 0, page, kv_h, off] = u[torch.from_numpy(seq_).to(dev()), kv_h]
        cache[:, 1, page, kv_h, off] += 2 * torch.randn(n_layers, len(rows), D, generator=g, device=dev())
        amp = torch.zeros(len(rows), D, device=dev())
        has = pl[:, 3] >= 0
        amp[torch.from_numpy(np.nonzero(has)[0]).to(dev()), torch.from_numpy(pl[has, 3].astype(np.int64)).to(dev())] = \
            torch.from_numpy(AMP * pl[has, 4]).float().to(dev())
        cache[:, 1, page, kv_h, off] += amp
        self.kv = cache.to(torch.bfloat16).contiguous()
        grp = nh // nkv
        qs = []
        for i, ql in enumerate(q_lens):
            if flat:
                qs.append(2.0 * torch.randn(ql, nh, D, generator=g, device=dev()))
            else:
                base = u[i].repeat_interleave(grp, dim=0)      # [nh, D]
                beta = 16.0 / math.sqrt(D)                     # planted score ~16 nats above the background's spread of ~beta
                qs.append(beta * (base[None] + 0.25 * torch.randn(ql, nh, D, generator=g, device=dev())))
        self.q = torch.cat(qs, 0).to(torch.bfloat16).contiguous()

    def run(self, L, layer=0, counters=None, n_ctas_target=0, force_splits=0):
        """oa_k_paged_attention_ex on this cache: decode when every q_len is 1, else causal prefill"""
        T = self.q.shape[0]
        out = torch.full((T, self.nh, self.D), float("nan"), dtype=torch.bfloat16, device=dev())
        ctx_a = np.array(self.ctx, np.int32); ql = np.array(self.q_lens, np.int32); bt = np.ascontiguousarray(self.bt.numpy())
        rc = L.oa_k_paged_attention_ex(ptr(self.q), ptr(out), ptr(self.kv), self.num_pages, self.n_layers, layer, bt.ctypes.data, self.maxp,
                                       ctx_a.ctypes.data, ql.ctypes.data, len(self.ctx), self.nh, self.nkv, self.D, force_splits, n_ctas_target,
                                       ptr(counters), None)
        assert rc == 0
        return out

    def _seq(self, layer, i):
        c, D = self.ctx[i], self.D
        pages = self.bt[i, : (c + 63) // 64].to(dev()).long()
        Kc = self.kv[layer, 0, pages].permute(0, 2, 1, 3).reshape(-1, self.nkv, D)[:c].double()
        Vc = self.kv[layer, 1, pages].permute(0, 2, 1, 3).reshape(-1, self.nkv, D)[:c].double()
        return Kc, Vc

    def _probs(self, qi, Kc, h, c, ql, rows=None):
        """unnormalised fp64 probabilities of head h for the query rows `rows` (default: all) of a sequence"""
        D, grp = self.D, self.nh // self.nkv
        r = torch.arange(ql, device=dev()) if rows is None else rows
        sc = (qi[r, h] @ Kc[:, h // grp].T) / math.sqrt(D)
        qpos = (c - ql + r)[:, None]; kpos = torch.arange(c, device=dev())[None, :]
        sc = sc.masked_fill(kpos > qpos, float("-inf"))
        return torch.exp(sc - sc.max(dim=1, keepdim=True).values)

    def ref(self, layer):
        """fp64 attention of every query row, head by head -> (out, sum_k p |v| / l): the second bounds the effect of the kernels' bf16 P"""
        outs, absw, row = [], [], 0
        grp = self.nh // self.nkv
        for i, (c, ql) in enumerate(zip(self.ctx, self.q_lens)):
            Kc, Vc = self._seq(layer, i)
            qi = self.q[row:row + ql].double()
            o = torch.empty(ql, self.nh, self.D, dtype=torch.float64, device=dev()); oa = torch.empty_like(o)
            for h in range(self.nh):
                p = self._probs(qi, Kc, h, c, ql)
                l = p.sum(1, keepdim=True)
                o[:, h] = (p @ Vc[:, h // grp]) / l
                oa[:, h] = (p @ Vc[:, h // grp].abs()) / l
            outs.append(o); absw.append(oa); row += ql
        return torch.cat(outs, 0), torch.cat(absw, 0)

    def piece_power(self, layer, ref, tol, items=None):
        """For every piece of every item in `items` (default: all (seq, kvh) with two or more pieces): the reference with that piece's
        tokens dropped, and with their weight doubled (the piece's m off by one in the log2 domain), must each move some output of the
        item's heads by more than 5x the tolerance.  Checked on the last query row of every 128-row tile (the rows that see the most keys)."""
        grp, D = self.nh // self.nkv, self.D
        starts = np.cumsum([0] + self.q_lens)
        keys = items if items is not None else [k for k, v in self.pieces.items() if len(v) > 1]
        assert keys, "no item with two or more pieces"
        by_seq = {}
        for (i, h) in keys:
            by_seq.setdefault(i, []).append(h)
        for i, kvhs in by_seq.items():
            c, ql = self.ctx[i], self.q_lens[i]
            Kc, Vc = self._seq(layer, i)
            qi = self.q[starts[i]:starts[i] + ql].double()
            rows = torch.tensor(sorted({min(r, ql - 1) for r in range(127, ql + 127, 128)}), device=dev())
            for kvh in kvhs:
                pcs = self.pieces[(i, kvh)]
                idx = torch.empty(c, dtype=torch.long, device=dev())
                for kk, (cb, ce) in enumerate(pcs):
                    idx[cb * 64:min(ce * 64, c)] = kk
                best = torch.zeros(len(pcs), 2, dtype=torch.float64, device=dev())
                for h in range(kvh * grp, (kvh + 1) * grp):
                    p = self._probs(qi, Kc, h, c, ql, rows)                            # [r, c]
                    l = p.sum(1)                                                       # [r]
                    O = p @ Vc[:, kvh]                                                 # [r, D]
                    Pk = torch.zeros(len(rows), len(pcs), dtype=torch.float64, device=dev()).index_add_(1, idx, p)
                    Ok = torch.zeros(len(rows), len(pcs), D, dtype=torch.float64, device=dev()).index_add_(1, idx, p[:, :, None] * Vc[None, :, kvh])
                    base = ref[starts[i] + rows, h].double()[:, None, :]               # [r, 1, D]
                    t = tol[starts[i] + rows, h].double()[:, None, :]
                    for j, sgn in enumerate((-1.0, 1.0)):
                        alt = (O[:, None, :] + sgn * Ok) / (l[:, None] + sgn * Pk)[:, :, None]
                        ratio = ((alt - base).abs() / t).nan_to_num(0.0)
                        best[:, j] = torch.maximum(best[:, j], ratio.amax(dim=(0, 2)))
                weak = (best <= 5).any(dim=1).nonzero().flatten().tolist()
                assert not weak, f"seq {i} kv head {kvh}: pieces {weak[:8]} of {len(pcs)} move no output by 5x the tolerance " \
                                 f"(drop / double: {best[weak[0]].tolist()})"
