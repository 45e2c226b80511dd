"""The decode-step kernels one at a time (sv_op_attention_decode / _prefill, sv_op_gemv_ring, sv_op_select) against float64
references, plus engine-level regressions at decoder widths the shipped configs do not use.

Whole-model parity (logits within 2x the bf16 oracle's error, greedy ids with tolerated flips) catches a broken kernel; the
tests here are built to catch a subtly wrong one: one key dropped at a CTA boundary, a LayerNorm skipped at one width, a tie
broken the wrong way, a sampled token one CDF cell off.
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle.pipeline import OracleStarVector, OracleStarVectorV2
from starvector_b200 import _lib
from starvector_b200 import engine as E
from starvector_b200.config import ModelDims, dims_tiny, dims_tiny_v2
from starvector_b200.engine import Engine, GenerationParams
from starvector_b200.weights import synthetic_images, synthetic_state_dict

pytestmark = pytest.mark.gpu
DEV = "cuda"
D = 128
F64 = torch.float64


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn(*shape, g, scale=1.0):
    return (torch.randn(*shape, generator=g, device=DEV, dtype=torch.float32) * scale).to(torch.bfloat16)


def _r(x):                      # a bf16 rounding point of the kernel, applied to an fp64 reference value
    return x.to(torch.bfloat16).to(F64)


def _ulp(x):                    # bf16 ulp of |x| (x in fp64)
    return torch.exp2(torch.floor(torch.log2(x.abs().clamp_min(1e-30))) - 7)


# ------------------------------------------------------------------------------------------------------------------------
# Decode attention
# ------------------------------------------------------------------------------------------------------------------------
KDEC_WARPS = 8        # warps per CTA of attention_decode_cluster_kernel
NKEYS = [1, 2, 31, 32, 33, 255, 256, 257, 2047, 2049, 4097]
SPLITS = [1, 2, 7, 128]


def _window_lengths(window):
    """Lengths where the window's first key falls inside a 32-key block (key_lo % 32 != 0)."""
    return [window + 1 + 5, window + 37] if window else []


def _cluster_boundaries(nkeys, key_lo, ncta):
    blk_lo, blk_hi = key_lo // 32, (nkeys + 31) // 32
    per = (blk_hi - blk_lo + ncta - 1) // ncta
    keys = set()
    for c in range(ncta):
        b0, b1 = blk_lo + c * per, min(blk_hi, blk_lo + (c + 1) * per)
        if b0 >= b1:
            continue
        keys |= {max(key_lo, b0 * 32), min(nkeys, b1 * 32) - 1}
        for w in range(KDEC_WARPS):                   # warp w of the CTA walks blocks b0 + w, b0 + w + 8, ...
            blks = list(range(b0 + w, b1, KDEC_WARPS))
            if blks:
                keys |= {max(key_lo, blks[0] * 32), min(nkeys, blks[-1] * 32 + 32) - 1}
    return keys


def _split_boundaries(nkeys, key_lo, nsplit):
    blk_lo = key_lo // 32
    blocks = (nkeys + 31) // 32 - blk_lo
    per = (blocks + nsplit - 1) // nsplit
    keys = set()
    for s in range(nsplit):
        k0, k1 = max(key_lo, (blk_lo + s * per) * 32), min(nkeys, (blk_lo + (s + 1) * per) * 32)
        if k0 < k1:
            keys |= {k0, k1 - 1}
    return keys


def _decode_case(B, n_head, n_kv, tcap, nkeys, window, spikes, seed):
    """q / K / V^T for one decode token per row.  Head r of a group reads only dims [8r, 8r+8) of the keys, so a "spike" key
    can be made to dominate one head alone: spikes[(b, head)] = key gets score ln(#valid keys) for that head (about half of its
    softmax mass), so dropping or double-counting it is an O(1) error.  Cache positions outside [key_lo, nkeys) hold large
    finite garbage whose score would dominate every head of the group."""
    g = _gen(seed)
    grp = n_head // n_kv
    key_lo = max(0, nkeys - window) if window else 0
    nvalid = nkeys - key_lo
    mag = torch.rand(B, n_kv, grp, 8, generator=g, device=DEV) + 0.5
    sgn = torch.randint(0, 2, (B, n_kv, grp, 8), generator=g, device=DEV) * 2 - 1
    qd = (mag * sgn).to(torch.bfloat16).float()                                   # [B, n_kv, grp, 8]
    q = torch.zeros(B, n_kv, grp, D, device=DEV)
    for r in range(grp):
        q[:, :, r, 8 * r: 8 * r + 8] = qd[:, :, r]
    K = torch.randn(B, n_kv, tcap, D, generator=g, device=DEV)
    V = torch.randn(B, n_kv, tcap, D, generator=g, device=DEV) * 0.5
    garbage = torch.ones(tcap, dtype=torch.bool, device=DEV)
    garbage[key_lo:nkeys] = False
    gk = torch.randn(B, n_kv, D, generator=g, device=DEV)
    for r in range(grp):
        gk[:, :, 8 * r: 8 * r + 8] = 16.0 * qd[:, :, r].sign()
    K[:, :, garbage] = gk[:, :, None, :]
    V[:, :, garbage] = 64.0 * torch.sign(torch.randn(B, n_kv, int(garbage.sum()), D, generator=g, device=DEV))
    for (b, h), key in spikes.items():
        kv, r = divmod(h, grp)
        alpha = math.log(max(nvalid, 2)) * math.sqrt(D) / float((qd[b, kv, r] ** 2).sum())
        K[b, kv, key, 8 * r: 8 * r + 8] = alpha * qd[b, kv, r]
        V[b, kv, key] = 4.0 * torch.sign(torch.randn(D, generator=g, device=DEV))
    qb = q.reshape(B, n_head * D).to(torch.bfloat16).contiguous()
    Kb = K.to(torch.bfloat16).contiguous()
    Vtb = V.to(torch.bfloat16).transpose(2, 3).contiguous()
    return qb, Kb, Vtb, key_lo


def _decode_ref(qb, Kb, Vtb, n_kv, key_lo, nkeys, drop=None):
    """Masked fp64 softmax attention; `drop` = {(b, head): key} removes those keys (the power check).  Returns the output
    [B, n_head*D] and the per-element bound sum_k p_k |v_k| used by the tolerance."""
    B = qb.shape[0]
    n_head = qb.shape[1] // D
    grp = n_head // n_kv
    q = qb.to(F64).view(B, n_kv, grp, D)
    k = Kb.to(F64)[:, :, key_lo:nkeys]
    v = Vtb.to(F64).transpose(2, 3)[:, :, key_lo:nkeys]
    s = torch.einsum("bkgd,bktd->bkgt", q, k) / math.sqrt(D)
    if drop:
        for (b, h), key in drop.items():
            s[b, h // grp, h % grp, key - key_lo] = -math.inf
    p = torch.softmax(s, dim=-1)
    out = torch.einsum("bkgt,bktd->bkgd", p, v).reshape(B, n_head * D)
    mag = torch.einsum("bkgt,bktd->bkgd", p, v.abs()).reshape(B, n_head * D)
    return out, mag


def _attn_tol(ref, mag):
    # P is rounded to bf16 before the P.V MMA (<= 2^-9 of each term) and the output to bf16 (<= 2^-9 of |out|)
    return 2.0 ** -8 * (ref.abs() + mag) + 1e-6


@pytest.mark.parametrize("window", [0, 24, 512, 4096])
@pytest.mark.parametrize("group", [1, 2, 9, 16])
def test_attention_decode_boundaries(group, window):
    """Both implementations (cluster at every forced size 1..8, split+merge at several split counts and the engine's own
    choice) at lengths around block, CTA and window edges, with a spike on every boundary key of every configuration."""
    n_kv = {1: 16, 2: 8, 9: 2, 16: 1}[group]             # 16 MQA-like heads; 8 kv heads of 2 (tiny-v2); 2 of 9 (8B-like); MQA
    n_head = group * n_kv
    lengths = NKEYS + _window_lengths(window)
    for i, nkeys in enumerate(lengths):
        B = (1, 3, 8)[i % 3]
        tcap = (nkeys + 31) // 32 * 32 + 32
        key_lo = max(0, nkeys - window) if window else 0
        configs = [(_lib.SV_ATTN_DECODE_CLUSTER, c) for c in range(1, 9)] + \
                  [(_lib.SV_ATTN_DECODE_SPLIT, s) for s in SPLITS + [0]]
        keys = {0, key_lo, nkeys - 1}
        for c in range(1, 9):
            keys |= _cluster_boundaries(nkeys, key_lo, c)
        for s in SPLITS + [max(1, min(128, (nkeys + 31) // 32))]:
            keys |= _split_boundaries(nkeys, key_lo, s)
        keys = sorted(k for k in keys if key_lo <= k < nkeys)
        slots = [(b, h) for b in range(B) for h in range(n_head)]
        for rnd in range(0, len(keys), len(slots)):
            chunk = keys[rnd: rnd + len(slots)]
            spikes = {slots[j]: key for j, key in enumerate(chunk)}
            qb, Kb, Vtb, _ = _decode_case(B, n_head, n_kv, tcap, nkeys, window, spikes, seed=1000 * i + rnd)
            ref, mag = _decode_ref(qb, Kb, Vtb, n_kv, key_lo, nkeys)
            tol = _attn_tol(ref, mag)
            if nkeys - key_lo > 1:                       # the test's power: every spike moves its head's output by >> tol
                nospike, _ = _decode_ref(qb, Kb, Vtb, n_kv, key_lo, nkeys, drop=spikes)
                for (b, h) in spikes:
                    sl = slice(h * D, h * D + D)
                    gap = ((nospike[b, sl] - ref[b, sl]).abs() / tol[b, sl]).max().item()
                    assert gap > 10, (nkeys, window, b, h, spikes[(b, h)], gap)
            for impl, parts in configs:
                out = E.op_attention_decode(qb, Kb, Vtb, nkeys, window, impl, parts).to(F64)
                bad = (out - ref).abs() > tol
                if bool(bad.any()):
                    b, col = [int(x) for x in bad.nonzero()[0]]
                    raise AssertionError(
                        f"impl {impl} parts {parts} nkeys {nkeys} window {window} group {group} B {B}: {int(bad.sum())} "
                        f"elements off, first row {b} head {col // D} (spike key {spikes.get((b, col // D))}), "
                        f"err {(out - ref).abs().max().item():.4f}")


def test_attention_decode_rejects_bad_arguments():
    q = torch.zeros(1, 2 * D, dtype=torch.bfloat16, device=DEV)
    kc = torch.zeros(1, 1, 64, D, dtype=torch.bfloat16, device=DEV)
    vt = torch.zeros(1, 1, D, 64, dtype=torch.bfloat16, device=DEV)
    for kw in (dict(nkeys=65), dict(nkeys=0), dict(nparts=9), dict(window=-1)):
        args = dict(nkeys=10, window=0, impl=_lib.SV_ATTN_DECODE_CLUSTER, nparts=0) | kw
        with pytest.raises(ValueError):
            E.op_attention_decode(q, kc, vt, **args)
    with pytest.raises(ValueError):
        E.op_attention_decode(q, kc, vt, 10, 0, _lib.SV_ATTN_DECODE_SPLIT, 129)
    with pytest.raises(ValueError):                      # group 17
        E.op_attention_decode(torch.zeros(1, 17 * D, dtype=torch.bfloat16, device=DEV), kc, vt, 10)
    with pytest.raises(ValueError):                      # 9 rows
        E.op_attention_decode(q.expand(9, -1).contiguous(), kc.expand(9, -1, -1, -1).contiguous(),
                              vt.expand(9, -1, -1, -1).contiguous(), 10)


# ------------------------------------------------------------------------------------------------------------------------
# Prefill attention with GQA and a sliding window
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("window", [0, 24, 257])
@pytest.mark.parametrize("group,n_kv", [(1, 4), (2, 4), (9, 2), (16, 1)])
def test_attention_prefill_gqa_window(group, n_kv, window):
    n_head = group * n_kv
    for B, T in ((1, 259), (2, 300)):
        g = _gen(7 + T)
        qkv = _randn(B * T, (n_head + 2 * n_kv) * D, g=g)
        out = E.op_attention_prefill(qkv, B, T, n_head, n_kv, window).to(F64).view(B, T, n_head, D)
        x = qkv.to(F64).view(B, T, -1)
        q = x[..., : n_head * D].view(B, T, n_kv, group, D)
        k = x[..., n_head * D: (n_head + n_kv) * D].view(B, T, n_kv, D)
        v = x[..., (n_head + n_kv) * D:].view(B, T, n_kv, D)
        s = torch.einsum("bqkgd,btkd->bkgqt", q, k) / math.sqrt(D)
        i, j = torch.arange(T, device=DEV)[:, None], torch.arange(T, device=DEV)[None, :]
        allowed = (j <= i) & ((j > i - window) if window else True)
        p = torch.softmax(s.masked_fill(~allowed, -math.inf), dim=-1)
        ref = torch.einsum("bkgqt,btkd->bqkgd", p, v).reshape(B, T, n_head, D)
        mag = torch.einsum("bkgqt,btkd->bqkgd", p, v.abs()).reshape(B, T, n_head, D)
        bad = (out - ref).abs() > _attn_tol(ref, mag)
        assert not bool(bad.any()), (B, T, int(bad.sum()), (out - ref).abs().max().item(), bad.nonzero()[:3].tolist())


# ------------------------------------------------------------------------------------------------------------------------
# Ring GEMV
# ------------------------------------------------------------------------------------------------------------------------
GEMV_K = [32, 96, 384, 640, 1280, 1536, 2048, 2304, 4608, 8192]
GEMV_N = [1, 147, 148, 149, 2368, 2369, 5632, 20000, 49157]
ACTS = [_lib.SV_ACT_NONE, _lib.SV_ACT_QUICKGELU, _lib.SV_ACT_GELU_TANH, _lib.SV_ACT_SILU]


def _ln_ref(x, w, b, eps=1e-5):
    # the LN output is a bf16 tensor, computed in fp32 as torch's bf16 LayerNorm does (an fp64 LN would flip the rounding of
    # a few elements per row, and their sum over K reaches an ulp of the small outputs)
    y = torch.nn.functional.layer_norm(x.float(), (x.shape[-1],), w.float(), b.float(), eps)
    return y.to(torch.bfloat16).to(F64)


def _gemv_epilogue(y, act, res):
    """The bf16 epilogue chain from the rounded GEMV value y: activation, then residual.  Also returns |value before the
    residual| (where a later cancellation keeps the ulp of a flip)."""
    if act == _lib.SV_ACT_QUICKGELU:
        y = _r(y * _r(torch.sigmoid(_r(1.702 * y))))
    elif act == _lib.SV_ACT_SILU:
        y = _r(y * _r(torch.sigmoid(y)))
    elif act == _lib.SV_ACT_GELU_TANH:
        y = _r(torch.nn.functional.gelu(y, approximate="tanh"))
    before_res = y.abs()
    if res is not None:
        y = _r(y + res.to(F64))
    return y, before_res


def _gemv_ref(x, w, bias, res, ln, act):
    """Returns the reference [B,N], the epilogue applied to the two bf16 neighbours of the rounded GEMV value [2,B,N], and
    the magnitude the ulp of the check is taken at."""
    xn = _ln_ref(x, *ln) if ln is not None else x.to(F64)
    acc = xn @ w.to(F64).t() + (bias.to(F64) if bias is not None else 0.0)
    floor = 2.0 ** -10 * (xn.abs() @ w.to(F64).abs().t())                         # sum |x_k w_k| per output
    pre = _r(acc)
    ref, before_res = _gemv_epilogue(pre, act, res)
    step = _ulp(torch.maximum(pre.abs(), floor))
    # a neighbour one step away, or half a step where pre sits on a binade edge; _r snaps both onto the bf16 grid
    nbr = torch.stack([_gemv_epilogue(_r(pre + k * step), act, res)[0] for k in (-1.0, -0.5, 0.5, 1.0)])
    return ref, nbr, torch.maximum(torch.maximum(ref.abs(), before_res), floor)


def _gemv_check(got, want, what):
    """At most 1 bf16 ulp from the rounded fp64 reference and >= 98 % bit-equal.
    The kernel sums in fp32: where the exact sum lies next to a bf16 rounding midpoint, its first rounding point (the
    GEMV + bias value) may land on the neighbouring bf16 value, which the activation and residual then carry forward.  So an
    output also passes within 1 ulp of the epilogue applied to that neighbour.  The ulp is taken at the largest magnitude on
    the way after that point (the value before the residual, whose rounding a cancellation keeps), and at least at
    2^-10 * sum|x w| (an output that cancels to near zero carries the fp32 accumulation error of its terms)."""
    ref, nbr, mag = want
    got = got.to(F64)
    tol = _ulp(mag)
    err = (got - ref).abs()
    err_nbr = (got[None] - nbr).abs().amin(0)
    bad = (err > tol) & (err_nbr > tol)
    if bool(bad.any()):
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} beyond 1 ulp, max err {err.max().item():.5f}, first at "
                             f"{list(i)}: got {got[i].item():.6g} ref {ref[i].item():.6g} tol {tol[i].item():.3g}")
    eq = (got == ref).double().mean().item()
    assert eq >= 0.98, f"{what}: only {eq:.4f} bit-equal"


@pytest.mark.parametrize("K", GEMV_K)
def test_gemv_ring_shapes(K):
    """Every N of the sweep at this K: LayerNorm + bias + activation + separate residual, and no LayerNorm with the residual
    in place (y aliasing it); each also from slab-tiled weights, which must give bit-identical y."""
    for i, N in enumerate(GEMV_N):
        B = (1, 5, 8)[(i + K // 32) % 3]
        act = ACTS[i % 4]
        g = _gen(K * 100003 + N)
        x = _randn(B, K, g=g)
        w = _randn(N, K, g=g, scale=1.0 / math.sqrt(K))
        bias = _randn(N, g=g, scale=0.2)
        res = _randn(B, N, g=g)
        ln = (_randn(K, g=g, scale=0.3) + 1.0, _randn(K, g=g, scale=0.2))
        what = f"K {K} N {N} B {B} act {act}"
        y = E.op_gemv_ring(x, w, bias, res, ln, act)
        _gemv_check(y, _gemv_ref(x, w, bias, res, ln, act), what + " LayerNorm")
        yt = E.op_gemv_ring(x, w, bias, res, ln, act, tiled=True)
        assert torch.equal(y, yt), what + ": tiled weights give other bits (LayerNorm)"
        buf = res.clone()
        E.op_gemv_ring(x, w, None, buf, None, _lib.SV_ACT_NONE, out=buf)
        _gemv_check(buf, _gemv_ref(x, w, None, res, None, _lib.SV_ACT_NONE), what + " in-place residual")
        buf_t = res.clone()
        E.op_gemv_ring(x, w, None, buf_t, None, _lib.SV_ACT_NONE, out=buf_t, tiled=True)
        assert torch.equal(buf, buf_t), what + ": tiled weights give other bits (in-place residual)"


@pytest.mark.parametrize("K,n_head,n_kv", [(640, 5, 1), (512, 4, 2), (2048, 16, 1), (2304, 18, 2), (384, 3, 1)])
def test_gemv_ring_qkv_appends_exactly_one_cache_position(K, n_head, n_kv):
    N = (n_head + 2 * n_kv) * D
    B, tcap = 3, 96
    g = _gen(K + n_head)
    x = _randn(B, K, g=g)
    w = _randn(N, K, g=g, scale=1.0 / math.sqrt(K))
    bias = _randn(N, g=g, scale=0.2)
    ln = (_randn(K, g=g, scale=0.3) + 1.0, _randn(K, g=g, scale=0.2))
    want = _gemv_ref(x, w, bias, None, ln, 0)
    for pos in (0, 37, tcap - 1):
        kc = _randn(B, n_kv, tcap, D, g=g, scale=100.0)          # sentinel fill
        vt = _randn(B, n_kv, D, tcap, g=g, scale=100.0)
        k0, v0 = kc.clone(), vt.clone()
        y = E.op_gemv_ring(x, w, bias, None, ln, 0, epi=_lib.SV_GEMV_EPI_QKV, kcache=kc, vtcache=vt, n_head=n_head, pos=pos)
        _gemv_check(y, want, f"QKV K {K} pos {pos}")
        kcols = y[:, n_head * D: (n_head + n_kv) * D].view(B, n_kv, D)
        vcols = y[:, (n_head + n_kv) * D:].view(B, n_kv, D)
        k0[:, :, pos, :] = kcols
        v0[:, :, :, pos] = vcols
        assert torch.equal(kc, k0), f"K cache differs from sentinel + row {pos}"
        assert torch.equal(vt, v0), f"V^T cache differs from sentinel + column {pos}"


@pytest.mark.parametrize("K,N", [(256, 500), (640, 2369), (2048, 49157), (4608, 20000)])
def test_gemv_ring_lmhead_partials_first_max(K, N):
    """Per-tile argmax partials reduce to the FIRST maximum of the bf16-rounded row: exact twins (equal rows of W) and
    near-twins (rows one bf16 ulp apart in one weight, equal after rounding) are placed as the row maximum, the later index
    of a near-twin pair being the larger before rounding."""
    B = 4
    g = _gen(K + N)
    x = _randn(B, K, g=g)
    w = _randn(N, K, g=g, scale=1.0 / math.sqrt(K))
    ln = (_randn(K, g=g, scale=0.3) + 1.0, _randn(K, g=g, scale=0.2))
    xn = _ln_ref(x, *ln)
    top = (xn[0] / xn[0].norm() * 4.0).to(torch.bfloat16)
    a, b, c, d = 3, N // 2 + 1, N // 3, N - 2                    # twins (a, b) for row 0; near-twins (c < d) for row 1
    w[a] = top
    w[b] = top
    top1 = (xn[1] / xn[1].norm() * 4.0).to(torch.bfloat16)
    w[c] = top1
    j = int(xn[1].abs().argmin())                                 # nudge the weight of the smallest activation by 1 ulp
    w[d] = top1
    w[d, j] = (top1[j].float() + torch.sign(xn[1, j]).float() * _ulp(top1[j].to(F64)).float()).to(torch.bfloat16)
    y, aval, aidx = E.op_gemv_ring(x, w, None, None, ln, 0, epi=_lib.SV_GEMV_EPI_LMHEAD)
    assert aval.shape[0] * 16 >= N and aval.shape[0] <= N
    yf = y.float().cpu().numpy()
    v = aval[:, :B].cpu().numpy()
    ix = aidx[:, :B].cpu().numpy()
    for r in range(B):
        best = v[:, r].max()
        idx = ix[v[:, r] == best, r].min()
        first = int(np.argmax(yf[r]))                             # numpy: the first maximal index
        assert idx == first, (r, idx, first, yf[r, idx], yf[r, first])
        assert best == yf[r, first]
    assert int(np.argmax(yf[0])) == a, "twin rows of the maximum: the lower index must win"
    assert yf[1, c] == yf[1, d] and int(np.argmax(yf[1])) == c, "near-twins equal after rounding: the lower index must win"
    # the fused select kernel reduces the same partials to the same token and writes its embedding
    wte = _randn(N, K, g=g)
    seen = torch.zeros(B, N, dtype=torch.uint8, device=DEV)
    p = GenerationParams(max_new_tokens=8, eos_token_id=None)
    tok, _ = E.op_select(_lib.SV_SELECT_FUSED_PARTIALS, y, seen, p, partials=(aval, aidx), wte=wte)
    assert tok.cpu().tolist() == [int(np.argmax(yf[r])) for r in range(B)]


def test_gemv_ring_rejects_bad_arguments():
    x = torch.zeros(9, 64, dtype=torch.bfloat16, device=DEV)
    w = torch.zeros(16, 64, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(ValueError):
        E.op_gemv_ring(x, w)                                       # 9 rows
    with pytest.raises(ValueError):
        E.op_gemv_ring(x[:2, :48].contiguous(), w[:, :48].contiguous())       # K % 32
    kc = torch.zeros(1, 1, 32, D, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(ValueError):                                # pos >= tcap
        E.op_gemv_ring(torch.zeros(1, 64, dtype=torch.bfloat16, device=DEV), torch.zeros(3 * D, 64, dtype=torch.bfloat16, device=DEV),
                       epi=_lib.SV_GEMV_EPI_QKV, kcache=kc, vtcache=kc.transpose(2, 3).contiguous(), n_head=1, pos=32)


# ------------------------------------------------------------------------------------------------------------------------
# Token selection
# ------------------------------------------------------------------------------------------------------------------------
def test_select_greedy_penalty_and_ties():
    """Greedy over penalised logits (HF RepetitionPenaltyLogitsProcessor in fp32) with ties: all three kernels pick the
    first maximum; the fused kernel's embedding row is wte[tok] + wpe[cur_len + 1] with one bf16 rounding."""
    B, V, H = 8, 49157, 256
    g = _gen(5)
    logits = _randn(B, V, g=g, scale=2.0).clamp(max=1.9)
    seen = (torch.rand(B, V, generator=g, device=DEV) < 0.3).to(torch.uint8)
    for b in range(B):                 # even rows: a seen 4.0 (penalised to 2.0 at rp 2) ties an unseen 2.0 later in the row;
        lo, hi = 100 + 7 * b, 30000 + 11 * b           # odd rows: two unseen 2.0; both beat the rest of the row
        logits[b, lo], seen[b, lo] = (4.0, 1) if b % 2 == 0 else (2.0, 0)
        logits[b, hi], seen[b, hi] = 2.0, 0
    wte = _randn(V, H, g=g)
    wpe = _randn(64, H, g=g)
    for rp in (2.0, 1.3):
        v = logits.float().cpu().numpy().copy()
        s = seen.bool().cpu().numpy()
        v = np.where(s, np.where(v < 0, v * np.float32(rp), v / np.float32(rp)), v).astype(np.float32)
        want = [int(np.argmax(v[b])) for b in range(B)]
        if rp == 2.0:
            assert want == [100 + 7 * b for b in range(B)]
        p = GenerationParams(max_new_tokens=8, eos_token_id=None, repetition_penalty=rp)
        got = E.op_select(_lib.SV_SELECT_GREEDY, logits, seen, p, step=3, cur_len=20)
        assert got.cpu().tolist() == want, rp
        for cur_len in (20, 63):
            tok, x = E.op_select(_lib.SV_SELECT_FUSED, logits, seen, p, step=3, cur_len=cur_len, wte=wte, wpe=wpe)
            assert tok.cpu().tolist() == want, rp
            pos = min(cur_len + 1, 63)
            emb = (wte[tok.long()].float() + wpe[pos].float()).to(torch.bfloat16)
            assert torch.equal(x, emb)


def _philox_uniform(seed, c0, c1):
    """Philox4x32-10 of the sampling kernel (counter (row, step, 0x5356, 0x42323030)), vectorised over c0 / c1."""
    M = np.uint64(0xFFFFFFFF)
    k0 = np.uint64(seed & 0xFFFFFFFF)
    k1 = np.uint64((seed >> 32) & 0xFFFFFFFF)
    x0 = np.asarray(c0, dtype=np.uint64)
    x1 = np.asarray(c1, dtype=np.uint64)
    x2 = np.full_like(x0, 0x5356)
    x3 = np.full_like(x0, 0x42323030)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * x0
        p1 = np.uint64(0xCD9E8D57) * x2
        hi0, lo0 = p0 >> np.uint64(32), p0 & M
        hi1, lo1 = p1 >> np.uint64(32), p1 & M
        x0, x1, x2, x3 = hi1 ^ x1 ^ k0, lo1, hi0 ^ x3 ^ k1, lo0
        k0 = (k0 + np.uint64(0x9E3779B9)) & M
        k1 = (k1 + np.uint64(0xBB67AE85)) & M
    return ((x0 >> np.uint64(8)).astype(np.float64) + 0.5) / 16777216.0


def _sample_ref(logits_row, seen_row, rp, temp, top_p, u):
    """HF's filtered distribution in fp64 (repetition penalty -> temperature -> top-p, a token kept iff the mass of strictly
    more probable tokens is < top_p) and the id-order inverse CDF at u * kept_mass.  Returns (token, ambiguous)."""
    v = logits_row.astype(np.float64)
    v = np.where(seen_row, np.where(v < 0, v * rp, v / rp), v) / temp
    p = np.exp(v - v.max())
    p /= p.sum()
    order = np.argsort(-p, kind="stable")
    ps = p[order]
    above = np.concatenate([[0.0], np.cumsum(ps)[:-1]])
    # mass strictly above each token (ties share the mass above the whole tie group)
    first = np.searchsorted(-ps, -ps, side="left")
    above = above[first]
    keep = np.zeros_like(p, dtype=bool)
    keep[order] = above < top_p if top_p < 1.0 else True
    near_nucleus = top_p < 1.0 and bool(np.any(np.abs(above - top_p) <= 1e-4))
    q = np.where(keep, p, 0.0)
    cdf = np.cumsum(q)
    mass = cdf[-1]
    t = u * mass
    tok = int(np.searchsorted(cdf, t, side="right"))
    tok = min(tok, len(p) - 1)
    while not keep[tok]:
        tok -= 1
    lo = cdf[tok] - q[tok]                                   # the chosen cell is [lo, cdf[tok])
    near_cdf = min(abs(t - lo), abs(cdf[tok] - t)) <= 1e-4 * mass
    return tok, near_nucleus or near_cdf


def _sampling_rows(V, g):
    """8 rows: peaked, flat over 20 ids, a tie group after a dominant id, penalised, and generic ones (a spread of 4 keeps
    the draws whose CDF cell is narrower than the 1e-4 ambiguity band rare)."""
    rows = torch.randn(8, V, generator=g, device=DEV) * 6.0
    rows[0, 17] = 60.0                                      # peaked
    rows[1] = -30.0
    rows[1, 40:60] = 1.0                                    # flat over 20 ids
    rows[2] = -30.0
    rows[2, 5] = 3.0
    rows[2, 100:110] = 1.5                                  # tied group after a dominant id
    rows[3, :50] += 6.0                                     # penalised ids are the likely ones
    return rows.to(torch.bfloat16)


@pytest.mark.parametrize("top_p,temp", [(1.0, 1.0), (0.9, 0.7)])
def test_select_sample_replays_philox_exactly(top_p, temp):
    B, V, steps, seed = 8, 500, 400, 0x1234_5678_9ABC
    g = _gen(11)
    logits = _sampling_rows(V, g)
    seen = torch.zeros(B, V, dtype=torch.uint8, device=DEV)
    seen[3, :50] = 1
    seen[5, ::3] = 1
    rp = 1.3
    p = GenerationParams(max_new_tokens=steps + 1, do_sample=True, temperature=temp, top_p=top_p, repetition_penalty=rp,
                         eos_token_id=None, seed=seed)
    lg = logits.float().cpu().numpy()
    sn = seen.bool().cpu().numpy()
    got = np.stack([E.op_select(_lib.SV_SELECT_SAMPLE, logits, seen, p, step=s, cur_len=30).cpu().numpy()
                    for s in range(steps)])                              # [steps, B]
    u = _philox_uniform(seed, np.arange(B)[None, :].repeat(steps, 0), np.arange(steps)[:, None].repeat(B, 1))
    n_amb = 0
    wrong = []
    for s in range(steps):
        for b in range(B):
            tok, amb = _sample_ref(lg[b], sn[b], rp, temp, top_p, u[s, b])
            n_amb += amb
            if got[s, b] != tok and not amb:
                wrong.append((s, b, int(got[s, b]), tok))
    # exceptions: the replayed target lies within 1e-4 (relative to the kept mass) of its cell's edge, or a token's mass-above
    # lies within 1e-4 of top_p; the kernel accumulates in fp32 (~1e-5 relative over 500 ids), so only those may differ
    assert not wrong, f"{len(wrong)} draws differ from the replay, e.g. (step, row, kernel, ref) {wrong[:5]}"
    assert n_amb < 0.01 * steps * B, f"{n_amb} ambiguous draws"
    assert len(set(got[:, 1].tolist())) > 10, "the flat row must spread its draws"


# ------------------------------------------------------------------------------------------------------------------------
# Engine-level regressions at widths the shipped configs do not use
# ------------------------------------------------------------------------------------------------------------------------
def _err(a, ref):
    d = (a.float().cpu() - ref.float().cpu()).abs()
    return d.max().item(), d.mean().item()


def _as_accurate_as_bf16(engine_out, oracle_bf16, oracle_fp32, slack=2.0, floor=3e-2):
    e_max, e_mean = _err(engine_out, oracle_fp32)
    o_max, o_mean = _err(oracle_bf16, oracle_fp32)
    assert e_max <= slack * o_max + floor, f"max err {e_max:.4f} vs bf16-oracle {o_max:.4f}"
    assert e_mean <= slack * o_mean + floor / 10, f"mean err {e_mean:.5f} vs bf16-oracle {o_mean:.5f}"


def _engine(d, sd, **env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        e = Engine(d, 0)
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
    e.load_state_dict(sd)
    return e


def _teacher_forced(e, img, prompt, forced):
    e.encode_images(img)
    out = [e.prefill(torch.tensor([prompt] * img.shape[0]), return_logits=True)]
    for j in range(forced.shape[1]):
        out.append(e.decode_step(forced[:, j]))
    return torch.stack(out, dim=1)


@pytest.mark.parametrize("hidden,n_head", [(640, 5), (384, 3)])
def test_v1_narrow_width_slab_layernorm(hidden, n_head):
    """Hidden widths whose ring-GEMV plan has more than two slabs (640 = 5 x 128, 384 = 3 x 128): teacher-forced logits
    against the oracle, and the graph, legacy and (where accepted) dataflow decode modes agree token for token."""
    d = dims_tiny(hidden=hidden, n_head=n_head, n_inner=4 * hidden)
    sd = synthetic_state_dict(d, seed=0, init="randomized")
    img = synthetic_images(d, 2, seed=1)
    prompt = [44, 78]
    forced = torch.randint(5, d.vocab - 5, (2, 12), generator=torch.Generator().manual_seed(3))
    o16 = OracleStarVector(d, sd, dtype=torch.bfloat16, eos_token_id=None, pad_token_id=d.vocab - 4)
    o32 = OracleStarVector(d, sd, dtype=torch.float32, eos_token_id=None, pad_token_id=d.vocab - 4)
    ref16 = o16.teacher_forced_logits(img, prompt, forced)
    ref32 = o32.teacher_forced_logits(img.float(), prompt, forced)
    outs = {}
    for name, env in (("graph", {}), ("legacy", {"SV_DECODE": "legacy"}), ("flow", {"SV_FLOW": "1"})):
        e = _engine(d, sd, **env)
        if name == "graph":
            assert "ring-gemv-graph" in e.describe(), e.describe()
        if name == "flow" and "dataflow" not in e.describe():
            e.close()
            continue
        got = _teacher_forced(e, img, prompt, forced)
        _as_accurate_as_bf16(got, ref16, ref32)
        e.encode_images(img)
        e.prefill(torch.tensor([prompt] * 2))
        outs[name] = e.generate(GenerationParams(max_new_tokens=16, eos_token_id=None, pad_token_id=d.vocab - 4)).cpu()
        e.close()
    for k in outs:
        assert torch.equal(outs[k], outs["graph"]), (k, outs[k].tolist(), outs["graph"].tolist())


def _v2_fused_case(d, seed, n_forced):
    sd = synthetic_state_dict(d, seed=seed, init="randomized")
    img = synthetic_images(d, 2, seed=seed + 1)
    prompt = [44, 78]
    forced = torch.randint(5, d.vocab - 5, (2, n_forced), generator=torch.Generator().manual_seed(seed + 2))
    assert d.query_length + len(prompt) + n_forced > d.sliding_window + 8           # the window is crossed
    e = _engine(d, sd, SV_DECODE="fused")
    assert "ring-gemv-graph" in e.describe(), e.describe()
    got = _teacher_forced(e, img, prompt, forced)
    e.close()
    o16 = OracleStarVectorV2(d, sd, dtype=torch.bfloat16)
    o32 = OracleStarVectorV2(d, sd, dtype=torch.float32)
    _as_accurate_as_bf16(got, o16.teacher_forced_logits(img, prompt, forced),
                         o32.teacher_forced_logits(img.float(), prompt, forced), floor=4e-2)


def test_v2_fused_decode_tiny():
    """SV_DECODE=fused on the tiny v2 model (GQA group 2, RoPE, window 24): rope_append + cluster attention + ring GEMVs."""
    _v2_fused_case(dims_tiny_v2(), seed=0, n_forced=20)


def test_v2_fused_decode_group9_wide():
    """hidden 2304, 18 heads over 2 kv heads (group 9): K > 2048, so the LN_BIGK ring GEMVs, rope_append and the group-9
    cluster attention all run."""
    _v2_fused_case(dims_tiny_v2(hidden=2304, n_head=18, n_kv_head=2, n_inner=1024), seed=4, n_forced=20)
