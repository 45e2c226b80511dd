"""Scoring path: `sv_extend` (teacher forcing over a chunk) and its lm_head with the fused log-prob epilogue
(`sv_op_lm_head_logps`), against float64 references for the kernel and against the CPU oracle for the engine.

The log-prob contract (DESIGN.md §3): logp = fp32 log_softmax(bf16 logits / temperature)[target], where the bf16 logits are
what HF's lm_head returns.  The kernel test therefore holds the log-probs to the fp64 log-softmax of the kernel's OWN bf16
logits (8 fp32 ulps of max(1, |lse|)), and the logits to 1 bf16 ulp of the fp64 product.
"""
import ctypes as C
import dataclasses
import os

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
F64 = torch.float64
PROMPT = [44, 78]


def _ulp_bf16(x):
    return torch.exp2(torch.floor(torch.log2(x.abs().clamp_min(1e-30))) - 7)


def _lp_tol(lse):                 # 8 fp32 ulps of max(1, |lse|)
    return 8 * torch.exp2(torch.floor(torch.log2(lse.abs().clamp_min(1.0))) - 23)


def _check_logps_of(logps, logits, ids, temperature):
    """logps (fp32 [R]) against the fp64 log-softmax of the given bf16-exact logits [R, N] / temperature at ids [R]."""
    z = logits.to(F64) / temperature
    lse = torch.logsumexp(z, dim=-1)
    ref = z.gather(1, ids.long().view(-1, 1)).squeeze(1) - lse
    err = (logps.to(F64) - ref).abs()
    tol = _lp_tol(lse)
    assert bool((err <= tol).all()), f"logp err {err.max().item():.3e} (tol {tol[err.argmax()].item():.3e}) at row {int(err.argmax())}"


# ------------------------------------------------------------------------------------------------------------------------
# 1. the kernel against float64
# ------------------------------------------------------------------------------------------------------------------------
def _op_case(M, N, K, seed):
    """x [M,K], w [N,K] (bf16) and targets.  Columns 0..7 of K are control channels: row 0 (M >= 3) has one huge logit,
    row 1 all logits equal, row 2 a near-tie of two logits one bf16 ulp apart; the other rows are random."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(M, K, generator=g, device=DEV) * 0.35
    w = torch.randn(N, K, generator=g, device=DEV) * 0.35
    x[:, :8] = 0
    w[:, :8] = 0
    if M >= 3:
        x[:3] = 0
        j_huge = (7 * N) // 11
        x[0, 0] = 48.0
        w[j_huge, 0] = 1.0                                  # row 0: logit j_huge = 48, every other logit 0
        x[1, 1] = 1.0
        w[:, 1] = 1.5                                       # row 1: all logits 1.5
        x[2, 2] = 1.0
        w[:, 2] = torch.rand(N, generator=g, device=DEV)
        if N >= 2:
            w[N // 3, 2] = 3.0
            w[(2 * N) // 3 if (2 * N) // 3 != N // 3 else N - 1, 2] = 3.015625   # one bf16 ulp above 3.0
    x, w = x.to(torch.bfloat16), w.to(torch.bfloat16)
    choices = [0, N - 1, min(128, N - 1), min(127, N - 1), min(255, N - 1), min(256, N - 1), (N // 128) * 128 if (N // 128) * 128 < N else 0]
    ids = torch.tensor([choices[r % len(choices)] for r in range(M)], device=DEV, dtype=torch.int32)
    rnd = torch.randint(0, N, (M,), generator=g, device=DEV, dtype=torch.int32)
    ids = torch.where(torch.arange(M, device=DEV) % 3 == 2, rnd, ids)
    return x, w, ids


@pytest.mark.parametrize("N", [1, 7, 500, 4099, 49156])
@pytest.mark.parametrize("M", [1, 127, 128, 129, 4096])
def test_lm_head_logps_vs_float64(M, N):
    K = 256 if M * N < 4096 * 4099 else 128
    x, w, ids = _op_case(M, N, K, seed=M * 7 + N)
    ref_logits = x.to(F64) @ w.to(F64).T
    # 1 bf16 ulp of the reference, and of 2^-10 where the product cancels to almost nothing (fp32 accumulation error)
    ulp = _ulp_bf16(ref_logits.to(torch.bfloat16).to(F64).abs().clamp_min(2.0 ** -10))
    for temp in (1.0, 0.7, 1.3):
        lp, lg = E.op_lm_head_logps(x, w, ids, temperature=temp, return_logits=True)
        assert lg.shape == (M, N) and lp.shape == (M,)
        assert torch.equal(lg, lg.to(torch.bfloat16).float()), "logits are not bf16-exact"
        d = (lg.to(F64) - ref_logits).abs()
        assert bool((d <= ulp).all()), f"logit off by {(d / ulp).max().item():.2f} bf16 ulp"
        _check_logps_of(lp, lg, ids, temp)
        lp2, lg2 = E.op_lm_head_logps(x, w, ids, temperature=temp, return_logits=True)
        assert torch.equal(lp, lp2) and torch.equal(lg, lg2), "not deterministic"
        assert torch.equal(E.op_lm_head_logps(x, w, ids, temperature=temp), lp), "the logits store changed the log-probs"


def test_lm_head_logps_out_of_range_ids_and_refusals():
    x, w, ids = _op_case(130, 500, 128, seed=5)
    ids[3], ids[4] = -1, 500
    lp = E.op_lm_head_logps(x, w, ids)
    assert torch.isnan(lp[3]) and torch.isnan(lp[4]) and bool(torch.isfinite(lp[5:]).all())
    for bad in (dict(temperature=0.0), dict(temperature=-1.0)):
        with pytest.raises(ValueError):
            E.op_lm_head_logps(x, w, ids, **bad)
    with pytest.raises(ValueError):
        E.op_lm_head_logps(x[:, :96].contiguous(), w[:, :96].contiguous(), ids)      # K % 64 != 0


# ------------------------------------------------------------------------------------------------------------------------
# 2./3. the engine against the oracle
# ------------------------------------------------------------------------------------------------------------------------
def _err(a, ref):
    d = (a.float().cpu() - ref.float().cpu()).abs()
    return d.max().item(), d.mean().item()


def _as_accurate_as_bf16(engine_out, oracle_bf16, oracle_fp32, slack=2.0, floor=3e-2):
    e_max, e_mean = _err(engine_out, oracle_fp32)
    o_max, o_mean = _err(oracle_bf16, oracle_fp32)
    assert e_max <= slack * o_max + floor, f"max err {e_max:.4f} vs bf16-oracle {o_max:.4f}"
    assert e_mean <= slack * o_mean + floor / 10, f"mean err {e_mean:.5f} vs bf16-oracle {o_mean:.5f}"


def _oracle_logps(tf, ids, temperature=1.0):
    """tf [B, T+1, V] teacher-forced oracle logits (position t predicts token t) -> [B, T] log-probs of ids."""
    z = torch.log_softmax(tf[:, :-1].double() / temperature, dim=-1)
    return z.gather(2, ids.long().unsqueeze(2)).squeeze(2)


@pytest.fixture(scope="module")
def tiny():
    d = dims_tiny()
    sd = synthetic_state_dict(d, seed=0, init="randomized")
    eng = Engine(d, 0)
    eng.load_state_dict(sd)
    pad = d.vocab - 4
    o16 = OracleStarVector(d, sd, dtype=torch.bfloat16, pad_token_id=pad)
    o32 = OracleStarVector(d, sd, dtype=torch.float32, pad_token_id=pad)
    img = synthetic_images(d, 4, seed=1)
    yield d, sd, eng, o16, o32, img
    eng.close()


def test_extend_v1_matches_oracle_and_splits(tiny):
    d, sd, eng, o16, o32, img = tiny
    B, T = 4, 40
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(1, d.vocab - 8, (B, T + 1), generator=g)
    forced, nxt = ids[:, :T], ids[:, T]
    eng.encode_images(img)
    lead = eng.prefill(torch.tensor([PROMPT] * B), return_logits=True)
    lg, lp = eng.extend(forced, keep_logits=T, logps=True)
    assert lg.shape == (B, T, d.vocab) and lp.shape == (B, T)
    after = eng.decode_step(nxt)                                   # a decode step continues where the chunk ended
    tf = {dt: o.teacher_forced_logits(img, PROMPT, ids) for dt, o in ((16, o16), (32, o32))}   # [B, T+2, V]
    _as_accurate_as_bf16(lg, tf[16][:, 1:T + 1], tf[32][:, 1:T + 1])
    _as_accurate_as_bf16(lp, _oracle_logps(tf[16][:, :T + 1], forced), _oracle_logps(tf[32][:, :T + 1], forced))
    _as_accurate_as_bf16(after, tf[16][:, T + 1], tf[32][:, T + 1])
    # the log-probs are the fp32 log-softmax of this call's own bf16 logits (t = 0: the prefill's)
    own = torch.cat([lead.unsqueeze(1), lg[:, :-1]], dim=1).reshape(B * T, -1)
    _check_logps_of(lp.reshape(-1), own, forced.to(DEV).reshape(-1), 1.0)
    # extend(17) + extend(23) == extend(40)
    eng.encode_images(img)
    eng.prefill(torch.tensor([PROMPT] * B))
    lg_a, lp_a = eng.extend(forced[:, :17], keep_logits=17)
    lg_b, lp_b = eng.extend(forced[:, 17:], keep_logits=23)
    lg_s, lp_s = torch.cat([lg_a, lg_b], 1), torch.cat([lp_a, lp_b], 1)
    assert bool(((lg_s - lg).abs() <= _ulp_bf16(lg.double()).float()).all()), "split call moved a logit by more than 1 bf16 ulp"
    lse = torch.logsumexp(own.double(), -1).view(B, T)
    assert bool(((lp_s - lp).abs().double() <= _lp_tol(lse)).all()), (lp_s - lp).abs().max().item()


def test_extend_v2_window_crossing():
    """StarCoder2 with sliding window 24: a 30-token prefix and a 50-token chunk cross the window edge (RoPE positions,
    window bounds and the KV scatter all at an offset)."""
    d = dims_tiny_v2()
    sd = synthetic_state_dict(d, seed=0, init="randomized")
    eng = Engine(d, 0)
    eng.load_state_dict(sd)
    B, T = 2, 50
    prompt = list(range(40, 40 + 30 - d.query_length))             # Q + 14 = 30 prefix tokens
    img = synthetic_images(d, B, seed=2)
    g = torch.Generator().manual_seed(4)
    ids = torch.randint(1, d.vocab - 8, (B, T), generator=g)
    eng.encode_images(img)
    eng.prefill(torch.tensor([prompt] * B))
    lg, lp = eng.extend(ids, keep_logits=T)
    tf = {dt: OracleStarVectorV2(d, sd, dtype=dt, eos_token_id=0).teacher_forced_logits(img, prompt, ids)
          for dt in (torch.bfloat16, torch.float32)}
    _as_accurate_as_bf16(lg, tf[torch.bfloat16][:, 1:], tf[torch.float32][:, 1:])
    _as_accurate_as_bf16(lp, _oracle_logps(tf[torch.bfloat16], ids), _oracle_logps(tf[torch.float32], ids))
    eng.close()


def test_extend_1b_dims_chunked():
    """1B decoder widths and vocabulary (2 layers, small ViT so the CPU oracle stays fast), B = 8 rows = 2 images x G = 4
    via expand_batch, T = 1100 = three internal chunks of 4096 / 8 = 512 tokens.  Logits just before / after every chunk
    boundary and at the end, and all log-probs, against the fp32 oracle (one forward per row)."""
    d = dataclasses.replace(ModelDims(max_batch=8, max_len=1400), n_layer=2, image_size=56, vit_width=128, vit_layers=1,
                            vit_heads=2, vit_mlp=512)
    sd = synthetic_state_dict(d, seed=0, init="randomized")
    eng = Engine(d, 0)
    eng.load_state_dict(sd)
    b, G, T = 2, 4, 1100
    img = synthetic_images(d, b, seed=1)
    g = torch.Generator().manual_seed(5)
    ids = torch.randint(1, d.vocab - 8, (b * G, T), generator=g)
    eng.encode_images(img)
    eng.prefill(torch.tensor([PROMPT] * b))
    eng.expand_batch([r % b for r in range(b * G)])
    lg, lp = eng.extend(ids, keep_logits=T, logps=True, temperature=1.0)
    steps = [510, 511, 512, 1022, 1023, 1024, T - 1]
    lg_chk = lg[:, steps].cpu()
    own_last = lg[:, :-1]
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    o = OracleStarVector(d, sd, dtype=torch.float32, pad_token_id=d.vocab - 4)
    errs_lg, errs_lp = [], []
    for r in range(b * G):
        im = img[r % b:r % b + 1]
        emb, _, _ = o.prepare_generation_inputs(im, PROMPT)
        t0 = emb.shape[1]
        hidden = o._body(inputs_embeds=torch.cat([emb, o._embed(ids[r:r + 1])], 1), use_cache=False).last_hidden_state
        ref_lg = o.llm.lm_head(hidden[0, t0 - 1:t0 + T - 1]).float()                    # [T, V]: row t predicts token t
        scale = ref_lg.abs().max().clamp_min(1.0).item()                                 # errors relative to the logit scale
        z = torch.log_softmax(ref_lg.double(), -1).gather(1, ids[r].long().view(-1, 1)).squeeze(1)
        errs_lp.append((lp[r].cpu().double() - z).abs() / scale)
        errs_lg.append((lg_chk[r] - o.llm.lm_head(hidden[0, [t0 + s for s in steps]]).float()).abs() / scale)
    e_lg, e_lp = torch.stack(errs_lg), torch.stack(errs_lp)
    # bf16 storage of 2 layers + the lm_head (a bf16 ulp is 2^-8 relative): a few ulps of the logit scale at most
    assert e_lg.max().item() < 0.05 and e_lg.mean().item() < 0.006, (e_lg.max().item(), e_lg.mean().item())
    assert e_lp.max().item() < 0.05 and e_lp.mean().item() < 0.006, (e_lp.max().item(), e_lp.mean().item())
    # and exactly the log-softmax of the call's own logits, across the chunk boundaries too
    for r in range(b * G):
        _check_logps_of(lp[r, 1:], own_last[r], ids[r, 1:].to(DEV), 1.0)
    eng.close()


# ------------------------------------------------------------------------------------------------------------------------
# 5. the facade
# ------------------------------------------------------------------------------------------------------------------------
def test_per_token_logps_matches_forward_and_oracle():
    from starvector_b200.modeling import StarVectorForCausalLM

    d = dims_tiny()
    sd = synthetic_state_dict(d, seed=0, init="randomized")
    m = StarVectorForCausalLM.from_config(dims=d, state_dict=sd)
    b, G, T, temp = 2, 2, 12, 0.8
    img = synthetic_images(d, b, seed=1).cuda()
    emb, _ = m.model.engine.encode_images(img, return_embeds=True)
    vision_embeds = torch.cat([emb, m.model._get_embeddings(torch.tensor([PROMPT] * b))], dim=1)
    g = torch.Generator().manual_seed(7)
    ids = torch.randint(1, d.vocab - 8, (b * G, T), generator=g)
    mask = torch.ones(b * G, vision_embeds.shape[1] + T, dtype=torch.long)
    mask[1, -3:] = 0
    lp = m.per_token_logps(vision_embeds, ids, num_generations=G, attention_mask=mask, temperature=temp)
    assert lp.shape == (b * G, T) and lp.dtype == torch.float32
    full = m.forward(vision_embeds, ids, num_generations=G, attention_mask=mask, num_logits_to_keep=T + 1).logits
    assert full.shape == (b * G, T + 1, d.vocab)
    plain = m.forward(vision_embeds, ids, num_generations=G, attention_mask=mask, num_logits_to_keep=T).logits
    assert torch.equal(full[:, 1:], plain), "the extra leading row moved the completion logits"
    lead = m.model.engine.prefill_embeds(vision_embeds, return_logits=True)
    assert torch.equal(full[:, 0], lead[[r % b for r in range(b * G)]])
    via_forward = torch.log_softmax(full[:, :-1].double() / temp, -1).gather(2, ids.to(DEV).long().unsqueeze(2)).squeeze(2)
    refs = {}
    for dt in (torch.bfloat16, torch.float32):
        o = OracleStarVector(d, sd, dtype=dt, pad_token_id=d.vocab - 4)
        e = torch.cat([vision_embeds.cpu().to(dt).repeat(G, 1, 1), o.llm.transformer.wte(ids)], dim=1)
        with torch.no_grad():
            logits = o.llm(inputs_embeds=e, use_cache=False).logits[:, -T - 1:-1].double()
        refs[dt] = torch.log_softmax(logits / temp, -1).gather(2, ids.long().unsqueeze(2)).squeeze(2)
    _as_accurate_as_bf16(lp, refs[torch.bfloat16], refs[torch.float32])
    _as_accurate_as_bf16(via_forward, refs[torch.bfloat16], refs[torch.float32])
    o_max = (refs[torch.bfloat16] - refs[torch.float32]).abs().max().item()
    assert (lp.double() - via_forward).abs().max().item() <= 4.0 * o_max + 3e-2
    with pytest.raises(NotImplementedError):
        left = mask.clone(); left[0, 0] = 0
        m.per_token_logps(vision_embeds, ids, G, left)
    with pytest.raises(ValueError):
        m.per_token_logps(vision_embeds, ids[:3], G)
    m.model.engine.close()


# ------------------------------------------------------------------------------------------------------------------------
# 6. refusals
# ------------------------------------------------------------------------------------------------------------------------
def test_extend_refusals_launch_nothing(tiny):
    d, sd, _, _, _, img = tiny
    eng = Engine(d, 0)
    eng.load_state_dict(sd)
    lib, h = eng._lib, eng._h
    ids = torch.ones(2, 8, dtype=torch.int32, device=DEV)
    lp = torch.empty(2, 8, device=DEV)

    def call(T=8, keep=0, temp=1.0, logits=None):
        return lib.sv_extend(h, C.c_void_p(ids.data_ptr()), T, C.c_void_p(logits.data_ptr() if logits is not None else 0),
                             keep, C.c_void_p(lp.data_ptr()), temp, None)

    n0 = eng.launch_count()
    assert call() == _lib.SV_ERR_STATE                                  # no prefill yet
    assert eng.launch_count() == n0
    eng.encode_images(img[:2])
    eng.prefill(torch.tensor([PROMPT] * 2))
    eng.generate(GenerationParams(max_new_tokens=4, eos_token_id=None, pad_token_id=d.vocab - 4))
    n0 = eng.launch_count()
    assert call() == _lib.SV_ERR_STATE                                  # the last generated token was never fed
    eng.encode_images(img[:2])
    eng.prefill(torch.tensor([PROMPT] * 2))
    n0 = eng.launch_count()
    assert call(T=d.max_len) == _lib.SV_ERR_INVALID                    # past max_len
    assert call(T=0) == _lib.SV_ERR_INVALID
    for t in (0.0, -1.0, float("nan"), float("inf")):
        assert call(temp=t) == _lib.SV_ERR_INVALID
    assert call(keep=9) == _lib.SV_ERR_INVALID                         # keep > T
    assert call(keep=2) == _lib.SV_ERR_INVALID                         # keep without a logits buffer
    assert eng.launch_count() == n0, "a refused call launched kernels"
    assert call() == _lib.SV_OK
    cp = GenerationParams(max_new_tokens=4, eos_token_id=None, pad_token_id=d.vocab - 4).to_c()
    out = torch.empty(2, 4, dtype=torch.int32, device=DEV)
    n0 = eng.launch_count()
    assert lib.sv_generate(h, C.byref(cp), C.c_void_p(out.data_ptr()), None, None) == _lib.SV_ERR_STATE
    assert eng.launch_count() == n0
    eng.close()
