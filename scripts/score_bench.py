"""Scoring throughput (not the headline bench): what a GRPO trainer pays to score its completions.

StarVector-1B dims, synthetic weights, 2 images x G = 4 completions, T completion tokens per row.  Two paths on the same
seeded inputs:
  * chunk   : `per_token_logps` = prefill once per image -> expand_batch -> sv_extend (4096-row tcgen05 GEMMs, lm_head with the
              fused log-prob epilogue);
  * decode  : `forward(..., num_logits_to_keep=T + 1)` (one sv_decode_step per token) + torch log_softmax / gather.
Times come from CUDA events around each call (median of --repeats after one warm-up).  FLOPs are counted from shapes (linear
layers, attention over the keys each token sees, lm_head).  A separate torch.profiler run of one chunk call at the largest T
splits its kernel time into attention, decoder GEMMs and lm_head + log-probs.  Prints one JSON object (and writes it to --out).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

PEAK_BF16_TFLOPS = 2250.0      # B200 data sheet, dense BF16, one GPU (HGX B200 figure / 8)


def extend_flops(d, B, prefix, T):
    """Multiply-adds x 2 of one sv_extend of T tokens on B rows after `prefix` cached tokens."""
    H, I, V, L = d.hidden, d.n_inner, d.vocab, d.n_layer
    qkv = H + 2 * d.n_kv_head * d.head_dim
    per_tok = 2 * L * (H * qkv + H * H + 2 * H * I) + 2 * H * V
    keys = sum(prefix + t + 1 for t in range(T))          # causal: token t sees prefix + t + 1 keys
    attn = 2 * 2 * L * d.n_head * d.head_dim * keys       # Q.K^T and P.V
    return B * (T * per_tok + attn)


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as exc:   # noqa: BLE001
        return f"unknown ({exc})"


def timed(fn, repeats):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return ms[len(ms) // 2], out


def classify(name):
    n = name.lower()
    if "attention_heads" in n:
        return "attention"
    logps_gemm = "linear_tc05_kernel" in n and ("<128, 1>" in n or "ili128eli1ee" in n)    # the EPI_LOGPS instantiation
    if logps_gemm or "logps_merge" in n or "row_logp" in n or "score_maps" in n or "float_rows_to_bf16" in n:
        return "lm_head_logps"
    if "linear_tc05" in n or "rowgroup" in n:
        return "decoder_gemm"
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, nargs="+", default=[256, 1024, 4096])
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--skip-decode-above", type=int, default=1 << 30, help="time the decode-step path only up to this T")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_bench needs a CUDA device: there is no CPU measurement path")
    from starvector_b200.config import dims_1b
    from starvector_b200.modeling import StarVectorForCausalLM
    from starvector_b200.weights import synthetic_images

    b, G, temp = 2, 4, 1.0
    Tmax = max(args.T)
    prompt = [44, 78]
    d = dims_1b(max_batch=b * G, max_len=257 + len(prompt) + Tmax + 8)
    m = StarVectorForCausalLM.from_config(dims=d)
    eng = m.model.engine
    dev = eng.device
    emb, _ = eng.encode_images(synthetic_images(d, b, seed=1).to(dev), return_embeds=True)
    vision = torch.cat([emb, m.model._get_embeddings(torch.tensor([prompt] * b))], dim=1)
    prefix = vision.shape[1]
    out = {"gpu": gpu_identity(), "workload": {"model": "StarVector-1B dims (24 layers, vocab 49156), synthetic weights",
                                              "images": b, "G": G, "rows": b * G, "prefix_tokens": prefix,
                                              "temperature": temp, "timing": f"CUDA events, median of {args.repeats} after 1 warm-up"},
           "peak_bf16_tflops_datasheet": PEAK_BF16_TFLOPS, "runs": []}
    g = torch.Generator().manual_seed(0)
    for T in sorted(args.T):
        ids = torch.randint(1, d.vocab - 8, (b * G, T), generator=g).to(dev)
        chunk_ms, lp = timed(lambda: m.per_token_logps(vision, ids, num_generations=G, temperature=temp), args.repeats)
        fl = extend_flops(d, b * G, prefix, T)
        run = {"T": T, "scored_tokens": b * G * T,
               "chunk_ms_per_call": round(chunk_ms, 3), "chunk_tokens_per_s": round(b * G * T / chunk_ms * 1e3, 1),
               "extend_tflop": round(fl / 1e12, 3),
               "chunk_achieved_tflops_whole_call": round(fl / chunk_ms / 1e9, 1),
               "chunk_share_of_datasheet_bf16_peak": round(fl / chunk_ms / 1e9 / PEAK_BF16_TFLOPS, 4)}
        if T <= args.skip_decode_above:
            def decode_path():
                lg = m.forward(vision, ids, num_generations=G, num_logits_to_keep=T + 1).logits
                return torch.log_softmax(lg[:, :-1] / temp, -1).gather(2, ids.long().unsqueeze(2)).squeeze(2)
            dec_ms, lp_dec = timed(decode_path, max(1, args.repeats - 1) if T >= 4096 else args.repeats)
            run.update({"decode_ms_per_call": round(dec_ms, 3), "decode_tokens_per_s": round(b * G * T / dec_ms * 1e3, 1),
                        "speedup_chunk_vs_decode": round(dec_ms / chunk_ms, 2),
                        "max_abs_dlogp_chunk_vs_decode": float((lp - lp_dec).abs().max().item()),
                        "mean_abs_dlogp_chunk_vs_decode": float((lp - lp_dec).abs().mean().item())})
            del lp_dec
            torch.cuda.empty_cache()
        else:
            run["decode_ms_per_call"] = "not measured"
        out["runs"].append(run)
        print(json.dumps(run), flush=True)
    # kernel-time split of one chunk call at the largest T, from a separate profiled run
    ids = torch.randint(1, d.vocab - 8, (b * G, Tmax), generator=g).to(dev)
    m.per_token_logps(vision, ids, num_generations=G, temperature=temp)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.per_token_logps(vision, ids, num_generations=G, temperature=temp)
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t:
            k = classify(ev.key)
            split[k] = split.get(k, 0.0) + t / 1e3
    total = sum(split.values()) or 1.0
    out["profile_split_T%d" % Tmax] = {k: {"kernel_ms": round(v, 3), "share": round(v / total, 4)} for k, v in sorted(split.items())}
    out["gpu_after"] = gpu_identity()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    eng.close()


if __name__ == "__main__":
    main()
