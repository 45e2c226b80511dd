#!/usr/bin/env python
"""bench.py — SVG tokens/sec of the im2svg hot path (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--max-new-tokens 4096] [--batch-per-gpu 1] [--no-cpu-baseline] [--dump-outputs DIR]

A "step" is one full `generate_im2svg` pass over one batch of synthetic 224x224 images with
random-init StarVector-1B weights: ViT -> adapter -> decoder prefill -> `max_new_tokens` greedy
decode steps (EOS/stop disabled so the length is deterministic, SURVEY.md §8d).
  value : whole-job new tokens / second, inputs already resident in HBM, CUDA events, max over ranks
  e2e   : same through the host-buffer entry point (pinned host image -> H2D -> ... -> D2H ids)
  roofline : decode step vs HBM (algorithmic bytes = W + kv*L per step, SURVEY.md §8d)
  cpu_baseline : the CPU oracle (HF generate on the host cores) on a bounded sample, rank 0, N=1
`--impl reference` times that CPU path as the reference arm (the reference is pure Python and has
no GPU-independent build; its own decoder is the installed `transformers` class).
`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float32), so that
two builds can be compared output for output: the inputs are seeded, identical from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

PROMPT_IDS = [44, 5678]          # stand-in for tokenizer('<svg') (no tokenizer files offline)
METRIC = "svg_tokens_per_sec"
WORKLOAD = "StarVector-1B im2svg greedy, batch={b}/GPU, 224x224 synthetic image, max_new_tokens={n}"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (profiling recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) == 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "reasons": reasons, "samples": len(self.rows)}


CPU_THREADS_CAP = 32      # decode on CPU is a GEMV stream: more threads than memory channels only adds contention
CONFIG1_NEW = 256         # BASELINE.json configs[0]: 1 image, greedy, max_new_tokens = 256, CPU via HF generate()


def _oracle_1b(dtype):
    from oracle.pipeline import OracleStarVector
    from starvector_b200.config import dims_1b
    from starvector_b200.weights import synthetic_images, synthetic_state_dict

    d = dims_1b(max_batch=1, max_len=8192)
    o = OracleStarVector(d, synthetic_state_dict(d, seed=0), dtype=dtype, eos_token_id=None, pad_token_id=49152)
    return d, o, synthetic_images(d, 1, seed=1).to(dtype)


def cpu_generate_seconds(o, d, img, n_new):
    t0 = time.perf_counter()
    ids = o.generate_im2svg_ids(img, PROMPT_IDS, (), use_nucleus_sampling=False, num_beams=1,
                                max_length=d.query_length + len(PROMPT_IDS) + n_new)
    assert ids.shape[1] == len(PROMPT_IDS) + n_new
    return time.perf_counter() - t0, ids[0, len(PROMPT_IDS):].tolist()


def cpu_reference_run(threads: int, steps: int = 1, warmup: int = 1, n_new: int = CONFIG1_NEW,
                      target_new: int = 4096, try_bf16: bool = True):
    """BASELINE.json configs[0] literally: the CPU oracle (reference ViT/adapter modules + the installed transformers
    `GPTBigCodeForCausalLM.generate`, oracle/pipeline.py) generates `n_new` = 256 greedy tokens for one image in fp32;
    every timed step is one whole such call (ViT + adapter + 259-token prefill + 256 decode steps), `steps` of them.
    A short generation (8 tokens) separates the fixed prefix cost from the per-token cost, so that the projection to the GPU arm's `target_new`-token workload can be stated next
    to the measured number.  bf16 (BASELINE.md §3 asks for both) is attempted on 8 tokens first and only run in full when
    the host executes bf16 matmuls natively (AMX); otherwise the reason is recorded."""
    torch.set_num_threads(threads)
    d, o, img = _oracle_1b(torch.float32)
    t_short = None
    for _ in range(max(1, warmup)):                      # warm-up: allocator, oneDNN primitive caches (short runs)
        t_short, _ = cpu_generate_seconds(o, d, img, 8)
    times, ids = [], None
    for _ in range(steps):
        t, ids = cpu_generate_seconds(o, d, img, n_new)
        times.append(t)
    sec = sum(times) / len(times)
    per_tok = max(sec - t_short, 1e-9) / (n_new - 8)
    prefix = max(t_short - 8 * per_tok, 0.0)
    out = {"seconds_per_step": sec, "steps_run": len(times), "tokens_per_s": n_new / sec, "per_token_s": per_tok, "prefix_s": prefix,
           "projected_tokens_per_s_at_target": target_new / (prefix + target_new * per_tok), "target_new": target_new, "ids": ids,
           "fp32_8tok_s": t_short}
    if try_bf16:
        try:
            # is bf16 native on this host (AMX / AVX512-BF16)?  one prefill-sized matmul in both dtypes decides
            a32, b32 = torch.randn(259, 2048), torch.randn(2048, 8192)
            a16, b16 = a32.bfloat16(), b32.bfloat16()

            def mm_time(a, b):
                torch.mm(a, b)
                t0 = time.perf_counter()
                for _ in range(3):
                    torch.mm(a, b)
                return (time.perf_counter() - t0) / 3

            t32, t16 = mm_time(a32, b32), mm_time(a16, b16)
            if t16 > 2.0 * t32:
                out["bf16"] = {"skipped": f"bf16 matmuls are emulated on this host ([259x2048]x[2048x8192]: {1e3 * t16:.1f} ms vs "
                                          f"{1e3 * t32:.1f} ms in fp32): a 256-token bf16 run would not finish in the bench budget"}
            else:
                d16, o16, img16 = _oracle_1b(torch.bfloat16)
                cpu_generate_seconds(o16, d16, img16, 2)
                t, _ = cpu_generate_seconds(o16, d16, img16, n_new)
                out["bf16"] = {"tokens_per_s": n_new / t, "seconds_per_step": t}
        except Exception as e:                           # noqa: BLE001 - a missing bf16 kernel must not kill the bench line
            out["bf16"] = {"skipped": f"{type(e).__name__}: {e}"[:200]}
    return out


def _cpu_sample_text(n_new, steps_run):
    return (f"BASELINE configs[0]: 1 image, greedy, {n_new} new tokens, fp32, reference ViT/adapter modules + HF GPTBigCode generate on "
            f"the host cores; {steps_run} full call(s) (ViT + adapter + 259-token prefill + {n_new} decode steps), wall clock")


def cpu_baseline_dict(r, threads):
    return {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": threads, "kind": "port",
            "sample": _cpu_sample_text(CONFIG1_NEW, r["steps_run"]), "seconds_per_step": r["seconds_per_step"],
            "per_token_ms": 1000 * r["per_token_s"], "prefix_s": r["prefix_s"],
            "projected_to_gpu_workload": {"max_new_tokens": r["target_new"], "tokens_per_s": r["projected_tokens_per_s_at_target"],
                                          "how": "prefix_s + n * per_token_s from the 8- and 256-token runs (context growth ignored: favours the CPU)"},
            "bf16": r.get("bf16")}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, CPU_THREADS_CAP)
    r = cpu_reference_run(threads, steps=args.steps, warmup=min(args.warmup, 2), target_new=args.max_new_tokens)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ids": torch.tensor([r["ids"]])})
    v = r["tokens_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s", "n_gpus": args.gpus, "steps": r["steps_run"],
        "warmup": min(args.warmup, 2), "ms_per_step": 1000 * r["seconds_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(b=1, n=args.max_new_tokens), "global_batch": 1,
                   "sample_of_workload": f"each step = the first {CONFIG1_NEW} new tokens of the workload (= BASELINE configs[0]) on the host CPU",
                   "note": ("a single CPU job on rank 0's host cores regardless of --gpus: ratios against it are only meaningful at N=1"
                            if args.gpus > 1 else "single CPU job")},
        "cpu_baseline": cpu_baseline_dict(r, threads),
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def ids_digest(ids: torch.Tensor) -> str:
    import hashlib

    return hashlib.sha256(ids.detach().to("cpu", torch.int32).contiguous().numpy().tobytes()).hexdigest()[:16]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """arrays: name -> tensor, written as out_dir/<name>.npy in float32 (token ids < 2**24 are exact)."""
    import numpy as np

    host = {k: v.detach().to("cpu", torch.float32).contiguous().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench: --dump-outputs would write {total} bytes, over the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def measure(model: str, B: int, n_new: int, steps: int, warmup: int, world: int, rank: int, local: int, sampling: bool = False,
            weights_on_device: bool = False):
    """One workload on this rank's GPU (all ranks run the same code): returns the numbers of the JSON line.

    Timing rules (profiling recipe): >= 3 warm-up passes, CUDA events on the launching stream bracketed by
    synchronize (+ barrier) on both sides, max over ranks; every pass streams the decoder weights (>> L2) once per token,
    so no explicit L2 flush is needed; nvidia-smi clocks are sampled during the timed region."""
    import torch.distributed as dist

    from starvector_b200.config import dims_1b, dims_8b
    from starvector_b200.engine import Engine, GenerationParams
    from starvector_b200.parallel import all_gather_generated
    from starvector_b200.weights import synthetic_images, synthetic_state_dict

    dev = torch.device("cuda", local)
    if model == "8b":
        d = dims_8b(max_batch=max(B, 1), max_len=min(16384, 576 + len(PROMPT_IDS) + n_new + 32))
    else:
        d = dims_1b(max_batch=max(B, 1), max_len=min(8192, 257 + len(PROMPT_IDS) + n_new + 32))
    sd = synthetic_state_dict(d, seed=0, device=dev if weights_on_device else None)   # every rank builds the same replica
    eng = Engine(d, local)
    eng.load_state_dict(sd)
    del sd
    gb = B * world
    img_host = synthetic_images(d, gb, seed=1)[rank * B:(rank + 1) * B].contiguous().pin_memory()
    img_dev = img_host.to(dev)
    prompt_host = torch.tensor([PROMPT_IDS] * B, dtype=torch.int32).pin_memory()
    prompt_dev = prompt_host.to(dev)
    if sampling:      # BASELINE configs[4]: temperature 0.8, reference default top_p 0.9
        params = GenerationParams(max_new_tokens=n_new, do_sample=True, temperature=0.8, top_p=0.9, eos_token_id=None, pad_token_id=49152,
                                  seed=1234 + rank)
    else:
        params = GenerationParams(max_new_tokens=n_new, eos_token_id=None, pad_token_id=49152)

    def step_resident():
        eng.encode_images(img_dev)
        eng.prefill(prompt_dev)
        ids = eng.generate(params)
        if world > 1:
            ids = all_gather_generated(ids, n_new, (), 49152, gb)
        return ids

    def step_host():
        ids, _ = eng.generate_im2svg_host(img_host, prompt_host, params)
        if world > 1:
            ids = all_gather_generated(ids.to(dev), n_new, (), 49152, gb).cpu()
        return ids

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, k):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        outs = [fn() for _ in range(k)]
        e1.record()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        sync_all()
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), outs

    for _ in range(warmup):
        step_resident()
    launches0 = eng.launch_count()
    dec_ms, dec_steps, digests = [], [], []
    first_ids = None
    with ClockSampler(local) as clocks:
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        passes = []
        for _ in range(steps):
            passes.append(step_resident())
            m, st = eng.last_decode_timing()
            dec_ms.append(m); dec_steps.append(st)
        e1.record()
        torch.cuda.synchronize(dev)
        ms_t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        sync_all()
        if world > 1:
            dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        total_ms = float(ms_t.item())
    launches = eng.launch_count() - launches0
    digests = [ids_digest(x) for x in passes]                 # after the timed region: what did the timed passes produce?
    first_ids, last_ids = passes[0].detach().cpu(), passes[-1].detach().cpu()
    del passes

    def prefill_only():
        eng.encode_images(img_dev)
        eng.prefill(prompt_dev)
    pf_ms, _ = timed(prefill_only, 5)
    for _ in range(min(warmup, 1)):
        step_host()
    e2e_ms, host_outs = timed(step_host, steps)
    digests_host = [ids_digest(x) for x in host_outs]
    del host_outs

    ms_per_step = total_ms / steps
    value = gb * n_new / (ms_per_step / 1000.0)
    e2e_value = gb * n_new / (e2e_ms / steps / 1000.0)
    # roofline of the decode step (the dominant cost: > 99% of a 4096-token pass)
    peak, peak_src = load_peaks()
    t0 = d.query_length + len(PROMPT_IDS)
    mean_ctx = t0 + (n_new - 1) / 2.0
    if d.sliding_window:                                      # SURVEY.md §8d: min(L_i, window) keys are read at every step
        mean_ctx = sum(min(t0 + i, d.sliding_window) for i in range(n_new)) / float(n_new)
    bytes_per_step = d.decoder_weight_bytes() + B * d.kv_bytes_per_token() * (mean_ctx + 1) + B * d.vocab * 2
    step_ms = sum(dec_ms) / max(1, sum(dec_steps))
    achieved = bytes_per_step / (step_ms / 1000.0) / 1e9 if step_ms > 0 else 0.0
    desc = eng.describe()
    eng.close()
    same = (not sampling) and len(set(digests + digests_host)) == 1
    return {
        "dims": d, "gb": gb, "t0": t0, "value": value, "e2e_value": e2e_value, "ms_per_step": ms_per_step, "prefill_ms_per_image": pf_ms / 5 / B,
        "step_ms": step_ms, "launches": int(launches), "engine": desc, "clocks": clocks.summary(), "achieved": achieved, "peak": peak,
        "peak_src": peak_src, "bytes_per_step": int(bytes_per_step), "first_ids": first_ids, "last_ids": last_ids,
        "ids": {"sha256_16_per_pass": digests, "host_path": digests_host,
                "identical_across_passes_and_paths": same if not sampling else None},
    }


def measure_beam(local: int, n_new: int = 512, num_beams: int = 2, passes: int = 2):
    """The reference's DEFAULT generate() mode (starvector_base.py:231-241: num_beams=2; do_sample, top_p 0.9 when
    use_nucleus_sampling) on this rank's GPU: 1 image x `num_beams` beams at StarVector-1B dims, the whole search on the device
    (sv_beam_search).  EOS / stop disabled so that every pass runs `n_new` steps.  No collective: every rank runs it alone."""
    from starvector_b200.beam_search import beam_search
    from starvector_b200.config import dims_1b
    from starvector_b200.engine import Engine
    from starvector_b200.weights import synthetic_images, synthetic_state_dict

    dev = torch.device("cuda", local)
    d = dims_1b(max_batch=num_beams, max_len=257 + len(PROMPT_IDS) + n_new + 32)
    eng = Engine(d, local)
    eng.load_state_dict(synthetic_state_dict(d, seed=0, device=dev))        # drawn on the GPU: seconds instead of ~15 s of host RNG
    img = synthetic_images(d, 1, seed=1).to(dev)
    prompt = torch.tensor([PROMPT_IDS], dtype=torch.int32, device=dev)
    out = {"workload": f"StarVector-1B dims, 1 image x {num_beams} beams, {n_new} steps, EOS/stop disabled, early_stopping='never'",
           "loop": "device-resident (sv_beam_search): candidates, bookkeeping and KV suffix copies inside the replayed decode graph"}
    for name, kw in (("beam_search", dict(do_sample=False)), ("beam_sample", dict(do_sample=True, top_p=0.9, temperature=1.0, seed=1234))):
        def run():
            return beam_search(eng, img, prompt, num_beams=num_beams, max_new_tokens=n_new, early_stopping="never", eos_token_id=None,
                               pad_token_id=49152, impl="device", **kw)
        run()
        torch.cuda.synchronize(dev)
        ms, toks, digs = [], [], []
        for _ in range(passes):
            ids = run()
            m, st = eng.last_decode_timing()
            ms.append(m / max(st, 1)); toks.append(int(ids.shape[1])); digs.append(ids_digest(ids))
        step_ms = sum(ms) / len(ms)
        out[name] = {"ms_per_beam_step": step_ms, "tokens_per_s": 1000.0 / step_ms, "tokens_returned": toks,
                     "timing": "CUDA events around the replayed graph loop on the engine's stream, mean of %d passes" % passes,
                     "identical_across_passes": len(set(digs)) == 1}
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--max-new-tokens", type=int, default=4096)
    ap.add_argument("--batch-per-gpu", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra BASELINE configs (configs[2] / configs[3] per-GPU slices)")
    ap.add_argument("--model", default="1b", choices=["1b", "8b"],
                    help="1b = StarVector-1B (headline, configs[1]); 8b = StarVector-8B family dims (SigLIP + StarCoder2)")
    ap.add_argument("--sampling", action="store_true", help="temperature 0.8 / top_p 0.9 sampling instead of greedy (BASELINE configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the generated ids of the last timed step as DIR/ids.npy (float32) after the timed steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run --nproc-per-node N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B, n_new = args.batch_per_gpu, args.max_new_tokens
    m = measure(args.model, B, n_new, args.steps, args.warmup, world, rank, local, sampling=args.sampling,
                weights_on_device=args.model == "8b")
    d = m["dims"]
    if m["ids"]["identical_across_passes_and_paths"] is False:
        raise SystemExit(f"bench: greedy passes produced different ids {m['ids']}: the timed work is not deterministic - refusing to report")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"ids": m["last_ids"]})
    workload = WORKLOAD if args.model == "1b" else WORKLOAD.replace("StarVector-1B", "StarVector-8B (SigLIP-L/16-384 + StarCoder2-7B dims)").replace("224x224", "384x384")
    if args.sampling:
        workload = workload.replace("greedy", "sampling T=0.8 top_p=0.9")
    line = {
        "metric": METRIC, "value": m["value"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": f"synthetic (random-init StarVector-{args.model.upper()} weights, seeded noise images)",
        "config": {"workload": workload.format(b=B, n=n_new), "global_batch": m["gb"], "parallelism": f"batch-shard x{world}",
                   "l2": f"no flush needed: {d.decoder_weight_bytes() / 1e9:.2f} GB of weights stream per decode step (>> 126 MB L2)",
                   "prompt_len": len(PROMPT_IDS), "prefix_len": m["t0"]},
        "prefill_ms_per_image": m["prefill_ms_per_image"],
        "decode_ms_per_token_step": m["step_ms"],
        "e2e": {"value": m["e2e_value"], "unit": "tokens/s",
                "h2d_bytes_per_step": int(B * 3 * d.image_size * d.image_size * 2 + B * len(PROMPT_IDS) * 4),
                "d2h_bytes_per_step": int(B * n_new * 4 + B * 4)},
        "gpu_launches": m["launches"],
        "engine": m["engine"],
        "clocks": m["clocks"],
        "roofline": {"bound": "hbm", "achieved": m["achieved"], "peak": m["peak"], "unit": "GB/s", "frac": m["achieved"] / m["peak"],
                     "traffic": None, "traffic_note": "not measured in this run (ncu captures: profiles/r02_*)",
                     "peak_source": m["peak_src"], "kernel": "decode step (" + m["engine"].split(" ")[0] + ")",
                     "algorithmic_bytes_per_step": m["bytes_per_step"]},
        "ids": m["ids"],
    }
    tpath = os.path.join(ROOT, "profiles", "r02_decode_step_traffic.json")
    if os.path.exists(tpath) and B == 1 and args.model == "1b":
        with open(tpath) as f:
            tj = json.load(f)
        line["roofline"]["traffic"] = int(tj["dram_bytes_read"] + tj["dram_bytes_write"])
        line["roofline"]["traffic_note"] = f"static: ncu dram__bytes of one decode step from profiles/r02_decode_step_traffic.json ({tj.get('how', '')}), not re-measured in this run"

    if not args.no_extras and args.model == "1b" and not args.sampling and B == 1:
        # the other GPU workloads BASELINE.json names, as per-GPU slices (same timing rules, shorter passes)
        extras = []
        for name, mdl, b, n, smp in (("configs[2]: StarVector-1B greedy, batch 64 over 8 GPUs = 8 images/GPU", "1b", 8, 1024, False),
                                     ("configs[3]: StarVector-8B bf16, batch 32 over 8 GPUs = 4 images/GPU", "8b", 4, 1024, False)):
            try:
                x = measure(mdl, b, n, 2, 3, world, rank, local, sampling=smp, weights_on_device=mdl == "8b")
                extras.append({"config": name, "max_new_tokens_run": n, "value": x["value"], "e2e": x["e2e_value"], "unit": "tokens/s",
                               "n_gpus": world, "decode_ms_per_token_step": x["step_ms"], "prefill_ms_per_image": x["prefill_ms_per_image"],
                               "roofline_frac": x["achieved"] / x["peak"], "engine": x["engine"].split(" ")[0], "ids": x["ids"]})
            except Exception as e:                        # noqa: BLE001 - an extra must never cost the headline line
                extras.append({"config": name, "error": f"{type(e).__name__}: {e}"[:300]})
        line["extra"] = {"configs": extras}
        try:
            line["extra"]["beam"] = measure_beam(local)
        except Exception as e:                            # noqa: BLE001 - an extra must never cost the headline line
            line["extra"]["beam"] = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.model == "1b" and not args.sampling:
        threads = min(os.cpu_count() or 1, CPU_THREADS_CAP)
        r = cpu_reference_run(threads, steps=1, warmup=1, target_new=n_new)
        line["cpu_baseline"] = cpu_baseline_dict(r, threads)
        # the timed passes' ids against the oracle's (same weights, same image): fp32 CPU vs bf16 GPU agree until two logits
        # come closer than bf16 resolves; the exhaustive contract lives in tests/ (this is a tripwire for the timed path)
        if B == 1:
            got = m["first_ids"][0, :len(r["ids"])].tolist()
            k = next((i for i, (a, b) in enumerate(zip(got, r["ids"])) if a != b), len(r["ids"]))
            line["ids"]["oracle_check"] = {"oracle": "fp32 CPU oracle, first %d greedy tokens" % len(r["ids"]), "matching_prefix": k,
                                           "all_match": k == len(r["ids"])}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
