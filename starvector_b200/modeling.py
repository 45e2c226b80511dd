"""Drop-in facade: the reference's `StarVectorForCausalLM` surface on top of the B200 engine.

Kept surface (SURVEY.md §8b; reference starvector/model/starvector_arch.py:133-193,
starvector/model/models/starvector_base.py:203-295, starvector_v1.py):
  StarVectorForCausalLM.from_pretrained / .from_config, .cuda()/.to()/.eval(), .process_images,
  .generate_im2svg(batch, **kw) -> list[str], .model.generate_im2svg, .model.generate_im2svg_grpo,
  .model.svg_transformer.tokenizer, .model.svg_transformer.transformer.generate(inputs_embeds=...),
  .model.processor, .model.query_length, .model.max_length, .model.image_encoder, .model.image_projection.
Errors are Python exceptions (ValueError for bad arguments, RuntimeError subclasses for CUDA
failures), as the reference's callers expect (serve/model_worker.py:183-207).
"""
from __future__ import annotations

import dataclasses
import json
import os
import warnings
from typing import Any, Dict, List, Optional

import torch

from .config import ModelDims, StarVectorConfig, refine_dims_from_state_dict
from .engine import Engine, GenerationParams
from .parallel import merge_generated
from .preprocess import ImageTrainProcessor, SiglipImageProcessor
from .tokenizer import load_tokenizer
from .weights import DEC, DEC2, synthetic_state_dict

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)


class _Transformer:
    """Stands where `svg_transformer.transformer` (the HF causal LM) is; only `.generate` is offered."""

    def __init__(self, owner: "StarVectorStarCoder"):
        self._o = owner
        self.config = owner.llm_config

    def generate(self, inputs_embeds: torch.Tensor = None, attention_mask: torch.Tensor = None, **kw) -> torch.Tensor:
        """`GenerationMixin.generate(inputs_embeds=...)` (starvector_base.py:255): returns NEW token ids only."""
        if inputs_embeds is None:
            raise ValueError("generate() on this engine takes inputs_embeds (the im2svg path); input_ids-only is not built")
        if attention_mask is not None and not bool(torch.all(attention_mask == 1)):
            raise NotImplementedError("padded prefixes never occur on the im2svg path and are not built")
        o = self._o
        params = self._hf_params(kw, prefix_len=inputs_embeds.shape[1])
        nb = int(kw.get("num_beams", 1))
        if nb > 1:
            es = kw.get("early_stopping", False)                                # HF: False (default) | True | "never"
            return o._beam_generate(params, kw, nb, inputs_embeds=inputs_embeds, early_stopping=es if es == "never" else bool(es))
        o.engine.prefill_embeds(inputs_embeds)
        return o.engine.generate(params).long()

    _HANDLED = {"do_sample", "top_p", "temperature", "num_beams", "max_length", "max_new_tokens", "min_length", "repetition_penalty",
                "length_penalty", "use_cache", "stopping_criteria", "early_stopping", "pad_token_id", "eos_token_id", "seed"}

    def _hf_params(self, kw: Dict[str, Any], prefix_len: int) -> GenerationParams:
        """HF `generate()` semantics for exactly the kwargs the reference passes (starvector_base.py:228-241, :292-295):
        HF defaults (greedy, top_p = 1, no stop sequence) unless given; anything else is refused instead of ignored."""
        o = self._o
        unknown = sorted(set(kw) - self._HANDLED)
        if unknown:
            raise NotImplementedError(f"generate(): unsupported arguments {unknown}")
        do_sample = bool(kw.get("do_sample", False))
        max_new = kw.get("max_new_tokens")
        if max_new is None:
            max_new = int(kw.get("max_length", 20)) - prefix_len                # generation/utils.py:1629-1638
        if max_new <= 0:
            raise ValueError(f"Input length of input_ids is 0, but `max_length` is set to {max_new}. Increase max_length "
                             "(it counts the visual prefix and the prompt).")
        if int(kw.get("min_length", 0)) - prefix_len > 0:                       # :1655-1660: becomes max(min_length - prefix, 0)
            raise NotImplementedError("min_length beyond the prefix (a MinLengthLogitsProcessor) is not built")
        stop_ids: List[int] = []
        for crit in (kw.get("stopping_criteria") or []):
            stops = getattr(crit, "stops", None)                                # StoppingCriteriaSub(stops=[ids]) (:9-20)
            if stops is None or len(stops) != 1:
                raise NotImplementedError("only the reference's StoppingCriteriaSub with one stop sequence is supported")
            stop_ids = [int(t) for t in (stops[0].tolist() if hasattr(stops[0], "tolist") else stops[0])]
        eos = kw.get("eos_token_id", o.eos_token_id)
        pad = kw.get("pad_token_id")
        if pad is None:
            pad = eos if eos is not None else o.svg_transformer.tokenizer.pad_token_id     # HF: pad falls back to eos
        return GenerationParams(max_new_tokens=int(max_new), do_sample=do_sample, temperature=float(kw.get("temperature", 1.0)),
                                top_p=float(kw.get("top_p", 1.0)) if do_sample else 1.0,
                                repetition_penalty=float(kw.get("repetition_penalty", 1.0)), eos_token_id=eos, pad_token_id=pad,
                                stop_ids=stop_ids, stop_row0_only=True, seed=int(kw.get("seed", o.seed)))


class _SvgTransformer:
    """`StarCoderModel` stand-in (llm/starcoder.py): tokenizer + transformer + prompt."""

    def __init__(self, owner: "StarVectorStarCoder", tokenizer):
        self.tokenizer = tokenizer
        self.transformer = _Transformer(owner)
        self.prompt = "<svg"                                   # starcoder.py:38
        self.svg_start_token = "<svg-start>"


class _ImageEncoder:
    """`ImageEncoder` stand-in: `process_images` (image_encoder.py:112-117) and a callable forward."""

    def __init__(self, owner: "StarVectorStarCoder"):
        self._o = owner

    def process_images(self, images):
        if self._o.v2:                                                          # image_encoder.py:119
            return self._o.processor(images=images, return_tensors="pt").pixel_values.unsqueeze(0)
        return [x.unsqueeze(0) for x in self._o.processor.batch(images)]        # image_encoder.py:113-117, one upload + 2 launches

    def __call__(self, image: torch.Tensor) -> torch.Tensor:
        _, vit = self._o.engine.encode_images(image, return_vit=True)
        return vit


class StarVectorStarCoder:
    """v1 model core (models/starvector_v1.py + starvector_base.py) bound to one Engine."""

    def __init__(self, config: StarVectorConfig, engine: Engine, tokenizer, wte: torch.Tensor, v2: bool = False):
        self.config = config
        self.engine = engine
        self.v2 = v2                                                            # models/starvector_v2.py semantics
        self.task = "im2svg"
        self.query_length = engine.query_length
        self.max_length = config.max_length_train - self.query_length - 4      # starvector_base.py:41
        self.llm_config = {"hidden_size": engine.dims.hidden, "vocab_size": engine.dims.vocab,
                           "n_positions": engine.dims.n_positions}
        # image_encoder.py:25 (clip: ImageTrainProcessor) / :32-48 (siglip: the hub's SiglipProcessor); both run on the GPU
        dev_index = engine.device.index or 0
        self.processor = (SiglipImageProcessor(size=engine.dims.image_size, device=dev_index) if v2
                          else ImageTrainProcessor(size=engine.dims.image_size, device=dev_index))
        self.svg_transformer = _SvgTransformer(self, tokenizer)
        self.image_encoder = _ImageEncoder(self)
        self.image_projection = self._project
        self._wte = wte                                                        # [V,H] on device, for _get_embeddings
        self.eos_token_id: Optional[int] = tokenizer.eos_token_id
        self.seed = 0

    # -- reference helpers ---------------------------------------------------------------
    def _project(self, *_a, **_k):
        raise NotImplementedError("the adapter runs fused with the image encoder: use engine.encode_images(..., return_embeds=True)")

    def _get_embeddings(self, input_ids: torch.Tensor) -> torch.Tensor:       # starvector_v1.py:16-18
        return self._wte[input_ids.to(self._wte.device)]

    def _tokenize_prompt(self, prompt: Optional[str], batch: int) -> torch.Tensor:
        if prompt is None:
            prompt = self.svg_transformer.prompt
        enc = self.svg_transformer.tokenizer([prompt] * batch, add_special_tokens=False, return_tensors="pt",
                                             padding="longest", truncation=True)
        return enc["input_ids"]

    def _stop_ids(self) -> List[int]:
        return list(self.svg_transformer.tokenizer("</svg>", add_special_tokens=False)["input_ids"])   # base:226

    def _gen_params(self, kw: Dict[str, Any], prefix_len: int) -> GenerationParams:
        """`_get_generation_kwargs` (:223-241) + `_get_im2svg_specific_kwargs` (:289-295) + HF length fix-up."""
        do_sample = bool(kw.get("use_nucleus_sampling", True))                # :231 — a `do_sample` kwarg is not in the whitelist
        max_length = int(kw.get("max_length", 30))
        max_new = kw.get("max_new_tokens")
        if max_new is None:
            max_new = max_length - prefix_len                                  # generation/utils.py:1629-1638
        if max_new <= 0:
            raise ValueError(
                f"Input length of input_ids is 0, but `max_length` is set to {max_length - prefix_len}. "
                "Increase max_length (it counts the visual prefix and the prompt).")
        tok = self.svg_transformer.tokenizer
        return GenerationParams(
            max_new_tokens=int(max_new), do_sample=do_sample,
            temperature=float(kw.get("temperature", 1)), top_p=float(kw.get("top_p", 0.9)) if do_sample else 1.0,
            repetition_penalty=float(kw.get("repetition_penalty", 1.0)),
            eos_token_id=self.eos_token_id,
            # v1 passes tokenizer.pad_token_id (starvector_base.py:294); v2 passes nothing and HF falls back to eos
            pad_token_id=(self.eos_token_id if self.v2 and self.eos_token_id is not None else tok.pad_token_id),
            stop_ids=kw.get("stop_ids", self._stop_ids()), stop_row0_only=True,
            seed=int(kw.get("seed", self.seed)),
        )

    def _beam_generate(self, params: GenerationParams, kw: Dict[str, Any], num_beams: int, image=None, prompt_ids=None,
                       inputs_embeds=None, early_stopping: Optional[bool] = None) -> torch.Tensor:
        """num_beams > 1 (the reference default is 2, starvector_base.py:234): beam search / beam-sample with the
        caller's `length_penalty`; `early_stopping=True` for v1 (:292), HF's default False for v2
        (starvector_v2.py:53-57) — bookkeeping in beam_search.py."""
        from .beam_search import beam_search

        return beam_search(
            self.engine, image, prompt_ids, inputs_embeds=inputs_embeds, num_beams=num_beams,
            max_new_tokens=params.max_new_tokens, do_sample=params.do_sample, temperature=params.temperature,
            top_p=params.top_p, repetition_penalty=params.repetition_penalty,
            length_penalty=float(kw.get("length_penalty", 1.0)),
            # v1 passes early_stopping=True (:292); v2's specific kwargs are {} -> HF default False
            early_stopping=(not self.v2) if early_stopping is None else early_stopping,
            eos_token_id=params.eos_token_id, pad_token_id=params.pad_token_id, stop_ids=params.stop_ids, seed=params.seed)

    # -- the path ------------------------------------------------------------------------
    @torch.no_grad()
    def generate_im2svg_ids(self, batch: Dict[str, torch.Tensor], **kwargs) -> torch.Tensor:
        """Token ids `[B, P + n_new]` (prompt + generated) — starvector_base.py:243-256."""
        image = batch["image"]
        prompt_ids = self._tokenize_prompt(kwargs.get("prompt"), image.shape[0])
        params = self._gen_params(kwargs, prefix_len=self.query_length + prompt_ids.shape[1])
        num_beams = int(kwargs.get("num_beams", 2))                             # reference default (:234)
        if num_beams > 1:
            if kwargs.get("streamer") is not None:                              # same rule and message as HF generate()
                raise ValueError("`streamer` cannot be used with beam search (yet!). Make sure that `num_beams` is set to 1.")
            out = self._beam_generate(params, kwargs, num_beams, image=image, prompt_ids=prompt_ids)
            return torch.cat([prompt_ids.to(out.device), out.long()], dim=1)
        mb = self.engine.dims.max_batch
        streamer = kwargs.get("streamer")                                       # serve/model_worker.py:131,172
        if streamer is not None:
            if image.shape[0] > mb:
                raise ValueError(f"streaming needs the batch ({image.shape[0]}) to fit the engine's max_batch ({mb})")
            self.engine.encode_images(image)
            self.engine.prefill(prompt_ids)

            def on_tokens(ids: torch.Tensor, first_step: int) -> bool:          # HF BaseStreamer protocol: put([B]) per step
                for j in range(ids.shape[1]):
                    streamer.put(ids[:, j].long())
                return False

            try:
                out = self.engine.generate(params, on_tokens=on_tokens)
            finally:
                streamer.end()
        elif image.shape[0] * int(kwargs.get("_share_prefix", 1)) <= mb:
            self.engine.encode_images(image)
            self.engine.prefill(prompt_ids)
            G = int(kwargs.get("_share_prefix", 1))
            if G > 1:      # num_return_sequences: the visual prefix is encoded and prefilled ONCE per image, its KV rows replicated
                self.engine.expand_batch([r // G for r in range(image.shape[0] * G)])
                prompt_ids = prompt_ids.repeat_interleave(G, dim=0)
            out = self.engine.generate(params)
        else:
            # More images than the engine holds at once: run max_batch-sized groups one after another and rebuild the
            # single-call rectangle with the rule the multi-GPU path uses (parallel.merge_generated): only the group that
            # contains global row 0 arms the row-0 `</svg>` stop, rows are independent, so prefixes are identical.
            groups = []
            for lo in range(0, image.shape[0], mb):
                p = params if lo == 0 else dataclasses.replace(params, stop_ids=(), seed=params.seed + lo)
                self.engine.encode_images(image[lo:lo + mb])
                self.engine.prefill(prompt_ids[lo:lo + mb])
                groups.append(self.engine.generate(p))
            out = merge_generated(groups, params.stop_ids, params.pad_token_id)
        return torch.cat([prompt_ids.to(out.device), out.long()], dim=1)

    def generate_im2svg(self, batch: Dict[str, torch.Tensor], **kwargs) -> List[str]:
        ids = self.generate_im2svg_ids(batch, **kwargs)
        return self.svg_transformer.tokenizer.batch_decode(ids, skip_special_tokens=True)          # :257

    def generate_im2svg_grpo(self, batch, **kwargs):                                               # :261-286
        """`num_return_sequences` completions per image (sampled independently, `num_beams` forced to 1, :277-280):
        HF's `_expand_inputs_for_generation` = every image row repeated G times, adjacent — here the image is encoded and
        prefilled once and its KV-cache rows are replicated (`sv_expand_batch`).  Returns the reference's dict;
        `outputs` is `[B*G, P + n_new]`, `inputs_embeds` the un-expanded `[B, Q+P, H]` prefix embeddings."""
        G = int(kwargs.get("num_return_sequences", 1))
        if G < 1:
            raise ValueError("num_return_sequences must be >= 1")
        image = batch["image"]
        if G > 1:
            if image.shape[0] * G > self.engine.dims.max_batch:
                raise ValueError(f"batch {image.shape[0]} x num_return_sequences {G} exceeds the engine's max_batch "
                                 f"{self.engine.dims.max_batch}")
            kwargs = dict(kwargs, num_beams=1)                 # :277-280 (only when num_return_sequences > 1)
        ids = self.generate_im2svg_ids({"image": image}, **(dict(kwargs, _share_prefix=G) if G > 1 else kwargs))
        emb, _ = self.engine.encode_images(image, return_embeds=True)
        prompt_ids = self._tokenize_prompt(kwargs.get("prompt"), image.shape[0])
        inputs_embeds = torch.cat([emb, self._get_embeddings(prompt_ids.to(emb.device))], dim=1)    # :217-219
        return {"raw_svg": self.svg_transformer.tokenizer.batch_decode(ids, skip_special_tokens=True),
                "outputs": ids, "inputs_embeds": inputs_embeds}


@dataclasses.dataclass
class _ScoreOutput:
    """The two fields of `CausalLMOutputWithCrossAttentions` the RLRF scoring callers read."""
    loss: Optional[torch.Tensor]
    logits: torch.Tensor


def read_checkpoint(path: str):
    """`(StarVectorConfig, state_dict)` from a local HF-style directory: config.json + every *.safetensors shard, or
    pytorch_model.bin.  Tensors stay on the CPU in their stored dtype; the engine converts to bf16 at load."""
    config = StarVectorConfig.from_pretrained(path)
    sd: Dict[str, torch.Tensor] = {}
    files = sorted(f for f in os.listdir(path) if f.endswith(".safetensors"))
    if files:
        from safetensors.torch import load_file

        for f in files:
            sd.update(load_file(os.path.join(path, f)))
    elif os.path.exists(os.path.join(path, "pytorch_model.bin")):
        sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu", weights_only=True)
    else:
        raise FileNotFoundError(f"no *.safetensors / pytorch_model.bin under {path}")
    return config, sd


def write_checkpoint(path: str, config: StarVectorConfig, state_dict: Dict[str, torch.Tensor]) -> None:
    """config.json + model.safetensors.  A TIED `lm_head.weight` (equal to the token embedding) is not stored twice — the
    reference pops it and re-ties at load (train/util.py:68-77); an un-tied head, which the engine supports, is kept so that
    a save / load round trip cannot silently change the logits."""
    from safetensors.torch import save_file

    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, "config.json"), "w") as f:
        json.dump(config.to_dict(), f, indent=1)

    def tied(k: str) -> bool:
        if not k.endswith("lm_head.weight"):
            return False
        pre = k[: -len("lm_head.weight")]
        emb = next((state_dict[c] for c in (pre + "transformer.wte.weight", pre + "model.embed_tokens.weight") if c in state_dict), None)
        return emb is not None and emb.shape == state_dict[k].shape and torch.equal(emb, state_dict[k])

    save_file({k: v.contiguous() for k, v in state_dict.items() if not tied(k)}, os.path.join(path, "model.safetensors"))


class StarVectorForCausalLM:
    """`StarVectorForCausalLM` facade (starvector_arch.py:133-193) — not an nn.Module: weights live in the engine."""

    config_class = StarVectorConfig

    def __init__(self, config: StarVectorConfig, state_dict: Dict[str, torch.Tensor], device: int = 0,
                 max_batch: int = 8, max_len: Optional[int] = None, tokenizer_path: Optional[str] = None):
        self.config = config
        dims = refine_dims_from_state_dict(config.to_dims(max_batch=max_batch, max_len=max_len), state_dict)
        self.dims = dims
        engine = Engine(dims, device)
        engine.load_state_dict(state_dict)
        v2 = dims.variant == 1
        wte = state_dict[(DEC2 + "embed_tokens.weight") if v2 else (DEC + "wte.weight")].to(device=engine.device,
                                                                                               dtype=torch.bfloat16)
        tok = load_tokenizer(tokenizer_path, dims.vocab, v2=v2)
        self.model = StarVectorStarCoder(config, engine, tok, wte, v2=v2)     # v2 = StarVectorStarCoder2 (starvector_arch.py:137-145)
        self.device = engine.device
        self.dtype = torch.bfloat16

    # -- construction --------------------------------------------------------------------
    @classmethod
    def from_config(cls, config: Optional[StarVectorConfig] = None, dims: Optional[ModelDims] = None, seed: int = 0,
                    init: str = "hf_default", device: int = 0, max_batch: int = 8, max_len: Optional[int] = None,
                    state_dict: Optional[Dict[str, torch.Tensor]] = None) -> "StarVectorForCausalLM":
        """Random-init model of the configured architecture (synthetic benchmark / tests)."""
        config = config or StarVectorConfig()
        if dims is not None:
            config.engine_dims = {k: v for k, v in dims.__dict__.items() if k not in ("max_batch", "max_len")}
            max_batch, max_len = dims.max_batch, dims.max_len
            if dims.variant == 1:
                config.starcoder_model_name, config.image_encoder_type = "bigcode/starcoder2-7b", "siglip_384"
        d = config.to_dims(max_batch=max_batch, max_len=max_len)
        sd = state_dict if state_dict is not None else synthetic_state_dict(d, seed=seed, init=init)
        return cls(config, sd, device=device, max_batch=max_batch, max_len=max_len)

    @classmethod
    def from_pretrained(cls, path: str, torch_dtype: Any = None, device: int = 0, max_batch: int = 8,
                        max_len: Optional[int] = None, **kw) -> "StarVectorForCausalLM":
        """Load a LOCAL checkpoint directory (config.json + *.safetensors / pytorch_model.bin).  No hub access."""
        config, sd = read_checkpoint(path)
        return cls(config, sd, device=device, max_batch=max_batch, max_len=max_len, tokenizer_path=path)

    def save_pretrained(self, path: str, state_dict: Dict[str, torch.Tensor]) -> None:
        write_checkpoint(path, self.config, state_dict)

    # -- scoring (starvector_arch.py:161-184) ------------------------------------------------
    def _scoring_rows(self, vision_embeds: torch.Tensor, input_ids: torch.Tensor, num_generations: int,
                      attention_mask: Optional[torch.Tensor]):
        """Shared argument rules of `forward` and `per_token_logps`: `b * G` completion rows in `.repeat` order, and only a
        right-padded tail may be masked.  Prefills the prefix ONCE per image and replicates its KV rows (row r <- r % b)."""
        eng = self.model.engine
        b, G = vision_embeds.shape[0], int(num_generations)
        ids = input_ids.to(eng.device)
        if ids.shape[0] != b * G:
            raise ValueError(f"input_ids has {ids.shape[0]} rows, expected vision rows {b} x num_generations {G}")
        if b * G > eng.dims.max_batch:
            raise ValueError(f"{b} x {G} rows exceed the engine's max_batch {eng.dims.max_batch}")
        T = ids.shape[1]
        if attention_mask is not None:
            m = attention_mask.to(torch.bool)
            tail = m[:, m.shape[1] - T:] if m.shape[1] >= T else m
            if not bool(torch.all(m[:, : m.shape[1] - T])) or bool(torch.any(tail[:, 1:] & ~tail[:, :-1])):
                raise NotImplementedError("only right-padded completions (mask = ones then zeros) are supported")
        return eng, b, G, ids, T

    @torch.no_grad()
    def forward(self, vision_embeds: torch.Tensor, input_ids: torch.Tensor, num_generations: int = 1,
                attention_mask: Optional[torch.Tensor] = None, num_logits_to_keep: int = 0):
        """Logits of `num_generations` completions per image over a shared visual prefix, as the reference's
        `StarVectorForCausalLM.forward`: `inputs_embeds = cat([vision_embeds.repeat(G, 1, 1), wte(input_ids)], 1)` -> decoder
        -> `lm_head` on the last `num_logits_to_keep` positions (all completion positions when 0; T + 1 adds the prefix's
        last position, TRL's `logits_to_keep + 1`).  Here the prefix is prefilled ONCE per image and its KV rows replicated
        (`sv_expand_batch`, rows r % b as `.repeat` orders them); the completion is teacher-forced through `sv_decode_step`.
        Returns an object with `.logits` fp32 `[b*G, n_keep, V]` and `.loss = None`.  `attention_mask` may only mask a
        right-padded tail (what GRPO completions carry).  Log-probs for RL: `per_token_logps` computes them without the logits."""
        eng, b, G, ids, T = self._scoring_rows(vision_embeds, input_ids, num_generations, attention_mask)
        n_keep = T if int(num_logits_to_keep) <= 0 else int(num_logits_to_keep)
        if n_keep > T + 1:
            raise NotImplementedError("num_logits_to_keep beyond the completion and the prefix's last position is not built")
        lead = eng.prefill_embeds(vision_embeds.to(eng.device, torch.bfloat16), return_logits=n_keep == T + 1)
        if G > 1:
            eng.expand_batch([r % b for r in range(b * G)])
        n_body = min(n_keep, T)
        out = torch.empty(b * G, n_body, eng.dims.vocab, dtype=torch.float32, device=eng.device)
        for t in range(T):
            keep = t >= T - n_body
            lg = eng.decode_step(ids[:, t], return_logits=keep)
            if keep:
                out[:, t - (T - n_body)] = lg
        if n_keep == T + 1:
            out = torch.cat([lead[[r % b for r in range(b * G)]].unsqueeze(1), out], dim=1)
        return _ScoreOutput(loss=None, logits=out)

    @torch.no_grad()
    def per_token_logps(self, vision_embeds: torch.Tensor, input_ids: torch.Tensor, num_generations: int = 1,
                        attention_mask: Optional[torch.Tensor] = None, temperature: float = 1.0) -> torch.Tensor:
        """What a GRPO trainer computes from `forward(..., num_logits_to_keep=T + 1).logits`: fp32 `[b*G, T]` with
        `[r, t] = log_softmax(logits[r, t] / temperature)[input_ids[r, t]]`, where logits[r, t] is the row predicting
        completion token t (t = 0: the prefix's last position).  Rows and mask rules as `forward`; the caller applies the
        mask to the result.  One prefill per image, then the completions in chunks through `sv_extend`, whose lm_head reduces
        its tiles to log-probs on the fly: the `[b*G, T, V]` logits are never written."""
        eng, b, G, ids, T = self._scoring_rows(vision_embeds, input_ids, num_generations, attention_mask)
        eng.prefill_embeds(vision_embeds.to(eng.device, torch.bfloat16))
        if G > 1:
            eng.expand_batch([r % b for r in range(b * G)])
        _, lp = eng.extend(ids, logps=True, temperature=temperature)
        return lp

    __call__ = forward

    # -- nn.Module-ish no-ops the callers use (quickstart.py:11-12) ------------------------
    def cuda(self, *a, **k): return self
    def to(self, *a, **k): return self
    def eval(self): return self
    def half(self): return self
    def bfloat16(self): return self

    # -- the surface ---------------------------------------------------------------------
    def generate_im2svg(self, batch, **kwargs) -> List[str]:                  # starvector_arch.py:186-187
        return self.model.generate_im2svg(batch, **kwargs)

    def generate_im2text(self, batch, **kwargs):                              # :189-190 (dangling in the reference too)
        raise AttributeError("generate_im2text has no implementation in the reference model core either")

    def process_images(self, images):                                         # :192-193
        return self.model.image_encoder.process_images(images)
