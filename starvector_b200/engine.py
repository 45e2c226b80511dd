"""`Engine`: the thin object around one `sv_engine*` (one model replica on one GPU).

PyTorch is used only for device memory, dtype views and the current stream handle; all
compute happens inside libstarvector_b200.so.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import threading
from typing import Dict, Iterable, Optional, Sequence, Tuple

import torch

from . import _lib
from .config import ModelDims

_DTYPES = {torch.bfloat16: _lib.SV_DTYPE_BF16, torch.float32: _lib.SV_DTYPE_F32, torch.float16: _lib.SV_DTYPE_F16}


@dataclasses.dataclass
class GenerationParams:
    """HF `generate()` kwargs after the reference's whitelist (starvector_base.py:223-241)."""

    max_new_tokens: int
    do_sample: bool = False
    temperature: float = 1.0
    top_p: float = 1.0
    repetition_penalty: float = 1.0
    eos_token_id: Optional[int] = 0
    pad_token_id: int = 0
    stop_ids: Sequence[int] = ()
    stop_row0_only: bool = True
    seed: int = 0
    poll_interval: int = 16

    def to_c(self) -> _lib.GenParams:
        if len(self.stop_ids) > 8:
            raise ValueError("stop sequence longer than 8 tokens")
        p = _lib.GenParams()
        p.max_new_tokens = int(self.max_new_tokens)
        p.do_sample = int(bool(self.do_sample))
        p.temperature = float(self.temperature)
        p.top_p = float(self.top_p)
        p.repetition_penalty = float(self.repetition_penalty)
        p.eos_token_id = -1 if self.eos_token_id is None else int(self.eos_token_id)
        p.pad_token_id = int(self.pad_token_id)
        p.n_stop_ids = len(self.stop_ids)
        for i, s in enumerate(self.stop_ids):
            p.stop_ids[i] = int(s)
        p.stop_row0_only = int(bool(self.stop_row0_only))
        p.seed = int(self.seed) & (2 ** 64 - 1)
        p.poll_interval = int(self.poll_interval)
        return p


def _stream_ptr(device: torch.device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    def __init__(self, dims: ModelDims, device: int | torch.device = 0):
        self._lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.EngineError("starvector_b200: no CUDA device visible; this engine has no CPU fallback")
        self.device = torch.device("cuda", device if isinstance(device, int) else (device.index or 0))
        self.dims = dims
        desc = _lib.ModelDesc(
            variant=dims.variant, image_size=dims.image_size, patch_size=dims.patch_size, vit_width=dims.vit_width,
            vit_layers=dims.vit_layers, vit_heads=dims.vit_heads, vit_mlp=dims.vit_mlp, adapter_norm=dims.adapter_norm,
            hidden=dims.hidden, n_layer=dims.n_layer, n_head=dims.n_head, n_kv_head=dims.n_kv_head,
            head_dim=dims.head_dim, n_inner=dims.n_inner, n_positions=dims.n_positions, vocab=dims.vocab,
            ln_eps=dims.ln_eps, max_batch=dims.max_batch, max_len=dims.max_len,
            rope_theta=dims.rope_theta, sliding_window=dims.sliding_window, vit_ln_eps=dims.vit_ln_eps,
        )
        h = C.c_void_p()
        torch.cuda.init()
        torch.zeros(1, device=self.device)        # make sure the primary context exists
        _lib.check(self._lib, self._lib.sv_engine_create(C.byref(desc), self.device.index, C.byref(h)))
        self._h = h
        self._lock = threading.Lock()             # engine is not re-entrant (SURVEY.md §3.3: threaded callers)
        self.query_length = dims.query_length
        self._batch = 0
        self._prompt_len = 0

    # -- lifecycle -----------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.sv_engine_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, code: int) -> None:
        _lib.check(self._lib, code, self._h)

    # -- weights -------------------------------------------------------------------------
    def load_state_dict(self, sd: Dict[str, torch.Tensor], strict: bool = True) -> None:
        """Copy a reference-named state dict (CPU or CUDA tensors; bf16/fp16/fp32) into the engine."""
        wte_key = ("model.svg_transformer.transformer.model.embed_tokens.weight" if self.dims.variant == 1
                   else "model.svg_transformer.transformer.transformer.wte.weight")
        lm_key = "model.svg_transformer.transformer.lm_head.weight"
        with self._lock:
            for name, t in sd.items():
                if name == lm_key and wte_key in sd and (t is sd[wte_key] or t.data_ptr() == sd[wte_key].data_ptr()
                                                          or torch.equal(t, sd[wte_key])):
                    continue                       # tied head: the engine aliases wte
                if not t.is_floating_point():
                    continue
                if t.dtype not in _DTYPES:
                    t = t.float()
                t = t.contiguous()
                shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
                code = self._lib.sv_engine_load_weight(self._h, name.encode(), C.c_void_p(t.data_ptr()), shape,
                                                       t.dim(), _DTYPES[t.dtype])
                if code == _lib.SV_ERR_INVALID and not strict:
                    continue
                self._ck(code)
            if self.dims.variant == 1:
                self._load_rope_tables()
            missing = self._lib.sv_engine_missing_weights(self._h)
            if missing and strict:
                names = self._lib.sv_last_error(self._h).decode()
                raise KeyError(f"{missing} weights missing from state dict, e.g. {names.splitlines()[:4]}")

    def _load_rope_tables(self) -> None:
        """cos/sin tables computed exactly as Starcoder2RotaryEmbedding does (fp32 outer product, cast to bf16), so the
        engine's RoPE inputs are bit-identical to the reference's; the engine's own on-device table is the fallback."""
        d = self.dims
        inv_freq = 1.0 / (d.rope_theta ** (torch.arange(0, d.head_dim, 2, dtype=torch.int64).float() / d.head_dim))
        freqs = torch.outer(torch.arange(d.n_positions, dtype=torch.float32), inv_freq)
        for name, t in (("engine.rope_cos", freqs.cos()), ("engine.rope_sin", freqs.sin())):
            t = t.to(torch.bfloat16).contiguous()
            shape = (C.c_int64 * 2)(*t.shape)
            self._ck(self._lib.sv_engine_load_weight(self._h, name.encode(), C.c_void_p(t.data_ptr()), shape, 2,
                                                     _lib.SV_DTYPE_BF16))

    # -- stages --------------------------------------------------------------------------
    def _dev(self, t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
        return t.to(device=self.device, dtype=dtype, non_blocking=True).contiguous()

    def encode_images(self, pixels: torch.Tensor, return_embeds: bool = False, return_vit: bool = False):
        """ViT + adapter. pixels [B,3,S,S] (any float dtype/device) -> resident visual prefix."""
        d = self.dims
        if pixels.dim() != 4 or tuple(pixels.shape[1:]) != (3, d.image_size, d.image_size):
            raise ValueError(f"image batch must be [B,3,{d.image_size},{d.image_size}], got {tuple(pixels.shape)}")
        px = self._dev(pixels, torch.bfloat16)
        B = px.shape[0]
        emb = torch.empty(B, d.query_length, d.hidden, dtype=torch.bfloat16, device=self.device) if return_embeds else None
        vit = torch.empty(B, d.query_length, d.vit_width, dtype=torch.bfloat16, device=self.device) if return_vit else None
        with self._lock:
            self._ck(self._lib.sv_encode_images(
                self._h, C.c_void_p(px.data_ptr()), B, C.c_void_p(emb.data_ptr() if emb is not None else 0),
                C.c_void_p(vit.data_ptr() if vit is not None else 0), _stream_ptr(self.device)))
            self._batch = B
        return emb, vit

    def prefill(self, prompt_ids: torch.Tensor, return_logits: bool = False) -> Optional[torch.Tensor]:
        ids = self._dev(prompt_ids, torch.int32)
        if ids.dim() != 2:
            raise ValueError("prompt_ids must be [B,P]")
        B, P = ids.shape
        logits = torch.empty(B, self.dims.vocab, dtype=torch.float32, device=self.device) if return_logits else None
        with self._lock:
            self._ck(self._lib.sv_prefill(self._h, C.c_void_p(ids.data_ptr()), B, P,
                                          C.c_void_p(logits.data_ptr() if logits is not None else 0),
                                          _stream_ptr(self.device)))
            self._prompt_len = P
            self._prefix_len = self.query_length + P
        return logits

    def prefill_embeds(self, inputs_embeds: torch.Tensor, return_logits: bool = False) -> Optional[torch.Tensor]:
        x = self._dev(inputs_embeds, torch.bfloat16)
        if x.dim() != 3 or x.shape[2] != self.dims.hidden:
            raise ValueError("inputs_embeds must be [B,T,hidden]")
        B, T, _ = x.shape
        logits = torch.empty(B, self.dims.vocab, dtype=torch.float32, device=self.device) if return_logits else None
        with self._lock:
            self._ck(self._lib.sv_prefill_embeds(self._h, C.c_void_p(x.data_ptr()), B, T,
                                                 C.c_void_p(logits.data_ptr() if logits is not None else 0),
                                                 _stream_ptr(self.device)))
            self._batch = B
            self._prefix_len = T
        return logits

    def decode_step(self, ids: torch.Tensor, return_logits: bool = True) -> Optional[torch.Tensor]:
        t = self._dev(ids, torch.int32).reshape(-1)
        if t.numel() != self._batch:
            raise ValueError("ids must have one entry per image of the current batch")
        logits = torch.empty(self._batch, self.dims.vocab, dtype=torch.float32, device=self.device) if return_logits else None
        with self._lock:
            self._ck(self._lib.sv_decode_step(self._h, C.c_void_p(t.data_ptr()),
                                              C.c_void_p(logits.data_ptr() if logits is not None else 0),
                                              _stream_ptr(self.device)))
        return logits

    def extend(self, ids: torch.Tensor, keep_logits: int = 0, logps: bool = True,
               temperature: float = 1.0) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """`sv_extend`: teacher-force ids `[B, T]` after the cached sequence of every row (after a prefill, `expand_batch`,
        `decode_step` or another `extend`).  Returns `(logits, logps)`: fp32 logits `[B, keep_logits, V]` of the last
        `keep_logits` new positions (None when 0) and fp32 `[B, T]` log-probs `log_softmax(L / temperature)[ids]`, where
        position t is scored by the logits that predict it (t = 0: the logits held before the call); None unless `logps`."""
        t = self._dev(ids, torch.int32)
        if t.dim() != 2 or t.shape[0] != self._batch:
            raise ValueError(f"ids must be [B, T] with B = {self._batch} rows of the current batch")
        B, T = t.shape
        keep = int(keep_logits)
        lg = torch.empty(B, keep, self.dims.vocab, dtype=torch.float32, device=self.device) if keep > 0 else None
        lp = torch.empty(B, T, dtype=torch.float32, device=self.device) if logps else None
        with self._lock:
            self._ck(self._lib.sv_extend(self._h, C.c_void_p(t.data_ptr()), T, _p(lg), keep, _p(lp), float(temperature),
                                         _stream_ptr(self.device)))
        return lg, lp

    def reorder_cache(self, src_rows: torch.Tensor) -> None:
        """KV-cache row permutation for beam search: row r <- row src_rows[r]."""
        idx = self._dev(src_rows, torch.int32).reshape(-1)
        if idx.numel() != self._batch:
            raise ValueError("src_rows must have one entry per cache row")
        with self._lock:
            self._ck(self._lib.sv_reorder_cache(self._h, C.c_void_p(idx.data_ptr()), _stream_ptr(self.device)))

    def beam_search_device(self, batch: int, *, num_beams: int, max_new_tokens: int, do_sample: bool = False,
                           temperature: float = 1.0, top_p: float = 1.0, repetition_penalty: float = 1.0,
                           length_penalty: float = 1.0, early_stopping=True, eos_token_id: Optional[int] = 0,
                           pad_token_id: int = 0, stop_ids: Sequence[int] = (), seed: int = 0,
                           poll_interval: int = 16) -> torch.Tensor:
        """`sv_beam_search`: the whole beam search / beam-sample on the device, after a prefill of batch * num_beams rows
        (every image repeated num_beams times, adjacent).  Returns int32 `[batch, n_generated]`, the best hypothesis per image.
        Raises NotImplementedError when the vocabulary does not fit the candidate kernel (use the host-stepped loop)."""
        if len(stop_ids) > 8:
            raise ValueError("stop sequence longer than 8 tokens")
        bp = _lib.BeamParams()
        bp.num_beams, bp.max_new_tokens, bp.do_sample = int(num_beams), int(max_new_tokens), int(bool(do_sample))
        bp.early_stopping = 2 if early_stopping == "never" else int(early_stopping is True)
        bp.temperature, bp.top_p = float(temperature), float(top_p)
        bp.repetition_penalty, bp.length_penalty = float(repetition_penalty), float(length_penalty)
        bp.eos_token_id = -1 if eos_token_id is None else int(eos_token_id)
        bp.pad_token_id = int(pad_token_id)
        bp.n_stop_ids = len(stop_ids)
        for i, t in enumerate(stop_ids):
            bp.stop_ids[i] = int(t)
        bp.poll_interval = int(poll_interval)
        bp.seed = int(seed) & (2 ** 64 - 1)
        out = torch.empty(batch, max(int(max_new_tokens), 1), dtype=torch.int32, device=self.device)
        olen = torch.empty(batch, dtype=torch.int32, device=self.device)
        with self._lock:
            self._ck(self._lib.sv_beam_search(self._h, C.byref(bp), int(batch), C.c_void_p(out.data_ptr()),
                                              C.c_void_p(olen.data_ptr()), _stream_ptr(self.device)))
        return out[:, : int(olen[0].item())]

    def expand_batch(self, src_rows) -> None:
        """Prefix-KV sharing: right after a prefill, row r of the new batch becomes a copy of prefilled row src_rows[r]."""
        rows = [int(r) for r in src_rows]
        arr = (C.c_int32 * len(rows))(*rows)
        with self._lock:
            self._ck(self._lib.sv_expand_batch(self._h, arr, len(rows), _stream_ptr(self.device)))
        self._batch = len(rows)

    def generate(self, params: GenerationParams, on_tokens=None) -> torch.Tensor:
        """Run the decode loop after a prefill. Returns int32 [B, n_generated] (new tokens only).

        `on_tokens(ids, first_step)` (optional) streams: it is called on this thread every `params.poll_interval` steps and
        once at the end with a CPU int32 tensor `[B, n]` of the tokens generated since the previous call (`sv_generate_stream`);
        returning a truthy value cancels the generation.  An exception raised by the callback cancels and is re-raised."""
        B, n = self._batch, int(params.max_new_tokens)
        out = torch.empty(B, max(n, 1), dtype=torch.int32, device=self.device)
        olen = torch.empty(B, dtype=torch.int32, device=self.device)
        cp = params.to_c()
        if on_tokens is None:
            with self._lock:
                self._ck(self._lib.sv_generate(self._h, C.byref(cp), C.c_void_p(out.data_ptr()), C.c_void_p(olen.data_ptr()),
                                               _stream_ptr(self.device)))
        else:
            failure = []

            def trampoline(_user, ids_ptr, batch, first_step, n_steps):
                try:
                    flat = torch.frombuffer(C.cast(ids_ptr, C.POINTER(C.c_int32 * (batch * n_steps))).contents, dtype=torch.int32)
                    return 1 if on_tokens(flat.view(batch, n_steps).clone(), int(first_step)) else 0
                except BaseException as exc:      # never let an exception unwind through the C frames
                    failure.append(exc)
                    return 1

            cb = _lib.TOKEN_CALLBACK(trampoline)
            with self._lock:
                self._ck(self._lib.sv_generate_stream(self._h, C.byref(cp), C.c_void_p(out.data_ptr()), C.c_void_p(olen.data_ptr()),
                                                      cb, None, _stream_ptr(self.device)))
            if failure:
                raise failure[0]
        n_gen = int(olen[0].item())
        return out[:, :n_gen]

    def generate_im2svg_host(self, pixels_host: torch.Tensor, prompt_ids_host: torch.Tensor,
                             params: GenerationParams) -> Tuple[torch.Tensor, int]:
        """Whole path on HOST buffers (pinned CPU tensors in, CPU tensors out): the e2e entry point."""
        d = self.dims
        if pixels_host.is_cuda or prompt_ids_host.is_cuda:
            raise ValueError("host entry point takes CPU tensors")
        px = pixels_host.to(torch.bfloat16).contiguous()
        ids = prompt_ids_host.to(torch.int32).contiguous()
        B, P = ids.shape
        out = torch.empty(B, int(params.max_new_tokens), dtype=torch.int32).pin_memory()
        olen = torch.empty(B, dtype=torch.int32).pin_memory()
        cp = params.to_c()
        with self._lock:
            self._ck(self._lib.sv_generate_im2svg_host(
                self._h, C.c_void_p(px.data_ptr()), B, C.c_void_p(ids.data_ptr()), P, C.byref(cp),
                C.c_void_p(out.data_ptr()), C.c_void_p(olen.data_ptr()), _stream_ptr(self.device)))
            self._batch = B
        n_gen = int(olen[0])
        return out[:, :n_gen], n_gen

    # -- introspection -------------------------------------------------------------------
    def launch_count(self) -> int:
        return int(self._lib.sv_launch_count(self._h))

    def describe(self) -> str:
        return self._lib.sv_engine_describe(self._h).decode()

    def debug_timeline(self, n: int = 1024, raw: bool = False):
        buf = (C.c_longlong * n)()
        self._ck(self._lib.sv_debug_read_timeline(self._h, buf, n))
        return [int(v) for v in buf] if raw else [int(v) for v in buf if v]

    def last_decode_timing(self) -> Tuple[float, int]:
        ms, steps = C.c_float(), C.c_int32()
        self._ck(self._lib.sv_last_decode_timing(self._h, C.byref(ms), C.byref(steps)))
        return float(ms.value), int(steps.value)


# -- single-kernel entry points (unit parity tests) --------------------------------------------
def _p(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(t.data_ptr() if t is not None else 0)


def op_layernorm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    lib = _lib.load()
    y = torch.empty_like(x)
    rows = x.numel() // x.shape[-1]
    _lib.check(lib, lib.sv_op_layernorm(_p(x), _p(w), _p(b), _p(y), rows, x.shape[-1], eps, _stream_ptr(x.device)))
    return y


def op_linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None,
              residual: Optional[torch.Tensor] = None, act: int = 0, impl: int = 0) -> torch.Tensor:
    lib = _lib.load()
    M, K = x.shape
    N = w.shape[0]
    y = torch.empty(M, N, dtype=torch.bfloat16, device=x.device)
    _lib.check(lib, lib.sv_op_linear(impl, _p(x), _p(w), _p(bias), _p(residual), _p(y), M, N, K, act, _stream_ptr(x.device)))
    return y


def op_attention_vit(qkv: torch.Tensor, batch: int, seq: int, heads: int) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(batch * seq, heads * 64, dtype=torch.bfloat16, device=qkv.device)
    _lib.check(lib, lib.sv_op_attention_vit(_p(qkv), _p(out), batch, seq, heads, _stream_ptr(qkv.device)))
    return out


def op_attention_mqa(qkv: torch.Tensor, batch: int, seq: int, heads: int) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(batch * seq, heads * 128, dtype=torch.bfloat16, device=qkv.device)
    _lib.check(lib, lib.sv_op_attention_mqa(_p(qkv), _p(out), batch, seq, heads, _stream_ptr(qkv.device)))
    return out


def op_attention_prefill(qkv: torch.Tensor, batch: int, seq: int, n_head: int, n_kv: int, window: int = 0) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(batch * seq, n_head * 128, dtype=torch.bfloat16, device=qkv.device)
    _lib.check(lib, lib.sv_op_attention_prefill(_p(qkv), _p(out), batch, seq, n_head, n_kv, window, _stream_ptr(qkv.device)))
    return out


def op_attention_decode(q: torch.Tensor, kcache: torch.Tensor, vtcache: torch.Tensor, nkeys: int, window: int = 0,
                        impl: int = _lib.SV_ATTN_DECODE_CLUSTER, nparts: int = 0) -> torch.Tensor:
    """q [B, n_head*128], kcache [B, n_kv, tcap, 128], vtcache [B, n_kv, 128, tcap] -> [B, n_head*128]."""
    lib = _lib.load()
    B, n_kv, tcap, _ = kcache.shape
    out = torch.empty_like(q)
    _lib.check(lib, lib.sv_op_attention_decode(impl, _p(q), _p(kcache), _p(vtcache), _p(out), B, q.shape[1] // 128, n_kv,
                                               tcap, nkeys, window, nparts, _stream_ptr(q.device)))
    return out


def op_gemv_ring(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None,
                 residual: Optional[torch.Tensor] = None, ln: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                 act: int = 0, ln_eps: float = 1e-5, tiled: bool = False, out: Optional[torch.Tensor] = None,
                 epi: int = _lib.SV_GEMV_EPI_PLAIN, kcache: Optional[torch.Tensor] = None,
                 vtcache: Optional[torch.Tensor] = None, n_head: int = 0, pos: int = 0):
    """One weight-ring decode GEMV.  `out` may alias `residual` (in-place residual).  Returns y, or for the lm_head
    epilogue (y, amax_val [ntiles, 8], amax_idx [ntiles, 8])."""
    lib = _lib.load()
    B, K = x.shape
    N = w.shape[0]
    y = torch.empty(B, N, dtype=torch.bfloat16, device=x.device) if out is None else out
    cap = N if epi == _lib.SV_GEMV_EPI_LMHEAD else 0
    aval = torch.empty(cap, 8, dtype=torch.float32, device=x.device) if cap else None
    aidx = torch.empty(cap, 8, dtype=torch.int32, device=x.device) if cap else None
    n_kv, tcap = (kcache.shape[1], kcache.shape[2]) if kcache is not None else (0, 0)
    ntiles = C.c_int32(0)
    lw, lb = ln if ln is not None else (None, None)
    _lib.check(lib, lib.sv_op_gemv_ring(_p(x), _p(w), _p(bias), _p(residual), _p(lw), _p(lb), _p(y), B, N, K, act, ln_eps, epi,
                                        int(tiled), _p(kcache), _p(vtcache), n_head, n_kv, tcap, pos, _p(aval), _p(aidx), cap,
                                        C.byref(ntiles), _stream_ptr(x.device)))
    if epi == _lib.SV_GEMV_EPI_LMHEAD:
        return y, aval[: ntiles.value], aidx[: ntiles.value]
    return y


def op_lm_head_logps(x: torch.Tensor, w: torch.Tensor, ids: torch.Tensor, temperature: float = 1.0,
                     return_logits: bool = False):
    """The scoring lm_head: x bf16 [M,K], w bf16 [N,K], ids int [M] -> fp32 logps [M] = log_softmax(bf16(x.w^T) / T)[ids]
    (NaN where an id is outside [0,N)); with `return_logits` also the fp32 [M,N] bf16-rounded logits."""
    lib = _lib.load()
    M, K = x.shape
    N = w.shape[0]
    tid = ids.to(device=x.device, dtype=torch.int32).contiguous()
    lp = torch.empty(M, dtype=torch.float32, device=x.device)
    lg = torch.empty(M, N, dtype=torch.float32, device=x.device) if return_logits else None
    _lib.check(lib, lib.sv_op_lm_head_logps(_p(x), _p(w), _p(tid), _p(lp), _p(lg), M, N, K, float(temperature),
                                            _stream_ptr(x.device)))
    return (lp, lg) if return_logits else lp


def op_select(mode: int, logits: torch.Tensor, seen: torch.Tensor, params: GenerationParams, step: int = 0,
              cur_len: int = 0, partials: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
              wte: Optional[torch.Tensor] = None, wpe: Optional[torch.Tensor] = None):
    """One token-selection kernel on bf16 logits [B,V] and a uint8 seen bitmap [B,V].  Returns the tokens int32 [B], and for
    the fused kernels also the embedding rows [B,h] it writes."""
    lib = _lib.load()
    B, V = logits.shape
    tok = torch.empty(B, dtype=torch.int32, device=logits.device)
    fused = mode in (_lib.SV_SELECT_FUSED, _lib.SV_SELECT_FUSED_PARTIALS)
    h = wte.shape[1] if wte is not None else 0
    x = torch.empty(B, h, dtype=torch.bfloat16, device=logits.device) if fused else None
    aval, aidx = partials if partials is not None else (None, None)
    cp = params.to_c()
    _lib.check(lib, lib.sv_op_select(mode, _p(logits), _p(seen), C.byref(cp), B, V, step, cur_len, _p(aval), _p(aidx),
                                     aval.shape[0] if aval is not None else 0, _p(wte), _p(wpe), h,
                                     wpe.shape[0] if wpe is not None else 0, _p(x), _p(tok), _stream_ptr(logits.device)))
    return (tok, x) if fused else tok
