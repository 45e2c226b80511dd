"""CPU tests of the host side: ABI surface, config/tokenizer/params plumbing, loud failure without a GPU."""
import ctypes as C
import os
import re
import subprocess

import pytest
import torch

from starvector_b200 import _lib
from starvector_b200.config import StarVectorConfig, dims_1b, dims_tiny
from starvector_b200.engine import GenerationParams
from starvector_b200.tokenizer import SyntheticTokenizer
from starvector_b200.weights import synthetic_state_dict, weight_shapes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "starvector_b200.h")).read()
    return set(re.findall(r"SV_API\s+[\w\s\*]+?\b(sv_\w+)\s*\(", text))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _header_symbols()
    assert declared, "no SV_API declarations parsed"
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (sv_\w+)", out))
    assert declared == exported, (declared ^ exported)
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    assert lib.sv_abi_version() == _lib.ABI_VERSION


def test_struct_layout_matches_header():
    assert C.sizeof(_lib.ModelDesc) == 22 * 4
    assert C.sizeof(_lib.GenParams) == 88 and _lib.GenParams.seed.offset == 72


def test_create_rejects_bad_descriptors_without_touching_cuda():
    lib = _lib.load()
    h = C.c_void_p()
    d = _lib.ModelDesc(variant=7)
    assert lib.sv_engine_create(C.byref(d), 0, C.byref(h)) == _lib.SV_ERR_UNSUPPORTED
    d = _lib.ModelDesc(variant=1, rope_theta=0.0)
    assert lib.sv_engine_create(C.byref(d), 0, C.byref(h)) == _lib.SV_ERR_INVALID
    assert b"rope_theta" in lib.sv_last_error(None)
    d = _lib.ModelDesc(vit_width=100, vit_heads=2)
    assert lib.sv_engine_create(C.byref(d), 0, C.byref(h)) == _lib.SV_ERR_INVALID


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_engine_fails_loudly_without_gpu():
    from starvector_b200.engine import Engine

    with pytest.raises(_lib.EngineError, match="no CPU fallback"):
        Engine(dims_tiny())
    lib = _lib.load()
    h = C.c_void_p()
    t = dims_tiny()
    d = _lib.ModelDesc(image_size=t.image_size, patch_size=t.patch_size, vit_width=t.vit_width, vit_layers=1,
                       vit_heads=t.vit_heads, vit_mlp=t.vit_mlp, hidden=t.hidden, n_layer=1, n_head=t.n_head,
                       n_kv_head=1, head_dim=128, n_inner=t.n_inner, n_positions=64, vocab=500, ln_eps=1e-5,
                       max_batch=1, max_len=64)
    assert lib.sv_engine_create(C.byref(d), 0, C.byref(h)) == _lib.SV_ERR_CUDA
    assert b"no CPU fallback" in lib.sv_last_error(None)


def test_1b_dimensions_match_survey():
    d = dims_1b()
    assert d.query_length == 257 and d.patch_k == 588 and d.patch_k_padded == 640
    assert d.decoder_weight_bytes() == 2_240_876_544          # SURVEY.md §8d `W`
    assert d.kv_bytes_per_token() == 12_288
    n = sum(int(torch.tensor(s).prod()) for _, s, _ in weight_shapes(d))
    assert 1.42e9 < n < 1.45e9                                  # ViT 290.6M + adapter ~7.3M(+norm) + decoder 1137M


def test_config_roundtrip_and_dims():
    c = StarVectorConfig()
    d = c.to_dims(max_batch=2, max_len=4096)
    assert (d.hidden, d.n_layer, d.vocab, d.max_len) == (2048, 24, 49156, 4096)
    d8 = StarVectorConfig(starcoder_model_name="bigcode/starcoder2-7b", image_encoder_type="siglip_384", image_size=384,
                          hidden_size=4608, num_attention_heads=36, max_length=16384).to_dims(max_batch=2)
    assert (d8.variant, d8.query_length, d8.hidden, d8.n_kv_head, d8.sliding_window) == (1, 576, 4608, 4, 4096)
    assert d8.decoder_weight_bytes() == 14_347_893_760 and d8.kv_bytes_per_token() == 65_536   # SURVEY.md §8d (8B)
    c2 = StarVectorConfig(**{k: v for k, v in c.to_dict().items() if k not in ("model_type", "_name_or_path")})
    assert c2.hidden_size == c.hidden_size


def test_synthetic_tokenizer_roundtrip():
    t = SyntheticTokenizer(49156)
    assert t("<svg", add_special_tokens=False)["input_ids"] == [44, 5678]
    assert t.pad_token_id == 49152 and t.eos_token_id == 0
    ids = t(["<svg"] * 3, return_tensors="pt")["input_ids"]
    assert ids.shape == (3, 2)
    s = t.batch_decode([[44, 5678, 9, 10, 1245, 7, 29, 0, 49152]])[0]
    assert s == "<svg<t9><t10></svg>" and t.encode(s) == [44, 5678, 9, 10, 1245, 7, 29]


def test_generation_params_to_c():
    p = GenerationParams(max_new_tokens=7, do_sample=True, temperature=0.8, top_p=0.9, repetition_penalty=3.1,
                         eos_token_id=None, pad_token_id=49152, stop_ids=[1, 2, 3], seed=5).to_c()
    assert (p.max_new_tokens, p.do_sample, p.eos_token_id, p.n_stop_ids, list(p.stop_ids)[:3]) == (7, 1, -1, 3, [1, 2, 3])
    with pytest.raises(ValueError):
        GenerationParams(max_new_tokens=1, stop_ids=list(range(9))).to_c()


def test_state_dict_names_follow_reference_tree():
    sd = synthetic_state_dict(dims_tiny(), seed=0)
    assert "model.image_encoder.visual_encoder.transformer.resblocks.0.attn.in_proj_weight" in sd
    assert "model.image_projection.norm.weight" in sd
    assert sd["model.svg_transformer.transformer.lm_head.weight"] is sd["model.svg_transformer.transformer.transformer.wte.weight"]


def test_real_tokenizer_directory_is_prepared_like_the_reference(tmp_path):
    """llm/starcoder.py:40-53: eos/pad added when missing, the three start tokens appended; the facade's calls on it."""
    from tokenizers import Tokenizer, decoders, models, pre_tokenizers, trainers
    from transformers import PreTrainedTokenizerFast

    from starvector_b200.tokenizer import load_tokenizer

    tk = Tokenizer(models.BPE(unk_token="<unk>"))
    tk.pre_tokenizer = pre_tokenizers.ByteLevel(add_prefix_space=False)
    tk.decoder = decoders.ByteLevel()
    corpus = ['<svg xmlns="http://www.w3.org/2000/svg" viewBox="0 0 24 24"><path d="M12 2L2 7l10 5 10-5z"/></svg>'] * 4
    tk.train_from_iterator(corpus, trainers.BpeTrainer(vocab_size=120, special_tokens=["<unk>"]))
    PreTrainedTokenizerFast(tokenizer_object=tk, unk_token="<unk>").save_pretrained(str(tmp_path))
    tok = load_tokenizer(str(tmp_path), vocab_size=500)
    assert not isinstance(tok, SyntheticTokenizer)
    assert tok.eos_token == "[EOS]" and tok.pad_token == "[PAD]" and tok.eos_token_id != tok.pad_token_id
    for t in ("<svg-start>", "<image-start>", "<caption-start>"):
        assert len(tok.encode(t)) == 1
    stop = tok("</svg>", add_special_tokens=False)["input_ids"]                 # starvector_base.py:226
    prompt = tok(["<svg"] * 2, add_special_tokens=False, return_tensors="pt", padding="longest", truncation=True)["input_ids"]
    assert prompt.shape[0] == 2 and 1 <= len(stop) <= 8
    ids = prompt[0].tolist() + tok(' viewBox="0 0 24 24">')["input_ids"] + stop + [tok.eos_token_id, tok.pad_token_id]
    assert tok.batch_decode([ids], skip_special_tokens=True)[0] == '<svg viewBox="0 0 24 24"></svg>'
    assert isinstance(load_tokenizer(None, 500), SyntheticTokenizer)
    assert isinstance(load_tokenizer(str(tmp_path / "missing"), 500), SyntheticTokenizer)


def test_checkpoint_directory_round_trip(tmp_path):
    """write_checkpoint -> read_checkpoint: config fields, every tensor bit for bit, tied lm_head stored once, shards merged."""
    from safetensors.torch import save_file

    from starvector_b200.config import StarVectorConfig, dims_tiny
    from starvector_b200.modeling import read_checkpoint, write_checkpoint
    from starvector_b200.weights import synthetic_state_dict

    d = dims_tiny()
    sd = dict(synthetic_state_dict(d, seed=0, init="randomized"))
    cfg = StarVectorConfig(max_length_train=100, image_size=d.image_size)
    write_checkpoint(str(tmp_path), cfg, sd)
    cfg2, sd2 = read_checkpoint(str(tmp_path))
    assert cfg2.to_dict() == {**cfg.to_dict(), "_name_or_path": str(tmp_path)} or cfg2.max_length_train == 100
    stored = {k for k in sd if not k.endswith("lm_head.weight")}
    assert set(sd2) == stored and all(torch.equal(sd2[k], sd[k]) for k in stored)
    # a second shard is merged in
    save_file({"extra.tensor": torch.arange(4, dtype=torch.float32)}, str(tmp_path / "model-00002.safetensors"))
    assert "extra.tensor" in read_checkpoint(str(tmp_path))[1]
    with pytest.raises(FileNotFoundError):
        read_checkpoint(str(tmp_path / "nowhere"))
    (tmp_path / "empty").mkdir()
    (tmp_path / "empty" / "config.json").write_text((tmp_path / "config.json").read_text())
    with pytest.raises(FileNotFoundError):
        read_checkpoint(str(tmp_path / "empty"))


def test_untied_lm_head_survives_a_checkpoint_round_trip(tmp_path):
    """The reference always re-ties (train/util.py:68-77); the engine also takes an un-tied head, so saving must keep it."""
    from starvector_b200.config import StarVectorConfig
    from starvector_b200.modeling import read_checkpoint, write_checkpoint

    d = dims_tiny()
    sd = dict(synthetic_state_dict(d, seed=0))
    head = "model.svg_transformer.transformer.lm_head.weight"
    write_checkpoint(str(tmp_path / "tied"), StarVectorConfig(), sd)
    assert head not in read_checkpoint(str(tmp_path / "tied"))[1]                 # equal to wte: stored once
    sd[head] = sd[head].clone() + 1.0
    write_checkpoint(str(tmp_path / "untied"), StarVectorConfig(), sd)
    back = read_checkpoint(str(tmp_path / "untied"))[1]
    assert head in back and torch.equal(back[head], sd[head])


def test_decoder_dims_follow_the_checkpoint_tensors():
    """config.json fields that disagree with the tensors (max_length vs wpe rows, another model size) must not break loading."""
    import dataclasses

    from starvector_b200.config import dims_tiny_v2, refine_dims_from_state_dict

    for d in (dims_tiny(), dims_tiny_v2()):
        sd = synthetic_state_dict(d, seed=0)
        wrong = dataclasses.replace(d, n_layer=7, n_inner=64, vocab=123, hidden=128 * 5, n_head=5,
                                    n_positions=999 if d.variant == 0 else d.n_positions)
        assert refine_dims_from_state_dict(wrong, sd) == d


def test_v2_tokenizer_preparation(tmp_path):
    """llm/starcoder2.py:36-53: four added tokens (incl. <svg-end>) and left padding; the synthetic stand-in mirrors both."""
    from tokenizers import Tokenizer, models, pre_tokenizers, trainers
    from transformers import PreTrainedTokenizerFast

    from starvector_b200.tokenizer import load_tokenizer

    tk = Tokenizer(models.BPE(unk_token="<unk>"))
    tk.pre_tokenizer = pre_tokenizers.ByteLevel(add_prefix_space=False)
    tk.train_from_iterator(["<svg></svg>"] * 4, trainers.BpeTrainer(vocab_size=60, special_tokens=["<unk>"]))
    PreTrainedTokenizerFast(tokenizer_object=tk, unk_token="<unk>").save_pretrained(str(tmp_path))
    tok = load_tokenizer(str(tmp_path), vocab_size=500, v2=True)
    assert tok.padding_side == "left"
    for t in ("<svg-start>", "<image-start>", "<caption-start>", "<svg-end>"):
        assert len(tok.encode(t)) == 1
    syn = load_tokenizer(None, 500, v2=True)
    assert isinstance(syn, SyntheticTokenizer) and syn.padding_side == "left" and syn.pad_token_id == 495


def test_bench_dump_outputs_writes_float32_arrays(tmp_path):
    """bench.py --dump-outputs: every array as <name>.npy in float32 with the values unchanged; over 64 MB in all is refused."""
    import numpy as np

    import bench

    ids = torch.tensor([[44, 49151, 0, 16777215]], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "out"), {"ids": ids})
    got = np.load(tmp_path / "out" / "ids.npy")
    assert got.dtype == np.float32 and got.shape == (1, 4) and np.array_equal(got, ids.numpy())
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"ids": torch.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, dtype=torch.int32)})
    assert not (tmp_path / "big").exists()
