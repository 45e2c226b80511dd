"""Pin the CPU oracle (oracle/) against fixtures produced by the reference's own modules.

tests/golden/tiny_v1_*.pt were written by `python -m oracle.make_golden` and
`python -m oracle.make_golden_reference`, which run VisionTransformer / LayerNorm / Adapter of the
reference checkout and drive the installed transformers GPTBigCode through generate().  The oracle
restatement must reproduce them: within 2 bf16 ulps of the fixtures taken with oneDNN on, and bit for
bit with oneDNN off on both sides.
"""
import os

import pytest
import torch

from oracle.pipeline import OracleStarVector
from starvector_b200.config import ModelDims
from starvector_b200.weights import synthetic_images, synthetic_state_dict


def _load(golden_dir, norm):
    g = torch.load(os.path.join(golden_dir, f"tiny_v1_{norm}.pt"), weights_only=False)
    d = ModelDims(**g["dims"])
    sd = synthetic_state_dict(d, seed=g["seed"], init=g["init"])
    img = synthetic_images(d, 2, seed=g["image_seed"])
    return g, d, sd, img


def _ulp_close(a, b, ulps=2):
    a, b = a.float(), b.float()
    tol = ulps * 2.0 ** -8 * torch.maximum(a.abs(), b.abs()) + 1e-6
    return bool(((a - b).abs() <= tol).all())


@pytest.mark.parametrize("norm", ["layer_norm", "batch_norm"])
def test_vision_restatement_matches_reference_fixture(golden_dir, norm):
    torch.set_num_threads(1)
    g, d, sd, img = _load(golden_dir, norm)
    o = OracleStarVector(d, sd, dtype=torch.bfloat16, pad_token_id=d.vocab - 4)
    vit = o.image_encoder(img)
    assert _ulp_close(vit, g["vit_out"]), "ViT restatement drifted from the reference module output"
    assert _ulp_close(o.image_projection(vit), g["adapter_out"], ulps=3)


def test_generate_restatement_matches_fixture(golden_dir):
    torch.set_num_threads(1)
    g, d, sd, img = _load(golden_dir, "layer_norm")
    o = OracleStarVector(d, sd, dtype=torch.float32, pad_token_id=d.vocab - 4)
    n_new = g["greedy_ids_fp32"].shape[1] - len(g["prompt_ids"])
    ids = o.generate_im2svg_ids(img, g["prompt_ids"], g["stop_ids"], use_nucleus_sampling=False, num_beams=1,
                                max_length=d.query_length + len(g["prompt_ids"]) + n_new)
    assert torch.equal(ids, g["greedy_ids_fp32"])
    tf = o.teacher_forced_logits(img, g["prompt_ids"], g["forced_ids"])
    torch.testing.assert_close(tf, g["tf_logits_fp32"], rtol=1e-4, atol=1e-4)


def test_hf_length_arithmetic(golden_dir):
    """D5: new tokens = max_length - (Q + P) (generation/utils.py:1629-1638)."""
    g, d, sd, img = _load(golden_dir, "layer_norm")
    o = OracleStarVector(d, sd, dtype=torch.float32, pad_token_id=d.vocab - 4, eos_token_id=None)
    ids = o.generate_im2svg_ids(img[:1], g["prompt_ids"], (), use_nucleus_sampling=False, num_beams=1,
                                max_length=d.query_length + 2 + 5)
    assert ids.shape == (1, 2 + 5)


def test_row0_stop_stops_whole_batch(golden_dir):
    """D6: StoppingCriteriaSub looks at row 0 only and ends the batch (starvector_base.py:15-20)."""
    g, d, sd, img = _load(golden_dir, "layer_norm")
    o = OracleStarVector(d, sd, dtype=torch.float32, pad_token_id=d.vocab - 4, eos_token_id=None)
    base = o.generate_im2svg_ids(img, g["prompt_ids"], (), use_nucleus_sampling=False, num_beams=1,
                                 max_length=d.query_length + 2 + 12)
    stop = base[0, 2 + 3: 2 + 6].tolist()            # tokens 3..5 of row 0 become the stop sequence
    out = o.generate_im2svg_ids(img, g["prompt_ids"], stop, use_nucleus_sampling=False, num_beams=1,
                                max_length=d.query_length + 2 + 12)
    first = next(i for i in range(2, base.shape[1] - 2) if base[0, i:i + 3].tolist() == stop)
    assert out.shape[1] == first + 3 and torch.equal(out, base[:, : first + 3])


@pytest.mark.parametrize("norm", ["layer_norm", "batch_norm"])
def test_restatement_bit_exact_vs_reference_outputs(golden_dir, norm):
    """Same operations in the same order as the reference modules: equal bits.  oneDNN stays off on both sides because its AMX
    and AVX kernels round bf16 matmuls differently (oracle/make_golden_reference.py)."""
    torch.set_num_threads(1)
    g, d, sd, img = _load(golden_dir, norm)
    ref = torch.load(os.path.join(golden_dir, "tiny_v1_reference_vision.pt"), weights_only=False)[norm]
    o = OracleStarVector(d, sd, dtype=torch.bfloat16, pad_token_id=d.vocab - 4)
    with torch.no_grad(), torch.backends.mkldnn.flags(enabled=False):
        assert torch.equal(o.image_encoder(img), ref["vit_out"])
        assert torch.equal(o.image_projection(ref["vit_out"]), ref["adapter_out"])


def test_v2_oracle_matches_fixture(golden_dir):
    """v2 family (SigLIP + StarCoder2 from the installed transformers, reference Adapter): regression pin."""
    from oracle.pipeline import OracleStarVectorV2

    torch.set_num_threads(1)
    g = torch.load(os.path.join(golden_dir, "tiny_v2_layer_norm.pt"), weights_only=False)
    d = ModelDims(**g["dims"])
    sd = synthetic_state_dict(d, seed=g["seed"], init=g["init"])
    img = synthetic_images(d, 2, seed=g["image_seed"])
    o = OracleStarVectorV2(d, sd, dtype=torch.float32)
    vit = o.image_encoder(img.float())
    torch.testing.assert_close(vit, g["vit_out_fp32"], rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(o.image_projection(vit), g["adapter_out_fp32"], rtol=1e-4, atol=1e-4)   # restated vs reference Adapter
    n_new = g["greedy_ids_fp32"].shape[1] - 2
    ids = o.generate_im2svg_ids(img, g["prompt_ids"], g["stop_ids"], use_nucleus_sampling=False, num_beams=1,
                                max_length=d.query_length + 2 + n_new)
    assert torch.equal(ids, g["greedy_ids_fp32"])
