"""CPU tests of the FLAVA encoder path: the oracle pinned to the reference goldens, and the drop-in parameter
containers (state-dict keys / seeded init) pinned through the parameter checksum the fixture generator recorded from
the REFERENCE model."""
import os

import pytest
import torch

import flava_cases as FC
from oracle import flava_oracle as FO

GOLD = os.path.join(os.path.dirname(__file__), "golden", "flava_golden.pt")


@pytest.fixture(scope="module")
def flava_golden():
    return torch.load(GOLD)


@pytest.mark.parametrize("name", list(FC.CASES))
def test_flava_oracle_and_init_mirror_match_reference_golden(flava_golden, name):
    from multimodal_b200.models.flava import flava_model

    g = flava_golden[name]
    m = FC.build(flava_model, name)
    # same parameter set, same creation order, same RNG consumption as the reference builder
    assert FC.param_checksum(m) == pytest.approx(g["param_checksum"], rel=1e-12)
    inp = FC.inputs(name)
    for k, v in g["inputs"].items():
        assert torch.equal(inp[k], v)
    out = FO.flava_forward(m.state_dict(), FC.CASES[name]["kwargs"], inp["image"], inp["text"],
                           inp["image_patches_mask"], inp["text_masked"], skip_unmasked_mm_encoder=False)
    assert set(out) == set(g["outputs"])
    for k, ref in g["outputs"].items():
        assert torch.allclose(FC.golden_view(out[k]), ref, rtol=1e-5, atol=1e-5), k


def test_flava_state_dict_keys_follow_reference_layout():
    from multimodal_b200.models.flava import flava_model

    m = FC.build(flava_model, "flava_small")
    keys = set(m.state_dict())
    for k in ("image_encoder.embeddings.cls_token", "image_encoder.embeddings.mask_token",
              "image_encoder.embeddings.patch_embeddings.projection.weight",
              "image_encoder.encoder.layer.1.attention.query.weight", "image_encoder.encoder.layer.0.attention.output.bias",
              "image_encoder.encoder.layer.0.feedforward.model.0.weight", "image_encoder.encoder.layer.0.feedforward.model.2.bias",
              "image_encoder.encoder.layer.0.attention_layernorm.weight", "image_encoder.encoder.layer.0.feedforward_layernorm.bias",
              "image_encoder.layernorm.weight", "image_encoder.pooler.dense.weight",
              "text_encoder.embeddings.word_embeddings.weight", "text_encoder.embeddings.position_embeddings.weight",
              "text_encoder.embeddings.token_type_embeddings.weight", "text_encoder.embeddings.layer_norm.weight",
              "mm_encoder.cls_token", "mm_encoder.encoder.layer.0.attention.key.weight",
              "image_to_mm_projection.weight", "text_to_mm_projection.bias", "text_projection.weight", "image_projection.bias"):
        assert k in keys, k


def test_flava_modules_refuse_cpu_execution():
    """No CPU fallback: the encoders fail loudly when asked to run off-GPU."""
    from multimodal_b200._lib import MMBError
    from multimodal_b200.models.flava import flava_model

    m = FC.build(flava_model, "flava_small")
    inp = FC.inputs("flava_small")
    with pytest.raises(MMBError):
        m(image=inp["image"], text=inp["text"])
    with pytest.raises(ValueError):
        m.image_encoder(None)
    with pytest.raises(ValueError):
        m.text_encoder()


def test_flava_text_oracle_reproduces_reference_known_answers():
    """tests/models/flava/test_text_encoder.py:26-125 of the reference: 2-d BERT encoder built under seed 0 from the
    drop-in containers (same RNG consumption as the reference's) + fixed embedding tables; hidden states with and without
    an explicit attention mask."""
    from functools import partial

    from torch import nn

    from multimodal_b200.models.flava.transformer import init_transformer_weights, TransformerEncoder
    from multimodal_b200.modules.encoders.bert_text_encoder import BERTTextEncoder
    from multimodal_b200.modules.layers.text_embedding import BERTTextEmbeddings

    torch.manual_seed(0)
    emb_w = torch.Tensor([[0, 1], [1, 0], [1, 1]])
    emb = BERTTextEmbeddings(hidden_size=2, vocab_size=3, max_position_embeddings=2, dropout=0)
    emb.word_embeddings = nn.Embedding.from_pretrained(emb_w)
    emb.position_embeddings = nn.Embedding.from_pretrained(emb_w)
    emb.token_type_embeddings = nn.Embedding.from_pretrained(emb_w)
    enc = TransformerEncoder(n_layer=1, d_model=2, n_head=1, dim_feedforward=1, activation=nn.GELU, norm_first=True)
    m = BERTTextEncoder(embeddings=emb, encoder=enc, layernorm=nn.LayerNorm(2), pooler=nn.Identity(),
                        weight_init_fn=partial(init_transformer_weights, initializer_range=0.02))
    sd = {"text_encoder." + k: v for k, v in m.state_dict().items()}
    cfg = dict(text_num_hidden_layers=1, text_num_attention_heads=1, pad_token_id=0, text_layer_norm_eps=1e-12)
    # the test's final LayerNorm is nn.LayerNorm(2) (eps 1e-5); the oracle applies one eps to all: irrelevant at 1e-4
    ids = torch.tensor([[0, 1]])
    out = FO.text_encoder(ids, sd, cfg)      # test_text_transformer: default mask = ids != pad (token 0 is the pad id)
    assert torch.allclose(out["hidden_states"][0], torch.Tensor([[[1.0, -1.0], [-1.0, 1.0]]]), atol=1e-4)
    assert torch.allclose(out["hidden_states"][1], torch.Tensor([[[1.0008, -0.9994], [-0.9997, 1.0012]]]), atol=1e-4)
    assert torch.allclose(out["last_hidden_state"], torch.Tensor([[[1.0, -1.0], [-1.0, 1.0]]]), atol=1e-3)
    out = FO.text_encoder(ids, sd, cfg, attention_mask=torch.tensor([[1, 0]]))   # test_text_transformer_attn_mask
    assert torch.allclose(out["hidden_states"][1], torch.Tensor([[[0.9997, -1.0012], [-1.0008, 0.9994]]]), atol=1e-4)


def test_flava_image_oracle_reproduces_reference_known_answers():
    """tests/models/flava/test_image_encoder.py:20-130 of the reference: 1x1-patch, 2-d image transformer built under
    seed 0 from the drop-in containers; embeddings and final hidden state for an all-ones image."""
    from torch import nn

    from multimodal_b200.models.flava.image_encoder import ImageEmbeddings, ImageTransformer
    from multimodal_b200.models.flava.transformer import TransformerEncoder

    torch.manual_seed(0)
    emb = ImageEmbeddings(image_size=2, patch_size=1, hidden_size=2)
    enc = TransformerEncoder(n_layer=1, d_model=2, n_head=1, dim_feedforward=1, activation=nn.GELU, norm_first=True)
    m = ImageTransformer(embeddings=emb, encoder=enc, layernorm=nn.LayerNorm(2), pooler=nn.Identity())
    sd = {"image_encoder." + k: v for k, v in m.state_dict().items()}
    cfg = dict(patch_size=1, image_num_hidden_layers=1, image_num_attention_heads=1, image_layer_norm_eps=1e-12,
               image_final_layer_norm_eps=1e-5)   # the test passes a plain nn.LayerNorm(2) as the final layernorm
    out = FO.image_encoder(torch.ones(2, 3, 2, 2), sd, cfg)
    e = torch.Tensor([[0.0, 0.0]] + [[0.0224, 0.0573]] * 4)
    assert torch.allclose(out["hidden_states"][0], e.expand(2, 5, 2), atol=1e-4)
    last = torch.Tensor([[-0.0040, 0.0040]] + [[-0.9840, 0.9840]] * 4)
    assert torch.allclose(out["last_hidden_state"], last.expand(2, 5, 2), atol=1e-4)
