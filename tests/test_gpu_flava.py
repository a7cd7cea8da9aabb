"""GPU parity of the FLAVA encoders' forward (BASELINE.json config 3) against the reference goldens and the oracle.

Tolerance: GEMM operands are rounded to bf16 (fp32 accumulate / residual stream / LayerNorm / softmax statistics), so
every compared tensor must agree with the fp32 reference to 2e-2 of that tensor's absmax and with cosine > 0.9995
(measured: ~3e-3 / 0.99999).  Masks, ids and gathers are bit-exact.
"""
import math
import os

import pytest
import torch

import flava_cases as FC
from oracle import flava_oracle as FO

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "flava_golden.pt")


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(autouse=True)
def _inference():
    """This file pins the INFERENCE runtime (engine_flava.py); with grad mode on, trainable modules take the training
    runtime instead (engine_flava_train.py, covered by tests/test_gpu_flava_train.py)."""
    with torch.no_grad():
        yield


def _close(got, ref, name, tol=2e-2):
    got, ref = got.float().cpu(), ref.float().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert torch.isfinite(got).all(), name
    err = (got - ref).abs().max().item() / max(ref.abs().max().item(), 1e-20)
    cos = torch.nn.functional.cosine_similarity(got.flatten(), ref.flatten(), dim=0).item()
    assert err < tol and cos > 0.9995, (name, err, cos)
    return err


def test_flava_helper_kernels(dev):
    from multimodal_b200 import ops

    torch.manual_seed(0)
    B, S, d, V = 5, 13, 256, 50
    ids = torch.randint(0, V, (B, S), device=dev)
    ids[1, 9:] = 3
    tt = torch.randint(0, 2, (B, S), device=dev)
    word, pos, typ = torch.randn(V, d, device=dev), torch.randn(32, d, device=dev), torch.randn(2, d, device=dev)
    gam, bet = torch.randn(d, device=dev), torch.randn(d, device=dev)
    x = torch.empty(B * S, d, device=dev)
    km = torch.empty(B * S, dtype=torch.uint8, device=dev)
    ops.bert_embed_ln_fwd(ids, tt, word, pos, typ, gam, bet, x, km, 3, B, S, d, V, 1e-12)
    ref = torch.nn.functional.layer_norm(word[ids] + pos[:S][None] + typ[tt], (d,), gam, bet, 1e-12)
    assert torch.allclose(x.view(B, S, d), ref, rtol=1e-4, atol=1e-4)
    assert torch.equal(km.view(B, S), (ids != 3).to(torch.uint8))
    # image token assembly with mask-token substitution
    P = S - 1
    po = torch.randn(B * P, d, device=dev).bfloat16()
    cls, posi, mt = torch.randn(1, 1, d, device=dev), torch.randn(1, S, d, device=dev), torch.randn(1, 1, d, device=dev)
    pm = (torch.rand(B, P, device=dev) < 0.5)
    xo = torch.empty(B * S, d, device=dev)
    ops.vit_assemble_fwd(po, cls, posi, mt, pm.to(torch.uint8), xo, B, S, d)
    e = torch.where(pm[..., None], mt.expand(B, P, d), po.float().view(B, P, d))
    assert torch.equal(xo.view(B, S, d), torch.cat([cls.expand(B, 1, d), e], 1) + posi)
    # concat / gather / tanh
    a, b = torch.randn(B, 4, d, device=dev), torch.randn(B, 6, d, device=dev)
    out = torch.empty(B * 11, d, device=dev)
    ops.concat_tokens(cls, a, b, out, B, 4, 6, d)
    assert torch.equal(out.view(B, 11, d), torch.cat([cls.expand(B, 1, d), a, b], 1))
    gb = torch.empty(B, d, device=dev, dtype=torch.bfloat16)
    ops.gather_rows_cast(out, gb, B, 11, 2, d)
    assert torch.equal(gb, out.view(B, 11, d)[:, 2].bfloat16())
    t = torch.randn(B, d, device=dev)
    r = torch.tanh(t)
    ops.tanh_(t)
    assert torch.allclose(t, r, atol=1e-6)


@pytest.mark.parametrize("B,S,H", [(3, 12, 2), (4, 77, 12), (2, 256, 4), (2, 200, 3)])
def test_attention_fwd_key_padding_mask(dev, B, S, H):
    from multimodal_b200 import ops

    torch.manual_seed(1)
    d = 64 * H
    qkv = torch.randn(B * S, 3 * d, device=dev).bfloat16()
    lens = torch.randint(1, S + 1, (B,), device=dev)
    lens[0] = S
    km = (torch.arange(S, device=dev)[None] < lens[:, None])
    km[-1, 0] = False  # a hole that is not right padding
    out = torch.empty(B * S, d, device=dev, dtype=torch.bfloat16)
    ops.attention_fwd_kmask(qkv, out, None, km.to(torch.uint8).contiguous().view(-1), B, S, H, False, 0.125)
    q, k, v = (t.view(B, S, H, 64).transpose(1, 2).float() for t in qkv.view(B, S, 3 * d).split(d, dim=-1))
    s = (q @ k.transpose(-1, -2)) * 0.125
    s = s.masked_fill(~km[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * S, d)
    err = (out.float() - ref).abs().max().item()
    assert err < 2e-2, err  # bf16 P and bf16 output rounding on |o| <~ 3
    # attention probabilities on request (TransformerOutput.attentions): recomputed from QKV + the forward's row LSE
    lse = torch.empty(B * H * S, device=dev)
    kmf = km.to(torch.uint8).contiguous().view(-1)
    ops.attention_fwd_kmask(qkv, out, lse, kmf, B, S, H, False, 0.125)
    probs = torch.empty(B, H, S, S, device=dev)
    ops.attention_probs(qkv, lse, kmf, probs, B, S, H, False, 0.125)
    torch.testing.assert_close(probs, torch.softmax(s, -1), rtol=2e-3, atol=2e-5)   # fp32 dot products, ex2.approx
    assert (probs.sum(-1) - 1).abs().max().item() < 1e-3
    assert probs.masked_select(~km[:, None, None, :].expand_as(probs)).abs().max().item() == 0.0


def test_flava_attentions_on_request(dev):
    """`TransformerOutput.attentions` (always returned by the reference: models/flava/image_encoder.py:220-233) is
    opt-in here: None by default, one [B, H, S, S] tensor per layer after `set_output_attentions()`; the probabilities
    must reproduce the layer's attention output when applied to V, i.e. they ARE what the fused kernel used."""
    from multimodal_b200.models.flava import flava_model

    name = "flava_small"
    g = torch.load(GOLD)[name]
    m = FC.build(flava_model, name).to(dev)
    inp = {k: v.to(dev) for k, v in g["inputs"].items()}
    o = m(image=inp["image"], text=inp["text"])
    assert o.image.attentions is None and o.text.attentions is None
    m.set_output_attentions(True)
    o2 = m(image=inp["image"], text=inp["text"], skip_unmasked_mm_encoder=False)
    for part, out in (("image", o2.image), ("text", o2.text), ("multimodal", o2.multimodal)):
        att = out.attentions
        n_layers = len(out.hidden_states) - 1
        assert att is not None and len(att) == n_layers, part
        B, S = out.last_hidden_state.shape[:2]
        for a in att:
            assert a.shape[0] == B and a.shape[2] == a.shape[3] == S and a.dtype == torch.float32
            rows = a.sum(-1)
            assert torch.isfinite(a).all() and (rows - 1).abs().max().item() < 2e-3, part
    torch.testing.assert_close(o2.image.last_hidden_state, o.image.last_hidden_state)   # asking does not change results


@pytest.mark.parametrize("name", list(FC.CASES))
def test_flava_forward_against_reference_golden(dev, name):
    from multimodal_b200.models.flava import flava_model

    g = torch.load(GOLD)[name]
    m = FC.build(flava_model, name)
    assert FC.param_checksum(m) == pytest.approx(g["param_checksum"], rel=1e-12)
    m = m.to(dev)
    inp = {k: v.to(dev) for k, v in g["inputs"].items()}
    o = m(image=inp["image"], text=inp["text"], image_patches_mask=inp["image_patches_mask"],
          text_masked=inp["text_masked"], skip_unmasked_mm_encoder=False)
    assert o.image.attentions is None
    got = FC.flatten_output(o)
    assert set(got) == set(g["outputs"])
    worst = max(_close(FC.golden_view(got[k]), ref, k) for k, ref in g["outputs"].items())
    print(f"{name}: worst rel-to-absmax error {worst:.2e}")
    # single-modality calls (model.py:136-142 required_embedding defaults)
    oi = m(image=inp["image"])
    assert oi.text.last_hidden_state is None and oi.multimodal_masked.last_hidden_state is None
    _close(FC.golden_view(oi.image.last_hidden_state), g["outputs"]["image.last_hidden_state"], "image-only")
    _close(oi.projected_image_embeddings, g["outputs"]["projected_image_embeddings"], "image-only proj")
    ot = m(text=inp["text"])
    assert ot.image.last_hidden_state is None
    _close(ot.text.pooler_output, g["outputs"]["text.pooler_output"], "text-only pooled")
    # explicit attention mask == the pad-derived default (bert_text_encoder.py:85-90)
    et = m.encode_text(inp["text"], text_mask=(inp["text"] != 0).long())
    _close(FC.golden_view(et.last_hidden_state), g["outputs"]["text.last_hidden_state"], "explicit mask")


def test_flava_base_width_against_oracle(dev):
    """d = 768 / 12 heads (the real FLAVA width) with 2+2+1 layers, 224x224 images: S = 197 / 275 as in config 3."""
    from multimodal_b200.models.flava import flava_model

    kw = dict(image_num_hidden_layers=2, text_num_hidden_layers=2, multimodal_num_hidden_layers=1, vocab_size=1000,
              max_position_embeddings=128)
    torch.manual_seed(0)
    m = flava_model(**kw).eval()
    gen = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(0.02 * torch.randn(p.shape, generator=gen))
    B, St = 2, 77
    image = torch.randn(B, 3, 224, 224, generator=gen)
    text = torch.randint(1, 1000, (B, St), generator=gen)
    text[1, 40:] = 0
    cfg = dict(patch_size=16, image_num_hidden_layers=2, image_num_attention_heads=12, text_num_hidden_layers=2,
               text_num_attention_heads=12, multimodal_num_hidden_layers=1, multimodal_num_attention_heads=12)
    ref = FO.flava_forward(m.state_dict(), cfg, image, text, None, text, skip_unmasked_mm_encoder=True)
    m = m.to(dev)
    o = m(image=image.to(dev), text=text.to(dev), text_masked=text.to(dev))
    got = FC.flatten_output(o)
    for k in ("image.last_hidden_state", "text.last_hidden_state", "multimodal_masked.last_hidden_state",
              "multimodal_masked.pooler_output", "projected_image_embeddings", "projected_text_embeddings",
              "image.hidden_states.2", "text.hidden_states.2"):
        _close(got[k], ref[k], k)
    assert got["multimodal_masked.last_hidden_state"].shape == (B, 1 + 197 + St, 768)
