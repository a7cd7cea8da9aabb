"""CPU: pins the oracle (oracle/clip_oracle.py) against (1) golden vectors produced by the unmodified reference
(tests/golden/make_golden.py) and (2) the reference's own known-answer tests, and checks that this package's module
constructors reproduce the reference initialisation / state-dict schema."""
import math

import pytest
import torch

import clip_cases as CC
from oracle import clip_oracle as O


def test_oracle_small_forward_and_grads_match_reference_golden(golden):
    g = golden["clip_small"]
    sd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in CC.small_state_dict(g).items()}
    scale = torch.tensor(math.log(1 / 0.07), requires_grad=True)
    a, b = O.clip_forward(g["image"], g["text"], sd, img_heads=2, txt_heads=2)
    loss, la, lb, _, _ = O.contrastive_loss(a, b, scale)
    torch.testing.assert_close(a, g["emb_a"], rtol=0, atol=2e-6)
    torch.testing.assert_close(b, g["emb_b"], rtol=0, atol=2e-6)
    torch.testing.assert_close(la, g["logits_a"], rtol=0, atol=5e-5)
    torch.testing.assert_close(lb, g["logits_b"], rtol=0, atol=5e-5)
    torch.testing.assert_close(loss, g["loss"], rtol=0, atol=1e-5)
    loss.backward()
    torch.testing.assert_close(scale.grad, g["logit_scale_grad"], rtol=1e-4, atol=1e-6)
    for k, ref in g["grads"].items():
        got = sd[k].grad
        if isinstance(ref, dict):
            assert tuple(got.shape) == ref["shape"]
            torch.testing.assert_close(got.reshape(-1)[::ref["stride"]], ref["sample"], rtol=1e-3, atol=2e-6)
            assert abs(got.double().abs().sum() - ref["abssum"]) <= 1e-4 * ref["abssum"] + 1e-6
        else:
            torch.testing.assert_close(got, ref, rtol=1e-3, atol=2e-6)


def test_oracle_b16_forward_matches_reference_golden_and_init_mirror(golden):
    """clip_vit_b16() of THIS package under manual_seed(0) must hold the reference's weights (same construction
    order), and the oracle forward on them must reproduce the reference outputs."""
    from multimodal_b200.models.clip.model import clip_vit_b16

    torch.manual_seed(0)
    m = clip_vit_b16()
    sd = m.state_dict()
    assert len(sd) == 301  # SURVEY.md §8(b)
    img, txt = O.synthetic_batch(2)
    with torch.no_grad():
        a, b = O.clip_forward(img, txt, sd, img_heads=12, txt_heads=8)
        loss, la, _, _, _ = O.contrastive_loss(a, b, torch.tensor(math.log(1 / 0.07)))
    g = golden["clip_b16_b2"]
    torch.testing.assert_close(a, g["emb_a"], rtol=0, atol=5e-6)
    torch.testing.assert_close(b, g["emb_b"], rtol=0, atol=5e-6)
    torch.testing.assert_close(la, g["logits_a"], rtol=0, atol=1e-4)
    torch.testing.assert_close(loss, g["loss"], rtol=0, atol=1e-5)


def test_fused_timing_variant_matches_oracle(golden):
    """bench.py's CPU arm uses oracle.clip_forward_fused (library-fused ops); it must be the same function."""
    g = golden["clip_small"]
    sd = CC.small_state_dict(g)
    with torch.no_grad():
        a, b = O.clip_forward(g["image"], g["text"], sd, 2, 2)
        af, bf = O.clip_forward_fused(g["image"], g["text"], sd, 2, 2)
    torch.testing.assert_close(af, a, rtol=0, atol=2e-6)
    torch.testing.assert_close(bf, b, rtol=0, atol=2e-6)


def test_reference_kat_contrastive_loss():
    """tests/modules/losses/test_contrastive_loss_with_temperature.py:75-82 (9.8753) and :112-123 (10.2524)."""
    torch.manual_seed(1234)
    scale = torch.tensor(math.log(1 / 0.07))
    a, b = torch.randn(3, 5), torch.randn(3, 5)
    loss = O.contrastive_loss(a, b, O.clamp_logit_scale(scale))[0]
    assert abs(loss.item() - 9.8753) < 1e-3
    loss = O.contrastive_loss(a, b, O.clamp_logit_scale(scale), label_smoothing=0.1)[0]
    assert abs(loss.item() - 10.2524) < 1e-3


def test_reference_kat_text_encoder():
    """tests/models/clip/test_text_encoder.py:107-120: seed 1234, text drawn BEFORE the encoder is built,
    CLIPTextEncoder(embedding_dim=4, heads=2, width=512) -> [[-1.3103,-0.6713,-0.9614,0.7010],[1.1780,...]]."""
    from multimodal_b200.models.clip.text_encoder import CLIPTextEncoder

    torch.manual_seed(1234)
    text = torch.randint(1, 10, (2, 77), dtype=torch.long)
    enc = CLIPTextEncoder(embedding_dim=4, use_clip_init=True, context_length=77, width=512, heads=2)
    with torch.no_grad():
        out = O.text_encoder(text, {"e." + k: v for k, v in enc.state_dict().items()}, "e.", heads=2)
    expected = torch.tensor([[-1.3103, -0.6713, -0.9614, 0.7010], [1.1780, 0.1888, 0.8019, 0.7287]])
    torch.testing.assert_close(out, expected, rtol=0, atol=1e-4)
    # causal mask (:96-105)
    m = CLIPTextEncoder(embedding_dim=4, context_length=4, width=512, heads=2).build_attention_mask()
    inf = float("inf")
    assert torch.equal(m, torch.tensor([[0, -inf, -inf, -inf], [0, 0, -inf, -inf], [0, 0, 0, -inf], [0, 0, 0, 0.0]]))


def test_reference_kat_clip_normalize():
    """tests/models/clip/test_clip.py:26-56 (seed 1234, Linear(5,3)/Linear(4,3) encoders)."""
    torch.manual_seed(1234)
    ea, eb = torch.nn.Linear(5, 3), torch.nn.Linear(4, 3)
    xa = torch.randint(1, 8, (2, 5), dtype=torch.float)
    xb = torch.randint(1, 8, (2, 4), dtype=torch.float)
    with torch.no_grad():
        a, b = O.normalize(ea(xa)), O.normalize(eb(xb))
    torch.testing.assert_close(a, torch.tensor([[-0.8066, -0.1749, 0.5647], [-0.7709, -0.1118, 0.6271]]), rtol=0, atol=1e-4)
    torch.testing.assert_close(b, torch.tensor([[-0.1719, 0.7932, 0.5842], [-0.2805, 0.8761, -0.3921]]), rtol=0, atol=1e-4)


def test_error_conventions_match_reference():
    from multimodal_b200.models.clip.image_encoder import CLIPViTEncoder
    from multimodal_b200.models.clip.text_encoder import CLIPTextEncoder
    from multimodal_b200.modules.losses.contrastive_loss_with_temperature import ContrastiveLossWithTemperature

    enc = CLIPViTEncoder(embedding_dim=64, patch_size=16, image_size=64, width=128, heads=2, layers=1)
    with pytest.raises(ValueError):
        enc(torch.ones(2, 3, 32, 32))      # image_encoder.py:83-86
    with pytest.raises(ValueError):
        enc(torch.ones(2, 1, 64, 64))      # :87-88
    t = CLIPTextEncoder(embedding_dim=64, vocab_size=100, width=128, dim_feedforward=256, heads=2, layers=1)
    with pytest.raises(ValueError):
        t(torch.ones(2, 78, dtype=torch.long))  # text_encoder.py:114-117
    with pytest.raises(ValueError):
        ContrastiveLossWithTemperature(logit_scale_max=None, logit_scale_min=None)  # :172-175
    with pytest.raises(ValueError):
        ContrastiveLossWithTemperature(logit_scale_min=0.0, logit_scale_max=None)   # truthiness quirk (:172)


def test_no_cpu_fallback():
    """The product path must fail loudly on CPU tensors instead of silently computing somewhere else."""
    from multimodal_b200._lib import MMBError
    from multimodal_b200.models.clip.image_encoder import CLIPViTEncoder

    enc = CLIPViTEncoder(embedding_dim=64, patch_size=16, image_size=64, width=128, heads=2, layers=1)
    with pytest.raises(MMBError):
        enc(torch.ones(2, 3, 64, 64))


def test_oracle_masked_loss_matches_reference_golden():
    """Row `mask` (contrastive_loss_with_temperature.py:97-100): oracle forward + autograd vs the reference's."""
    import os

    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "loss_mask_golden.pt"))
    for name, c in g.items():
        a, b = c["a"].clone().requires_grad_(True), c["b"].clone().requires_grad_(True)
        s = torch.tensor(math.log(1 / 0.07), requires_grad=True)
        loss, la, lb, loss_a, loss_b = O.contrastive_loss(a, b, s, label_smoothing=c["smoothing"], mask=c["mask"])
        loss.backward()
        assert torch.allclose(loss, c["loss"], atol=1e-5), name
        assert torch.allclose(la, c["logits_a"], atol=1e-5) and torch.allclose(lb, c["logits_b"], atol=1e-5)
        assert torch.allclose(loss_a, c["loss_a"], atol=1e-5) and torch.allclose(loss_b, c["loss_b"], atol=1e-5)
        assert torch.allclose(a.grad, c["dA"], atol=1e-6) and torch.allclose(b.grad, c["dB"], atol=1e-6)
        assert torch.allclose(s.grad, c["dS"], atol=1e-4)
