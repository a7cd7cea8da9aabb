"""Shared definition of the small CLIP parity case (see tests/flava_cases.py for the scheme).  The fixture generator
(tests/golden/make_golden.py) builds it from the reference's classes, the tests from multimodal_b200's: both hold the
same weights because the parameter containers are created in the same order under the same seed.  The fixture stores
per-tensor checksums of the reference's state dict instead of the weights themselves."""
import pytest
import torch


def build_small(CLIP, CLIPViTEncoder, CLIPTextEncoder):
    """CLIP with 64x64 images, width 128, 2 layers / 2 heads per tower: reference init under torch.manual_seed(0) plus a
    seeded perturbation."""
    torch.manual_seed(0)
    m = CLIP(CLIPViTEncoder(embedding_dim=64, patch_size=16, image_size=64, width=128, heads=2, layers=2),
             CLIPTextEncoder(embedding_dim=64, vocab_size=512, width=128, dim_feedforward=512, heads=2, layers=2))
    with torch.no_grad():  # break the "all layers identical" symmetry of nn.TransformerEncoder's deepcopy init
        g = torch.Generator().manual_seed(7)
        for p in m.parameters():
            p.add_(0.02 * torch.randn(p.shape, generator=g))
    return m


def state_dict_checksum(sd) -> dict:
    return {k: float(v.double().abs().sum()) for k, v in sd.items()}


def small_state_dict(case) -> dict:
    """The small model's weights, rebuilt with this package's constructors (the global RNG state is left as it was) and
    checked key by key against the checksums the generator recorded from the reference model."""
    from multimodal_b200.models.clip.image_encoder import CLIPViTEncoder
    from multimodal_b200.models.clip.model import CLIP
    from multimodal_b200.models.clip.text_encoder import CLIPTextEncoder

    with torch.random.fork_rng(devices=[]):
        sd = build_small(CLIP, CLIPViTEncoder, CLIPTextEncoder).state_dict()
    ref = case["state_dict_checksum"]
    assert list(sd) == list(ref)   # the reference's state-dict keys, in the reference's order
    for k, v in state_dict_checksum(sd).items():
        assert v == pytest.approx(ref[k], rel=1e-12), k
    return sd
