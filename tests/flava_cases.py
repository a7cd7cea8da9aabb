"""Shared definitions of the FLAVA parity cases: builder kwargs, seeded weights and inputs.  Used by the fixture
generator (tests/golden/make_flava_golden.py, which feeds them to the reference) and by the parity tests (which feed
them to multimodal_b200) — both sides construct bit-identical models because the parameter containers are created in
the same order under the same seed (checked by the param checksum stored in the fixture)."""
import torch

CASES = {
    # S_image = 17, S_text = 12, S_mm = 30: every encoder on the tcgen05 attention path
    "flava_small": dict(
        kwargs=dict(image_hidden_size=128, image_num_attention_heads=2, image_num_hidden_layers=2,
                    image_intermediate_size=256, image_size=32, patch_size=8,
                    text_hidden_size=128, text_num_attention_heads=2, text_num_hidden_layers=2,
                    text_intermediate_size=256, vocab_size=100, max_position_embeddings=32,
                    multimodal_hidden_size=256, multimodal_num_attention_heads=4, multimodal_num_hidden_layers=1,
                    multimodal_intermediate_size=512, text_and_image_proj_size=64),
        batch=3, text_len=12),
    # S_image = 257, S_mm = 274: sequence lengths of the real model class (197 / 275) that exceed one 256-row tile
    "flava_long": dict(
        kwargs=dict(image_hidden_size=128, image_num_attention_heads=2, image_num_hidden_layers=1,
                    image_intermediate_size=256, image_size=64, patch_size=4,
                    text_hidden_size=128, text_num_attention_heads=2, text_num_hidden_layers=1,
                    text_intermediate_size=256, vocab_size=100, max_position_embeddings=32,
                    multimodal_hidden_size=128, multimodal_num_attention_heads=2, multimodal_num_hidden_layers=1,
                    multimodal_intermediate_size=256, text_and_image_proj_size=64),
        batch=2, text_len=16),
}


def build(builder, name: str):
    """builder = reference or multimodal_b200 `flava_model`.  Seeded init + a seeded perturbation so that biases,
    LayerNorm affine terms, cls/mask tokens and position embeddings (all zero/one at init) take part in the test."""
    torch.manual_seed(0)
    m = builder(**CASES[name]["kwargs"])
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=g))
    return m.eval()


def param_checksum(m) -> float:
    return float(sum(p.detach().double().abs().sum() for p in m.parameters()))


def inputs(name: str):
    c = CASES[name]
    kw, B, St = c["kwargs"], c["batch"], c["text_len"]
    g = torch.Generator().manual_seed(5)
    image = torch.randn(B, 3, kw["image_size"], kw["image_size"], generator=g)
    text = torch.randint(1, kw["vocab_size"], (B, St), generator=g)
    for b in range(B):  # ragged right padding with pad_token_id = 0 (row 0 keeps full length)
        n_pad = (3 * b) % (St - 2)
        if n_pad:
            text[b, St - n_pad:] = 0
    text_masked = text.clone()
    text_masked[:, 2] = kw["vocab_size"] - 1  # stand-in for [MASK]
    P = (kw["image_size"] // kw["patch_size"]) ** 2
    patches_mask = torch.rand(B, P, generator=g) < 0.4
    return dict(image=image, text=text, text_masked=text_masked, image_patches_mask=patches_mask)


def flatten_output(out) -> dict:
    """FLAVAOutput -> {name: tensor} of everything the parity test compares."""
    res = {}
    for field in ("image", "image_masked", "text", "text_masked", "multimodal", "multimodal_masked"):
        t = getattr(out, field)
        if t is None or t.last_hidden_state is None:
            continue
        res[f"{field}.last_hidden_state"] = t.last_hidden_state
        res[f"{field}.pooler_output"] = t.pooler_output
        for i, h in enumerate(t.hidden_states):
            res[f"{field}.hidden_states.{i}"] = h
    res["projected_image_embeddings"] = out.projected_image_embeddings
    res["projected_text_embeddings"] = out.projected_text_embeddings
    return {k: v.detach().float().cpu().clone() for k, v in res.items() if v is not None}


GOLDEN_TOKENS = 8


def golden_view(t: torch.Tensor) -> torch.Tensor:
    """The part of an output the fixture stores, so that it stays small: of a [B, S, D] sequence output with more than
    GOLDEN_TOKENS positions, the first, the last and evenly spaced positions between them; anything else whole."""
    if t.dim() != 3 or t.shape[1] <= GOLDEN_TOKENS:
        return t
    return t[:, torch.linspace(0, t.shape[1] - 1, GOLDEN_TOKENS).round().long().to(t.device)]
