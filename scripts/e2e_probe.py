"""GPU bring-up probe: per-kernel checks (attention, LayerNorm) + end-to-end small CLIP vs the reference golden."""
import math
import os
import sys
import time
import traceback

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import clip_cases as CC  # noqa: E402
from multimodal_b200 import ops  # noqa: E402
from oracle import clip_oracle as O  # noqa: E402

dev = torch.device("cuda:0")
lines = []


def log(*a):
    s = " ".join(str(x) for x in a)
    print(s, flush=True)
    lines.append(s)


def rel(got, ref):
    got, ref = got.float(), ref.float()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-12)).item(), (got - ref).abs().max().item()


def attn_ref(qkv, B, S, H, causal):
    d = H * 64
    q, k, v = qkv.float().view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    att = q @ k.transpose(-1, -2) / 8.0
    if causal:
        att = att + torch.full((S, S), float("-inf"), device=qkv.device).triu(1)
    p = torch.softmax(att, -1)
    o = (p @ v).transpose(1, 2).reshape(B * S, d)
    return o


def check_attention(B, S, H, causal):
    d = H * 64
    torch.manual_seed(1)
    qkv = (torch.randn(B * S, 3 * d, device=dev) * 0.7).bfloat16()
    out = torch.empty(B * S, d, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B * H * S, device=dev)
    ops.attention_fwd(qkv, out, lse, B, S, H, causal, 0.125)
    qf = qkv.float().requires_grad_(True)
    ref = attn_ref(qf, B, S, H, causal)
    r, a = rel(out, ref)
    log(f"attn_fwd B{B} S{S} H{H} causal={causal}: rel={r:.3e} abs={a:.3e}")
    dout = (torch.randn(B * S, d, device=dev) * 0.5).bfloat16()
    ref.backward(dout.float())
    dqkv = torch.empty_like(qkv)
    ops.attention_bwd(qkv, out, dout, lse, dqkv, B, S, H, causal, 0.125)
    for i, n in enumerate("qkv"):
        r, a = rel(dqkv[:, i * d:(i + 1) * d], qf.grad[:, i * d:(i + 1) * d])
        log(f"   attn_bwd d{n}: rel={r:.3e} abs={a:.3e}")


def check_ln(M, d):
    torch.manual_seed(2)
    x = torch.randn(M, d, device=dev)
    y = torch.randn(M, d, device=dev).bfloat16()
    g = torch.randn(d, device=dev)
    b = torch.randn(d, device=dev)
    xo = torch.empty_like(x)
    ln = torch.empty(M, d, device=dev, dtype=torch.bfloat16)
    mean = torch.empty(M, device=dev)
    rstd = torch.empty(M, device=dev)
    ops.add_layernorm_fwd(x, y, xo, ln, None, g, b, mean, rstd, M, d, 1e-5)
    xs = (x + y.float()).requires_grad_(True)
    gp = g.clone().requires_grad_(True)
    bp = b.clone().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(xs, (d,), gp, bp, 1e-5)
    log(f"ln_fwd M{M} d{d}: x_out {rel(xo, xs)}  ln {rel(ln, ref)}")
    dy = torch.randn(M, d, device=dev).bfloat16()
    ref.backward(dy.float())
    gin = torch.randn(M, d, device=dev)
    gout = torch.empty_like(gin)
    gb = torch.empty(M, d, device=dev, dtype=torch.bfloat16)
    dg = torch.zeros(d, device=dev)
    db = torch.zeros(d, device=dev)
    ops.layernorm_bwd(xo, dy, None, mean, rstd, g, gin, gout, gb, dg, db, M, d)
    log(f"ln_bwd: dx {rel(gout - gin, xs.grad)} dgamma {rel(dg, gp.grad)} dbeta {rel(db, bp.grad)} gb {rel(gb, gout)}")


def e2e_small():
    from multimodal_b200.models.clip.image_encoder import CLIPViTEncoder
    from multimodal_b200.models.clip.model import CLIP
    from multimodal_b200.models.clip.text_encoder import CLIPTextEncoder
    from multimodal_b200.modules.losses.contrastive_loss_with_temperature import (
        ContrastiveLossWithTemperature, contrastive_loss_with_temperature)

    gold = torch.load(os.path.join(ROOT, "tests/golden/clip_golden.pt"), map_location="cpu", weights_only=False)["clip_small"]
    m = CLIP(CLIPViTEncoder(64, 16, 64, 128, 2, 2),
             CLIPTextEncoder(embedding_dim=64, vocab_size=512, width=128, dim_feedforward=512, heads=2, layers=2))
    m.load_state_dict(CC.small_state_dict(gold))
    m = m.to(dev).train()
    loss_mod = ContrastiveLossWithTemperature().to(dev)
    img, txt = gold["image"].to(dev), gold["text"].to(dev)
    out = m(img, txt)
    log("emb_a", rel(out.embeddings_a, gold["emb_a"].to(dev)), "emb_b", rel(out.embeddings_b, gold["emb_b"].to(dev)))
    res = contrastive_loss_with_temperature(out.embeddings_a, out.embeddings_b, loss_mod.logit_scale)
    log("loss", res.loss.item(), "golden", gold["loss"].item(), "logits_a", rel(res.logits_a, gold["logits_a"].to(dev)))
    res.loss.backward()
    log("logit_scale grad", loss_mod.logit_scale.grad.item(), "golden", gold["logit_scale_grad"].item())
    worst = []
    for k, p in m.named_parameters():
        ref = gold["grads"][k]
        if p.grad is None:
            log("  MISSING grad", k)
            continue
        if isinstance(ref, dict):
            samp = p.grad.reshape(-1)[::ref["stride"]]
            r = (((samp - ref["sample"].to(dev)).abs().max() / ref["absmax"].to(dev)).item(), 0.0)
            asum = p.grad.double().abs().sum().item()
            worst.append((r[0], k, f"abssum {asum:.6e} vs {ref['abssum'].item():.6e}"))
        else:
            r = rel(p.grad, ref.to(dev))
            worst.append((r[0], k, f"abs {r[1]:.3e} refmax {ref.abs().max().item():.3e}"))
    worst.sort(reverse=True)
    for w in worst[:14]:
        log("  grad", f"{w[0]:.3e}", w[1], w[2])
    log("  median grad rel err", sorted(x[0] for x in worst)[len(worst) // 2])


def e2e_b16(B=8):
    from multimodal_b200.models.clip.model import clip_vit_b16
    from multimodal_b200.modules.losses.contrastive_loss_with_temperature import ContrastiveLossWithTemperature

    torch.manual_seed(0)
    m = clip_vit_b16()
    sd = {k: v.to(dev) for k, v in m.state_dict().items()}
    m = m.to(dev).train()
    img, txt = O.synthetic_batch(B, device=dev)
    with torch.no_grad():
        ra, rb = O.clip_forward(img, txt, sd, 12, 8)
        rl = O.contrastive_loss(ra, rb, torch.tensor(math.log(1 / 0.07), device=dev))[0]
    t0 = time.time()
    out = m(img, txt)
    loss = ContrastiveLossWithTemperature().to(dev)(out.embeddings_a, out.embeddings_b)
    loss.backward()
    torch.cuda.synchronize()
    log(f"b16 B={B}: emb_a {rel(out.embeddings_a, ra)} emb_b {rel(out.embeddings_b, rb)} loss {loss.item():.6f} ref {rl.item():.6f}  ({time.time()-t0:.2f}s)")


for fn, args in [(check_attention, (2, 197, 12, False)), (check_attention, (3, 77, 8, True)), (check_attention, (2, 5, 2, False)),
                 (check_attention, (2, 257, 16, False)), (check_ln, (1000, 768)), (check_ln, (77, 512)), (e2e_small, ()), (e2e_b16, ())]:
    try:
        fn(*args)
    except Exception:  # noqa: BLE001
        log("EXC in", fn.__name__, args)
        log(traceback.format_exc())
        break
os.makedirs("gpurun_out", exist_ok=True)
open("gpurun_out/e2e_probe.log", "w").write("\n".join(lines) + "\n")
