"""Generates tests/golden/clip_golden.pt by running the UNMODIFIED reference (a TorchMultimodal checkout, given as the
argument) on small deterministic inputs.  Committed together with its outputs; the tests only ever read the .pt file.

    python tests/golden/make_golden.py <path to the TorchMultimodal checkout>

Cases (kept tiny so the fixture stays small; weights are regenerated from seeds, only inputs/outputs are stored):
  clip_small : tests/clip_cases.py's small CLIP (64x64 images, width 128, 2 layers per tower), B=4; fp32 forward, loss,
               and all gradients (per-tensor float64 sums + a few raw tensors), and per-tensor checksums of the weights.
  clip_b16_b2: clip_vit_b16() under torch.manual_seed(0), B=2 synthetic batch; embeddings + loss only.
"""
import math
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle", "iopath_shim"))
sys.path.insert(0, os.path.abspath(sys.argv[1]))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from torchmultimodal.models.clip.image_encoder import CLIPViTEncoder  # noqa: E402
from torchmultimodal.models.clip.model import CLIP, clip_vit_b16  # noqa: E402
from torchmultimodal.models.clip.text_encoder import CLIPTextEncoder  # noqa: E402
from torchmultimodal.modules.losses.contrastive_loss_with_temperature import (  # noqa: E402
    ContrastiveLossWithTemperature,
    contrastive_loss_with_temperature,
)

import clip_cases as CC  # noqa: E402
from oracle import clip_oracle as O  # noqa: E402


def main():
    torch.set_num_threads(8)
    out = {}
    # ---------------- clip_small: forward + loss + grads ----------------
    m = CC.build_small(CLIP, CLIPViTEncoder, CLIPTextEncoder).train()
    img, txt = O.synthetic_batch(4, image_size=64, vocab=512)
    loss_mod = ContrastiveLossWithTemperature()
    o = m(img, txt)
    res = contrastive_loss_with_temperature(o.embeddings_a, o.embeddings_b, loss_mod.logit_scale)
    res.loss.backward()
    out["clip_small"] = {
        "image": img, "text": txt,
        "state_dict_checksum": CC.state_dict_checksum(m.state_dict()),
        "emb_a": o.embeddings_a.detach().clone(), "emb_b": o.embeddings_b.detach().clone(),
        "loss": res.loss.detach().clone(), "logits_a": res.logits_a.detach().clone(),
        "logits_b": res.logits_b.detach().clone(),
        # full gradients for small tensors; (abs-sum, abs-max, 4096 evenly strided samples) for the large ones
        "grads": {k: (p.grad.detach().clone() if p.numel() <= 20000 else
                      {"abssum": p.grad.double().abs().sum(), "absmax": p.grad.abs().max(),
                       "stride": max(1, p.numel() // 4096),
                       "sample": p.grad.reshape(-1)[::max(1, p.numel() // 4096)].clone(), "shape": tuple(p.shape)})
                  for k, p in m.named_parameters()},
        "logit_scale_grad": loss_mod.logit_scale.grad.detach().clone(),
    }
    # ---------------- clip_b16_b2: full-size forward ----------------
    torch.manual_seed(0)
    big = clip_vit_b16().eval()
    img, txt = O.synthetic_batch(2)
    with torch.no_grad():
        big.train()  # python MHA path (SURVEY.md §7 'three numerics paths'); dropout is 0
        ob = big(img, txt)
        lb = contrastive_loss_with_temperature(ob.embeddings_a, ob.embeddings_b, torch.tensor(math.log(1 / 0.07)))
    out["clip_b16_b2"] = {"emb_a": ob.embeddings_a.clone(), "emb_b": ob.embeddings_b.clone(), "loss": lb.loss.clone(),
                          "logits_a": lb.logits_a.clone()}
    torch.save(out, os.path.join(HERE, "clip_golden.pt"))
    print("wrote", os.path.join(HERE, "clip_golden.pt"), os.path.getsize(os.path.join(HERE, "clip_golden.pt")) / 1e6, "MB")


if __name__ == "__main__":
    main()
