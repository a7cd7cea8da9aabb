"""GPU probe for the FLAVA forward path: per-tensor parity against the committed reference goldens and timing of
BASELINE.json config 3 (FLAVA full forward, bs=256).  Run under gpurun; writes gpurun_out/flava_probe.log."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import flava_cases as FC  # noqa: E402
from multimodal_b200 import ops  # noqa: E402
from multimodal_b200.models.flava import flava_model  # noqa: E402

lines = []


def log(*a):
    s = " ".join(str(x) for x in a)
    print(s, flush=True)
    lines.append(s)


@torch.no_grad()   # inference runtime (with grad mode on, trainable modules take the training runtime)
def main():
    dev = torch.device("cuda:0")
    gold = torch.load(os.path.join(ROOT, "tests", "golden", "flava_golden.pt"))
    for name in FC.CASES:
        g = gold[name]
        m = FC.build(flava_model, name).to(dev)
        inp = {k: v.to(dev) for k, v in g["inputs"].items()}
        o = m(image=inp["image"], text=inp["text"], image_patches_mask=inp["image_patches_mask"],
              text_masked=inp["text_masked"], skip_unmasked_mm_encoder=False)
        got = FC.flatten_output(o)
        for k, ref in g["outputs"].items():
            err = (FC.golden_view(got[k]) - ref).abs().max().item()
            log(f"{name} {k}: abs_err={err:.3e} ref_absmax={ref.abs().max().item():.3e} rel={err / ref.abs().max().item():.3e}")
    # ---- config 3 timing
    B = int(os.environ.get("FLAVA_BS", "256"))
    torch.manual_seed(0)
    m = flava_model().to(dev).eval()
    image = torch.randn(B, 3, 224, 224, device=dev)
    text = torch.randint(1, 30522, (B, 77), device=dev)
    pm = torch.rand(B, 196, device=dev) < 0.4

    def timed(fn, n=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    t_img = timed(lambda: m.image_encoder(image))
    t_txt = timed(lambda: m.text_encoder(input_ids=text, return_hidden_states=True))
    ih = m.image_encoder(image).hidden_states[-1].clone()
    th = m.text_encoder(input_ids=text, return_hidden_states=True).hidden_states[-1].clone()
    t_mm = timed(lambda: m.encode_mm(ih, th))
    t_full = timed(lambda: m(image=image, text=text, image_patches_mask=pm, text_masked=text))
    ops.GEMM_TIMING = []
    m(image=image, text=text, image_patches_mask=pm, text_masked=text)
    torch.cuda.synchronize()
    gt = ops.GEMM_TIMING
    ops.GEMM_TIMING = None
    gemm_ms = sum(ev[0].elapsed_time(ev[1]) for _, _, ev in gt)
    gemm_fl = sum(f for f, _, _ in gt)
    # model flops of one full forward: GEMMs + attention (4*S^2*d per layer per sample)
    att = lambda S, L: 4.0 * S * S * 768 * L * B  # noqa: E731
    fl_full = gemm_fl + 2 * att(197, 12) + 2 * att(77, 12) + att(275, 6)
    log(f"FLAVA bs={B}: image_encoder {t_img:.2f} ms | text_encoder {t_txt:.2f} ms | encode_mm {t_mm:.2f} ms")
    log(f"FLAVA bs={B}: FLAVAModel.forward(image,text,patches_mask,text_masked) {t_full:.2f} ms = {B / t_full * 1e3:.0f} samples/s; "
        f"{fl_full / t_full / 1e9:.1f} TFLOP/s model (GEMM kernels {gemm_ms:.2f} ms at {gemm_fl / gemm_ms / 1e9:.1f} TFLOP/s, {len(gt)} launches)")
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/flava_probe.log", "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
