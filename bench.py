#!/usr/bin/env python
"""Headline benchmark: image-text pairs/sec of one CLIP ViT-B/16 contrastive pre-training step (forward + loss +
backward + gradient all-reduce + AdamW), bs=1024 per GPU, bf16 tensor-core math, synthetic 224x224x3 / 77-token data.

    python bench.py --gpus 1 --steps 5 --warmup 3                  # ours, one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                     # ours, N GPUs (weak scaling)
    python bench.py --impl reference --steps 3 --warmup 1          # reference arm: CPU fp32 port of the reference path
    python bench.py --steps 5 --warmup 3 --dump-outputs DIR        # also write the last timed step's outputs as DIR/*.npy

Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for every field.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Algorithmic FLOPs per pair, CLIP ViT-B/16 (SURVEY.md §8d / BASELINE.md §5): forward 41.01 GF, step = 3x forward.
F_FWD_B16 = 35.127e9 + 5.887e9
F_STEP_B16 = 3.0 * F_FWD_B16
METRIC = "image-text pairs/sec (CLIP ViT-B/16 contrastive pretrain step, bs=1024/GPU)"
# BASELINE.json configs[3] (a parity / capability case, not the headline line): CLIP ViT-L/14, 4096 pairs per GPU
# (global 32 768 on 8 GPUs), two-pass activation recompute in micro-batches.  SURVEY.md §8d: 175.22 GF forward per pair.
F_STEP_L14 = 3.0 * (162.03e9 + 13.19e9)
CONFIGS = {
    "b16": {"builder": "clip_vit_b16", "f_step": F_STEP_B16, "batch": 1024, "micro_batch": None, "metric": METRIC,
            "workload": "CLIP ViT-B/16 contrastive pretrain step (fwd+loss+bwd+grad-allreduce+AdamW)"},
    "l14": {"builder": "clip_vit_l14", "f_step": F_STEP_L14, "batch": 4096, "micro_batch": 256,
            "metric": "image-text pairs/sec (CLIP ViT-L/14 contrastive pretrain step, bs=4096/GPU, global 32768 on 8 GPUs)",
            "workload": "CLIP ViT-L/14 contrastive pretrain step (two-pass recompute in micro-batches of 256: "
                        "no-save forward of all slices -> global loss -> re-forward+backward per slice; +grad-allreduce+AdamW)"},
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-eager-gpu"])
    ap.add_argument("--config", default="b16", choices=sorted(CONFIGS),
                    help="b16 = the headline BASELINE.json configs[1]; l14 = configs[3] (ViT-L/14, 4096/GPU, recompute)")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default = the config's)")
    ap.add_argument("--micro-batch", type=int, default=None, help="recompute slice size (default = the config's)")
    ap.add_argument("--cpu-batch", type=int, default=4, help="sample size of the CPU reference/port legs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true",
                    help="skip the info-only same-box torch eager bf16-autocast leg of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["bf16_tflops_sustained"]), float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, sustained cuBLAS bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md: 1.4 PFLOP/s sustained)"


# ----------------------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the oracle port (fp32, all host threads) of the reference's own path
# ----------------------------------------------------------------------------------------------------------------
def cpu_port_run(steps, warmup, batch, budget_s=None):
    """Returns (pairs/s, seconds/step, threads, timed steps).  budget_s bounds the timed part of the cpu_baseline leg (the
    --impl reference arm times exactly `steps` steps as the driver asks)."""
    import torch
    from oracle import clip_oracle as O  # test-infrastructure port; allowed here (cpu_baseline / --impl reference)
    from multimodal_b200.models.clip.model import clip_vit_b16

    # Threads: the schedulable CPUs, capped at 32 — on the pool's 128-vCPU boxes the eager fp32 port at these small
    # batches runs ~10x SLOWER with 128 intra-op threads than with 32 (oversubscription), so the cap favours the CPU arm.
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cores = max(1, min(avail, 32))
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    sd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in clip_vit_b16().state_dict().items()}
    scale = torch.tensor(math.log(1 / 0.07), requires_grad=True)
    img, txt = O.synthetic_batch(batch)
    params = [v for v in sd.values() if v.requires_grad] + [scale]

    def step():
        a, b = O.clip_forward_fused(img, txt, sd, 12, 8)   # library-fused form: what the reference dispatches to on CPU
        loss = O.contrastive_loss(a, b, O.clamp_logit_scale(scale))[0]
        loss.backward()
        with torch.no_grad():  # plain SGD update: the cheapest possible optimizer (favours the CPU arm)
            for p in params:
                p -= 1e-4 * p.grad
                p.grad = None
        return float(loss.detach())

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        step()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = (time.perf_counter() - t0) / max(done, 1)
    return batch / dt, dt, cores, done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    val, dt, cores, _ = cpu_port_run(args.steps, args.warmup, args.cpu_batch)
    sample = f"{args.cpu_batch} pairs/step x {args.steps} steps (fwd+loss+bwd+SGD), fp32 eager, {cores} threads"
    # SURVEY.md §8(d) also asks for a B=64 throughput point of the CPU path: one warm-up + up to 2 timed steps,
    # bounded to ~60 s so that the arm still ends within minutes (reported beside the line's own B=4 value)
    b64 = None
    try:
        v64, dt64, _, done64 = cpu_port_run(2, 1, 64, budget_s=45.0)
        b64 = {"value": v64, "unit": "pairs/s", "per_step_batch": 64, "timed_steps": done64, "s_per_step": dt64}
    except Exception as e:  # noqa: BLE001 — the extra point must never cost the arm its line
        b64 = {"error": str(e)[:200]}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "CLIP ViT-B/16 contrastive pretrain step (fwd+loss+bwd+update), CPU port of the reference path",
                   "per_gpu_batch": args.cpu_batch, "image": "224x224x3", "text_len": 77},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample,
                         "b64_point": b64},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------------------------
# Info-only leg: "what PyTorch gives today" on the same B200 (BASELINE.md §4, SURVEY.md §8d) — stock torch modules
# (torch.nn.TransformerEncoder fast path, flash SDPA, cuBLAS), bf16 autocast, torch's fused AdamW, same batch.
# None of this repo's kernels run here; it is context for the kernels' numbers, not an arm the driver scores.
# ----------------------------------------------------------------------------------------------------------------
def torch_eager_gpu_run(batch, steps, warmup, dev):
    import torch
    import torch.nn.functional as F
    from multimodal_b200.models.clip.model import clip_vit_b16
    from oracle import clip_oracle as O  # synthetic-input generator only

    torch.manual_seed(0)
    model = clip_vit_b16().to(dev).train()       # the drop-in modules HOLD stock torch layers (state-dict contract)
    ia, tb = model.encoder_a, model.encoder_b

    class QuickGELU(torch.nn.Module):   # plain torch ops (activation.py:24-25); the drop-in's own SiLU is a fused-kernel stub
        def forward(self, x):
            return torch.sigmoid(1.702 * x) * x

    for layer in list(ia.encoder.layers) + list(tb.encoder.layers):
        layer.activation = QuickGELU()
    logit_scale = torch.nn.Parameter(torch.tensor(math.log(1 / 0.07), device=dev))
    opt = torch.optim.AdamW(list(model.parameters()) + [logit_scale], lr=5e-4, betas=(0.9, 0.98), eps=1e-6,
                            weight_decay=0.2, fused=True)
    causal = torch.full((77, 77), float("-inf"), device=dev).triu(1)

    def ln32(mod, x):   # Fp32LayerNorm semantics with the module's parameters (upcast, fp32 layer_norm, cast back)
        return F.layer_norm(x.float(), x.shape[-1:], mod.weight, mod.bias, mod.eps).type_as(x)

    def forward(img, txt):
        x = ia.conv(img).flatten(2).transpose(1, 2)                                  # [B, 196, d]
        x = torch.cat([ia.cls_token_embedding.expand(x.shape[0], 1, -1).to(x.dtype), x], dim=1) + ia.positional_embedding
        x = ia.encoder(ln32(ia.ln_pre, x))
        a = ln32(ia.ln_post, x[:, 0, :]) @ ia.projection
        y = tb.token_embedding(txt) + tb.positional_embedding
        y = tb.encoder(y.transpose(0, 1), mask=causal, is_causal=True).transpose(0, 1)   # seq-first layers
        y = ln32(tb.ln_final, y)
        b = tb.projection(y[torch.arange(y.shape[0], device=dev), txt.argmax(dim=-1)])
        return F.normalize(a.float(), dim=1), F.normalize(b.float(), dim=1)

    def step(img, txt):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            a, b = forward(img, txt)
        logits = a @ b.t() * logit_scale.exp()
        labels = torch.arange(a.shape[0], device=dev)
        loss = 0.5 * (F.cross_entropy(logits, labels) + F.cross_entropy(logits.t(), labels))
        loss.backward()
        opt.step()
        return loss

    B = batch
    while True:
        try:
            img, txt = O.synthetic_batch(B, device=dev)
            for _ in range(max(warmup, 1)):
                step(img, txt)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                loss = step(img, txt)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            return {"value": B / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms, "per_gpu_batch": B,
                    "final_loss": float(loss.item()), "tflops_step_level": B / (ms * 1e-3) * F_STEP_B16 / 1e12,
                    "what": "stock torch modules (nn.TransformerEncoder, SDPA, cuBLAS), bf16 autocast, fused AdamW; "
                            "fwd+loss+bwd+step, device-resident synthetic batch"}
        except torch.cuda.OutOfMemoryError:
            opt.zero_grad(set_to_none=True)
            torch.cuda.empty_cache()
            if B <= 64:
                raise
            B //= 2   # eager autograd keeps far more activations than the fused schedule: fall back, and say so


def run_torch_eager(args):
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    r = torch_eager_gpu_run(args.batch or 1024, args.steps, args.warmup, dev)
    print(json.dumps({"impl": "torch-eager-gpu", "metric": METRIC, "value": r["value"], "unit": "pairs/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                      "dtype": "bf16 autocast", "data": "synthetic",
                      "config": {"workload": "CLIP ViT-B/16 contrastive pretrain step, stock PyTorch eager on the same B200",
                                 "per_gpu_batch": r["per_gpu_batch"], "requested_batch": args.batch or 1024}, "detail": r}))


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# outputs of the timed path, for comparing two builds (the inputs and the initial weights are seeded)
# ----------------------------------------------------------------------------------------------------------------
def dump_outputs(dirname, model, loss_mod, loss, n_sample=1 << 23):
    """Writes what the last timed step computed, as its caller receives it, in float32: loss.npy (the step's loss),
    logit_scale.npy (the updated temperature parameter) and weights.npy, the updated weights at a fixed seeded sample of
    n_sample positions of the model's parameters in named_parameters() order (~600 MB in full, 32 MB as sampled).  The
    parameters' .grad views hold nothing by then: the fused AdamW step clears them.  The training step is not yet
    bit-reproducible: split-K GEMMs (TMA reduce-add) and the LayerNorm / bias / embedding / logit-scale gradient
    reductions accumulate with fp32 atomics, and AdamW turns last-bit differences in near-zero gradients into weight
    differences of up to 2 * lr, so two runs of one build differ by up to ~1e-3 in the weights."""
    import numpy as np
    import torch

    params = [p for _, p in model.named_parameters()]
    sizes = torch.tensor([p.numel() for p in params])
    ends = sizes.cumsum(0)
    pos = torch.randint(0, int(ends[-1]), (n_sample,), generator=torch.Generator().manual_seed(0)).sort().values
    cut = torch.searchsorted(pos, ends).tolist()   # pos[cut[i - 1]:cut[i]] fall into params[i]
    weights, lo = [], 0
    for p, hi, start in zip(params, cut, (ends - sizes).tolist()):
        weights.append(p.detach().reshape(-1)[(pos[lo:hi] - start).to(p.device)])
        lo = hi
    out = {"loss": loss.detach().reshape(1), "logit_scale": loss_mod.logit_scale.detach().reshape(1),
           "weights": torch.cat(weights)}
    os.makedirs(dirname, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(dirname, name + ".npy"), t.float().cpu().numpy())


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from multimodal_b200 import _lib, ops
    from multimodal_b200.models.clip import model as clip_models
    from multimodal_b200.modules.losses.contrastive_loss_with_temperature import ContrastiveLossWithTemperature
    from multimodal_b200.train import ContrastiveTrainer
    from oracle import clip_oracle as O  # only for the synthetic-input generator + the bounded cpu_baseline leg

    if not _lib.LIB_PATH.exists():  # harness convenience on a fresh checkout: local rank 0 builds, the others wait
        if int(os.environ.get("LOCAL_RANK", "0")) == 0:
            _lib.build()
        else:
            t_wait = time.time()
            while not _lib.LIB_PATH.exists() and time.time() - t_wait < 900:
                time.sleep(2)
            time.sleep(2)
    _lib.lib()  # fail loudly right away if the CUDA library is missing
    cfg = CONFIGS[args.config]
    B = args.batch or cfg["batch"]
    MB = args.micro_batch or cfg["micro_batch"]
    if MB is not None and MB >= B:
        MB = None
    F_STEP = cfg["f_step"]
    torch.manual_seed(0)
    model = getattr(clip_models, cfg["builder"])().to(dev)
    loss_mod = ContrastiveLossWithTemperature().to(dev)
    trainer = ContrastiveTrainer(model, loss_mod)

    img_h, txt_h = O.synthetic_batch(B, rank=rank)
    img_h, txt_h = img_h.pin_memory(), txt_h.pin_memory()
    img_d, txt_d = img_h.to(dev, non_blocking=True), txt_h.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up (allocations, first-touch, clocks) ----
    for _ in range(max(args.warmup, 3)):
        loss = trainer.step(img_d, txt_d, micro_batch=MB)
    barrier()

    # ---- timed: device-resident inputs (no per-launch instrumentation inside this region) ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = trainer.step(img_d, txt_d, micro_batch=MB)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_dev = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    launches = (_lib.LAUNCHES - launches0) // args.steps
    final_loss = float(loss.item())
    if args.dump_outputs and rank == 0:   # before the steps below change the weights again
        dump_outputs(args.dump_outputs, model, loss_mod, loss)

    # ---- per-kernel-family breakdown: INSTR_STEPS more steps with every GEMM / attention / LayerNorm launch bracketed
    # by CUDA events on the launching stream (kept out of the region above: ~1000 event records per step) ----
    INSTR_STEPS = 2
    ops.GEMM_TIMING, ops.FAMILY_TIMING = [], []
    barrier()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for _ in range(INSTR_STEPS):
        trainer.step(img_d, txt_d, micro_batch=MB)
    i1.record()
    barrier()
    ms_instr = i0.elapsed_time(i1) / INSTR_STEPS
    gemm_log, ops.GEMM_TIMING = ops.GEMM_TIMING, None
    fam_log, ops.FAMILY_TIMING = ops.FAMILY_TIMING, None

    peak_tf, peak_gbs, peak_src = measured_peaks()
    tot_f, tot_ms, by_kind = 0.0, 0.0, {}
    for flops, kind, (a, b) in gemm_log:
        ms = a.elapsed_time(b)
        tot_f += flops; tot_ms += ms
        k = by_kind.setdefault(str(kind), [0.0, 0.0, 0]); k[0] += flops; k[1] += ms; k[2] += 1
    fams = {"gemm": [tot_f, tot_ms, len(gemm_log), "F"]}
    for fam, work, unit, (a, b) in fam_log:
        f = fams.setdefault(fam, [0.0, 0.0, 0, unit]); f[0] += work; f[1] += a.elapsed_time(b); f[2] += 1
    by_kernel = {}
    for fam, (work, ms, n, unit) in fams.items():
        if ms <= 0:
            continue
        if unit == "F":
            ach, pk, u = work / (ms * 1e-3) / 1e12, peak_tf, "TFLOP/s"
        else:
            ach, pk, u = work / (ms * 1e-3) / 1e9, peak_gbs, "GB/s"
        by_kernel[fam] = {"ms_per_step": ms / INSTR_STEPS, "share_of_step": (ms / INSTR_STEPS) / ms_instr,
                          "launches_per_step": n // INSTR_STEPS, "achieved": ach, "unit": u, "peak": pk, "frac": ach / pk,
                          "algorithmic_work_per_step": work / INSTR_STEPS, "work_unit": "flop" if unit == "F" else "byte"}
    covered = sum(v["ms_per_step"] for v in by_kernel.values())
    by_kernel["other"] = {"ms_per_step": ms_instr - covered, "share_of_step": (ms_instr - covered) / ms_instr,
                          "note": "embedding / patchify / loss / column-sum / optimizer kernels, launch gaps and (N > 1) "
                                  "exposed all-reduce"}

    # ---- timed: end to end through the public step() with host inputs (H2D of inputs + D2H of the loss every step) ----
    from multimodal_b200.train import HostPrefetcher
    # the box's own pinned-host -> device copy rate for this batch (context for e2e: when the copy of one batch takes
    # longer than a step, e2e is bound by the host link, not by the kernels)
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(2):
        img_d.copy_(img_h, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    h2d_ms = c0.elapsed_time(c1) / 2
    h2d_gbps = img_h.numel() * 4 / (h2d_ms * 1e-3) / 1e9
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    # Every step's loss is read back to the host inside the timed region — through pinned memory, asynchronously, and
    # consumed one step later (what a training loop's logging does): a blocking .item() per step would drain the launch
    # queue and leave the GPU waiting for the host at the start of every step (measured: e2e 175-191 ms at N = 1 and
    # 210 ms at N = 2 against 173-183 ms device-resident, purely from that bubble; the H2D copy alone is 11 ms).
    loss_h = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    pend, k, losses_read = None, 0, 0
    for xi, xt in HostPrefetcher(((img_h, txt_h) for _ in range(args.steps)), dev):  # every H2D copy is inside t0..t1
        loss_d = trainer.step(xi, xt, micro_batch=MB)
        buf = loss_h[k & 1]
        buf.copy_(loss_d.reshape(1), non_blocking=True)                               # D2H of the loss, every step
        ev = torch.cuda.Event(); ev.record()
        if pend is not None:
            pend[0].synchronize(); l_host = float(pend[1][0]); losses_read += 1       # previous step's loss, now on the host
        pend, k = (ev, buf), k + 1
    pend[0].synchronize(); l_host = float(pend[1][0]); losses_read += 1
    assert losses_read == args.steps and math.isfinite(l_host)
    t1.record()
    barrier()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1) / args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = B * world / (ms_dev * 1e-3)
    e2e_val = B * world / (ms_e2e * 1e-3)
    step_tf = value * F_STEP / 1e12 / world
    burst_tf = None
    try:
        burst_tf = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:  # noqa: BLE001
        pass
    # DRAM traffic of the dominant kernel's benchmarked launch, from the committed `ncu --set full` capture
    traffic, traffic_src = None, "no committed capture found (profiles/r2_ncu_kernels.json)"
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_kernels.json")))
        k = cap["kernels"]["gemm_qkv_fwd"]
        traffic = k["dram_bytes_read"] + k["dram_bytes_write"]
        traffic_src = (f"{k['name']} {k['shape']}: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch, "
                       f"{cap['source']}; algorithmic bytes of that launch {k['algorithmic_bytes']:.4g}")
    except Exception:  # noqa: BLE001
        pass
    out = {
        "metric": cfg["metric"], "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": args.config, "micro_batch": MB,
                   "per_gpu_batch": B, "global_batch": B * world, "image": "224x224x3 fp32", "text_len": 77,
                   "parallelism": f"dp{world}", "l2": "activations (~84 GB/step) and inputs (616 MB) exceed the 126 MB L2; no flush needed",
                   "final_loss": final_loss},
        "e2e": {"value": e2e_val, "unit": "pairs/s", "h2d_bytes_per_step": img_h.numel() * 4 + txt_h.numel() * 8,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e,
                "h2d_copy_alone_ms": h2d_ms, "h2d_copy_alone_gbps": h2d_gbps,
                "note": "the H2D copy of step i+1 (pinned fp32 images, side stream) overlaps the kernels of step i; every "
                        "step's loss is copied to pinned host memory inside the timed region and consumed one step later "
                        "(no per-step host sync draining the launch queue)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        # STEP-LEVEL roofline: algorithmic FLOPs of the whole step (SURVEY.md §8d: 123.04 GF per pair) over the
        # CUDA-event time of the timed region, against the measured sustained cuBLAS bf16 peak.
        "roofline": {"bound": "tensor", "achieved": step_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": step_tf / peak_tf if peak_tf else None,
                     "frac_of_burst_peak": step_tf / burst_tf if burst_tf else None,
                     "definition": f"pairs/s/GPU x {F_STEP / 1e9:.2f} GF (3 x forward GEMM+attention FLOPs, SURVEY.md §8d; a "
                                   "recompute pass is NOT counted as useful work) / measured sustained bf16 peak",
                     "peak_source": peak_src,
                     "traffic": traffic, "traffic_launch": traffic_src,
                     "dominant_kernel": "mmb::gemm_kernel (tcgen05, all instantiations)",
                     "by_kernel": by_kernel,
                     "by_kernel_note": f"CUDA events around every launch during {INSTR_STEPS} extra instrumented steps "
                                       f"({ms_instr:.1f} ms/step with the events) right after the timed region",
                     "gemm_by_kind": {k: {"tflops": v[0] / (v[1] * 1e-3) / 1e12, "ms_per_step": v[1] / INSTR_STEPS,
                                          "n": v[2] // INSTR_STEPS} for k, v in by_kind.items()}},
    }
    if world == 1 and not args.no_eager_baseline and args.config == "b16":
        # info-only: stock PyTorch eager bf16-autocast on the same GPU, same batch (needs the trainer's memory back)
        try:
            del trainer, model, loss_mod
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            out["gpu_eager_baseline"] = torch_eager_gpu_run(B, 3, 2, dev)
        except Exception as e:  # noqa: BLE001 — never lose the line to the info leg
            out["gpu_eager_baseline"] = {"error": f"{type(e).__name__}: {str(e)[:160]}"}
    if world == 1 and not args.no_cpu_baseline and args.config == "b16":
        val, dt, cores, done = cpu_port_run(3, 1, args.cpu_batch, budget_s=20.0)
        out["cpu_baseline"] = {"value": val, "unit": "pairs/s", "cores": cores, "kind": "port",
                               "sample": f"{args.cpu_batch} pairs/step x {done} steps (fwd+loss+bwd+SGD), fp32 eager oracle port"}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "torch-eager-gpu":
        run_torch_eager(a)
    else:
        run_ours(a)
