"""Training rate of the vanilla Diff model (UNet ch_mult [1, 2, 4, 8], 64x64, a_dim 32) -- the step of
run.py --model vanilla --mode train: loss_fn -> backward -> fused clip_grad_norm_(1.0) + AdamW.

For each batch size: samples/s over CUDA events after warm-up and the library's own launches per step; then one
step under torch.profiler (a separate run, so the profiler does not slow the timed one) with the summed device time
per kernel class; then, labelled as such, the same step eagerly through the fp32 oracle under torch autograd on the
same GPU (TF32 on as the reference's run.py:19-20 sets it, cuDNN autotuning, torch.optim.AdamW).  The GPU's name and
power limit are read in the same call.

    python tools/vanilla_train_bench.py [--batches 32,64] [--steps 10] [--warmup 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from collections import defaultdict
from pathlib import Path

sys.dont_write_bytecode = True
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import torch  # noqa: E402

# kernel classes of the profile, first match wins (substrings of the demangled kernel names)
CLASSES = [
    ("attn_fwd_wide_cuda_core", ("attn_generic_kernel",)),
    ("attn_fwd_tcgen05", ("attn_tma_kernel",)),
    ("attn_fwd_small", ("attn_small_kernel",)),
    ("attn_bwd_tcgen05", ("attn_bwd_scores", "attn_bwd_grads")),
    ("attn_bwd_small", ("attn_small_bwd",)),
    ("conv", ("conv_",)),
    ("wgrad", ("wgrad",)),
    ("adagn_bwd", ("adagn_bwd",)),
    ("adagn_fwd", ("adagn",)),
    ("optimizer", ("adamw_kernel", "grad_sqsum", "grad_norm")),
    ("other_idf", ("idf::",)),
]


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = (q.stdout.strip().splitlines()[0].split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?",) * 3
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clk}


def run_args():
    import run as idf_run
    args = idf_run.parse_args(["--model", "vanilla", "--mode", "train", "--prior", "regular", "--dataset", "celeba",
                               "--a_dim", "32", "--mmd_weight", "0"])
    shape = idf_run.get_dataset_config(args)
    idf_run._check_widths(args)
    return args, shape


def kernel_class(name: str) -> str:
    for cls, keys in CLASSES:
        if any(k in name for k in keys):
            return cls
    return "torch"


def time_steps(step, steps: int, warmup: int):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


def profile_step(step) -> dict:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    acc = defaultdict(lambda: [0.0, 0])
    for e in prof.key_averages():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        c = acc[kernel_class(e.key)]
        c[0] += us / 1000.0
        c[1] += e.count
    tot = sum(v[0] for v in acc.values())
    return {"total_kernel_ms": tot,
            "classes": {k: {"ms": v[0], "share": v[0] / tot if tot else 0.0, "launches": v[1]}
                        for k, v in sorted(acc.items(), key=lambda kv: -kv[1][0])}}


def own_step(B: int, steps: int, warmup: int) -> dict:
    from infodiffusion_b200 import _lib
    from infodiffusion_b200.models import Diff
    from infodiffusion_b200.optim import ClipAdamW
    dev = "cuda:0"
    args, shape = run_args()
    torch.manual_seed(64)
    model = Diff(args, dev, shape)
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    opt = ClipAdamW(params, lr=args.learning_rate, weight_decay=1e-5, max_norm=1.0)
    x = torch.rand(B, *shape, generator=torch.Generator().manual_seed(7)).mul(2).sub(1).to(dev)

    def step():
        loss = model.loss_fn(args=args, x=x)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss.detach()
    ms, loss = time_steps(step, 1, warmup)              # plans, graphs, warm-up
    l0 = _lib.launches()
    ms, loss = time_steps(step, steps, 0)
    launches = (_lib.launches() - l0) // steps
    prof = profile_step(step)
    out = {"batch": B, "ms_per_step": ms, "samples_per_s": B / (ms / 1000.0), "idf_launches_per_step": launches,
           "final_loss": loss, "profile": prof}
    del model, opt
    torch.cuda.empty_cache()
    return out


def eager_step(B: int, steps: int, warmup: int) -> dict:
    """The reference's arithmetic (oracle UNet, fp32 params) under torch autograd on the GPU: cuDNN / cuBLAS with TF32."""
    from infodiffusion_b200.models import Diff
    from oracle import infodiff_oracle as orc
    dev = "cuda:0"
    args, shape = run_args()
    torch.manual_seed(64)
    sd = {k: v.to(dev) for k, v in Diff(args, "cpu", shape).state_dict().items()}
    names = [k for k, v in sd.items() if v.is_floating_point() and "timembedding.0" not in k]
    for k in names:
        sd[k].requires_grad_(True)
    opt = torch.optim.AdamW([sd[k] for k in names], lr=args.learning_rate, weight_decay=1e-5)
    sch = orc.Schedule.make(args.beta1, args.betaT, args.diffusion_steps)
    sch = orc.Schedule(*(t.to(dev) for t in (sch.betas, sch.alphas, sch.alpha_bars, sch.alpha_prev_bars)))
    x = torch.rand(B, *shape, generator=torch.Generator().manual_seed(7)).mul(2).sub(1).to(dev)
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark = torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True

    def step():
        idx = torch.randint(0, args.diffusion_steps, (B,), device=dev)
        eps = torch.randn_like(x)
        loss = (orc.unet_forward(sd, orc.q_sample(sch, x, idx, eps), idx) - eps).square().mean()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_([sd[k] for k in names], 1.0)
        opt.step()
        return loss.detach()
    try:
        ms, loss = time_steps(step, steps, warmup)
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    out = {"batch": B, "ms_per_step": ms, "samples_per_s": B / (ms / 1000.0), "final_loss": loss,
           "kind": "eager baseline: oracle UNet (reference arithmetic) under torch autograd, fp32 + TF32, cuDNN autotuned, "
                   "torch.optim.AdamW + clip_grad_norm_"}
    del sd, opt
    torch.cuda.empty_cache()
    return out


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--batches", default="32,64")
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--out", default=None, help="also write the JSON result here")
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vanilla_train_bench.py measures on a CUDA device; none is visible")
    from infodiffusion_b200 import _lib
    _lib.check(_lib.load().idf_init())
    res = {"workload": "run.py --model vanilla --mode train step: Diff (UNet ch 64, ch_mult [1,2,4,8]) at 64x64, a_dim 32, "
                       "T=1000, dropout 0.1, fused clip(1.0) + AdamW(1e-4, wd 1e-5), one GPU",
           "gpu": gpu_info(), "steps": a.steps, "warmup": a.warmup, "own": [], "eager": []}
    for B in (int(b) for b in a.batches.split(",")):
        res["own"].append(own_step(B, a.steps, a.warmup))
        res["eager"].append(eager_step(B, a.steps, a.warmup))
        r, e = res["own"][-1], res["eager"][-1]
        print(f"B={B}: {r['samples_per_s']:.1f} samples/s ({r['ms_per_step']:.2f} ms/step, {r['idf_launches_per_step']} "
              f"launches/step); eager baseline {e['samples_per_s']:.1f} samples/s", file=sys.stderr)
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")


if __name__ == "__main__":
    main()
