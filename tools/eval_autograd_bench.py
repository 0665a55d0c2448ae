"""Cost of a differentiable eval-mode call: AuxiliaryUNet of bench.py's workload (a_dim 256, 64x64, T = 1000) in eval()
at batch `--batch`, forward + backward of (eps * G).sum() with x and a requiring grad (the training plan with dropout
off), against the no-grad inference forward at the same batch.

Reported: CUDA-event ms per call for both (every window, alternating), the library's launches per call, and the device
memory the eval-mode training plan adds (torch's allocated bytes after its first forward + backward, minus those after
the inference plan exists).  The GPU's name and power limit are read in the same call.

    python tools/eval_autograd_bench.py [--batch 32] [--iters 20] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.dont_write_bytecode = True
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import torch  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = (q.stdout.strip().splitlines()[0].split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?",) * 3
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clk}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    o = ap.parse_args()
    from infodiffusion_b200 import _lib
    from infodiffusion_b200.models import AuxiliaryUNet
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = AuxiliaryUNet(T=1000, ch=64, ch_mult=[1, 2, 2, 2], a_dim=256, shape=(3, 64, 64)).to(dev).eval()
    B = o.batch
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 3, 64, 64, generator=g).to(dev)
    t = torch.randint(0, 1000, (B,), generator=g).to(dev)
    a = torch.randn(B, 256, generator=g).to(dev)
    G = torch.randn(B, 3, 64, 64, generator=g).to(dev)

    def infer():
        with torch.no_grad():
            net(x, t, a)

    def grad_call():
        xd, ad = x.clone().requires_grad_(), a.clone().requires_grad_()
        net.zero_grad(set_to_none=True)
        (net(xd, t, ad) * G).sum().backward()

    for _ in range(3):
        infer()
    torch.cuda.synchronize()
    mem0 = torch.cuda.memory_allocated(dev)
    grad_call()
    torch.cuda.synchronize()
    net.zero_grad(set_to_none=True)
    mem_plan = torch.cuda.memory_allocated(dev) - mem0
    for _ in range(3):                                   # graph capture of forward and backward, then replays
        grad_call()
    res = {"gpu": gpu_info(), "batch": B, "eval_train_plan_bytes": mem_plan, "infer_ms": [], "grad_ms": []}
    for name, fn in (("infer", infer), ("grad", grad_call)):
        torch.cuda.synchronize()
        n0 = _lib.launches()
        fn()
        torch.cuda.synchronize()
        res[f"{name}_launches"] = _lib.launches() - n0
    for _ in range(o.rounds):
        for name, fn in (("infer", infer), ("grad", grad_call)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(o.iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[f"{name}_ms"].append(round(e0.elapsed_time(e1) / o.iters, 3))
    print(json.dumps(res))
    if o.out:
        Path(o.out).parent.mkdir(parents=True, exist_ok=True)
        Path(o.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
