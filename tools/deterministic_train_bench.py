"""Cost of deterministic training: bench.py's training workload (InfoDiff, a_dim 256, 64x64, batch 32, T = 1000, dropout
0.1, fused clip + AdamW) with torch.use_deterministic_algorithms off and on, alternating in one process.

Two models with the same initial weights, one per mode, are warmed up (plan building, graph capture); then `--rounds`
timed windows of `--steps` steps alternate between them.  Reported per mode: CUDA-event ms per step (every window),
the library's launches per step, and the workspace the ordered plans own (the split-K / bias scratch of the side
stream, the AdaGN dgamma / dbeta scratch and the tickets; the Linear and MMD ordered calls allocate theirs per call from
torch's caching allocator and are not counted).  The GPU's name and power limit are read in the same call.

    python tools/deterministic_train_bench.py [--steps 10] [--rounds 4] [--warmup 3] [--out FILE]
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
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from bench import make_args_ns
    from infodiffusion_b200 import _lib
    from infodiffusion_b200 import train as T
    from infodiffusion_b200.models import InfoDiff
    from infodiffusion_b200.optim import ClipAdamW
    dev = torch.device("cuda", 0)
    args = make_args_ns(1000)
    args.mode = "train"
    x = (torch.rand(a.batch, 3, 64, 64, generator=torch.Generator().manual_seed(7)) * 2 - 1).to(dev)
    runs = {}
    for det in (False, True):
        torch.manual_seed(64)
        model = InfoDiff(args, "cpu", (3, 64, 64)).to(dev)
        model.device = dev
        for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
            setattr(model, n, getattr(model, n).to(dev))
        model.train()
        params = [p for p in model.parameters() if p.requires_grad]
        runs[det] = dict(model=model, params=params, ms=[], launches=0,
                         opt=ClipAdamW(params, lr=1e-4, weight_decay=1e-5, max_norm=1.0))

    def window(det: bool, n: int):
        r = runs[det]
        torch.use_deterministic_algorithms(det)
        try:
            l0 = _lib.launches()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                loss = r["model"].loss_fn(args, x)
                r["opt"].zero_grad(set_to_none=True)
                loss.backward()
                r["opt"].step()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n, (_lib.launches() - l0) // n
        finally:
            torch.use_deterministic_algorithms(False)

    for det in (False, True):
        window(det, a.warmup)
    for _ in range(a.rounds):
        for det in (False, True):
            ms, launches = window(det, a.steps)
            runs[det]["ms"].append(ms)
            runs[det]["launches"] = launches
    result = {"gpu": gpu_info(), "batch": a.batch, "steps_per_window": a.steps, "rounds": a.rounds}
    for det, r in runs.items():
        ws = 0
        for net in (r["model"].backbone, r["model"].encoder):
            for key, plan in net._plans().items():
                if str(key[0]).startswith("train") and hasattr(plan, "_bwd"):
                    st = T._state(plan)
                    ws += sum(t.numel() * t.element_size() for t in (st.side_ws, st.main_ws, st.tickets) if t is not None)
        ms = sorted(r["ms"])
        result["deterministic" if det else "default"] = {
            "ms_per_step": r["ms"], "median_ms_per_step": ms[len(ms) // 2],
            "samples_per_sec": a.batch / (ms[len(ms) // 2] / 1000.0),
            "idf_launches_per_step": r["launches"], "plan_workspace_bytes": ws}
    result["median_cost"] = result["deterministic"]["median_ms_per_step"] / result["default"]["median_ms_per_step"] - 1
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        Path(a.out).write_text(text)


if __name__ == "__main__":
    main()
