"""The library's launch counter against the device: over each region below, the change of _lib.launches() (bench.py's
idf_launches_per_step) equals the number of idf:: kernels torch.profiler records on the GPU.

Regions: an inference eps forward; a sampler step, eager and graph-replayed; InfoDiff training steps (loss_fn, backward,
ClipAdamW.step) eager, captured and replayed, in default and in deterministic mode; the same for the vanilla 32x32 Diff
model, whose 4x4 attention backward takes the small-map kernel and whose 512-channel AdaGN backward the wide one.

The profiling runs in a subprocess (`python -m tests.test_gpu_launch_count` prints one JSON line per region), so the
profiler's CUPTI session stays out of the other tests' process."""
import collections
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _profiled(name, fn):
    """{region, counted, kernels, names}: the counter's change over fn() and the idf:: kernels the GPU ran."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from infodiffusion_b200 import _lib
    torch.cuda.synchronize()
    n0 = _lib.launches()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    counted = _lib.launches() - n0
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        events = json.load(open(path))["traceEvents"]
    names = collections.Counter(e["name"].split("<")[0].split("(")[0].replace("void ", "") for e in events
                                if e.get("cat") == "kernel" and "idf::" in e["name"])
    return dict(region=name, counted=counted, kernels=sum(names.values()), names=dict(names))


def _train_regions(tag, make, B):
    import torch
    from infodiffusion_b200.optim import ClipAdamW
    from oracle.golden_util import SEED
    out = []
    for det in (False, True):
        torch.manual_seed(SEED)
        args, model, data = make()
        x = data(torch.Generator().manual_seed(5), B).to("cuda:0")
        params = [p for p in model.parameters() if p.requires_grad]
        opt = ClipAdamW(params, lr=1e-4, weight_decay=1e-5, max_norm=1.0)
        model.train()

        def step():
            loss = model.loss_fn(args, x)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
        torch.use_deterministic_algorithms(det)
        try:
            for phase in ("eager", "captured", "replayed"):
                out.append(_profiled(f"{tag} train step {phase}{' deterministic' if det else ''}", step))
        finally:
            torch.use_deterministic_algorithms(False)
            model.eval()
    return out


def main():
    import torch
    from oracle.golden_util import make_args
    from infodiffusion_b200.models import InfoDiff
    from infodiffusion_b200.sampling import DiffusionProcess
    from tests.test_gpu_deterministic_training import MODELS
    dev = "cuda:0"
    B = 4
    torch.manual_seed(0)
    args = make_args(a_dim=32, diffusion_steps=10, deterministic=True)
    m = InfoDiff(args, "cpu", (3, 64, 64)).to(dev).eval()
    x, t, a = torch.randn(B, 3, 64, 64, device=dev), torch.randint(0, 10, (B,), device=dev), torch.randn(B, 32, device=dev)
    with torch.no_grad():
        m.backbone(x, t, a)                                  # builds the plan
        res = [_profiled("eps forward", lambda: m.backbone(x, t, a))]
        s = DiffusionProcess(args, m, dev, (3, 64, 64))._sampler("ddim", B)
        s.x.copy_(x)
        s.set_latent(a)
        s.run_step(5, use_graph=False)
        res.append(_profiled("sampler step eager", lambda: s.run_step(5, use_graph=False)))
        s.run_step(5)                                        # captures the graph
        res.append(_profiled("sampler step replayed", lambda: s.run_step(4)))
    res += _train_regions("infodiff", MODELS["infodiff_mmd"], B)
    res += _train_regions("vanilla 32x32", MODELS["vanilla_32"], B)
    for r in res:
        print(json.dumps(r), flush=True)


def test_launch_counter_matches_the_kernels_the_gpu_runs():
    r = subprocess.run([sys.executable, "-m", "tests.test_gpu_launch_count"], cwd=ROOT, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stderr[-4000:]
    rows = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(rows) == 15
    bad = [row for row in rows if row["counted"] != row["kernels"]]
    for row in rows:
        print(f"\n[launches] {row['region']}: counted {row['counted']}, idf kernels on the GPU {row['kernels']}")
    assert not bad, "launch counter differs from the device:\n" + "\n".join(json.dumps(b) for b in bad)
    assert all(row["kernels"] > 0 for row in rows)


if __name__ == "__main__":
    main()
