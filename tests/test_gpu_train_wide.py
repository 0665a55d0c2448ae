"""Training the vanilla Diff model at the widths it hard-wires (UNet ch_mult [1, 2, 4, 8]: 512-channel levels, GroupNorms
over concatenations of up to 1024 channels, attention heads of 256 and 512 channels) on the B200.

Op level: the wide instantiations of the AdaGN backward, the tcgen05 attention backward at d = 256 / 512 and weight-
gradient plans of more than 64 work units, each through the same check and tolerances as its narrow counterpart in
test_gpu_ops.py.  Network level: every parameter gradient of the [1, 2, 4, 8] UNet against torch autograd through the
fp32 CPU oracle (64x64 and 32x32), three optimizer steps of the reference recipe, and run.py's vanilla training feeding
the two-phase eval_fid sampler."""
import math
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest
import torch

from oracle import infodiff_oracle as orc
from oracle.golden_util import SEED, make_args, perturb_state_dict
from tests import test_gpu_ops as ops
from tests.test_gpu_network import _patched_draws
from tests.test_gpu_ops import lib  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = Path(__file__).resolve().parent.parent


# ------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("save", [False, True])
@pytest.mark.parametrize("mod,silu,drop", [(False, True, 0.0), (True, True, 0.0), (True, False, 0.0), (True, True, 0.1)])
@pytest.mark.parametrize("H", [8, 16])
@pytest.mark.parametrize("c0,c1", [(512, 0), (512, 256), (512, 512)])
def test_adagn_backward_wide(lib, c0, c1, H, mod, silu, drop, save):
    """The wide AdaGN backward (C = 512, and the 768 / 1024 up-path concatenations): dx, the fused gamma / beta /
    modulation gradients, the closed forms of (S1, S2) and the accumulate flag, as test_adagn_backward checks them."""
    ops.test_adagn_backward(lib, c0, c1, H, 2, mod, silu, drop, save)


@pytest.mark.parametrize("H,B,d", [(16, 3, 256), (16, 80, 256), (8, 5, 256), (8, 3, 512), (16, 2, 512)])
def test_attention_backward_wide_heads(lib, H, B, d):
    """tcgen05 attention backward with the head width walked in 128-wide chunks (scores) and split over CTAs (grads);
    at B = 80, S = 256, d = 256 the grads grid (2 x 80 x 2 CTAs) is larger than the machine."""
    ops.test_attention_backward(lib, H, B, d)


@pytest.mark.parametrize("cin,cout,H,B", [(1024, 512, 8, 2), (768, 512, 8, 2), (768, 256, 16, 2)])
def test_conv_weight_gradient_many_units(lib, cin, cout, H, B):
    """Weight-gradient plans of 96, 72 and 36 work units (co tiles x ci chunks x tap clusters; the kernel derives its
    unit's coordinates from the block index)."""
    ops.test_conv_weight_gradient(lib, cin, cout, H, B)


# ------------------------------------------------------------------------------------------------
# the network
# ------------------------------------------------------------------------------------------------
def _vanilla(size: int, T: int = 1000):
    from infodiffusion_b200.models import Diff
    args = make_args(a_dim=32, diffusion_steps=T, model="vanilla", input_size=size)
    torch.manual_seed(SEED)
    m = Diff(args, "cpu", (3, size, size))
    assert m.backbone.ch_mult == [1, 2, 4, 8]
    sd = perturb_state_dict(m.state_dict())
    m.load_state_dict(sd)
    m.device = DEV
    for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
        setattr(m, n, getattr(m, n).to(DEV))
    return args, m.to(DEV).eval(), sd


def _oracle_loss(sd, sch, x, idx, eps):
    """Diff.loss_fn (reference models.py:763-779) through the oracle UNet."""
    return (orc.unet_forward(sd, orc.q_sample(sch, x, idx, eps), idx) - eps).square().mean()


def _draws(B: int, size: int, g: torch.Generator, T: int = 1000):
    return dict(x=torch.rand(B, 3, size, size, generator=g) * 2 - 1, idx=torch.randint(0, T, (B,), generator=g),
                eps=torch.randn(B, 3, size, size, generator=g))


@pytest.mark.parametrize("size", [64, 32])
def test_vanilla_training_gradients_at_native_widths(size):
    """Diff(model='vanilla').loss_fn in train() mode (dropout 0): the loss and every parameter gradient against torch
    autograd through the oracle.  64x64 runs attention backward at (S=256, d=256) and (S=64, d=512) on tcgen05; 32x32
    at (S=64, d=256) on tcgen05 and (S=16, d=512) on the small-map kernel."""
    args, m, sd = _vanilla(size)
    d = _draws(2, size, torch.Generator().manual_seed(31 + size))
    sch = orc.Schedule.make(args.beta1, args.betaT, args.diffusion_steps)
    sdg = {k: v.clone().requires_grad_(v.is_floating_point() and "timembedding.0" not in k) for k, v in sd.items()}
    loss_o = _oracle_loss(sdg, sch, d["x"], d["idx"], d["eps"])
    loss_o.backward()
    m.train()
    m.backbone.dropout_p = 0.0
    m.zero_grad(set_to_none=True)
    try:
        with _patched_draws(d["idx"].to(DEV), [d["eps"].clone()]):
            loss = m.loss_fn(args, d["x"].to(DEV))
        loss.backward()
    finally:
        m.eval()
    print(f"\n[parity] vanilla [1,2,4,8] {size}x{size} loss: cuda {float(loss.detach()):.6f} vs oracle {float(loss_o.detach()):.6f}")
    assert abs(float(loss) - float(loss_o)) / abs(float(loss_o)) < 2e-2
    rels = []
    for name, p in m.named_parameters():
        g_ref = sdg[name].grad
        if g_ref is None or float(g_ref.abs().max()) == 0.0 or name.endswith("attn.proj_k.bias"):
            continue
        assert p.grad is not None, name
        g, r = p.grad.cpu().double().flatten(), g_ref.double().flatten()
        rels.append((float((g - r).norm() / r.norm()), float((g @ r) / (g.norm() * r.norm())), name))
    rels.sort(reverse=True)
    med = sorted(r[0] for r in rels)[len(rels) // 2]
    print(f"[parity] vanilla {size}x{size} gradients: {len(rels)} checked, median rel-L2 {med:.3e}, worst {rels[0]}, "
          f"min cosine {min(c for _, c, _ in rels):.5f}")
    assert len(rels) > 300 and med < 5e-2 and all(c > 0.98 for _, c, _ in rels), rels[:3]


def test_vanilla_three_training_steps_track_the_reference_recipe():
    """run.py:195-200 for three steps of the vanilla model -- loss_fn, backward, clip_grad_norm_(1.0), AdamW(lr, wd 1e-5)
    -- with the fused ClipAdamW on the GPU and torch autograd + torch.optim.AdamW on the oracle, identical draws."""
    from infodiffusion_b200.optim import ClipAdamW
    args, m, sd = _vanilla(64)
    B, steps, lr = 2, 3, 1e-4
    gl = torch.Generator().manual_seed(78)
    draws = [_draws(B, 64, gl) for _ in range(steps)]
    names = [k for k, v in sd.items() if v.is_floating_point() and "timembedding.0" not in k]
    sdo = {k: (v.clone().requires_grad_(True) if k in names else v.clone()) for k, v in sd.items()}
    opt_o = torch.optim.AdamW([sdo[k] for k in names], lr=lr, weight_decay=1e-5)
    sch = orc.Schedule.make(args.beta1, args.betaT, args.diffusion_steps)
    loss_o = []
    for d in draws:
        loss = _oracle_loss(sdo, sch, d["x"], d["idx"], d["eps"])
        opt_o.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_([sdo[k] for k in names if sdo[k].grad is not None], 1.0)
        opt_o.step()
        loss_o.append(float(loss))
    m.train()
    m.backbone.dropout_p = 0.0
    opt = ClipAdamW(m.parameters(), lr=lr, weight_decay=1e-5, max_norm=1.0)
    loss_g = []
    try:
        for d in draws:
            with _patched_draws(d["idx"].to(DEV), [d["eps"].clone()]):
                loss = m.loss_fn(args, d["x"].to(DEV))
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            loss_g.append(float(loss.detach()))
        torch.cuda.synchronize()
    finally:
        m.eval()
    print(f"\n[parity] vanilla, 3 training steps: loss cuda {['%.5f' % v for v in loss_g]} vs oracle {['%.5f' % v for v in loss_o]}")
    for a_, b_ in zip(loss_g, loss_o):
        assert abs(a_ - b_) / abs(b_) < 2e-2
    num = den_g = den_o = 0.0
    for name, p in m.named_parameters():
        if name not in names or sdo[name].grad is None:
            continue
        dg = (p.detach().cpu().double() - sd[name].double()).flatten()
        do = (sdo[name].detach().double() - sd[name].double()).flatten()
        num += float(dg @ do); den_g += float(dg @ dg); den_o += float(do @ do)
    cos = num / (den_g ** 0.5 * den_o ** 0.5)
    print(f"[parity] vanilla accumulated parameter update: cosine {cos:.4f}, norm ratio {(den_g / den_o) ** 0.5:.4f}")
    assert cos > 0.97 and 0.95 < (den_g / den_o) ** 0.5 < 1.05


def test_run_py_vanilla_train_feeds_two_phase_eval_fid(tmp_path):
    """run.py --model vanilla --mode train --mmd_weight 0 writes the checkpoint where the reference's eval_fid looks for
    it (models/diff/{dataset}_{a_dim}d/model-{epochs}.pth); eval_fid of the InfoDiff model then runs the two-phase
    sampler without --single_phase."""
    common = ["--prior", "regular", "--dataset", "synthetic", "--a_dim", "32", "--batch_size", "4", "--epochs", "1",
              "--save_epochs", "1", "--diffusion_steps", "4", "--synthetic_size", "8", "--r_seed", "64",
              "--model_folder", "./models", "--img_folder", "./imgs"]

    def run(*extra):
        r = subprocess.run([sys.executable, str(ROOT / "run.py"), *common, *extra], cwd=tmp_path, capture_output=True,
                           text=True, timeout=900, env={**os.environ, "PYTHONPATH": str(ROOT)})
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return r.stdout
    out = run("--model", "vanilla", "--mode", "train", "--mmd_weight", "0")
    losses = [float(v) for v in re.findall(r"Loss (\S+)", out)]
    assert losses and all(math.isfinite(v) for v in losses), out
    assert (tmp_path / "models" / "diff" / "synthetic_32d" / "model-1.pth").exists()
    run("--model", "diff", "--mode", "train")
    out = run("--model", "diff", "--mode", "eval_fid", "--sampling_number", "2")
    assert "--single_phase" not in out
    pngs = sorted((tmp_path / "imgs" / "synthetic_32d_0.1mmd" / "eval-fid-fast").glob("sample-*.png"))
    assert [p.name for p in pngs] == ["sample-000000.png", "sample-000001.png"]
