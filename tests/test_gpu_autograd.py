"""Autograd through the networks beyond the training step: eval-mode calls whose inputs require grad run the training
plan with dropout off and return input and parameter gradients, and train-mode calls return the input gradient.  The
references are torch autograd through the fp32 CPU oracle on perturb_state_dict weights.  Tolerances are 1.2x the
value measured on a B200; every test prints what it measured."""
import contextlib

import pytest
import torch

from oracle import infodiff_oracle as orc
from oracle.golden_util import SEED, make_args, perturb_state_dict, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# 1.2 x measured on B200 (rel-L2; for the cosine, 1.2 x the measured 1 - cosine): input gradients of the eval-mode
# backbones and the encoder, measured 2.66e-2 / 2.87e-2 / 2.98e-2 / 2.00e-2 (x) and 3.39e-2 / 3.53e-2 (a)
TOL_DX = {"aux": (3.2e-2, 0.99958), "bottleneck": (3.4e-2, 0.99950), "unet32": (3.6e-2, 0.99947),
          "encoder": (2.4e-2, 0.99976)}
TOL_DA = {"aux": (4.1e-2, 0.99931), "bottleneck": (4.2e-2, 0.99927)}
TOL_FWD = 1.2e-2         # eval-mode differentiable forward vs the inference plan (upsample not folded): 9.97e-3
TOL_DX_TRAIN = (3.5e-2, 0.99948)   # x.grad through InfoDiff.loss_fn (encoder + x_t + reconstruction term): 2.95e-2
TOL_IDENTITY = 1.06e-2   # <x.grad, x> = <head.weight.grad, head.weight> with dropout on: 8.8e-3 (encoder)
TOL_DZ_LATENT = 1e-5     # LatentUNet, the fp32 path: the project's fp32 tolerance (measured 6.6e-7)


def _to_dev(m):
    m.device = DEV
    for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
        setattr(m, n, getattr(m, n).to(DEV))
    return m.to(DEV).eval()


def _infodiff(**kw):
    from infodiffusion_b200.models import InfoDiff
    args = make_args(a_dim=32, diffusion_steps=1000, **kw)
    torch.manual_seed(SEED)
    m = InfoDiff(args, "cpu", (3, 64, 64))
    sd = perturb_state_dict(m.state_dict())
    m.load_state_dict(sd)
    return args, _to_dev(m), sd


@pytest.fixture(scope="module")
def aux():
    return _infodiff()


def _backbone(kind, aux):
    """(network, state dict with 'backbone.' keys, oracle forward, takes a, image size)"""
    if kind == "aux":
        _, m, sd = aux
        return m.backbone, sd, orc.aux_unet_forward, True, 64
    if kind == "bottleneck":
        _, m, sd = _infodiff(is_bottleneck=True)
        return m.backbone, sd, orc.bottleneck_unet_forward, True, 64
    from infodiffusion_b200.models import UNet
    torch.manual_seed(SEED)
    u = UNet(T=1000, ch=64, ch_mult=[1, 2, 4, 8], shape=(3, 32, 32))
    sd = perturb_state_dict({"backbone." + k: v for k, v in u.state_dict().items()})
    u.load_state_dict({k[len("backbone."):]: v for k, v in sd.items()})
    return u.to(DEV).eval(), sd, orc.unet_forward, False, 32


def _grad_sd(sd):
    return {k: v.clone().requires_grad_(v.is_floating_point() and "timembedding.0" not in k) for k, v in sd.items()}


def _rel_cos(got, ref):
    g, r = got.detach().cpu().double().flatten(), ref.detach().double().flatten()
    return float((g - r).norm() / r.norm().clamp_min(1e-30)), float((g @ r) / (g.norm() * r.norm()).clamp_min(1e-30))


def _check_param_grads(net, sdg, prefix, what):
    """The criteria of test_gpu_network.py::test_training_step_gradients_match_oracle_autograd."""
    rows = []
    for name, p in net.named_parameters():
        g_ref = sdg[prefix + name].grad
        if g_ref is None or float(g_ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-6 or "crossattn" in name, name
            continue
        if name.endswith("attn.proj_k.bias"):
            continue    # softmax is invariant to a per-row shift of the scores: this gradient is exactly 0 in theory
        assert p.grad is not None, f"no gradient for {name}"
        rows.append((*_rel_cos(p.grad, g_ref), name))
    rows.sort(reverse=True)
    med = sorted(r[0] for r in rows)[len(rows) // 2]
    print(f"[autograd] {what} parameter gradients: {len(rows)} checked, median rel-L2 {med:.3e}, worst {rows[0]}, "
          f"min cosine {min(r[1] for r in rows):.5f}")
    assert len(rows) > 100 and med < 5e-2 and all(r[1] > 0.98 for r in rows), rows[:3]


def _check_input_grad(what, got, ref, tol):
    rel, cos = _rel_cos(got, ref)
    print(f"[autograd] {what}: rel-L2 {rel:.3e}, cosine {cos:.6f}")
    assert torch.isfinite(got).all()
    assert rel < tol[0] and cos > tol[1], (rel, cos)


@contextlib.contextmanager
def _injected_randn_like(queue):
    real = torch.randn_like
    torch.randn_like = lambda t, **k: queue.pop(0).to(t.device, t.dtype)
    try:
        yield
    finally:
        torch.randn_like = real


@contextlib.contextmanager
def _train(*nets, dropout_p=None):
    saved = [(n, n.dropout_p) for n in nets]
    for n in nets:
        n.train()
        if dropout_p is not None:
            n.dropout_p = dropout_p
    try:
        yield
    finally:
        for n, p in saved:
            n.dropout_p = p
            n.eval()


@contextlib.contextmanager
def _deterministic():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


def _inputs(B, size, seed=41):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, size, size, generator=g) * 2 - 1
    t = torch.randint(0, 1000, (B,), generator=g)
    a = torch.randn(B, 32, generator=g)
    G = torch.randn(B, 3, size, size, generator=g)
    return x, t, a, G


# ------------------------------------------------------------------------------------------------
# eval mode against oracle autograd
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["aux", "bottleneck", "unet32"])
def test_eval_backbone_gradients_match_oracle_autograd(aux, kind):
    """eval() backbone with x and a requiring grad: x.grad, a.grad and every parameter gradient of (eps . G).sum()."""
    net, sd, fwd, has_a, size = _backbone(kind, aux)
    x, t, a, G = _inputs(2, size)
    sdg = _grad_sd(sd)
    xr, ar = x.clone().requires_grad_(), a.clone().requires_grad_()
    ((fwd(sdg, xr, t, ar) if has_a else fwd(sdg, xr, t)) * G).sum().backward()
    net.zero_grad(set_to_none=True)
    xd, ad = x.to(DEV).requires_grad_(), a.to(DEV).requires_grad_()
    args = (xd, t.to(DEV), ad) if has_a else (xd, t.to(DEV))
    eps = net(*args)
    assert not net.training and eps.requires_grad
    (eps * G.to(DEV)).sum().backward()
    with torch.no_grad():
        ref_eps = net(*args)
    e = rel_l2(eps.detach().cpu(), ref_eps.cpu())
    print(f"\n[autograd] {kind}: differentiable eval forward vs inference plan rel-L2 {e:.3e}")
    assert e < TOL_FWD
    _check_input_grad(f"{kind} x.grad", xd.grad, xr.grad, TOL_DX[kind])
    if has_a:
        _check_input_grad(f"{kind} a.grad", ad.grad, ar.grad, TOL_DA[kind])
    _check_param_grads(net, sdg, "backbone.", kind)


def test_eval_encoder_image_gradient_matches_oracle_autograd(aux):
    """eval() Encoder: gradient of <a,G1> + <mu,G2> + <log_var,G3> with respect to the image, with the encoder's one
    randn_like draw injected on both sides."""
    _, m, sd = aux
    x, _, _, _ = _inputs(2, 64, seed=43)
    g = torch.Generator().manual_seed(44)
    G1, G2, G3, noise = (torch.randn(2, 32, generator=g) for _ in range(4))
    sdg = _grad_sd(sd)
    xr = x.clone().requires_grad_()
    a_o, aq_o, mu_o, lv_o = orc.encoder_forward(sdg, xr, noise=noise)
    ((a_o * G1).sum() + (mu_o * G2).sum() + (lv_o * G3).sum()).backward()
    m.encoder.zero_grad(set_to_none=True)
    xd = x.to(DEV).requires_grad_()
    with _injected_randn_like([noise.clone()]):
        a, a_q, mu, lv = m.encoder(xd)
    ((a * G1.to(DEV)).sum() + (mu * G2.to(DEV)).sum() + (lv * G3.to(DEV)).sum()).backward()
    print(f"\n[autograd] encoder a_q vs oracle rel-L2 {rel_l2(a_q.detach().cpu(), aq_o.detach()):.3e}")
    _check_input_grad("encoder x.grad", xd.grad, xr.grad, TOL_DX["encoder"])
    _check_param_grads(m.encoder, sdg, "encoder.", "encoder")


def test_eval_latent_unet_gradient_matches_oracle_autograd():
    """eval() LatentUNet with z requiring grad: the fp32 autograd composite (Dropouts are identities)."""
    from infodiffusion_b200.models import Diff
    D = 32
    args = make_args(a_dim=D, diffusion_steps=10, model="vanilla", is_latent=True)
    torch.manual_seed(SEED)
    lat = Diff(args, "cpu", (1, D, D))
    lat.load_state_dict(perturb_state_dict(lat.state_dict()))
    sd = {k: v.clone() for k, v in lat.state_dict().items()}
    lat = _to_dev(lat)
    g = torch.Generator().manual_seed(17)
    z, G = torch.randn(5, D, generator=g), torch.randn(5, D, generator=g)
    tz = torch.randint(0, 10, (5,), generator=g)
    zr = z.clone().requires_grad_()
    (orc.latent_unet_forward(sd, zr, tz) * G).sum().backward()
    zd = z.to(DEV).requires_grad_()
    eps = lat.backbone(zd, tz.to(DEV))
    (eps * G.to(DEV)).sum().backward()
    with torch.no_grad():
        assert rel_l2(eps.detach().cpu(), lat.backbone(zd, tz.to(DEV)).cpu()) < 1e-5
    rel, cos = _rel_cos(zd.grad, zr.grad)
    print(f"\n[autograd] latent z.grad: rel-L2 {rel:.3e}, cosine {cos:.8f}")
    assert rel < TOL_DZ_LATENT


# ------------------------------------------------------------------------------------------------
# train mode: the input gradient
# ------------------------------------------------------------------------------------------------
def test_train_loss_fn_input_gradient_matches_oracle_autograd(aux):
    """x.grad of InfoDiff.loss_fn in train() mode with dropout 0: x reaches the loss through the encoder, through x_t and
    through the reconstruction term."""
    args, m, sd = aux
    gl = torch.Generator().manual_seed(21)
    B = 4
    xb = torch.rand(B, 3, 64, 64, generator=gl) * 2 - 1
    idx = torch.randint(0, 1000, (B,), generator=gl)
    eps = torch.randn(B, 3, 64, 64, generator=gl)
    encn = torch.randn(B, 32, generator=gl)
    prior = torch.randn(B, 32, generator=gl)
    sdg = _grad_sd(sd)
    xr = xb.clone().requires_grad_()
    sch = orc.Schedule.make(args.beta1, args.betaT, args.diffusion_steps)
    orc.infodiff_loss(sdg, sch, xr, idx, eps, encn, prior, args.mmd_weight, args.kld_weight,
                      args.diffusion_steps)["loss"].backward()
    xd = xb.to(DEV).requires_grad_()
    real_ri, queue = torch.randint, [eps.clone(), encn.clone(), prior.clone()]
    torch.randint = lambda *a, **k: idx.to(DEV)
    try:
        with _train(m.backbone, m.encoder, dropout_p=0.0), _injected_randn_like(queue):
            m.zero_grad(set_to_none=True)
            m.train()
            m.loss_fn(args, xd).backward()
    finally:
        torch.randint = real_ri
        m.eval()
    _check_input_grad("train loss_fn x.grad", xd.grad, xr.grad, TOL_DX_TRAIN)


def test_train_input_gradient_with_dropout_satisfies_the_head_identity(aux):
    """With dropout on the oracle has no reference.  For a linear first layer h = W * x + b,
    <dL/dx, x> = <dL/dW, W> exactly; here x.grad comes from the head's data-gradient conv and head.weight.grad from the
    weight-gradient kernel, both over the same head-output gradient."""
    _, m, _ = aux
    x, t, a, G = _inputs(2, 64, seed=45)
    g = torch.Generator().manual_seed(46)
    G1 = torch.randn(2, 32, generator=g)
    torch.manual_seed(7)
    for name, net in (("backbone", m.backbone), ("encoder", m.encoder)):
        xd = x.to(DEV).requires_grad_()
        with _train(net):
            net.zero_grad(set_to_none=True)
            out = net(xd, t.to(DEV), a.to(DEV)) if name == "backbone" else net(xd)
            loss = (out * G.to(DEV)).sum() if name == "backbone" else (out[0] * G1.to(DEV)).sum() + out[2].square().sum()
            loss.backward()
        lhs = float((xd.grad.double() * xd.detach().double()).sum())
        w = net.head.weight
        rhs = float((w.grad.double() * w.detach().double()).sum())
        rel = abs(lhs - rhs) / abs(rhs)
        print(f"\n[autograd] {name} train, dropout {net.dropout_p}: <x.grad, x> = {lhs:.6e}, "
              f"<W.grad, W> = {rhs:.6e}, relative difference {rel:.3e}")
        assert rel < TOL_IDENTITY


# ------------------------------------------------------------------------------------------------
# nothing else moves
# ------------------------------------------------------------------------------------------------
def test_eval_call_without_input_grad_keeps_the_inference_plan(aux):
    """Grad mode on, eval(), inputs that need no gradient (run.py's save_latent): the inference plan, bit for bit,
    a result without a graph and no training plan."""
    _, m, _ = aux
    x, t, a, _ = _inputs(3, 64, seed=47)
    x, t, a = x.to(DEV), t.to(DEV), a.to(DEV)
    for net, call in ((m.backbone, lambda: m.backbone(x, t, a)), (m.encoder, lambda: m.encoder(x))):
        torch.cuda.manual_seed(5)
        with torch.no_grad():
            ref = call()
        keys = set(net._plans())
        torch.cuda.manual_seed(5)
        assert torch.is_grad_enabled()
        got = call()
        for r, o in zip(ref if isinstance(ref, tuple) else (ref,), got if isinstance(got, tuple) else (got,)):
            assert not o.requires_grad and torch.equal(o, r)
        assert set(net._plans()) == keys
        assert not any(str(k[0]).startswith("train") and k[1] == 3 for k in keys)


def test_differentiable_eval_call_leaves_the_generators_as_the_inference_call(aux):
    _, m, _ = aux
    x, t, a, _ = _inputs(2, 64, seed=48)
    x, t, a = x.to(DEV), t.to(DEV), a.to(DEV)
    calls = (("backbone", lambda xx: m.backbone(xx, t, a)), ("encoder", lambda xx: m.encoder(xx)[1]))
    for name, call in calls:
        torch.manual_seed(11)
        with torch.no_grad():
            call(x)
        want = torch.get_rng_state(), torch.cuda.get_rng_state()
        torch.manual_seed(11)
        out = call(x.clone().requires_grad_())
        assert out.requires_grad, name
        got = torch.get_rng_state(), torch.cuda.get_rng_state()
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), name


def test_input_gradient_adds_exactly_one_backward_launch(aux):
    """Two identical train steps, the second with x requiring grad: one launch more in backward, the rest unchanged."""
    from infodiffusion_b200 import _lib
    _, m, _ = aux
    net = m.backbone
    x, t, a, G = _inputs(2, 64, seed=49)
    x, t, a, G = x.to(DEV), t.to(DEV), a.to(DEV), G.to(DEV)
    counts = []
    with _train(net):
        for step in range(4):                   # eager, graph capture, then two replays
            xx = x.clone().requires_grad_() if step == 3 else x
            net.zero_grad(set_to_none=True)
            loss = (net(xx, t, a) * G).sum()
            torch.cuda.synchronize()
            n0 = _lib.launches()
            loss.backward()
            torch.cuda.synchronize()
            counts.append(_lib.launches() - n0)
            assert (xx.grad is not None) == (step == 3)
    print(f"\n[autograd] backward launches per step: {counts}")
    assert counts[3] == counts[2] + 1


def test_eval_input_gradients_are_reproducible_in_deterministic_mode(aux):
    _, m, _ = aux
    x, t, a, G = _inputs(2, 64, seed=50)
    x, t, a, G = x.to(DEV), t.to(DEV), a.to(DEV), G.to(DEV)
    runs = []
    with _deterministic():
        for _ in range(2):
            xd, ad = x.clone().requires_grad_(), a.clone().requires_grad_()
            (m.backbone(xd, t, ad) * G).sum().backward()
            xe = x.clone().requires_grad_()
            a_e, _, mu, _ = m.encoder(xe)
            (a_e.square().sum() + mu.sum()).backward()
            runs.append((xd.grad, ad.grad, xe.grad))
    m.zero_grad(set_to_none=True)
    for g0, g1 in zip(*runs):
        assert torch.equal(g0, g1)
