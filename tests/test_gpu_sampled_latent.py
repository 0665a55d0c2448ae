"""Reverse DDIM of a KLD model (kld_weight != 0) on the B200: every re-encoding step conditions the backbone on the
sampled latent a_q = mu + randn_like(mu) * exp(0.5 * log_var) (reference models.py:515, 714-721), computed by
idf_reparameterize_f32 inside the captured step.  The op against torch's composite, the trajectory against the fp32
CPU oracle with injected encoder noise, the random stream against the reference's, graph replay, chunking, the
unchanged MMD-only path and run.py's analysis modes."""
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch

from oracle import infodiff_oracle as orc
from oracle.golden_util import SEED, make_args, perturb_state_dict, rel_l2, step_noise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = Path(__file__).resolve().parent.parent
TOL_X = 4.3e-3        # 1.2 x the worst measured value, see tests/test_gpu_network.py
# eps of the re-encoding step on a_q: 2.24e-2 measured on B200, above the 2.1e-2 bound of the deterministic latent (a_q
# carries the encoder's error in both mu and log_var into the backbone); pinned at 1.2 x the measured value
TOL_EPS_KLD = 2.7e-2
T = 10
A_DIM = 32


def build(kld_weight, a_dim=A_DIM, steps=T):
    from infodiffusion_b200.models import InfoDiff
    args = make_args(a_dim=a_dim, diffusion_steps=steps, kld_weight=kld_weight)
    torch.manual_seed(SEED)
    m = InfoDiff(args, "cpu", (3, 64, 64))
    sd = perturb_state_dict(m.state_dict())
    m.load_state_dict(sd)
    m.device = DEV
    for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
        setattr(m, n, getattr(m, n).to(DEV))
    return args, m.to(DEV).eval(), sd


@pytest.fixture(scope="module")
def kld10():
    return build(0.5)


def _proc(args, m, graph=True, chunk=None):
    from infodiffusion_b200.sampling import DiffusionProcess
    args = make_args(**{**vars(args), "deterministic": True})
    args.cuda_graph = graph
    args.sample_chunk = chunk
    return DiffusionProcess(args, m, DEV, (3, 64, 64))


def _x0(B, seed=4):
    return torch.rand(B, 3, 64, 64, generator=torch.Generator().manual_seed(seed)) * 2 - 1


def _enc_noise(idx, B):
    return step_noise(idx, (B, A_DIM), seed=7)


def _torch_composite(mu, log_var, noise):
    return mu + noise * torch.exp(0.5 * log_var)


def _ulp_diff(a, b):
    ia, ib = a.view(torch.int32).long(), b.view(torch.int32).long()
    ia = torch.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = torch.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return int((ia - ib).abs().max()) if a.numel() else 0


def test_reparameterize_op_matches_torch_composite():
    """idf_reparameterize_f32 == mu + noise * torch.exp(0.5 * log_var) computed by torch on the GPU, bit for bit: float4
    body, scalar tail (n % 4 != 0) and the all-scalar path for pointers that are not 16-byte aligned."""
    from infodiffusion_b200 import _lib
    lib = _lib.load()
    _lib.check(lib.idf_init())
    g = torch.Generator(device=DEV).manual_seed(31)
    stream = torch.cuda.current_stream().cuda_stream
    for n in (1, 3, 4, 7, 2 * 32, 2 * 32 + 1, 64 * 256, 64 * 256 + 3, 1 << 20):
        for off in (0, 1):                                  # off = 1: every pointer 4 bytes past a 16-byte boundary
            mu, lv, z = (torch.randn(n + off, device=DEV, generator=g) * s for s in (1.0, 3.0, 1.0))
            out = torch.full((n + off,), float("nan"), device=DEV)
            _lib.check(lib.idf_reparameterize_f32(mu[off:].data_ptr(), lv[off:].data_ptr(), z[off:].data_ptr(),
                                                  out[off:].data_ptr(), n, stream))
            want = _torch_composite(mu[off:], lv[off:], z[off:])
            ulp = _ulp_diff(out[off:], want)
            assert torch.equal(out[off:], want), f"n={n} off={off}: differs from torch's composite by up to {ulp} ulp"
    # the edge of exp's range: overflow to inf, underflow to 0, and nan propagate like torch's
    lv = torch.tensor([200.0, -300.0, float("nan"), 0.0, 177.0, -207.0, 1e-30, -1e-30], device=DEV)
    mu, z = torch.ones_like(lv), torch.full_like(lv, -0.5)
    out = torch.empty_like(lv)
    _lib.check(lib.idf_reparameterize_f32(mu.data_ptr(), lv.data_ptr(), z.data_ptr(), out.data_ptr(), lv.numel(), stream))
    assert torch.equal(out.nan_to_num(7.0), _torch_composite(mu, lv, z).nan_to_num(7.0))


def test_encoder_forward_sampled_latent_is_the_torch_composite(kld10):
    """Encoder.forward (eval) draws randn_like(mu) once per call, as before, and its a_q equals the torch composite on
    the returned mu / log_var with that draw, bit for bit."""
    args, m, sd = kld10
    x = _x0(2).to(DEV)
    for B in (2, 1):
        torch.manual_seed(5)
        a, a_q, mu, lv = m.encoder(x[:B])
        state = torch.cuda.get_rng_state()
        torch.manual_seed(5)
        z = torch.randn_like(mu)
        assert torch.equal(torch.cuda.get_rng_state(), state)
        assert torch.equal(a_q, _torch_composite(mu, lv, z))


def _oracle_reverse(sd, args, x0, enc_noise):
    """reverse DDIM (sampling.py:62-87) with the re-encoding call conditioned on a_q (models.py:515, 714-721)."""
    def eps_fn(x, idx):
        t = torch.full((x.shape[0],), idx, dtype=torch.long)
        _, a_q, _, _ = orc.encoder_forward(sd, x, noise=enc_noise(idx))
        return orc.aux_unet_forward(sd, x, t, a_q)
    sch = orc.Schedule.make(args.beta1, args.betaT, args.diffusion_steps)
    with torch.no_grad():
        return [r for r in orc.ddim_reverse_steps(sch, eps_fn, x0) if r[0] > 0]


def test_kld_reverse_ddim_against_the_oracle(kld10):
    args, m, sd = kld10
    B = 2
    x0 = _x0(B)
    rec = _oracle_reverse(sd, args, x0, lambda idx: _enc_noise(idx, B))
    p = _proc(args, m)
    p.latent_noise_fn = lambda idx, out: out.copy_(_enc_noise(idx, B))
    trace = []
    xT = p.reverse_sampling(x0.to(DEV), trace=trace)
    assert [i for i, _, _ in trace] == [i for i, _, _ in rec] == list(range(1, T - 1))
    worst_e = max(rel_l2(e.cpu(), e_o) for (_, e, _), (_, e_o, _) in zip(trace, rec))
    worst_x = max(rel_l2(x.cpu(), x_o) for (_, _, x), (_, _, x_o) in zip(trace, rec))
    # the latent noise is live: the same trajectory with mu alone (zero noise) is far away
    mu_only = _oracle_reverse(sd, args, x0, lambda idx: torch.zeros(B, A_DIM))
    gap = rel_l2(xT.cpu(), mu_only[-1][2])
    print(f"\n[parity] KLD reverse-DDIM-{T}: worst per-step rel-L2 eps = {worst_e:.3e}, x_t = {worst_x:.3e}; "
          f"x_T vs the mu-only trajectory {gap:.3e}")
    assert torch.isfinite(xT).all()
    assert worst_e < TOL_EPS_KLD and worst_x < TOL_X
    assert gap > 5 * TOL_X


def test_default_draws_follow_the_reference_stream(kld10):
    """Default latent_noise_fn = one randn_like(mu) of [B, a_dim] on torch's CUDA generator per model call and no
    other draw: identical to a hook that copies successive torch.randn(B, a_dim) draws, generator state included."""
    args, m, sd = kld10
    B = 3
    x0 = _x0(B, seed=12).to(DEV)
    p = _proc(args, m)
    p.reverse_sampling(x0)                                   # plans built and graph captured outside the window

    def run(hook):
        p.latent_noise_fn = hook if hook is not None else (lambda idx, out: out.normal_())
        torch.manual_seed(77)
        xT = p.reverse_sampling(x0)
        return xT, torch.cuda.get_rng_state()
    x_def, st_def = run(None)
    x_hook, st_hook = run(lambda idx, out: out.copy_(torch.randn(B, A_DIM, device=DEV)))
    assert torch.equal(x_def, x_hook)
    assert torch.equal(st_def, st_hook)
    torch.manual_seed(77)
    for _ in range(T - 2):
        torch.randn(B, A_DIM, device=DEV)
    assert torch.equal(torch.cuda.get_rng_state(), st_def), "reverse DDIM drew something besides one latent per step"


def test_graph_replay_equals_eager_and_is_deterministic(kld10):
    args, m, sd = kld10
    B = 4
    x0 = _x0(B, seed=5).to(DEV)
    outs = []
    for graph in (True, False, True):
        p = _proc(args, m, graph=graph)
        p.latent_noise_fn = lambda idx, out: out.copy_(_enc_noise(idx, B))
        outs.append(p.reverse_sampling(x0))
    assert torch.equal(outs[0], outs[1]), "CUDA-graph replay differs from eager launches"
    assert torch.equal(outs[0], outs[2]), "run-to-run non-determinism"


def test_chunked_plans_read_the_same_latent_noise(kld10):
    """sample_chunk = B/2: each chunk's encoder plan reads its rows of the one full-batch noise buffer, so the result
    agrees with the unchunked run to round-off.  A sample's GroupNorm statistics are summed in a different order at a
    different batch position (tests/test_gpu_network.py bounds that at 2e-3 for sampling with a given latent); the
    re-encoding steps feed that difference back through the encoder and a_q, measured 2.5e-3 worst sample on B200
    (a wrong noise row would move a sample by ~1e-1), pinned at 1.2 x."""
    args, m, sd = kld10
    B = 8
    x0 = _x0(B, seed=6).to(DEV)

    def run(chunk):
        p = _proc(args, m, chunk=chunk)
        p.latent_noise_fn = lambda idx, out: out.copy_(_enc_noise(idx, B))
        s = p._sampler("reverse", B, with_encoder=True)
        assert s.latent_noise is not None and s.latent_noise.shape == (B, A_DIM)
        return p.reverse_sampling(x0), s
    full, s_full = run(None)
    half, s_half = run(B // 2)
    assert len(s_half.plans) == 2 * len(s_full.plans)
    err = rel_l2(half.cpu(), full.cpu())
    per = ((half - full).flatten(1).norm(dim=1) / full.flatten(1).norm(dim=1)).cpu()
    print(f"\n[property] KLD reverse DDIM, chunk {B // 2} vs {B}: rel-L2 {err:.3e}, worst sample {float(per.max()):.3e}")
    assert float(per.max()) < 3e-3


def test_mmd_reverse_path_is_unchanged():
    """kld_weight = 0: the re-encoding reverse sampler builds today's plans (encoder -> latent MLP on `a` -> backbone),
    allocates no latent noise, draws nothing, and its result equals those plans run by hand bit for bit."""
    from infodiffusion_b200.engine import (BackbonePlan, EncoderPlan, ModulationPack, ModulationTables, Plan, Workspace,
                                           conditioned_blocks)
    from infodiffusion_b200.sampling import step_coefficients
    args, m, sd = build(0.0)
    B = 2
    x0 = _x0(B).to(DEV)
    p = _proc(args, m, graph=False)
    p.latent_noise_fn = lambda idx, out: pytest.fail("an MMD model drew a latent")
    state = torch.cuda.get_rng_state()
    got = p.reverse_sampling(x0)
    assert torch.equal(torch.cuda.get_rng_state(), state)
    s = p._sampler("reverse", B, with_encoder=True)
    assert s.latent_noise is None
    assert all(op.tag != "reparameterize" for pl in s.plans for op in pl.ops)
    # the same step assembled from plans built without latent_noise
    net, dev = m.backbone, torch.device(DEV)
    x = x0.clone()
    step = torch.zeros(1, dtype=torch.int32, device=dev)
    coef = step_coefficients("reverse", p.betas.cpu(), p.alphas.cpu(), p.alpha_bars.cpu(),
                             p.alpha_prev_bars.cpu()).to(dev).contiguous()
    pack = ModulationPack(conditioned_blocks(net), dev)
    tables = ModulationTables(net, dev, pack, T)
    tables.run()
    mod_z = torch.zeros(B, pack.ncol, device=dev)
    ws = Workspace(B, dev)
    ep = EncoderPlan(m.encoder, B, dev, ws=ws, x_in=x)
    zp = Plan(B, dev, ws=ws)
    zp._emit_latent_mlp(net, pack, ep.a, mod_z)
    bp = BackbonePlan(net, B, dev, mode="sampler", ws=ws, x_io=x, coef=coef, step=step, mod_t_table=tables.table,
                      mod_z=mod_z, pack=pack)
    assert s.n_launch == sum(op.kernels for pl in (ep, zp, bp) for op in pl.ops)
    for idx in range(1, T - 1):
        step.fill_(idx)
        for pl in (ep, zp, bp):
            pl.run()
    assert torch.equal(got, x)


def test_run_py_analysis_modes_on_a_kld_model(tmp_path):
    """run.py --kld_weight 0.5: train, then latent_quality / interpolate / disentangle exit 0 and write their files
    under the _0.5kld experiment name."""
    common = ["--model", "diff", "--prior", "regular", "--dataset", "synthetic", "--a_dim", "32", "--batch_size", "4",
              "--epochs", "1", "--save_epochs", "1", "--diffusion_steps", "4", "--synthetic_size", "8", "--r_seed", "64",
              "--kld_weight", "0.5", "--model_folder", "./models", "--img_folder", "./imgs"]

    def run(args, *extra):
        r = subprocess.run([sys.executable, str(ROOT / "run.py"), *args, *extra], cwd=tmp_path, capture_output=True,
                           text=True, timeout=600, env={**os.environ, "PYTHONPATH": str(ROOT)})
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return r.stdout
    out = run(common, "--mode", "train")
    assert "Loss" in out and "nan" not in out.lower()
    exp = "synthetic_32d_0.5kld_0.1mmd"
    assert (tmp_path / "models" / exp / "model-1.pth").exists()
    run(common, "--mode", "latent_quality", "--sampling_number", "3")
    assert len(list((tmp_path / "imgs" / exp / "latent_quality").glob("sample-*.png"))) == 3
    run(common, "--mode", "interpolate", "--img_id", "1")
    assert (tmp_path / "imgs" / exp / "interpolate-1" / "sample0.png").exists()
    short = [c if c != "32" else "4" for c in common]            # a_dim 4: disentangle renders one grid per latent dim
    exp4 = "synthetic_4d_0.5kld_0.1mmd"
    run(short, "--mode", "train")
    run(short, "--mode", "disentangle", "--img_id", "0")
    assert sorted(p.name for p in (tmp_path / "imgs" / exp4 / "disentangle-0").glob("*.png")) == \
        [f"sample{k}.png" for k in range(4)]


def test_two_phase_reverse_sampling_on_a_kld_model(kld10):
    from infodiffusion_b200.models import Diff
    from infodiffusion_b200.sampling import TwoPhaseDiffusionProcess
    args, m, sd = kld10
    vargs = make_args(**{**vars(args), "model": "vanilla", "mmd_weight": 0.0, "kld_weight": 0.0})
    torch.manual_seed(SEED)
    vanilla = Diff(vargs, "cpu", (3, 64, 64)).to(DEV).eval()
    proc = TwoPhaseDiffusionProcess(make_args(**{**vars(args), "deterministic": True}), m, vanilla, DEV, (3, 64, 64))
    x0 = _x0(2).to(DEV)
    xT = proc.reverse_sampling(x0)
    assert xT.shape == x0.shape and torch.isfinite(xT).all()
    assert float((xT - x0).abs().mean()) > 1e-3
