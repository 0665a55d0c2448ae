"""DDPM / DDIM / reverse-DDIM step loops -- mirror of the reference's ``sampling.py``.

Same class and method names as the reference (sampling.py:3-101): ``DiffusionProcess(args,
diffusion_fn, device, shape)`` with ``.sampling(sampling_number, xT, a)`` and
``.reverse_sampling(x0, a)``.  The loop body is different: one step is a single CUDA-graph replay of
the whole UNet with the x_{t-1} update fused into the output convolution's epilogue; per-step values
come from device tables indexed by a device-resident step counter, so the host does nothing per
step except (for stochastic steps, and for the sampled latent of a KLD model's re-encoding reverse
steps) drawing that step's noise with torch's generator, in the reference's order, so identical
seeds give identical noise.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import _lib
from .engine import (BackbonePlan, EncoderPlan, ModulationPack, ModulationTables, Plan, Workspace,
                     conditioned_blocks)


def make_schedule(beta1: float, betaT: float, T: int):
    """fp32 schedule exactly as the reference builds it (sampling.py:12-15)."""
    betas = torch.linspace(start=beta1, end=betaT, steps=T)
    alphas = 1 - betas
    alpha_bars = torch.cumprod(1 - torch.linspace(start=beta1, end=betaT, steps=T), dim=0)
    alpha_prev_bars = torch.cat([torch.Tensor([1]), alpha_bars[:-1]])
    return betas, alphas, alpha_bars, alpha_prev_bars


def step_coefficients(kind: str, betas, alphas, alpha_bars, alpha_prev_bars) -> torch.Tensor:
    """[T, 3] table (cx, ce, cn) with  x_next = cx*x + ce*eps + cn*noise  for step index idx.

    Derived from the reference's update formulas (DDPM sampling.py:30-37, DDIM 52-59 with eta = 0.01
    and alpha_prev_bars[idx] as the current abar, reverse DDIM 71-72); evaluated in float64 from the
    fp32 schedule so the collapsed form carries no extra cancellation error.
    """
    b, al, ab, apb = (t.double() for t in (betas, alphas, alpha_bars, alpha_prev_bars))
    T = len(ab)
    out = torch.zeros(T, 3, dtype=torch.float64)
    for i in range(T):
        if kind == "ddpm":
            cx = torch.sqrt(1 / al[i])
            ce = -cx * b[i] / torch.sqrt(1 - ab[i])
            cn = torch.sqrt((1 - apb[i]) / (1 - ab[i]) * b[i]) if i > 0 else torch.zeros(())
        elif kind == "ddim":
            inv = 1 / torch.sqrt(apb[i])
            if i == 0:
                cx, ce, cn = inv, -torch.sqrt(1 - apb[0]) * inv, torch.zeros(())
            else:
                sigma = 0.01 * torch.sqrt((1 - apb[i - 1]) / (1 - ab[i - 1])) * torch.sqrt(b[i - 1])
                cx = torch.sqrt(apb[i - 1]) * inv
                ce = torch.sqrt(1 - apb[i - 1] - sigma ** 2) - torch.sqrt(apb[i - 1]) * torch.sqrt(1 - apb[i]) * inv
                cn = sigma
        elif kind == "reverse":
            if i == 0 or i + 1 >= T:
                cx, ce, cn = torch.ones(()), torch.zeros(()), torch.zeros(())   # idx 0 yields x unchanged
            else:
                inv = 1 / torch.sqrt(apb[i])
                cx = torch.sqrt(apb[i + 1]) * inv
                ce = torch.sqrt(1 - apb[i + 1]) - torch.sqrt(apb[i + 1]) * torch.sqrt(1 - apb[i]) * inv
                cn = torch.zeros(())
        else:
            raise ValueError(kind)
        out[i, 0], out[i, 1], out[i, 2] = cx, ce, cn
    return out.float()


def _capture_step(enqueue, x: torch.Tensor, step: torch.Tensor, idx: int) -> torch.cuda.CUDAGraph:
    """CUDA graph of one sampler step.  `enqueue` runs once on a side stream first (kernel attributes are set outside
    the capture); that warm-up updates the live buffer x in place, so x is restored and the step counter refilled."""
    dev = x.device
    keep = x.clone()
    torch.cuda.synchronize(dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        enqueue()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enqueue()
    x.copy_(keep)
    step.fill_(idx)
    return g


class _FusedSampler:
    """Graph-captured step for an InfoDiff model: UNet forward + fused x update, for a fixed batch."""

    def __init__(self, proc: "DiffusionProcess", kind: str, batch: int, chunk: Optional[int] = None,
                 record_eps: bool = False, with_encoder: bool = False):
        model = proc.diffusion_fn
        net = model.backbone
        dev = proc.device
        self.kind, self.B = kind, batch
        T = len(proc.alpha_bars)
        self.T = T
        Cimg, H, W = net.shape
        f32 = dict(dtype=torch.float32, device=dev)
        self.x = torch.zeros(batch, Cimg, H, W, **f32)
        self.noise = torch.zeros(batch, Cimg, H, W, **f32) if kind != "reverse" else None
        self.eps = torch.zeros(batch, Cimg, H, W, **f32) if record_eps else None
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.coef = step_coefficients(kind, proc.betas.cpu(), proc.alphas.cpu(), proc.alpha_bars.cpu(),
                                      proc.alpha_prev_bars.cpu()).to(dev).contiguous()
        self.pack = ModulationPack(conditioned_blocks(net), dev)
        self.tables = ModulationTables(net, dev, self.pack, T)
        self.tables.run()
        self.mod_z = torch.zeros(batch, self.pack.ncol, **f32)
        # a KLD model conditions the re-encoded step on a_q = mu + noise * exp(0.5 * log_var) (models.py:515, 714-721):
        # one full-batch noise buffer, refilled before every step, so chunked plans read the same values
        sampled = with_encoder and model._uses_sampled_latent()
        self.latent_noise = torch.zeros(batch, model.encoder.a_dim, **f32) if sampled else None
        chunk = batch if chunk is None else min(chunk, batch)
        assert batch % chunk == 0, "chunk must divide the batch"
        # lanes: micro-batches on different lanes run on different streams (own workspace each), so the small
        # latency-bound layers of one micro-batch overlap with the other's work
        n_lanes = max(1, min(int(getattr(proc, "lanes", 1)), batch // chunk))
        self.lane_ws = [Workspace(chunk, dev) for _ in range(n_lanes)]
        self.lane_plans: List[List[Plan]] = [[] for _ in range(n_lanes)]
        self.lane_streams = [None] + [torch.cuda.Stream(dev) for _ in range(n_lanes - 1)]
        self.ws = self.lane_ws[0]
        self.plans: List[Plan] = []
        for ci, c0 in enumerate(range(0, batch, chunk)):
            sl = slice(c0, c0 + chunk)
            lane = ci % n_lanes
            self.ws = self.lane_ws[lane]
            n_before = len(self.plans)
            if with_encoder:
                # bug-compatible reverse DDIM: re-encode the current x_t every step (sampling.py:84,
                # models.py:709-710) and derive this chunk's z-modulation rows from the fresh latent
                ep = EncoderPlan(model.encoder, chunk, dev, ws=self.ws, x_in=self.x[sl],
                                 latent_noise=self.latent_noise[sl] if sampled else None)
                zp = Plan(chunk, dev, ws=self.ws)
                zp._emit_latent_mlp(net, self.pack, ep.a_q if sampled else ep.a, self.mod_z[sl])
                self.plans += [ep, zp]
            bp = BackbonePlan(net, chunk, dev, mode="sampler", ws=self.ws, x_io=self.x[sl],
                              noise=None if self.noise is None else self.noise[sl], coef=self.coef, step=self.step,
                              mod_t_table=self.tables.table, mod_z=self.mod_z[sl],
                              eps_out=None if self.eps is None else self.eps[sl], pack=self.pack)
            self.plans.append(bp)
            self.lane_plans[lane] += self.plans[n_before:]
        self.ws = self.lane_ws[0]
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.n_launch = sum(op.kernels for p in self.plans for op in p.ops)

    def set_latent(self, a: torch.Tensor) -> None:
        self.tables.latent_rows(a.contiguous().float(), self.mod_z)

    def _enqueue(self) -> None:
        if len(self.lane_plans) == 1:
            for p in self.plans:
                p.run()
            return
        cur = torch.cuda.current_stream(self.x.device)
        for st in self.lane_streams[1:]:                 # fork (also valid inside a graph capture)
            st.wait_stream(cur)
        for plans, st in zip(self.lane_plans, self.lane_streams):
            with torch.cuda.stream(st if st is not None else cur):
                for p in plans:
                    p.run()
        for st in self.lane_streams[1:]:                 # join
            cur.wait_stream(st)

    def run_step(self, idx: int, use_graph: bool = True) -> None:
        self.step.fill_(idx)
        if not use_graph:
            self._enqueue()
            return
        if self.graph is None:
            self.graph = _capture_step(self._enqueue, self.x, self.step, idx)
        self.graph.replay()
        _lib.count_launch(self.n_launch)


class DiffusionProcess():
    """Drop-in for the reference's DiffusionProcess (sampling.py:3-101)."""

    def __init__(self, args, diffusion_fn, device, shape):
        self.betas, self.alphas, ab, apb = make_schedule(args.beta1, args.betaT, args.diffusion_steps)
        self.alpha_bars = ab.to(device=device)
        self.alpha_prev_bars = apb.to(device=device)
        self.shape = shape
        self.deterministic = args.deterministic
        self.a_dim = args.a_dim
        self.model = args.model
        self.diffusion_fn = diffusion_fn.to(device=device)
        self.device = device
        self.chunk = getattr(args, "sample_chunk", None)      # micro-batch per graph segment (None = whole batch)
        self.lanes = int(getattr(args, "sample_lanes", 1))    # concurrent streams the micro-batches are spread over
        self.use_graph = getattr(args, "cuda_graph", True)
        self.honor_latent_in_reverse = getattr(args, "reverse_uses_given_latent", False)
        # noise_fn(idx, out) fills `out` with the step's N(0,1) noise; the default draws from torch's CUDA
        # generator exactly where the reference calls torch.randn_like (parity tests inject fixed tensors)
        self.noise_fn = lambda idx, out: out.normal_()
        # latent_noise_fn(idx, out) fills `out` [B, a_dim] with the N(0,1) draw of the encoder's sampled latent before
        # every re-encoding reverse step of a KLD model: the reference's one randn_like(mu) per model call (models.py:515)
        self.latent_noise_fn = lambda idx, out: out.normal_()
        self._samplers = {}

    # ------------------------------------------------------------------------------------------
    def _sampler(self, kind: str, batch: int, record_eps: bool = False, with_encoder: bool = False) -> _FusedSampler:
        net = getattr(self.diffusion_fn, "backbone", None)
        if net is None or not hasattr(net, "head"):
            raise NotImplementedError("DiffusionProcess drives the image UNets (InfoDiff / Diff over a UNet backbone); "
                                      "use LatentDiffusionProcess for a LatentUNet")
        if net.training:
            raise RuntimeError("sampling runs the inference forward; call model.eval() first")
        sig = tuple(m.weights_signature() for m in self.diffusion_fn.children() if hasattr(m, "weights_signature"))
        if getattr(self, "_sig", None) != sig:          # the weights moved since the samplers packed them
            self._samplers.clear()
            self._sig = sig
        key = (kind, batch, record_eps, with_encoder)
        if key not in self._samplers:
            self._samplers[key] = _FusedSampler(self, kind, batch, self.chunk, record_eps, with_encoder)
        return self._samplers[key]

    def _iter(self, kind: str, x: torch.Tensor, a: Optional[torch.Tensor], record_eps: bool = False):
        """Generator over the steps of one trajectory: yields (idx, sampler) after every update; sampler.x is the
        live x buffer (clone it to keep a step)."""
        B = x.shape[0]
        T = len(self.alpha_bars)
        vanilla = self.model == 'vanilla'                  # diffusion_fn(x, idx): no latent (sampling.py:31-32)
        with_encoder = (kind == "reverse") and (a is None) and not vanilla
        s = self._sampler(kind, B, record_eps=record_eps, with_encoder=with_encoder)
        s.x.copy_(x)
        if a is not None and not vanilla:
            s.set_latent(a)
        if kind == "reverse":
            order = range(1, T - 1)                     # idx 0 yields x unchanged (sampling.py:64-65)
        else:
            order = reversed(range(T))
        for idx in order:
            if kind != "reverse" and idx > 0:
                # ddpm: drawn BEFORE the model call (sampling.py:29); ddim: the reference draws it after the model
                # call (sampling.py:56) -- the model call consumes no random numbers, so the stream is identical
                self.noise_fn(idx, s.noise)
            if s.latent_noise is not None:
                self.latent_noise_fn(idx, s.latent_noise)
            s.run_step(idx, use_graph=self.use_graph)
            yield idx, s

    def _run(self, kind: str, x: torch.Tensor, a: Optional[torch.Tensor], trace=None) -> torch.Tensor:
        s = None
        for idx, s in self._iter(kind, x, a, record_eps=trace is not None):
            if trace is not None:
                trace.append((idx, s.eps.clone(), s.x.clone()))
        return s.x.clone() if s is not None else x.clone()

    # ---- the reference's generator methods: one x per step (sampling.py:23-79) --------------------------
    @torch.no_grad()
    def _ddpm_one_diffusion_step(self, x, a=None):
        for _, s in self._iter("ddpm", x, a):
            yield s.x.clone()

    @torch.no_grad()
    def _ddim_one_diffusion_step(self, x, a=None):
        for _, s in self._iter("ddim", x, a):
            yield s.x.clone()

    @torch.no_grad()
    def _ddim_one_reverse_diffusion_step(self, x, a=None):
        yield x                                          # idx == 0 (sampling.py:64-65)
        for _, s in self._iter("reverse", x, a):
            yield s.x.clone()

    def _one_diffusion_step(self, sample, a=None, deterministic=False):
        return self._ddim_one_diffusion_step(sample, a) if deterministic else self._ddpm_one_diffusion_step(sample, a)

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def reverse_sampling(self, x0, a=None, trace=None):
        """x0 -> xT by deterministic reverse DDIM (reference sampling.py:81-87).  The reference drops
        ``a`` and re-encodes x_t at every step (SURVEY H5a); that is the default here too.  Set
        ``args.reverse_uses_given_latent = True`` to honour the caller's ``a`` instead.  A KLD model
        (kld_weight != 0) conditions each re-encoded step on the sampled latent a_q, whose noise
        ``latent_noise_fn`` draws before the step (models.py:515, 714-721)."""
        if not self.honor_latent_in_reverse:
            a = None
        return self._run("reverse", x0, a, trace)

    @torch.no_grad()
    def sampling(self, sampling_number=16, xT=None, a=None, trace=None):
        """reference sampling.py:89-101: draws xT then a (in that order) when they are not given."""
        if xT is None:
            xT = torch.randn([sampling_number, *self.shape]).to(device=self.device)
        if self.model != 'vanilla' and a is None:          # sampling.py:93-95: a vanilla model draws no latent
            a = torch.randn([sampling_number, self.a_dim]).to(device=self.device)
        return self._run("ddim" if self.deterministic else "ddpm", xT, a, trace)


class TwoPhaseDiffusionProcess():
    """Drop-in for the reference's TwoPhaseDiffusionProcess (sampling.py:104-204): diffusion_fn_1 is the InfoDiff
    model (x, idx, a), diffusion_fn_2 the vanilla Diff model (x, idx).

    Bug compatibility (SURVEY H5b): the reference hands the step counter to its generators by value when they
    are created (t = 0, sampling.py:198-201), so `t <= split_step` never changes and diffusion_fn_2 runs every
    step whenever split_step >= 0.  That is the default here.  `args.two_phase_fix = True` makes the counter
    advance: steps with t <= split_step use diffusion_fn_2, later steps diffusion_fn_1."""

    def __init__(self, args, diffusion_fn_1, diffusion_fn_2, device, shape):
        import copy
        self.split_step = args.split_step
        self.deterministic = args.deterministic
        self.a_dim = args.a_dim
        self.shape = shape
        self.device = device
        self.fix = bool(getattr(args, "two_phase_fix", False))
        a1, a2 = copy.copy(args), copy.copy(args)
        a1.model, a2.model = "diff", "vanilla"
        self.p1 = DiffusionProcess(a1, diffusion_fn_1, device, shape)
        self.p2 = DiffusionProcess(a2, diffusion_fn_2, device, shape)
        self.diffusion_fn_1, self.diffusion_fn_2 = self.p1.diffusion_fn, self.p2.diffusion_fn
        self.betas, self.alphas = self.p1.betas, self.p1.alphas
        self.alpha_bars, self.alpha_prev_bars = self.p1.alpha_bars, self.p1.alpha_prev_bars
        self.noise_fn = lambda idx, out: out.normal_()

    @torch.no_grad()
    def sampling(self, sampling_number=16, xT=None, a=None):
        if xT is None:
            xT = torch.randn([sampling_number, *self.shape]).to(device=self.device)
        if a is None:
            a = torch.randn([sampling_number, self.a_dim]).to(device=self.device)
        kind = "ddim" if self.deterministic else "ddpm"
        self.p1.noise_fn = self.p2.noise_fn = self.noise_fn
        if not self.fix:
            proc = self.p2 if 0 <= self.split_step else self.p1
            return proc._run(kind, xT, a)
        # intended behaviour: switch networks along the trajectory; x moves between the two samplers' buffers
        B, T = xT.shape[0], len(self.alpha_bars)
        s1, s2 = self.p1._sampler(kind, B), self.p2._sampler(kind, B)
        s1.set_latent(a)
        cur = None
        x = xT
        for t, idx in enumerate(reversed(range(T))):
            s, proc = (s2, self.p2) if t <= self.split_step else (s1, self.p1)
            if s is not cur:
                s.x.copy_(x if cur is None else cur.x)
                cur = s
            if idx > 0:
                self.noise_fn(idx, s.noise)
            s.run_step(idx, use_graph=proc.use_graph)
        return cur.x.clone()

    @torch.no_grad()
    def reverse_sampling(self, x0, a=None):
        """reference sampling.py:189-195: diffusion_fn_1 with a dropped (the encoder is re-run every step)."""
        return self.p1.reverse_sampling(x0, None)


class LatentDiffusionProcess():
    """Drop-in for the reference's LatentDiffusionProcess (sampling.py:207-291): DDPM / DDIM / reverse DDIM over the
    latent z [B, a_dim] with diffusion_fn(z, idx) = Diff over a LatentUNet.  One CUDA graph per (kind, batch): 20
    launches of the MLP plus the fused z update, the timestep entering through a device-side step counter."""

    def __init__(self, args, diffusion_fn, device):
        self.betas, self.alphas, ab, apb = make_schedule(args.beta1, args.betaT, args.diffusion_steps)
        self.alpha_bars = ab.to(device=device)
        self.alpha_prev_bars = apb.to(device=device)
        self.deterministic = args.deterministic
        self.a_dim = args.a_dim
        self.model = args.model
        self.diffusion_fn = diffusion_fn.to(device=device)
        self.device = device
        self.use_graph = getattr(args, "cuda_graph", True)
        self.noise_fn = lambda idx, out: out.normal_()
        self._samplers = {}

    def _sampler(self, kind: str, batch: int):
        from .engine import LatentPlan
        net = self.diffusion_fn.backbone
        if net.training:
            raise RuntimeError("sampling runs the inference forward; call model.eval() first")
        sig = net.weights_signature()
        if getattr(self, "_sig", None) != sig:
            self._samplers.clear()
            self._sig = sig
        key = (kind, batch)
        if key not in self._samplers:
            dev = self.device
            T = len(self.alpha_bars)
            D = net.layers[0].linear.in_features
            s = type("LatentSampler", (), {})()
            s.x = torch.zeros(batch, D, dtype=torch.float32, device=dev)
            s.noise = torch.zeros_like(s.x) if kind != "reverse" else None
            s.eps = torch.zeros_like(s.x)
            s.step = torch.zeros(1, dtype=torch.int32, device=dev)
            s.coef = step_coefficients(kind, self.betas.cpu(), self.alphas.cpu(), self.alpha_bars.cpu(),
                                       self.alpha_prev_bars.cpu()).to(dev).contiguous()
            s.plan = LatentPlan(net, batch, dev, mode="sampler", T=T, z_io=s.x, noise=s.noise, coef=s.coef, step=s.step,
                                eps_out=s.eps)
            s.graph = None
            self._samplers[key] = s
        return self._samplers[key]

    def _step(self, s, idx: int) -> None:
        s.step.fill_(idx)
        if not self.use_graph:
            s.plan.run()
            return
        if s.graph is None:
            s.graph = _capture_step(s.plan.run, s.x, s.step, idx)
        s.graph.replay()
        _lib.count_launch(sum(op.kernels for op in s.plan.ops))

    def _iter(self, kind: str, x: torch.Tensor):
        T = len(self.alpha_bars)
        s = self._sampler(kind, x.shape[0])
        s.x.copy_(x)
        order = range(1, T - 1) if kind == "reverse" else reversed(range(T))
        for idx in order:
            if kind != "reverse" and idx > 0:
                self.noise_fn(idx, s.noise)
            self._step(s, idx)
            yield idx, s

    @torch.no_grad()
    def _ddpm_one_diffusion_step(self, x):
        for _, s in self._iter("ddpm", x):
            yield s.x.clone()

    @torch.no_grad()
    def _ddim_one_diffusion_step(self, x):
        for _, s in self._iter("ddim", x):
            yield s.x.clone()

    @torch.no_grad()
    def _ddim_one_reverse_diffusion_step(self, x):
        yield x
        for _, s in self._iter("reverse", x):
            yield s.x.clone()

    def _one_diffusion_step(self, sample, deterministic=False):
        return self._ddim_one_diffusion_step(sample) if deterministic else self._ddpm_one_diffusion_step(sample)

    @torch.no_grad()
    def reverse_sampling(self, x0):
        s = None
        for _, s in self._iter("reverse", x0):
            pass
        return s.x.clone() if s is not None else x0.clone()

    @torch.no_grad()
    def sampling(self, sampling_number=16, xT=None):
        if xT is None:
            xT = torch.randn([sampling_number, self.a_dim]).to(device=self.device)
        s = None
        for _, s in self._iter("ddim" if self.deterministic else "ddpm", xT):
            pass
        return s.x.clone()
