"""InfoDiffusion networks and model wrappers -- host-side mirror of the reference's ``models.py``.

Same class names, constructor arguments, ``forward`` signatures, attributes and ``state_dict`` keys
as the reference (models.py:7-779), so ``run.py``-style callers and checkpoints switch over
unchanged.  All tensor arithmetic is executed by the sm_100a kernels of libidf_b200.so through
``infodiffusion_b200.engine``; nothing here falls back to PyTorch ops or to the CPU.
"""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.nn import init

from .modules import (AuxResBlock, DownSample, ResBlock, ResBlock_encoder, TimeEmbedding, UpSample,
                      timestep_embedding)
from .utils import compute_mmd


def _unet_stacks(make_block, ch, ch_mult, attn, num_res_blocks, mid_factory):
    """Shared down / middle / up topology of every UNet-shaped network in the reference
    (models.py:16-46, 248-278, 342-372, 432-462)."""
    down, up = nn.ModuleList(), nn.ModuleList()
    widths = [ch]
    cur = ch
    for level, mult in enumerate(ch_mult):
        out = ch * mult
        for _ in range(num_res_blocks):
            down.append(make_block(cur, out, level in attn))
            cur = out
            widths.append(cur)
        if level != len(ch_mult) - 1:
            down.append(DownSample(cur))
            widths.append(cur)
    mid = mid_factory(cur)
    for level, mult in reversed(list(enumerate(ch_mult))):
        out = ch * mult
        for _ in range(num_res_blocks + 1):
            up.append(make_block(widths.pop() + cur, out, level in attn))
            cur = out
        if level != 0:
            up.append(UpSample(cur))
    assert not widths
    return down, mid, up, cur


def _tail(cur, out_ch):
    return nn.Sequential(nn.GroupNorm(32, cur), nn.SiLU(), nn.Conv2d(cur, out_ch, 3, stride=1, padding=1))


class _EngineNet(nn.Module):
    """Common plumbing: lazily builds (and caches per batch size) the kernel plan for this network."""

    def weights_signature(self):
        """Changes whenever a parameter is updated in place (optimizer step), replaced (.to(), load_state_dict) or
        written by the fused optimizer; inference plans hold packed bf16 copies of the weights and are keyed on it."""
        from ._lib import weight_epoch
        ver = ptr = 0
        for p in self.parameters():
            ver += p._version
            ptr += p.data_ptr()
        return (weight_epoch(), ver, ptr)

    def _plans(self):
        d = self.__dict__.setdefault("_idf_plans", {})
        sig = self.weights_signature()
        if self.__dict__.get("_idf_sig") != sig:
            for k in [k for k in d if not str(k[0]).startswith("train")]:   # training plans re-pack every step
                del d[k]
            self.__dict__["_idf_sig"] = sig
        return d

    def invalidate_plans(self):
        """Drop packed bf16 weights / workspaces (call after the fp32 parameters change)."""
        self._plans().clear()
        self.__dict__.pop("_idf_stack_params", None)

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self.invalidate_plans()
        return out

    def _differentiable(self, *inputs) -> bool:
        """The routing rule of every forward: autograd through the kernels' backward when grad mode is on and either
        the module is in train mode or a tensor input requires grad.  Every other call keeps the fused inference plan,
        including an eval() call whose inputs need no gradient (parameters that require grad do not count, or every
        such call would run on a training plan)."""
        return torch.is_grad_enabled() and (self.training or any(torch.is_tensor(v) and v.requires_grad for v in inputs))

    def _dropout(self):
        """(seed, p) of the differentiable forward.  train(): the hash-dropout seed comes from torch's CPU generator, so
        it follows torch.manual_seed.  eval(): dropout is off and nothing is drawn, so the call leaves torch's
        generators where the inference call leaves them."""
        if not self.training:
            return 0, 0.0
        return int(torch.empty((), dtype=torch.int64).random_().item()), self.dropout_p


class AuxiliaryUNet(_EngineNet):
    """eps-network conditioned on timestep t and auxiliary latent a (reference models.py:237-326)."""

    def __init__(self, T, ch=64, ch_mult=[1, 2, 4, 8], attn=[2], num_res_blocks=2, dropout=0.1, a_dim=32, shape=None):
        super().__init__()
        assert all(i < len(ch_mult) for i in attn), 'attn index out of bound'
        tdim = ch * 4
        self.a_dim = a_dim
        self.dropout_p = float(dropout)
        self.T, self.ch, self.ch_mult, self.shape = T, ch, list(ch_mult), tuple(shape)
        self.time_embedding = TimeEmbedding(T, ch, tdim)
        self.fc_a = nn.Linear(a_dim, tdim)
        self.head = nn.Conv2d(shape[0], ch, kernel_size=3, stride=1, padding=1)
        self.downblocks, self.middleblocks, self.upblocks, cur = _unet_stacks(
            lambda i, o, at: AuxResBlock(in_ch=i, out_ch=o, tdim=tdim, dropout=dropout, attn=at),
            ch, ch_mult, attn, num_res_blocks,
            lambda c: nn.ModuleList([AuxResBlock(c, c, tdim, dropout, attn=True, crossattn=False),
                                     AuxResBlock(c, c, tdim, dropout, attn=False, crossattn=False)]))
        self.tail = _tail(cur, shape[0])
        init.xavier_uniform_(self.head.weight)
        init.zeros_(self.head.bias)
        init.xavier_uniform_(self.fc_a.weight)
        init.zeros_(self.fc_a.bias)
        init.xavier_uniform_(self.tail[-1].weight, gain=1e-5)
        init.zeros_(self.tail[-1].bias)

    def forward(self, x, t, a):
        """x [B,C,H,W] fp32, t int64 [B], a [B,a_dim] -> eps [B,C,H,W] fp32 (reference models.py:296).
        train() with grad: dropout on and autograd through the kernels' backward.  eval() with grad and x or a
        requiring grad: the same path with dropout off.  Otherwise: the inference plan."""
        if self._differentiable(x, a):
            from .train import backbone_train_forward
            return backbone_train_forward(self, x, t, a, *self._dropout())
        from .engine import backbone_forward
        return backbone_forward(self, x, t, a)


class UNet(_EngineNet):
    """Unconditional eps-network of the vanilla diffusion model (reference models.py:7-88).  The reference's
    constructor crashes at HEAD (it passes crossattn= to ResBlock, models.py:32-33); here ResBlock accepts and
    ignores the keyword, everything else -- names, init order, forward(x, t) -- is the reference's."""

    def __init__(self, T, ch=64, ch_mult=[1, 2, 4, 8], attn=[2], num_res_blocks=2, dropout=0.1, shape=None):
        super().__init__()
        assert all(i < len(ch_mult) for i in attn), 'attn index out of bound'
        tdim = ch * 4
        self.dropout_p = float(dropout)
        self.T, self.ch, self.ch_mult, self.shape = T, ch, list(ch_mult), tuple(shape)
        self.time_embedding = TimeEmbedding(T, ch, tdim)
        self.head = nn.Conv2d(shape[0], ch, kernel_size=3, stride=1, padding=1)
        self.downblocks, self.middleblocks, self.upblocks, cur = _unet_stacks(
            lambda i, o, at: ResBlock(in_ch=i, out_ch=o, tdim=tdim, dropout=dropout, attn=at),
            ch, ch_mult, attn, num_res_blocks,
            lambda c: nn.ModuleList([ResBlock(c, c, tdim, dropout, attn=True, crossattn=False),
                                     ResBlock(c, c, tdim, dropout, attn=False, crossattn=False)]))
        self.tail = _tail(cur, shape[0])
        init.xavier_uniform_(self.head.weight)
        init.zeros_(self.head.bias)
        init.xavier_uniform_(self.tail[-1].weight, gain=1e-5)
        init.zeros_(self.tail[-1].bias)

    def forward(self, x, t):
        """x [B,C,H,W] fp32, t int64 [B] -> eps (reference models.py:62)."""
        if self._differentiable(x):
            from .train import backbone_train_forward
            return backbone_train_forward(self, x, t, None, *self._dropout())
        from .engine import backbone_forward
        return backbone_forward(self, x, t, None)


class BottleneckAuxUNet(_EngineNet):
    """eps-network whose only latent-conditioned blocks are the two middle AuxResBlocks; down / up blocks are
    plain ResBlocks and fc_a = SiLU -> Linear with kaiming init (reference models.py:329-421)."""

    def __init__(self, T, ch=64, ch_mult=[1, 2, 4, 8], attn=[2], num_res_blocks=2, dropout=0.1, a_dim=32, shape=None):
        super().__init__()
        assert all(i < len(ch_mult) for i in attn), 'attn index out of bound'
        tdim = ch * 4
        self.a_dim = a_dim
        self.dropout_p = float(dropout)
        self.T, self.ch, self.ch_mult, self.shape = T, ch, list(ch_mult), tuple(shape)
        self.time_embedding = TimeEmbedding(T, ch, tdim)
        self.fc_a = nn.Sequential(nn.SiLU(), nn.Linear(self.a_dim, tdim))
        self.head = nn.Conv2d(shape[0], ch, kernel_size=3, stride=1, padding=1)
        self.downblocks, self.middleblocks, self.upblocks, cur = _unet_stacks(
            lambda i, o, at: ResBlock(in_ch=i, out_ch=o, tdim=tdim, dropout=dropout, attn=at),
            ch, ch_mult, attn, num_res_blocks,
            lambda c: nn.ModuleList([AuxResBlock(c, c, tdim, dropout, attn=True, crossattn=False),
                                     AuxResBlock(c, c, tdim, dropout, attn=False, crossattn=False)]))
        self.tail = _tail(cur, shape[0])
        init.xavier_uniform_(self.head.weight)
        init.zeros_(self.head.bias)
        init.kaiming_normal_(self.fc_a[1].weight, a=0, nonlinearity='relu')
        init.xavier_uniform_(self.tail[-1].weight, gain=1e-5)
        init.zeros_(self.tail[-1].bias)

    def forward(self, x, t, a):
        if self._differentiable(x, a):
            from .train import backbone_train_forward
            return backbone_train_forward(self, x, t, a, *self._dropout())
        from .engine import backbone_forward
        return backbone_forward(self, x, t, a)


class Encoder(_EngineNet):
    """UNet-shaped encoder x -> (a, a_q, mu, log_var) (reference models.py:424-518)."""

    def __init__(self, ch=64, ch_mult=[1, 2, 4, 8, 8], attn=[2], num_res_blocks=2, dropout=0.1, a_dim=32, shape=None):
        super().__init__()
        assert all(i < len(ch_mult) for i in attn), 'attn index out of bound'
        self.shape = shape
        self.a_dim = a_dim
        self.dropout_p = float(dropout)
        self.ch, self.ch_mult = ch, list(ch_mult)
        self.head = nn.Conv2d(shape[0], ch, kernel_size=3, stride=1, padding=1)
        self.downblocks, self.middleblocks, self.upblocks, cur = _unet_stacks(
            lambda i, o, at: ResBlock_encoder(in_ch=i, out_ch=o, dropout=dropout, attn=at),
            ch, ch_mult, attn, num_res_blocks,
            lambda c: nn.ModuleList([ResBlock_encoder(c, c, dropout, attn=True),
                                     ResBlock_encoder(c, c, dropout, attn=False)]))
        self.tail = _tail(cur, 1)
        self.fc_a = nn.Linear(self.shape[1] * self.shape[2], self.a_dim)
        self.fc_mu = nn.Linear(self.a_dim, self.a_dim)
        self.fc_var = nn.Linear(self.a_dim, self.a_dim)
        for m in (self.head, self.fc_a, self.fc_mu, self.fc_var):
            init.xavier_uniform_(m.weight)
            init.zeros_(m.bias)
        init.xavier_uniform_(self.tail[-1].weight, gain=1e-5)
        init.zeros_(self.tail[-1].bias)

    def forward(self, x):
        if self._differentiable(x):
            from .train import encoder_train_forward
            return encoder_train_forward(self, x, *self._dropout())
        from .engine import encoder_forward
        return encoder_forward(self, x)


class MLPLNAct(nn.Module):
    """Linear -> x * (condition_bias + Linear(act(cond))) -> LayerNorm -> act -> Dropout: one layer of the latent
    eps-network (reference models.py:91-163).  Parameter container; `linear_emb` is registered twice (also as
    cond_layers.1) exactly like the reference, so the state_dict carries both aliases."""

    def __init__(self, in_channels, out_channels, norm, use_cond, activation=None, cond_channels=None,
                 condition_bias=0, dropout=0):
        super().__init__()
        self.activation = activation
        self.act = nn.SiLU() if activation is not None else nn.Identity()
        self.condition_bias = condition_bias
        self.use_cond = use_cond
        self.linear = nn.Linear(in_channels, out_channels)
        if self.use_cond:
            self.linear_emb = nn.Linear(cond_channels, out_channels)
            self.cond_layers = nn.Sequential(self.act, self.linear_emb)
        self.norm = nn.LayerNorm(out_channels) if norm else nn.Identity()
        self.dropout = nn.Dropout(dropout) if dropout > 0 else nn.Identity()
        gains = {'relu': (0, 'relu'), 'leaky_relu': (0.2, 'leaky_relu'), 'silu': (0, 'relu')}
        if activation in gains:                       # reference init_weights (models.py:127-145)
            a, nl = gains[activation]
            for module in self.modules():
                if isinstance(module, nn.Linear):
                    init.kaiming_normal_(module.weight, a=a, nonlinearity=nl)

    def forward(self, x, cond=None):
        raise RuntimeError("MLPLNAct is a parameter container; it runs inside LatentUNet.forward")


class LatentUNet(_EngineNet):
    """10-layer skip-MLP eps-network over the latent z (reference models.py:166-234): layer i >= 1 reads
    cat([h, x]); time embedding = Linear(SiLU(Linear(sinusoid(t))))."""

    def __init__(self, T, num_layers=10, dropout=0.1, shape=None, activation='silu', num_time_emb_channels: int = 64,
                 num_time_layers: int = 2):
        super().__init__()
        self.num_time_emb_channels = num_time_emb_channels
        self.shape = shape
        self.T = T
        D = shape[-1]
        layers = []
        for i in range(num_time_layers):
            layers.append(nn.Linear(num_time_emb_channels if i == 0 else D, D))
            if i < num_time_layers - 1:
                layers.append(nn.SiLU())
        self.time_embed = nn.Sequential(*layers)
        self.skip_layers = list(range(1, num_layers))
        self.layers = nn.ModuleList([])
        for i in range(num_layers):
            if i == 0:
                act, norm, cond, (a, b), drop = activation, True, True, (D, D * 4), dropout
            elif i == num_layers - 1:
                act, norm, cond, (a, b), drop = None, False, False, (D * 4, D), 0
            else:
                act, norm, cond, (a, b), drop = 'silu', True, True, (D * 4, D * 4), dropout
            if i in self.skip_layers:
                a += D
            self.layers.append(MLPLNAct(a, b, norm=norm, activation=act, cond_channels=D, use_cond=cond,
                                        condition_bias=1, dropout=drop))

    def forward(self, x, t):
        """x [B, D] fp32, t int64 [B] -> eps [B, D] (reference models.py:223).  eval(): fused kernels
        (engine.LatentPlan); train() with grad, or eval() with grad and x requiring grad: the same arithmetic as a torch
        autograd composite on the GPU (its Dropouts are identities in eval())."""
        from .engine import latent_forward, latent_forward_autograd
        if self._differentiable(x):
            return latent_forward_autograd(self, x, t)
        return latent_forward(self, x, t)


class InfoDiff(nn.Module):
    """Model wrapper: noise schedule, q(x_t|x_0), z routing and losses (reference models.py:605-723)."""

    def __init__(self, args, device, shape):
        super().__init__()
        self.device = device
        lin = lambda: torch.linspace(start=args.beta1, end=args.betaT, steps=args.diffusion_steps)
        self.alpha_bars = torch.cumprod(1 - lin(), dim=0).to(device=device)
        self.betas = lin().to(device=device)
        self.alphas = 1 - self.betas
        self.alpha_prev_bars = torch.cat([torch.Tensor([1]).to(device=device), self.alpha_bars[:-1]])
        ch_mult = [1, 2, 4] if args.input_size == 28 else [1, 2, 2, 2]
        net_cls = BottleneckAuxUNet if getattr(args, "is_bottleneck", False) else AuxiliaryUNet   # models.py:623-626
        self.backbone = net_cls(ch_mult=ch_mult, T=args.diffusion_steps, ch=args.unets_channels,
                                a_dim=args.a_dim, shape=shape)
        self.encoder = Encoder(ch_mult=ch_mult, ch=args.encoder_channels, a_dim=args.a_dim, shape=shape)
        self.mmd_weight: float = args.mmd_weight
        self.kld_weight: float = args.kld_weight
        self.to(device)

    def _uses_sampled_latent(self) -> bool:
        # reference models.py:714-721: a_q whenever the KLD term is on, the deterministic a otherwise
        return self.kld_weight != 0

    def forward(self, x, idx=None, a=None, get_target=False):
        epsilon = mu = log_var = None
        if idx is None:
            idx = torch.randint(0, len(self.alpha_bars), (x.size(0),)).to(device=self.device)
            used = self.alpha_bars[idx][:, None, None, None]
            epsilon = torch.randn_like(x)
            x_tilde = torch.sqrt(used) * x + torch.sqrt(1 - used) * epsilon
        else:
            if not torch.is_tensor(idx):
                idx = torch.full((x.size(0),), int(idx), dtype=torch.long, device=self.device)
            x_tilde = x
        if a is None:
            a, a_q, mu, log_var = self.encoder(x)
        else:
            a_q = a
        output = self.backbone(x_tilde, idx, a_q if self._uses_sampled_latent() else a)
        return (output, epsilon, a, mu, log_var) if get_target else output

    def loss_fn(self, args, x, idx=None, curr_epoch=0):
        """Training objective (reference models.py:632-696), prior='regular'.  In train() mode the returned
        scalar carries an autograd graph whose heavy nodes are the sm_100a backward kernels
        (infodiffusion_b200.train); in eval() mode it is the forward value only, unless x requires grad."""
        output, epsilon, a, mu, log_var = self.forward(x, idx=idx, get_target=True)
        loss = (output - epsilon).square().mean()
        x_0 = torch.sqrt(1 / self.alphas[0]) * (x - self.betas[0] / torch.sqrt(1 - self.alpha_bars[0]) * output)
        loss = loss + (x_0 - x).square().mean() / args.diffusion_steps
        if args.mmd_weight != 0:
            if args.prior != 'regular':
                raise NotImplementedError("only --prior regular is in scope (SURVEY section 2)")
            true_samples = torch.randn_like(a, device=self.device)
            loss = loss + args.mmd_weight * compute_mmd(true_samples, mu if args.kld_weight != 0 else a)
        if args.kld_weight != 0:
            kld = torch.sum(-0.5 * torch.sum(1 + log_var - mu ** 2 - log_var.exp(), dim=1), dim=0)
            if getattr(args, "use_C", False):
                c_max = torch.tensor([args.C_max], dtype=torch.float32, device=self.device)
                cc = torch.clamp(c_max / args.epochs * curr_epoch, torch.zeros_like(c_max), c_max)
                loss = loss + args.kld_weight * (kld - cc.squeeze(dim=0)).abs()
            else:
                loss = loss + args.kld_weight * kld
        return loss


class Diff(nn.Module):
    """Plain DDPM wrapper: eps-MSE loss only; UNet backbone over images or LatentUNet over z
    (reference models.py:726-779)."""

    def __init__(self, args, device, shape):
        super().__init__()
        self.device = device
        lin = lambda: torch.linspace(start=args.beta1, end=args.betaT, steps=args.diffusion_steps)
        self.alpha_bars = torch.cumprod(1 - lin(), dim=0).to(device=device)
        self.betas = lin().to(device=device)
        self.alphas = 1 - self.betas
        self.alpha_prev_bars = torch.cat([torch.Tensor([1]).to(device=device), self.alpha_bars[:-1]])
        self.is_latent = bool(args.is_latent) or args.mode == "train_latent_ddim"
        ch_mult = [1, 2, 4] if args.input_size == 28 else [1, 2, 4, 8]
        if self.is_latent:
            self.backbone = LatentUNet(T=args.diffusion_steps, num_layers=10, dropout=0.1, shape=shape, activation='silu')
        else:
            self.backbone = UNet(ch_mult=ch_mult, T=args.diffusion_steps, ch=args.unets_channels, shape=shape)
        self.to(device)

    def loss_fn(self, args, x, idx=None, curr_epoch=0):
        output, epsilon = self.forward(x, idx=idx, get_target=True)
        return (output - epsilon).square().mean()

    def forward(self, x, idx=None, get_target=False):
        epsilon = None
        if idx is None:
            idx = torch.randint(0, len(self.alpha_bars), (x.size(0),)).to(device=self.device)
            used = self.alpha_bars[idx][:, None] if self.is_latent else self.alpha_bars[idx][:, None, None, None]
            epsilon = torch.randn_like(x)
            x_tilde = torch.sqrt(used) * x + torch.sqrt(1 - used) * epsilon
        else:
            if not torch.is_tensor(idx):
                idx = torch.full((x.size(0),), int(idx), dtype=torch.long, device=self.device)
            x_tilde = x
        output = self.backbone(x_tilde, idx)
        return (output, epsilon) if get_target else output
