"""Entry points of the reference's run.py for the hot path: --mode train / eval_fid / save_latent /
train_latent_ddim / eval, same option names and defaults (reference run.py:25-97), same folder and file naming
(models/<exp>/model-N.pth, imgs/<exp>/eval-fid-*/sample-%06d.png, <model>_<exp>_latent.npz), on the sm_100a kernels.

What differs, on purpose:
  * data: the reference downloads torchvision datasets (data.py); there is no network here and data loading is out
    of scope (SURVEY section 2), so images come from --data_npz (array `images`: N x H x W x C uint8 or N x C x H x W
    float in [-1, 1], optional `labels`) or are synthetic U[-1, 1] (--synthetic_size images);
  * shapes: the kernels cover the 64x64 / 64-channel configuration (celeba, ffhq, chairs-sized data with
    --unets_channels 64) and the 32x32 cifar10 one; other dataset names raise.  The vanilla Diff model (UNet
    ch_mult [1,2,4,8], GroupNorms over up to 1024 channels) trains and samples at these widths; wider ones raise early;
  * eval_fid without --is_latent is the reference's two-phase sampler and, like the reference, loads the vanilla model
    from ./models/diff/{dataset}_{a_dim}d/model-{epochs}.pth.  `--model vanilla --mode train` saves under
    {model_folder}/diff/<experiment string>, which carries `_0.1mmd` unless --mmd_weight is 0 (reference naming, kept):
    train the vanilla model with --mmd_weight 0 to write the file eval_fid reads;
  * torchrun: under WORLD_SIZE > 1 training is data parallel (--batch_size per GPU, like BASELINE configs[2]);
    sampling / encoding shard every round of --batch_size images over the ranks, all ranks drawing the round's full
    batch from the same seed, so the written images do not depend on the number of GPUs (checked by
    tools/check_run_py_multigpu.sh: 2 GPUs vs 1 GPU differ by at most one uint8 level in 0.01 % of the pixels).
The analysis modes latent_quality / disentangle / interpolate (run.py:310-341, 371-414, 444-481) are thin callers of
the encoder, reverse DDIM and the sampler and are built; the VAE baseline, plot_latent (matplotlib) and save_original_img
are not.
"""
from __future__ import annotations

import argparse
import os
import random

import numpy as np
import torch

from infodiffusion_b200 import io as idf_io
from infodiffusion_b200.distributed import gather_batch, local_slice
from infodiffusion_b200.layout import shard_range
from infodiffusion_b200.models import Diff, InfoDiff
from infodiffusion_b200.optim import ClipAdamW
from infodiffusion_b200.sampling import DiffusionProcess, LatentDiffusionProcess, TwoPhaseDiffusionProcess
from infodiffusion_b200.train import GradSync, set_grad_sync


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument('--r_seed', type=int, default=0)
    p.add_argument('--img_id', type=int, default=0)
    p.add_argument('--model', required=True, choices=['diff', 'vae', 'vanilla'])
    p.add_argument('--mode', required=True, choices=['train', 'eval', 'eval_fid', 'save_latent', 'disentangle', 'interpolate',
                                                     'save_original_img', 'latent_quality', 'train_latent_ddim', 'plot_latent'])
    p.add_argument('--prior', required=True, choices=['regular', '10mix', 'roll'])
    p.add_argument('--kld_weight', type=float, default=0)
    p.add_argument('--mmd_weight', type=float, default=0.1)
    p.add_argument('--use_C', action='store_true', default=False)
    p.add_argument('--C_max', type=float, default=25)
    p.add_argument('--dataset', required=True, choices=['fmnist', 'mnist', 'celeba', 'cifar10', 'dsprites', 'chairs', 'ffhq',
                                                        'synthetic'])
    p.add_argument('--img_folder', default='./imgs')
    p.add_argument('--log_folder', default='./logs')
    p.add_argument('-e', '--epochs', type=int, default=20)
    p.add_argument('--save_epochs', type=int, default=5)
    p.add_argument('--batch_size', type=int, default=64)
    p.add_argument('--learning_rate', type=float, default=0.0001)
    p.add_argument('--optimizer', default='adam', choices=['adam'])
    p.add_argument('--model_folder', default='./models')
    p.add_argument('--deterministic', action='store_true', default=False)
    p.add_argument('--input_channels', type=int, default=1)
    p.add_argument('--unets_channels', type=int, default=64)
    p.add_argument('--encoder_channels', type=int, default=64)
    p.add_argument('--input_size', type=int, default=32)
    p.add_argument('--a_dim', type=int, default=32, required=True)
    p.add_argument('--beta1', type=float, default=1e-5)
    p.add_argument('--betaT', type=float, default=1e-2)
    p.add_argument('--diffusion_steps', type=int, default=1000)
    p.add_argument('--split_step', type=int, default=500)
    p.add_argument('--sampling_number', type=int, default=16)
    p.add_argument('--data_dir', type=str, default='./data')
    p.add_argument('--tb_logger', action='store_true')
    p.add_argument('--is_latent', action='store_true')
    p.add_argument('--is_bottleneck', action='store_true')
    # additions (see module docstring)
    p.add_argument('--data_npz', type=str, default=None, help='images (and labels) to train on / encode')
    p.add_argument('--synthetic_size', type=int, default=256, help='number of synthetic images when no --data_npz is given')
    p.add_argument('--single_phase', action='store_true',
                   help='eval_fid without --is_latent: skip the vanilla model / two-phase sampler (the reference requires it)')
    p.add_argument('--allow_random_init', action='store_true',
                   help='evaluate the seeded random initialisation when the checkpoint is missing (the reference raises)')
    p.add_argument('--deterministic_training', action='store_true',
                   help='train / train_latent_ddim: torch.use_deterministic_algorithms(True), so the seed pins the run '
                        '(bitwise reproducible on one GPU model; the gradient reductions run in a fixed order)')
    return p.parse_args(argv)


def generate_exp_string(args) -> str:
    """reference utils.py:49-61"""
    root = f'{args.dataset}_{args.a_dim}d'
    if args.kld_weight != 0:
        root += f'_{args.kld_weight}kld'
        if args.use_C:
            root += f'_{args.C_max}C'
    if args.mmd_weight != 0:
        root += f'_{args.mmd_weight}mmd'
    if args.prior != 'regular':
        root += f'_{args.prior}'
    if args.is_bottleneck:
        root += '_bottleneck'
    return root


def seed_everything(r_seed: int) -> None:
    """reference utils.py:64-71"""
    random.seed(r_seed)
    np.random.seed(r_seed)
    torch.manual_seed(r_seed)
    torch.cuda.manual_seed_all(r_seed)


def get_dataset_config(args):
    """reference data.py:63-108, restricted to what the kernels cover."""
    if args.dataset in ('celeba', 'ffhq', 'synthetic'):
        args.input_channels, args.unets_channels, args.encoder_channels, args.input_size = 3, 64, 64, 64
    elif args.dataset == 'cifar10':
        args.input_channels, args.unets_channels, args.encoder_channels, args.input_size = 3, 64, 64, 32
    else:
        raise NotImplementedError(f"--dataset {args.dataset}: the sm_100a plans cover 64x64 / 32x32 inputs with 64-channel "
                                  "UNets (celeba / ffhq / cifar10 shapes); see DESIGN.md section 7")
    return (args.input_channels, args.input_size, args.input_size)


def _world():
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not torch.distributed.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        torch.distributed.init_process_group("nccl")
    return rank, world


def load_images(args, shape):
    """[N, C, H, W] fp32 in [-1, 1] on the CPU (+ labels or None)."""
    if args.data_npz:
        z = np.load(args.data_npz)
        x = z["images"]
        x = torch.from_numpy(x)
        if x.dtype == torch.uint8:
            x = x.permute(0, 3, 1, 2).float() / 127.5 - 1.0
        labels = z["labels"] if "labels" in z.files else None
    else:
        g = torch.Generator().manual_seed(args.r_seed)
        x = torch.rand(args.synthetic_size, *shape, generator=g) * 2 - 1
        labels = None
    assert tuple(x.shape[1:]) == tuple(shape), f"data shape {tuple(x.shape[1:])} != {shape}"
    return x.float(), labels


class GradualWarmupScheduler(torch.optim.lr_scheduler._LRScheduler):
    """reference utils.py:133-160 (linear warm-up to multiplier x base lr over warm_epoch epochs, then the wrapped
    scheduler)."""

    def __init__(self, optimizer, multiplier, warm_epoch, after_scheduler=None):
        self.multiplier, self.total_epoch, self.after_scheduler, self.finished = multiplier, warm_epoch, after_scheduler, False
        super().__init__(optimizer)

    def get_lr(self):
        if self.last_epoch > self.total_epoch:
            if self.after_scheduler:
                if not self.finished:
                    self.after_scheduler.base_lrs = [b * self.multiplier for b in self.base_lrs]
                    self.finished = True
                return self.after_scheduler.get_lr()
            return [b * self.multiplier for b in self.base_lrs]
        return [b * ((self.multiplier - 1.) * self.last_epoch / self.total_epoch + 1.) for b in self.base_lrs]

    def step(self, epoch=None):
        if self.finished and self.after_scheduler:
            self.after_scheduler.step(None if epoch is None else epoch - self.total_epoch)
        else:
            super().step(epoch)


def _model_root(args, latent: bool = False) -> str:
    root = args.model_folder
    if args.model == 'vanilla':
        root = os.path.join(root, 'diff')
    root = os.path.join(root, generate_exp_string(args))
    return root + ('_latent' if latent else '')


def _fit(args, model, batches, device, rank, world, latent=False):
    """The reference's epoch loop (run.py:187-211 / 503-526): loss_fn -> backward -> clip(1.0) -> AdamW, cosine schedule
    with one warm-up epoch, checkpoint every save_epochs."""
    opt = ClipAdamW(model.parameters(), lr=args.learning_rate, weight_decay=1e-5, max_norm=1.0)
    cosine = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer=opt, T_max=args.epochs, eta_min=0, last_epoch=-1)
    warm = GradualWarmupScheduler(optimizer=opt, multiplier=2., warm_epoch=1, after_scheduler=cosine)
    sync = GradSync(world) if world > 1 else None
    set_grad_sync(sync)
    params = [p for p in model.parameters() if p.requires_grad]
    model.train()
    for epoch in range(args.epochs):
        total, n = torch.zeros((), device=device), 0
        for data in batches(epoch):
            loss = model.loss_fn(args=args, x=data.to(device, non_blocking=True), curr_epoch=epoch)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            if sync is not None:
                sync.finish(params)
            opt.step()
            total += loss.detach()                      # no host sync inside the epoch
            n += 1
        if rank == 0:
            print(f"Epoch [{epoch}/{args.epochs}] Loss {float(total) / max(n, 1):.4f}  lr {opt.param_groups[0]['lr']:.3e}")
        warm.step()
        if (epoch + 1) % args.save_epochs == 0 and rank == 0:
            root = _model_root(args, latent)
            os.makedirs(root, exist_ok=True)
            torch.save(model.state_dict(), os.path.join(root, f'model-{epoch + 1}.pth'))
    set_grad_sync(None)
    model.eval()


def _reseed_rank(r_seed: int, rank: int) -> None:
    """After the model has been built from the COMMON seed (identical initial weights on every rank), give every rank
    its own random stream: InfoDiff.forward draws the timesteps (CPU generator), eps, the dropout seeds, the encoder's
    a_q noise and the MMD prior sample from torch's generators, and with one shared seed a global batch of B*world would
    contain only B distinct (t, eps) draws."""
    if rank > 0 or int(os.environ.get("WORLD_SIZE", "1")) > 1:
        torch.manual_seed(r_seed + 1000 * rank)
        torch.cuda.manual_seed(r_seed + 1000 * rank)


def _batches(x, batch_size, rank, world, seed):
    usable = (x.shape[0] // (batch_size * world)) * batch_size * world
    if usable == 0:
        raise ValueError(f"{x.shape[0]} samples give no full batch of {batch_size} x {world} rank(s): lower --batch_size "
                         "(plans are built per batch size, the tail batch is dropped)")
    if usable < x.shape[0] and rank == 0:
        print(f"[run.py] dropping the tail batch: {x.shape[0] - usable} of {x.shape[0]} samples per epoch are not used")

    def it(epoch):
        g = torch.Generator().manual_seed(seed * 1000 + epoch)
        perm = torch.randperm(x.shape[0], generator=g)
        usable = (x.shape[0] // (batch_size * world)) * batch_size * world      # fixed batch shape: plans are per batch size
        for i in range(0, usable, batch_size * world):
            idx = perm[i + rank * batch_size: i + (rank + 1) * batch_size]
            yield x[idx].pin_memory()
    return it


def train(args):
    rank, world = _world()
    seed_everything(args.r_seed)
    if args.deterministic_training:
        torch.use_deterministic_algorithms(True)
    device = torch.device("cuda", torch.cuda.current_device())
    shape = get_dataset_config(args)
    x, _ = load_images(args, shape)
    _check_widths(args)
    model = InfoDiff(args, device, shape) if args.model == 'diff' else Diff(args, device, shape)
    _reseed_rank(args.r_seed, rank)
    _fit(args, model, _batches(x, args.batch_size, rank, world, args.r_seed), device, rank, world)


def train_latent_ddim(args):
    rank, world = _world()
    seed_everything(args.r_seed)
    if args.deterministic_training:
        torch.use_deterministic_algorithms(True)
    device = torch.device("cuda", torch.cuda.current_device())
    z = torch.from_numpy(np.load("{}_{}_latent.npz".format(args.model, generate_exp_string(args).replace(".", "_")))["all_a"]).float()
    model = Diff(args, device, (1, args.a_dim, args.a_dim))
    _reseed_rank(args.r_seed, rank)
    _fit(args, model, _batches(z, args.batch_size, rank, world, args.r_seed), device, rank, world, latent=True)


def _check_widths(args, vanilla: bool = None) -> None:
    """Fail EARLY and clearly for configurations the kernels do not cover (instead of deep inside plan creation)."""
    from infodiffusion_b200.engine import MAX_GN_CHANNELS
    vanilla = (args.model == 'vanilla') if vanilla is None else vanilla
    if vanilla and not args.is_latent and args.mode != 'train_latent_ddim':
        widest = 8 * args.unets_channels                      # Diff hard-wires ch_mult = [1, 2, 4, 8] (models.py:746)
        if 2 * widest > MAX_GN_CHANNELS:
            raise NotImplementedError(
                f"the vanilla image model (Diff over UNet, ch_mult [1,2,4,8], {widest} channels, GroupNorm over "
                f"{2 * widest}) exceeds the kernels' limit of {MAX_GN_CHANNELS} GroupNorm channels "
                f"(--mode {args.mode}; training and inference alike); see DESIGN.md section 7")


def _load(args, device, shape):
    _check_widths(args)
    model = InfoDiff(args, device, shape) if args.model == 'diff' else Diff(args, device, shape)
    path = os.path.join(_model_root(args), f'model-{args.epochs}.pth')
    if os.path.exists(path):
        model.load_state_dict(torch.load(path, map_location=device), strict=False)
    elif not args.allow_random_init:
        raise FileNotFoundError(f"no checkpoint at {path} (reference run.py:233 fails the same way); pass "
                                "--allow_random_init to evaluate the seeded random initialisation")
    elif int(os.environ.get("RANK", "0")) == 0:
        print(f"[run.py] no checkpoint at {path}: using the seeded random initialisation (--allow_random_init)")
    return model.eval()


def evaluate(args):
    rank, world = _world()
    seed_everything(args.r_seed)
    device = torch.device("cuda", torch.cuda.current_device())
    shape = get_dataset_config(args)
    model = _load(args, device, shape)
    exp = generate_exp_string(args)
    if args.mode in ('eval', 'eval_fid'):
        process = DiffusionProcess(args, model, device, shape)
        process_latent = None
        if args.mode == 'eval_fid' and args.model == 'diff':
            if args.is_latent:                                   # run.py:234-243, 278
                model2 = Diff(args, device, (1, args.a_dim, args.a_dim))
                p2 = f'./models/{exp}_latent/model-{args.epochs}.pth'
                if not os.path.exists(p2):
                    raise FileNotFoundError(f"The file path {p2} does not exist, please train the latent diffusion model first.")
                model2.load_state_dict(torch.load(p2, map_location=device), strict=True)
                process_latent = LatentDiffusionProcess(args, model2.eval(), device)
            else:                                                # run.py:244-252, 280: two-phase with the vanilla model
                p2 = f'./models/diff/{args.dataset}_{args.a_dim}d/model-{args.epochs}.pth'
                if os.path.exists(p2):
                    _check_widths(args, vanilla=True)
                    model2 = Diff(args, device, shape)
                    model2.load_state_dict(torch.load(p2, map_location=device), strict=True)
                    process = TwoPhaseDiffusionProcess(args, model, model2.eval(), device, shape)
                elif not getattr(args, "single_phase", False):
                    raise FileNotFoundError(f"The file path {p2} does not exist, please train the vanilla diffusion model "
                                            "first (reference run.py:249); pass --single_phase to sample with the "
                                            "InfoDiff model alone instead of the two-phase sampler")
                elif rank == 0:
                    print("[run.py] --single_phase: sampling with the InfoDiff model alone (NOT the reference's two-phase "
                          "procedure)")
        # run.py:265-274 (eval_fid: imgs/<exp>/eval-fid-latent|eval-fid-fast) and save_images (eval: imgs[/diff]/<exp>/eval)
        if args.mode == 'eval_fid':
            root = os.path.join(args.img_folder, exp, 'eval-fid-latent' if args.is_latent else 'eval-fid-fast')
        else:
            root = os.path.join(args.img_folder, 'diff' if args.model == 'vanilla' else '', exp, 'eval')
        total = args.sampling_number
        for first in range(0, total, args.batch_size):               # --batch_size is the GLOBAL batch of a round
            n_round = min(args.batch_size, total - first)
            lo, hi = shard_range(n_round, rank, world)
            # every rank draws the round's FULL batch from the same seed (x_T, then a, on the CPU generator like
            # sampling.py:92-95; per-step noise on the CUDA generator) and keeps its slice: the images do not depend
            # on the number of GPUs, and with one GPU the draws are the reference's
            if process_latent is not None:
                a_full = process_latent.sampling(sampling_number=n_round)
            else:
                a_full = None
            xT_full = torch.randn([n_round, *shape]).to(device=device)
            if a_full is None:
                a_full = torch.randn([n_round, args.a_dim]).to(device=device)
            if hi == lo:
                continue
            if world > 1:
                noise = lambda idx, out: out.copy_(torch.randn(n_round, *shape, device=device)[lo:hi])
                for pr in (process, getattr(process, "p1", None), getattr(process, "p2", None)):
                    if pr is not None:
                        pr.noise_fn = noise
            batch = process.sampling(sampling_number=hi - lo, xT=xT_full[lo:hi].contiguous(), a=a_full[lo:hi].contiguous())
            idf_io.save_eval_images(batch, root, first_index=first + lo, limit=total)     # every rank writes its own range
        if rank == 0:
            print("DONE", root)
    elif args.mode == 'save_latent':
        x, labels = load_images(args, shape)
        outs = []
        for i in range(0, x.shape[0], args.batch_size * world):
            chunk = x[i:i + args.batch_size * world]
            part = local_slice(chunk, chunk.shape[0]).to(device)
            a, _, mu, _ = model.encoder(part) if part.shape[0] else (torch.zeros(0, args.a_dim, device=device),) * 4
            z = mu if args.kld_weight != 0 else a                # run.py:428-437
            outs.append(gather_batch(z.contiguous(), chunk.shape[0]).cpu())
        if rank == 0:
            attr = labels if labels is not None else np.array(['No Attributes'] * x.shape[0])
            idf_io.save_latents_npz("{}_{}_latent".format(args.model, exp.replace(".", "_")), outs, [attr])
    elif args.mode in ('latent_quality', 'disentangle', 'interpolate'):
        _analysis_modes(args, model, device, shape, rank)
    else:
        raise NotImplementedError(f"--mode {args.mode}: plot_latent / save_original_img need matplotlib / the torchvision "
                                  "datasets and are outside the hot path (SURVEY section 8f rank 4)")


def _nth_batch(args, shape, n):
    """The reference iterates its DataLoader (batch_size = args.batch_size, in order) and keeps batch `n` -- or the last
    one when the data are shorter (run.py:316-321, 373-383, 446-451)."""
    x, _ = load_images(args, shape)
    nb = (x.shape[0] + args.batch_size - 1) // args.batch_size
    i = min(n, nb - 1) * args.batch_size
    return x[i:i + args.batch_size]


def _encode(args, model, data, for_quality=False):
    """run.py:322-329 / 386-392 / 452-461: the latent the analysis modes condition on."""
    with torch.no_grad():
        a, _, mu, log_var = model.encoder(data)
    if args.kld_weight != 0:
        return mu + torch.exp(0.5 * log_var) if for_quality else mu      # latent_quality adds the std (run.py:325)
    return a


def _save_grid(args, sample, name):
    """reference save_images (run.py:103-143) for disentangle / interpolate: one row, normalised from [-1, 1]."""
    from torchvision.utils import save_image
    root = os.path.join(args.img_folder, 'diff' if args.model == 'vanilla' else '', generate_exp_string(args),
                        f'{args.mode}-{args.img_id}')
    os.makedirs(root, exist_ok=True)
    path = os.path.join(root, name)
    save_image(sample.float().cpu(), path, normalize=True, value_range=(-1, 1), nrow=sample.shape[0])
    return path


def _analysis_modes(args, model, device, shape, rank):
    """latent_quality (run.py:310-341), disentangle (371-414), interpolate (444-481): thin callers of the encoder, the
    reverse DDIM and the sampler.  Single process (the reference pins batch_size to 1 / 1 / 2, run.py:535-538)."""
    if args.model != 'diff':
        raise NotImplementedError("the analysis modes are built for --model diff (InfoDiff)")
    process = DiffusionProcess(args, model, device, shape)
    exp = generate_exp_string(args)
    if args.mode == 'latent_quality':
        data = _nth_batch(args, shape, 10).to(device)
        a = _encode(args, model, data, for_quality=True)
        xT = process.reverse_sampling(data, a)
        xT_original = xT.repeat(args.sampling_number, 1, 1, 1)
        a_original = a.repeat(args.sampling_number, 1)
        xT = torch.randn_like(xT_original)
        batch = process.sampling(xT=xT, a=a_original)
        root = os.path.join(args.img_folder, exp, 'latent_quality')
        # the reference joins the file name onto an undefined `path` here (run.py:340, NameError); the evident intent
        # -- sample-%06d.png under <img_folder>/<exp>/latent_quality -- is what is written
        idf_io.save_eval_images(batch, root)
        if rank == 0:
            print("DONE", root)
    elif args.mode == 'disentangle':
        data = _nth_batch(args, shape, args.img_id).to(device)
        eta = [-1.5, -1.2, -0.9, -0.6, -0.3, 0.0, 0.3, 0.6, 0.9, 1.2, 1.5]
        a = _encode(args, model, data)
        xT = process.reverse_sampling(data, a).repeat(len(eta), 1, 1, 1)
        for k in range(args.a_dim):
            rows = []
            for e in eta:
                a_k = _encode(args, model, data).clone()
                a_k[0][k] = e                                        # run.py:408: first image of the batch, dimension k
                rows.append(a_k)
            a_all = torch.stack(rows).squeeze(dim=1)
            sample = process.sampling(xT=xT, a=a_all)
            path = _save_grid(args, sample, f"sample{k}.png")
        if rank == 0:
            print("DONE", os.path.dirname(path))
    else:                                                            # interpolate
        data = _nth_batch(args, shape, args.img_id).to(device)
        assert data.shape[0] >= 2, "interpolate needs two images (the reference sets batch_size = 2)"
        a = _encode(args, model, data)
        xT = process.reverse_sampling(data, a)
        u, v = xT[0].reshape(-1), xT[1].reshape(-1)
        theta = torch.arccos((torch.nn.functional.normalize(u, dim=0) * torch.nn.functional.normalize(v, dim=0)).sum())
        etas = [0.0, 0.11, 0.22, 0.33, 0.44, 0.55, 0.66, 0.77, 0.88, 1.0]
        intp_a = torch.stack([float(np.cos(e * np.pi / 2)) * a[0] + float(np.sin(e * np.pi / 2)) * a[1] for e in etas])
        intp_x = torch.stack([(torch.sin((1 - e) * theta) * xT[0] + torch.sin(e * theta) * xT[1]) / torch.sin(theta)
                              for e in etas])
        sample = process.sampling(xT=intp_x, a=intp_a)
        path = _save_grid(args, sample, "sample0.png")
        if rank == 0:
            print("DONE", path)


if __name__ == '__main__':
    args = parse_args()
    if args.model == 'vae':
        raise NotImplementedError("the VAE baseline is out of scope (SURVEY section 2)")
    if args.mode in ('disentangle', 'latent_quality'):               # reference run.py:535-538
        args.batch_size = 1
    elif args.mode == 'interpolate':
        args.batch_size = 2
    if args.mode == 'train':
        train(args)
    elif args.mode == 'train_latent_ddim':
        train_latent_ddim(args)
    else:
        evaluate(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()
