"""Headline benchmark: 100-step DDIM sampling of 64x64 images (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling strong|weak]
                    [--dump-outputs DIR]

One "step" = one complete DDIM-100 sampling pass over the job's batch of synthetic images (InfoDiff a_dim=256, T=100,
random-init weights, xT and a ~ N(0,1)).  Sampling is per-sample independent, so N GPUs run N batch shards with no
data-path collective until the final gather.  Default = the configuration BASELINE.json names: ONE global batch of 256
split 256/N per GPU ("scaling": "strong"); at N > 1 the weak-scaling number (256 images per GPU) is reported beside it
under "weak_scaling".  --scaling weak makes that the headline instead.

 value        : images/s with xT and a already resident in HBM (device-timed with CUDA events, max over ranks)
 e2e          : same metric through the public API (DiffusionProcess.sampling) with pinned HOST inputs and a host
                read-back of the samples inside the timed region
 roofline     : dominant kernel class (tcgen05 implicit-GEMM conv), algorithmic FLOPs / CUDA-event time
 cpu_baseline : the reference's own modules (oracle/_ref, "reference") or the oracle port ("port") on this box's
                cores, bounded sample, extrapolated to DDIM-100
 eager_gpu    : the SAME reference modules on this GPU through cuDNN / cuBLAS -- fp32 with TF32 + cudnn.benchmark as
                run.py:19-20 sets them, and under torch.autocast(bf16) -- the bar the hand-written path has to beat
 train        : BASELINE configs[2] (training samples/s, data parallel)
 save_latent  : BASELINE configs[3] (encoder + reverse DDIM-100 at 64 images/GPU, both variants)
 ddpm1000     : BASELINE configs[4] (1000-step DDPM at 128 images/GPU: image sampler, latent + image sampler, two-phase)
 dp_check     : N > 1 only: N-rank averaged gradients vs rank 0's single-process gradients on the concatenated batch,
                and sharded sampling vs single-GPU sampling (correctness evidence for the scaling runs)
--impl reference times the CPU path alone and prints the same line with "impl": "reference".
--dump-outputs DIR writes the images the last timed step returned as DIR/samples.npy (float32), so that two builds
can be compared output for output.  Compare only runs with the same arguments: the weights are seeded, xT and a are
drawn per rank (seed 1000 + rank, so --gpus, --scaling and --batch change them), and the DDIM noise (eta 0.01) comes
from torch's CUDA generator, seeded once before the warm-up (so --warmup and --steps change it).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)

import torch  # noqa: E402

A_DIM, T_STEPS, BATCH = 256, 100, 256
METRIC = "ddim100_64x64_images_per_sec"
UNIT = "images/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="global batch (strong scaling) / batch per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the secondary legs (eager_gpu, save_latent, ddpm1000, dp_check, weak_scaling)")
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("IDF_SAMPLE_CHUNK", "0")) or None)
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("IDF_SAMPLE_LANES", "1")),
                    help="streams the micro-batches of a step are spread over (needs --chunk < batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pdl", type=int, default=int(os.environ.get("IDF_PDL", "1")),
                    help="1: launch conv / AdaGN kernels with programmatic dependent launch")
    ap.add_argument("--fuse-adagn", action="store_true", help="fold EVERY AdaGN into its consumer conv (A/B comparison; "
                    "the default folds the 64x64 maps only, engine.FUSE_ADAGN_MIN_H)")
    ap.add_argument("--no-fuse-adagn", action="store_true", help="stand-alone AdaGN kernels everywhere (A/B comparison)")
    ap.add_argument("--no-train", action="store_true", help="skip the secondary training-throughput measurement")
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the samples of the last timed step to DIR/samples.npy; the inputs "
                    "and noise are the same only for runs with the same --gpus, --scaling, --batch, --warmup and --steps")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference leg times a bounded sample, not whole sampling passes)")
    return a


DUMP_BYTES = 64 << 20


def dump_samples(out_dir: str, x: torch.Tensor) -> None:
    """x -> out_dir/samples.npy in float32.  Beyond DUMP_BYTES only a fixed, seeded choice of images is kept (the same
    images for the same batch size), in batch order."""
    import numpy as np
    x = x.detach().float().cpu()
    keep = DUMP_BYTES // (x[0].numel() * 4)
    if x.shape[0] > keep:
        rows = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        x = x[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "samples.npy"), x.numpy())


def ncu_traffic(kind: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the captured kernel, from the newest committed
    `ncu --set full` raw page under profiles/ (None if there is none)."""
    import csv
    files = sorted((ROOT / "profiles").glob(f"*_ncu_{kind}_raw.csv"))
    if not files:
        return None, None
    rows = list(csv.reader(files[-1].open()))
    if len(rows) < 3:
        return None, None
    hdr, units = rows[0], rows[1]
    try:
        ir, iw, ik = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("Kernel Name")
    except ValueError:
        return None, None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    vals = [float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0) for r in rows[2:]]
    return sum(vals) / len(vals), f"{files[-1].name}: mean over {len(vals)} captured launches of {rows[2][ik].split('(')[0]}"


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def make_args_ns(T):
    import types
    return types.SimpleNamespace(beta1=1e-5, betaT=1e-2, diffusion_steps=T, input_size=64, is_bottleneck=False,
                                 unets_channels=64, encoder_channels=64, a_dim=A_DIM, mmd_weight=0.1, kld_weight=0.0,
                                 is_latent=False, mode="eval_fid", prior="regular", batch_size=BATCH, use_C=False,
                                 C_max=25.0, epochs=1, deterministic=True, model="diff", split_step=0)


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the reference itself (oracle/_ref, see oracle/build_ref.py) or the oracle port
# ------------------------------------------------------------------------------------------------
_REF = None


def reference_modules():
    """(models, sampling) modules of the UNMODIFIED reference from oracle/_ref, or None when that directory did not
    travel (then the oracle port stands in).  Test / baseline infrastructure: never used by the product path."""
    global _REF
    if _REF is None:
        d = ROOT / "oracle" / "_ref"
        _REF = False
        if all((d / f).exists() for f in ("modules.py", "models.py", "sampling.py", "utils.py")):
            sys.path.insert(0, str(d))
            try:
                import importlib
                _REF = (importlib.import_module("models"), importlib.import_module("sampling"))
            except Exception as e:      # e.g. a dependency of utils.py missing on the box
                print(f"[bench] oracle/_ref present but not importable ({e!r}); using the oracle port", file=sys.stderr)
            finally:
                sys.path.remove(str(d))
    return _REF or None


def reference_unet_step(device: str, batch: int):
    """One DDIM step of the reference path at `batch` on `device`: returns (step_fn, kind).  step_fn() runs one
    UNet evaluation + update of the T=100 schedule (the generator of sampling.py:41-60 / its oracle port)."""
    torch.manual_seed(64)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(batch, 3, 64, 64, generator=g).to(device)
    a = torch.randn(batch, A_DIM, generator=g).to(device)
    ref = reference_modules()
    if ref is not None:
        models, sampling = ref
        args = make_args_ns(T_STEPS)
        model = models.InfoDiff(args, device, (3, 64, 64)).eval()
        proc = sampling.DiffusionProcess(args, model, device, (3, 64, 64))
        state = {"it": proc._ddim_one_diffusion_step(x, a)}

        def step():
            try:
                next(state["it"])
            except StopIteration:
                state["it"] = proc._ddim_one_diffusion_step(x, a)
                next(state["it"])
        return step, "reference"
    from oracle import infodiff_oracle as orc
    from infodiffusion_b200.models import InfoDiff
    m = InfoDiff(make_args_ns(T_STEPS), "cpu", (3, 64, 64))
    sd = {k: v.detach().to(device) for k, v in m.state_dict().items()}
    t_dev = torch.full((batch,), T_STEPS // 2, dtype=torch.long, device=device)
    sch = orc.Schedule.make(1e-5, 1e-2, T_STEPS)
    if device == "cpu":
        state = {"it": orc.ddim_steps(sch, orc.infodiff_eps_fn(sd, a), x)}

        def step():
            try:
                next(state["it"])
            except StopIteration:
                state["it"] = orc.ddim_steps(sch, orc.infodiff_eps_fn(sd, a), x)
                next(state["it"])
        return step, "port"
    return (lambda: orc.aux_unet_forward(sd, x, t_dev, a)), "port"


def cpu_ddim_rate(batch: int, min_seconds: float, max_evals: int):
    """CPU images/s for DDIM-100 from a bounded sample of UNet evaluations at `batch` on all host cores."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind = reference_unet_step("cpu", batch)
    with torch.no_grad():
        step()                                       # warm-up evaluation (oneDNN primitive creation)
        t0 = time.perf_counter()
        n = 0
        while True:
            step()
            n += 1
            if n >= max_evals or time.perf_counter() - t0 >= min_seconds:
                break
        dt = time.perf_counter() - t0
    per_eval = dt / n
    what = "the reference's DiffusionProcess (oracle/_ref)" if kind == "reference" else "the oracle port"
    return (batch / (per_eval * T_STEPS), cores, kind,
            f"{n} DDIM steps of the T={T_STEPS} schedule at batch {batch} through {what} ({dt:.1f} s), x{T_STEPS}/{n} extrapolated")


def eager_gpu_rates(dev: str, batch: int, evals: int = 3):
    """The reference path on THIS GPU with the libraries it would use (cuDNN convs, cuBLAS bmm / Linear, ATen
    GroupNorm): fp32 with TF32 + cudnn.benchmark exactly as run.py:19-20, and under torch.autocast(bfloat16)."""
    out = {"batch": batch, "evals": evals}
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = True
    try:
        step, kind = reference_unet_step(dev, batch)
        out["kind"] = kind
        for name, ctx in (("tf32", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            def run():
                with torch.no_grad():
                    if ctx is None:
                        step()
                    else:
                        with ctx:
                            step()
            for _ in range(3):                       # cudnn.benchmark autotunes on the first calls
                run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(evals):
                run()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / evals
            out[f"{name}_ms_per_unet_eval"] = ms
            out[f"{name}_img_s"] = batch / (ms / 1000.0 * T_STEPS)
    except Exception as e:                           # never take the headline down with it
        out["error"] = repr(e)[:300]
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        torch.cuda.empty_cache()
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, times, sample, cores, kind = [], [], "", 1, "port"
    for i in range(a.warmup + a.steps):
        # one step = a bounded sample of the workload (batch 256 like the GPU arm): 1-2 UNet evaluations (>= 3 s)
        t0 = time.perf_counter()
        v, cores, kind, sample = cpu_ddim_rate(a.batch, 3.0, 2)
        if i >= a.warmup:
            vals.append(v)
            times.append(time.perf_counter() - t0)
    v = statistics.mean(vals)
    ms = 1000.0 * statistics.mean(times)            # wall time of one bounded-sample step (NOT a full DDIM-100 pass)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"eval_fid-style DDIM-{T_STEPS} sampling, global batch {a.batch}, 64x64x3, InfoDiff a_dim {A_DIM} "
                               f"(BASELINE configs[1]) on the host CPU; a step = a bounded sample (model build + 1-2 of the 100 UNet "
                               f"evaluations), value = batch / (seconds per evaluation x {T_STEPS})",
                   "global_batch": a.batch},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
# training throughput (secondary metric)
# ------------------------------------------------------------------------------------------------
def train_throughput(a, dev, world, rank, steps=6, warmup=3):
    import torch.distributed as dist
    from infodiffusion_b200 import _lib
    from infodiffusion_b200.models import InfoDiff
    from infodiffusion_b200.optim import ClipAdamW
    from infodiffusion_b200.train import GradSync, set_grad_sync
    B = a.train_batch
    args = make_args_ns(1000)
    args.mode = "train"
    torch.manual_seed(64)
    model = InfoDiff(args, "cpu", (3, 64, 64)).to(dev)
    model.device = dev
    for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
        setattr(model, n, getattr(model, n).to(dev))
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    opt = ClipAdamW(params, lr=1e-4, weight_decay=1e-5, max_norm=1.0)     # clip_grad_norm_(1.0) + AdamW (run.py:199-200)
    sync = GradSync(world) if world > 1 else None
    set_grad_sync(sync)
    g = torch.Generator().manual_seed(7 + rank)
    x_h = (torch.rand(B, 3, 64, 64, generator=g) * 2 - 1).pin_memory()

    def step():
        x = x_h.to(dev, non_blocking=True)
        loss = model.loss_fn(args, x)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if sync is not None:
            sync.finish(params)                  # all-reduces were started inside backward
        opt.step()
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    l0 = _lib.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    set_grad_sync(None)
    flops = 3 * (15.318e9 + 11.774e9) * B * world * steps      # fwd + bwd ~ 3 x fwd (BASELINE.md)
    return {"metric": "train_samples_per_sec", "value": world * B * steps / (ms / 1000.0), "unit": "samples/s",
            "ms_per_step": ms / steps, "batch_per_gpu": B, "n_gpus": world, "final_loss": float(loss.detach()),
            "tflops": flops / (ms / 1000.0) / 1e12, "idf_launches_per_step": (_lib.launches() - l0) // steps,
            "config": "InfoDiff a_dim 256, T=1000, bf16 kernels / fp32 params, dropout 0.1, fused clip(1.0)+AdamW(1e-4, "
                      "wd 1e-5), data-parallel all-reduce overlapped with backward" + (" (NCCL)" if world > 1 else " (single GPU)")}


# ------------------------------------------------------------------------------------------------
# secondary legs: BASELINE configs[3] / configs[4], data-parallel correctness
# ------------------------------------------------------------------------------------------------
def _timed_region(fn, dev, world):
    """fn() once untimed (plan building, graph capture), then once between barriers; returns (ms max over ranks,
    idf launches of the timed call, result)."""
    import torch.distributed as dist
    from infodiffusion_b200 import _lib
    fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    l0 = _lib.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, _lib.launches() - l0, out


def save_latent_throughput(dev, world, rank, per_gpu=64):
    """BASELINE configs[3]: encoder z + reverse DDIM x0 -> xT (T = 100) on 64 images per GPU; both the reference's
    behaviour (reverse_sampling drops `a` and re-encodes x_t every step, sampling.py:84) and the a-honouring variant."""
    from infodiffusion_b200.models import InfoDiff
    from infodiffusion_b200.sampling import DiffusionProcess
    args = make_args_ns(T_STEPS)
    args.mode = "save_latent"
    torch.manual_seed(64)
    model = InfoDiff(args, "cpu", (3, 64, 64)).to(dev).eval()
    model.device = dev
    g = torch.Generator().manual_seed(2000 + rank)
    x_h = (torch.rand(per_gpu, 3, 64, 64, generator=g) * 2 - 1).pin_memory()
    out = {"metric": "save_latent_images_per_sec", "unit": UNIT, "batch_per_gpu": per_gpu, "n_gpus": world,
           "config": f"encoder z + reverse DDIM-{T_STEPS} x0->xT, {per_gpu} images/GPU (BASELINE configs[3]), host x in, host z and xT out"}
    for key, honour in (("reencode_every_step", False), ("given_latent", True)):
        a2 = make_args_ns(T_STEPS)
        a2.reverse_uses_given_latent = honour
        proc = DiffusionProcess(a2, model, dev, (3, 64, 64))

        def job():
            x = x_h.to(dev, non_blocking=True)
            z = model.encoder(x)[0]
            xT = proc.reverse_sampling(x, z)
            return z.cpu(), xT.cpu()
        ms, launches, _ = _timed_region(job, dev, world)
        out[key] = {"value": world * per_gpu / (ms / 1000.0), "ms": ms, "idf_launches_per_step": launches // max(1, T_STEPS - 2)}
        del proc
    return out


def ddpm1000_throughput(dev, world, rank, per_gpu=128, T=1000):
    """BASELINE configs[4]: 1000-step DDPM, 128 images per GPU -- InfoDiff image sampler; latent sampler
    (LatentDiffusionProcess over z) followed by the image sampler (eval_fid --is_latent); two-phase sampler
    (bug-compatible: every step on the vanilla model, SURVEY H5b)."""
    from infodiffusion_b200.models import Diff, InfoDiff
    from infodiffusion_b200.sampling import DiffusionProcess, LatentDiffusionProcess, TwoPhaseDiffusionProcess
    import copy
    args = make_args_ns(T)
    args.deterministic = False
    torch.manual_seed(64)
    model = InfoDiff(args, "cpu", (3, 64, 64)).to(dev).eval()
    model.device = dev
    largs = copy.copy(args)
    largs.model, largs.is_latent = "vanilla", True
    lat = Diff(largs, "cpu", (1, A_DIM, A_DIM)).to(dev).eval()
    lat.device = dev
    proc = DiffusionProcess(args, model, dev, (3, 64, 64))
    proc_lat = LatentDiffusionProcess(largs, lat, dev)
    g = torch.Generator().manual_seed(3000 + rank)
    xT = torch.randn(per_gpu, 3, 64, 64, generator=g).to(dev)
    a = torch.randn(per_gpu, A_DIM, generator=g).to(dev)
    out = {"metric": "ddpm1000_64x64_images_per_sec", "unit": UNIT, "batch_per_gpu": per_gpu, "n_gpus": world,
           "config": f"DDPM-{T} sampling, {per_gpu} images/GPU (BASELINE configs[4]), inputs resident in HBM"}
    legs = {"image_sampler": lambda: proc.sampling(per_gpu, xT=xT, a=a),
            "latent_plus_image_sampler": lambda: proc.sampling(per_gpu, xT=xT, a=proc_lat.sampling(sampling_number=per_gpu))}
    try:
        vargs = copy.copy(args)
        vargs.model = "vanilla"
        van = Diff(vargs, "cpu", (3, 64, 64)).to(dev).eval()
        van.device = dev
        two = TwoPhaseDiffusionProcess(args, model, van, dev, (3, 64, 64))
        two.sampling(2, xT=xT[:2], a=a[:2])            # builds the plans: raises here if the widths are not covered
        legs["two_phase_sampler"] = lambda: two.sampling(per_gpu, xT=xT, a=a)
    except Exception as e:
        out["two_phase_sampler"] = {"unavailable": repr(e)[:200]}
    for key, fn in legs.items():
        ms, launches, _ = _timed_region(fn, dev, world)
        out[key] = {"value": world * per_gpu / (ms / 1000.0), "ms": ms, "idf_launches_per_step": launches // T}
    return out


def dp_check(dev, world, rank):
    """Correctness evidence for the multi-GPU runs (the driver's GPU tests see one GPU):
      gradients : InfoDiff eps-MSE loss (mmd_weight 0: batch-separable), dropout off, identical (x, t, eps) on all
                  ranks; every rank back-propagates its shard with GradSync (NCCL all-reduce AVG overlapped with the
                  backward); rank 0 then back-propagates the CONCATENATED batch alone.  Reported: rel-L2 of the whole
                  gradient vector and the worst tensor.
      sampling  : 3-step DDIM of world*4 images sharded over the ranks + all_gather vs rank 0 sampling all of them."""
    import torch.distributed as dist
    from infodiffusion_b200.models import InfoDiff
    from infodiffusion_b200.sampling import DiffusionProcess
    from infodiffusion_b200.train import GradSync, set_grad_sync
    b = 4
    args = make_args_ns(1000)
    args.a_dim, args.mmd_weight, args.mode = 32, 0.0, "train"
    torch.manual_seed(64)
    model = InfoDiff(args, "cpu", (3, 64, 64)).to(dev)
    model.device = dev
    for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
        setattr(model, n, getattr(model, n).to(dev))
    model.backbone.dropout_p = 0.0
    model.encoder.dropout_p = 0.0
    model.train()
    g = torch.Generator().manual_seed(11)
    G = world * b
    x = (torch.rand(G, 3, 64, 64, generator=g) * 2 - 1).to(dev)
    idx = torch.randint(0, 1000, (G,), generator=g).to(dev)
    eps = torch.randn(G, 3, 64, 64, generator=g).to(dev)
    params = [p for p in model.parameters() if p.requires_grad]

    def grads(sl, sync):
        set_grad_sync(sync)
        for p in params:
            p.grad = None
        used = model.alpha_bars[idx[sl]][:, None, None, None]
        x_t = torch.sqrt(used) * x[sl] + torch.sqrt(1 - used) * eps[sl]
        a_lat = model.encoder(x[sl])[0]
        loss = (model.backbone(x_t, idx[sl], a_lat) - eps[sl]).square().mean()
        loss.backward()
        if sync is not None:
            sync.finish(params)
        set_grad_sync(None)
        return [None if p.grad is None else p.grad.detach().clone() for p in params]

    sync = GradSync(world)
    g_dp = grads(slice(rank * b, (rank + 1) * b), sync)
    res = {"ranks": world, "batch_per_rank": b, "grad_views_fixed_up": sync.fixed_up}
    # every rank must hold the same reduced gradient
    flat = torch.cat([t.flatten() for t in g_dp if t is not None]).double()
    cs = torch.stack([flat.sum(), flat.abs().sum()])
    lo, hi = cs.clone(), cs.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    res["grad_checksum_spread_over_ranks"] = float(((hi - lo).abs() / hi.abs().clamp_min(1e-30)).max())
    if rank == 0:
        g_one = grads(slice(0, G), None)
        pairs = [(float((u.double() - v.double()).square().sum()), float(v.double().square().sum()))
                 for u, v in zip(g_dp, g_one) if u is not None and v is not None]
        num, den = sum(d for d, _ in pairs), sum(n for _, n in pairs)
        # tensors whose exact gradient is (analytically) zero -- e.g. the key bias of an attention block, softmax is
        # shift invariant -- hold only rounding noise: the per-tensor figure covers tensors above 1e-4 of the total norm
        worst = max(((d / n) ** 0.5 for d, n in pairs if n > 1e-8 * den), default=0.0)
        res["grad_rel_l2_vs_single_process"] = (num / max(den, 1e-300)) ** 0.5
        res["grad_worst_tensor_rel_l2"] = worst
        res["grad_tensors_compared"] = len(pairs)
    dist.barrier()
    # ---- sharded sampling == single-GPU sampling
    model.eval()
    sargs = make_args_ns(3)
    sargs.a_dim = 32
    proc = DiffusionProcess(sargs, model, dev, (3, 64, 64))
    xT = torch.randn(G, 3, 64, 64, generator=g).to(dev)
    a = torch.randn(G, 32, generator=g).to(dev)
    noise = {i: torch.randn(G, 3, 64, 64, generator=g).to(dev) for i in range(3)}
    sl = slice(rank * b, (rank + 1) * b)
    proc.noise_fn = lambda i, out: out.copy_(noise[i][sl])
    mine = proc.sampling(b, xT=xT[sl].contiguous(), a=a[sl].contiguous())
    gathered = torch.empty(G, 3, 64, 64, device=dev)
    dist.all_gather_into_tensor(gathered, mine.contiguous())
    if rank == 0:
        proc.noise_fn = lambda i, out: out.copy_(noise[i])
        full = proc.sampling(G, xT=xT, a=a)
        res["sharded_sampling_rel_l2_vs_single_gpu"] = float((gathered - full).double().norm() / full.double().norm())
    dist.barrier()
    del model, proc
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------
# GPU path
# ------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch.distributed as dist
    from infodiffusion_b200 import _lib
    from infodiffusion_b200.layout import shard_range
    from infodiffusion_b200.models import InfoDiff
    from infodiffusion_b200.sampling import DiffusionProcess

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product path has no CPU fallback)"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner to fd 1 while the communicator is
        # created, so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(dev))
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    args = make_args_ns(T_STEPS)
    args.sample_chunk = a.chunk
    args.sample_lanes = a.lanes
    torch.manual_seed(64)
    model = InfoDiff(args, "cpu", (3, 64, 64)).to(dev).eval()
    model.device = dev
    proc = DiffusionProcess(args, model, dev, (3, 64, 64))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(global_batch, k, warmup):
        """DDIM-100 over `global_batch` images sharded contiguously over the ranks: (ms device-resident, ms end to
        end, launches, bytes in, bytes out), every time the max over ranks."""
        lo, hi = shard_range(global_batch, rank, world)
        B = hi - lo
        g = torch.Generator().manual_seed(1000 + rank)
        xT_h = torch.randn(B, 3, 64, 64, generator=g).pin_memory()
        a_h = torch.randn(B, A_DIM, generator=g).pin_memory()
        xT_d, a_d = xT_h.to(dev), a_h.to(dev)
        out_h = torch.empty(B, 3, 64, 64).pin_memory()
        sizes = [shard_range(global_batch, r, world) for r in range(world)]
        even = len({h - l for l, h in sizes}) == 1
        gathered = torch.empty(global_batch, 3, 64, 64, device=dev) if world > 1 else None

        def job_device():
            x = proc.sampling(B, xT=xT_d, a=a_d)
            if world > 1:
                if even:
                    dist.all_gather_into_tensor(gathered, x)
                    return gathered
                from infodiffusion_b200.distributed import gather_batch
                return gather_batch(x, global_batch)
            return x

        def job_e2e():
            x = proc.sampling(B, xT=xT_h.to(dev, non_blocking=True), a=a_h.to(dev, non_blocking=True))
            out_h.copy_(x, non_blocking=True)
            return x

        def timed(job, n):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = _lib.launches()
            e0.record()
            for _ in range(n):
                out = job()
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms, _lib.launches() - l0, out

        for _ in range(warmup):
            job_device()
        ms, launches, out = timed(job_device, k)
        job_e2e()
        ms_e2e, _, _ = timed(job_e2e, k)
        return dict(ms=ms, ms_e2e=ms_e2e, launches=launches, B=B, h2d=xT_h.numel() * 4 + a_h.numel() * 4,
                    d2h=out_h.numel() * 4, out=out)

    strong = a.scaling == "strong"
    global_batch = a.batch if strong else a.batch * world
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    m = measure(global_batch, a.steps, max(a.warmup, 3))
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_samples(a.dump_outputs, m["out"])
    B = m["B"]
    value = global_batch * a.steps / (m["ms"] / 1000.0)
    e2e = global_batch * a.steps / (m["ms_e2e"] / 1000.0)
    other = None
    if world > 1 and not a.no_extras:            # the other scaling mode beside the headline
        gb2 = a.batch * world if strong else a.batch
        m2 = measure(gb2, 2, 3)
        other = {"scaling": "weak" if strong else "strong", "global_batch": gb2, "batch_per_gpu": m2["B"],
                 "value": gb2 * 2 / (m2["ms"] / 1000.0), "e2e": gb2 * 2 / (m2["ms_e2e"] / 1000.0), "unit": UNIT,
                 "ms_per_step": m2["ms"] / 2}

    # ---- per-kernel-class timing of one UNet evaluation (CUDA events around every launch)
    roof, breakdown = None, None
    if rank == 0:
        pk = peaks()
        s = proc._sampler("ddim", B)
        for _ in range(2):
            for p in s.plans:
                p.run()
        torch.cuda.synchronize()
        acc = {}
        reps = 3
        for _ in range(reps):
            for p in s.plans:
                for tag, t_ms, fl, by in p.run_timed():
                    d = acc.setdefault(tag, dict(ms=0.0, flops=0, bytes=0, n=0))
                    d["ms"] += t_ms; d["flops"] += fl; d["bytes"] += by; d["n"] += 1
        tot = sum(d["ms"] for d in acc.values())
        c = acc["conv_igemm"]
        tfs = c["flops"] / (c["ms"] * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv_halo_kernel (tcgen05 implicit GEMM, CTA pairs)", "achieved": tfs,
                "peak": pk["tf_sus"], "unit": "TFLOP/s", "frac": tfs / pk["tf_sus"], "traffic": ncu_traffic("conv")[0],
                "traffic_source": ncu_traffic("conv")[1],
                "peak_source": pk["src"] + " bf16_tflops_sustained (kernel timed inside a long step)",
                "share_of_step": c["ms"] / tot, "launches_per_unet_eval": c["n"] // reps,
                "avg_launch_ms": c["ms"] / c["n"], "batch_per_gpu": B}
        breakdown = {k: {"ms_per_unet_eval": v["ms"] / reps, "launches": v["n"] // reps} for k, v in acc.items()}
        if "adagn" in acc:       # the stand-alone AdaGN kernels, HBM-bound (default; --fuse-adagn folds them into the convs)
            g_ = acc["adagn"]
            gbs = g_["bytes"] / (g_["ms"] * 1e-3) / 1e9
            breakdown["adagn"].update({"bound": "hbm", "achieved_GBps": gbs, "peak_GBps": pk["hbm"], "frac": gbs / pk["hbm"],
                                       "traffic": ncu_traffic("adagn")[0], "traffic_source": ncu_traffic("adagn")[1]})
        if "conv_igemm_xf" in acc:   # convs that also apply a fused AdaGN+SiLU to their A operand: tensor work AND the HBM pass they replace
            x_ = acc["conv_igemm_xf"]
            breakdown["conv_igemm_xf"].update({"bound": "tensor + shared memory", "achieved_TFLOPs": x_["flops"] / (x_["ms"] * 1e-3) / 1e12,
                                               "frac_of_tensor_peak": x_["flops"] / (x_["ms"] * 1e-3) / 1e12 / pk["tf_sus"],
                                               "adagn_hbm_bytes_replaced_per_unet_eval": x_["bytes"] // reps})
        if "adagn_coef" in acc:
            roof["note"] = (f"{acc['adagn_coef']['n'] // reps} of the 73 AdaGN+SiLU are applied to the consumer conv's A operand "
                            "in shared memory (transform warps): those normalised activations are never written to or read "
                            "from HBM, only their per-image coefficient kernels (adagn_coef) remain")
    ws_gb = sum(w.bytes for w in proc._sampler("ddim", B).lane_ws) / 1e9
    del proc
    model.backbone.invalidate_plans()
    torch.cuda.empty_cache()
    # ---- secondary metrics: BASELINE configs[2] training, configs[3] save_latent, configs[4] DDPM-1000
    train = None
    if not a.no_train:
        train = train_throughput(a, dev, world, rank)
        torch.cuda.empty_cache()
    c4 = c5 = dpc = eager = None
    if not a.no_extras:
        c4 = save_latent_throughput(dev, world, rank)
        torch.cuda.empty_cache()
        c5 = ddpm1000_throughput(dev, world, rank)
        torch.cuda.empty_cache()
        if world > 1:
            dpc = dp_check(dev, world, rank)
        if rank == 0:
            eager = eager_gpu_rates(dev, BATCH)
    cpu = None
    if rank == 0 and not a.no_cpu_baseline:
        v, cores, kind, sample = cpu_ddim_rate(32, 15.0, 40)     # ~15 s of host work on all cores
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": m["ms"] / a.steps, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"eval_fid-style DDIM-{T_STEPS} sampling, global batch {global_batch} = {B}/GPU x {world}, "
                                   f"64x64x3, InfoDiff a_dim {A_DIM} (BASELINE configs[1]); random-init weights",
                       "global_batch": global_batch, "batch_per_gpu": B,
                       "parallelism": f"batch-sharded x{world}, final all_gather",
                       "sample_chunk": a.chunk or B, "sample_lanes": a.lanes,
                       "l2": f"no explicit flush: {ws_gb:.1f} GB of activations are rewritten per UNet evaluation "
                             f"(>> 126 MB L2) and every step consumes the previous step's output"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"]},
            "gpu_launches": m["launches"], "clocks": clk, "roofline": roof, "kernel_breakdown": breakdown,
            "cpu_baseline": cpu, "eager_gpu": eager, ("weak_scaling" if strong else "strong_scaling"): other,
            "train": train, "save_latent": c4, "ddpm1000": c5, "dp_check": dpc,
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # stdout carries exactly one JSON line: NCCL's version / debug banner (NCCL_DEBUG=VERSION|INFO) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        if a.fuse_adagn:
            from infodiffusion_b200 import engine
            engine.FUSE_ADAGN = True
        if a.no_fuse_adagn:
            from infodiffusion_b200 import engine
            engine.FUSE_ADAGN_MIN_H = 0
        if os.environ.get("IDF_XF_DEBUG"):
            from infodiffusion_b200 import _lib
            _lib.check(_lib.load().idf_set_option(b"xf_debug", int(os.environ["IDF_XF_DEBUG"])))
        from infodiffusion_b200 import _lib
        _lib.check(_lib.load().idf_set_option(b"pdl", 1 if a.pdl else 0))
        run_ours(a)
