"""Network-level execution engine: lowers the UNets (AuxiliaryUNet, BottleneckAuxUNet, UNet), the Encoder and the
LatentUNet onto the libidf_b200 kernels.

A *plan* is a static list of kernel launches over a preallocated workspace, built once per
(network, batch).  It is CUDA-graph capturable: no allocation, no host sync, every per-step value
(timestep row of the modulation table, sampler coefficients) is read from device memory through a
device-resident step counter.

Data layout in HBM (see include/idf_b200.h): activations are bf16 "pad-flat" NHWC -- image n,
pixel (y, x) lives at row (n*(H+1) + y)*(W+1) + x of a [rows, C] matrix; the extra row / column
per image is a shared zero border, which turns every 3x3 tap into a constant row offset and makes
`padding=1` free.  Weights are packed once to bf16 [Cout, K] with K = (tap, cin) order.

Fusions relative to the reference's one-op-per-kernel execution (modules.py / models.py):
  * GroupNorm + (1+s_t),b_t + (1+s_z),b_z + SiLU + torch.cat        -> one AdaGN kernel
  * conv + bias + residual add (+ 1x1 shortcut conv as extra K-blocks) -> one implicit-GEMM kernel
  * q,k,v 1x1 convs -> one N=384 GEMM; QK^T, softmax, PV -> one attention kernel
  * proj 1x1 conv + attention residual                               -> GEMM epilogue
  * tail conv + DDPM/DDIM/reverse-DDIM update of x                   -> GEMM epilogue (sampler mode)
  * every temb_proj / aemb_proj Linear of all 22 blocks              -> two batched GEMMs, hoisted out
    of the step loop (the timestep side becomes a [T, 4992] table, the z side is step-invariant)
  * nearest x2 upsampling + conv (inference)                         -> one 4-tap GEMM per output parity on the input grid
  * AdaGN + SiLU of the 64x64 maps (inference, batch >= 128)         -> applied to the consumer conv's A operand in
    shared memory (transform warps); the normalised activation never exists in HBM
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import _lib
from ._lib import EPI_BF16, EPI_F32_NCHW, EPI_SAMPLER, AdaGNArgs, ConvDesc
from .layout import (ParamIndex, pack_conv1x1, pack_conv3x3, pack_conv3x3_up2, pad_cols as _pad_cols, pad_rows as _pad_rows,
                     probing, pv, tap_offsets3x3, taps_stride2, taps_up2, window_records_exact)
from .modules import AttnBlock, AuxResBlock, DownSample, ResBlock, UpSample, timestep_embedding

BF16 = torch.bfloat16


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{what} must live on a CUDA (sm_100) device: infodiffusion_b200 has no CPU path")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------------------------------------
# workspace
# ------------------------------------------------------------------------------------------------
class Act:
    """A pad-flat bf16 activation buffer [phases * B*(H+1)*(W+1), C]."""
    __slots__ = ("t", "H", "C", "phases", "rows", "stats", "has_stats", "stats_unit", "stats_planes", "stats_rows")

    def __init__(self, t, H, C, phases, rows):
        self.t, self.H, self.C, self.phases, self.rows = t, H, C, phases, rows
        self.stats = None          # fp32 [2, ceil(rows/128)*4, C, 2] GroupNorm partial sums (conv epilogues)
        self.has_stats = False     # True while `stats` describes the current contents of `t`
        self.stats_unit = 32       # rows per statistics unit of the records in `stats` (idf_conv_plan_stats_unit)
        self.stats_planes = 0      # > 0: records written by an up2 conv (parity planes, producer grid of stats_rows rows / image)
        self.stats_rows = 0

    def stats_buffer(self, min_floats: int = 0) -> torch.Tensor:
        """Allocated once per buffer (plans keep raw pointers to it): sized for the map's own tiles plus the slack an
        up2 producer needs (its records cover the input grid's tiles, 4 parity planes wide: <= 1.13x for H >= 16)."""
        if self.stats is None:
            tiles = (self.rows + 127) // 128
            self.stats = torch.zeros(2 * (tiles + tiles // 4 + 8) * 4 * self.C * 2, dtype=torch.float32, device=self.t.device)
        assert self.stats.numel() >= min_floats, "statistics buffer too small for this producer"
        return self.stats


class VAct:
    """The output of an AdaGN (+SiLU) that is never materialised: the raw source activation(s) plus per-image
    (A, B) coefficients [B, C, 2]; the consuming conv applies bf16(act(A*x + B)) to its A operand in shared memory."""
    __slots__ = ("srcs", "coef", "silu", "H", "C")

    def __init__(self, srcs, coef, silu, H, C):
        self.srcs, self.coef, self.silu, self.H, self.C = srcs, coef, silu, H, C


# Inference plans can fold an AdaGN into its consumer conv (transform warps rewrite the A operand in shared memory; the
# normalised activation never touches HBM).  The transform shares the shared-memory port with the tensor core's operand
# fetch, so it is not free: measured per layer at batch 256 (tools/conv_microbench.py, IDF_MB_XF=1) the fused conv
# beats conv + stand-alone AdaGN on the 64x64 maps (125 vs 80 + 55 us for 64->64, 208 vs 135 + 120 us for the 128-channel
# concatenations), ties on 32x32 and loses on the 16x16 / 8x8 maps, where the extra coefficient kernel costs as much as
# the AdaGN launch it replaces.  FUSE_ADAGN = True fuses every layer (bench.py --fuse-adagn all); FUSE_ADAGN_MIN_H fuses
# the maps of at least that size when the batch is large enough to fill the machine (the default: 64x64 maps).
FUSE_ADAGN = False
FUSE_ADAGN_MIN_H = 64
FUSE_ADAGN_MIN_ROWS = 128 * 65 * 65      # ... and only from this many pad-flat rows (batch 128 at 64x64)
MAX_GN_CHANNELS = 1024       # widest GroupNorm the AdaGN kernels take, forward and backward (kMaxCWide, kBMaxCWide)


class Workspace:
    """Pool of zero-initialised pad-flat buffers.  Buffers are only ever recycled for the same
    (H, C, phases) geometry, so the zero border written at allocation time is never disturbed
    (kernels write interior rows only)."""

    def __init__(self, batch: int, device, recycle: bool = True):
        self.batch, self.device = batch, device
        self.recycle = recycle       # training keeps every activation alive for the backward pass
        self.free_lists: Dict[Tuple[int, int, int], List[Act]] = {}
        self.bytes = 0

    def alloc(self, H: int, C_: int, phases: int = 1) -> Act:
        key = (H, C_, phases)
        fl = self.free_lists.get(key)
        if fl:
            a = fl.pop()
            a.has_stats = False
            a.stats_planes = a.stats_rows = 0
            return a
        rows = self.batch * (H + 1) * (H + 1)
        t = torch.zeros(phases * rows, C_, dtype=BF16, device=self.device)
        self.bytes += t.numel() * 2
        return Act(t, H, C_, phases, rows)

    def free(self, a: Act) -> None:
        if self.recycle:
            self.free_lists.setdefault((a.H, a.C, a.phases), []).append(a)


# ------------------------------------------------------------------------------------------------
# op records and their runner
# ------------------------------------------------------------------------------------------------
@dataclass
class Op:
    """One launch of a plan: `fn(*args, stream)` is a library call that launches `kernels` kernels; with kernels = 0
    it is a torch op, `fn(*args)` on the current stream.  `side`: a leaf of the backward graph (weight / bias
    gradient) that may run on the side stream."""
    tag: str
    fn: object
    args: tuple
    kernels: int = 1
    flops: int = 0
    bytes: int = 0
    side: bool = False


def run_ops(ops: Sequence[Op], device, side: Optional[torch.cuda.Stream] = None) -> None:
    """Enqueue `ops` in order on the current stream, check every return code and count the declared kernels.  With a
    `side` stream, each op marked `side` runs there after everything enqueued before it; the side stream is joined
    at the end."""
    main = torch.cuda.current_stream(device)
    stream, side_stream = main.cuda_stream, side.cuda_stream if side is not None else None
    if side is not None:
        side.wait_stream(main)
    n = 0
    for op in ops:
        if not op.kernels:
            op.fn(*op.args)
        elif op.side and side is not None:
            side.wait_stream(main)
            _lib.check(op.fn(*op.args, side_stream))
        else:
            _lib.check(op.fn(*op.args, stream))
        n += op.kernels
    if side is not None:
        main.wait_stream(side)
    _lib.count_launch(n)


# ------------------------------------------------------------------------------------------------
# plan builder
# ------------------------------------------------------------------------------------------------
class _GatherArena:
    """Bump allocator for packed training operands: tensors are slices of a few large buffers, and each
    buffer carries the int32 gather map (1-based indices into Plan.flat_params, 0 = zero) that re-packs it."""

    def __init__(self, dtype, capacity: int, device):
        self.dtype, self.capacity, self.device = dtype, capacity, device
        self._chunks: List[dict] = []

    def alloc(self, shape, idx: List[torch.Tensor]) -> torch.Tensor:
        n = 1
        for d in shape:
            n *= d
        span = (n + 127) // 128 * 128                       # 256-byte alignment for bf16 (TMA base), 512 for fp32
        ch = self._chunks[-1] if self._chunks else None
        if ch is None or ch["used"] + span > ch["buf"].numel():
            cap = max(self.capacity if ch is None else self.capacity // 2, span)
            ch = dict(buf=torch.zeros(cap, dtype=self.dtype, device=self.device), used=0, parts=[], maps=None)
            self._chunks.append(ch)
        off = ch["used"]
        ch["used"] += span
        ch["parts"].append((off, n, idx))
        ch["maps"] = None
        return ch["buf"][off:off + n].view(*shape)

    def chunks(self):
        for ch in self._chunks:
            if ch["maps"] is None:
                i1 = torch.zeros(ch["used"], dtype=torch.int32, device=self.device)
                i2 = None
                for off, n, idx in ch["parts"]:
                    i1[off:off + n] = idx[0]
                    if len(idx) > 1:
                        if i2 is None:
                            i2 = torch.zeros(ch["used"], dtype=torch.int32, device=self.device)
                        i2[off:off + n] = idx[1]
                ch["maps"] = (i1, i2)
            yield ch["buf"], ch["maps"][0], ch["maps"][1], ch["used"]


class Plan:
    """Ordered list of kernel launches + everything they reference."""

    def __init__(self, batch: int, device, ws: Optional[Workspace] = None, training: bool = False,
                 ordered: bool = False):
        self.lib = _lib.load()
        _lib.check(self.lib.idf_init())
        self.B = batch
        self.device = device
        self.training = training
        if training:
            # the training step is a chain of ~1000 small dependent kernels: let each conv / AdaGN kernel run its
            # prologue (barriers, TMEM, bias, weight tiles) while its predecessor drains (+2.5 % step rate, bitwise
            # neutral: tests/test_gpu_network.py::test_programmatic_dependent_launch_is_bitwise_neutral)
            _lib.check(self.lib.idf_set_option(b"pdl", 1))
        self.fuse_adagn = FUSE_ADAGN and not training
        self.ws = ws if ws is not None else Workspace(batch, device, recycle=not training)
        self.tape: List = []         # training: backward emitters, one per forward composite, replayed in reverse
        self.bwd = None              # training: the backward op lists (infodiffusion_b200.train.BwdState)
        if training:
            from .train import BwdState
            self.bwd = BwdState(self, ordered)
        self.pindex: Optional[ParamIndex] = None   # training: flat parameter layout the packing gathers read
        self.recipes: List = []      # training: (packed tensor, recipe) pairs (kept for verification)
        self.dropout_p = 0.0
        self.dropout_seed = None     # device int64 scalar
        self._drop_layers = 0
        self.ops: List[Op] = []
        self.keep: List = []         # tensors / ctypes structs that must outlive the plan
        self.conv_plans: List[int] = []
        self.flops = 0               # algorithmic conv/attention FLOPs of one run
        self.conv_tiles = 0
        self.adagn_bytes = 0         # algorithmic AdaGN bytes (1 read + 1 write) of one run

    def __del__(self):
        try:
            for h in self.conv_plans:
                self.lib.idf_conv_plan_destroy(h)
        except Exception:
            pass

    def _emit(self, tag: str, fn, args: tuple, flops: int = 0, nbytes: int = 0, emit: bool = True) -> Op:
        """Record one launch; with emit=False the record is only returned (backward ops, kept outside this plan)."""
        op = Op(tag, fn, args, flops=flops, bytes=nbytes)
        if emit:
            self.ops.append(op)
            self.flops += flops
            self.adagn_bytes += nbytes if tag == "adagn" else 0
        return op

    # ---- execution -----------------------------------------------------------------------------
    def run_timed(self, run_ahead_ms: float = 8.0) -> List[Tuple[str, float, int, int]]:
        """Eager run with a CUDA-event pair around every launch (on the launching stream).  The stream is first
        blocked by a spin kernel of ~run_ahead_ms so that the host enqueues all launches and events ahead of the
        GPU: the event deltas are then GPU durations, not host launch intervals (a ctypes launch costs ~10 us,
        more than the small kernels run).  Returns [(kernel class, milliseconds, algorithmic flops, bytes)]."""
        st = torch.cuda.current_stream(self.device)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(self.ops) + 1)]
        if run_ahead_ms > 0:
            torch.cuda._sleep(int(run_ahead_ms * 1.9e6))          # cycles at ~1.9 GHz
        evs[0].record(st)
        for i, op in enumerate(self.ops):
            run_ops([op], self.device)
            evs[i + 1].record(st)
        st.synchronize()
        return [(op.tag, evs[i].elapsed_time(evs[i + 1]), op.flops, op.bytes) for i, op in enumerate(self.ops)]

    def run(self) -> None:
        run_ops(self.ops, self.device)

    # ---- op emitters ---------------------------------------------------------------------------
    def weight(self, m) -> torch.Tensor:
        """bf16 device copy of a packed weight.  `m` may be a recipe (callable returning the fp32 tensor, reading
        parameters through layout.pv): a training plan re-packs all recipes before every forward with one
        gather launch so the kernels see the current parameters."""
        return self._packed(m, BF16)

    def f32(self, m) -> torch.Tensor:
        """fp32 device copy (biases, GroupNorm affine); a recipe may return a tuple of tensors to be summed."""
        return self._packed(m, torch.float32)

    def _packed(self, m, dtype) -> torch.Tensor:
        src = m() if callable(m) else m
        if isinstance(src, tuple):
            src = sum(x.detach().double() for x in src)
        if not (callable(m) and self.training):
            t = src.detach().to(device=self.device, dtype=dtype).contiguous()
            self.keep.append(t)
            return t
        assert self.pindex is not None, "training plan: bind_params() before the first weight"
        with probing(self.pindex):
            idx = m()
        idx = idx if isinstance(idx, tuple) else (idx,)
        assert len(idx) <= 2 and all(i.dtype == torch.int64 for i in idx), "recipe must be a pure re-ordering of parameters"
        arena = self._arena_bf16 if dtype == BF16 else self._arena_f32
        t = arena.alloc(src.shape, [i.reshape(-1).to(torch.int32) for i in idx])
        t.copy_(src.detach())
        self.recipes.append((t, m))
        return t

    def bind_params(self, params) -> None:
        """Training plans: the parameters the recipes read, in a fixed flat fp32 layout."""
        self.pindex = ParamIndex(params, self.device)
        self.flat_params = torch.zeros(self.pindex.total, dtype=torch.float32, device=self.device)
        self._flat_views = self.pindex.views(self.flat_params)
        total = self.pindex.total
        self._arena_bf16 = _GatherArena(BF16, int(2.3 * total) + (4 << 20), self.device)
        self._arena_f32 = _GatherArena(torch.float32, 1 << 20, self.device)

    def refresh_ops(self) -> List[Op]:
        """flat_params <- parameters (one multi-tensor copy), then one gather launch per arena chunk."""
        ops = [Op("param_copy", torch._foreach_copy_, (self._flat_views, [p.detach() for p in self.pindex.params]),
                  kernels=0)]
        for arena in (self._arena_bf16, self._arena_f32):
            for buf, idx, idx2, used in arena.chunks():
                ops.append(Op("repack", self.lib.idf_gather_elems,
                              (self.flat_params.data_ptr(), idx.data_ptr(), idx2.data_ptr() if idx2 is not None else None,
                               buf.data_ptr(), used, 1 if arena.dtype == BF16 else 0, 0)))
        return ops

    def conv(self, srcs: Sequence[Act], kblocks: Sequence[Tuple[int, int, int]], wp: torch.Tensor,
             bias: torch.Tensor, H: int, cout: int, block_n: int, out: Optional[Act] = None,
             residual: Optional[Act] = None, epilogue: int = EPI_BF16, out_f32=None, x_io=None, noise=None,
             coef=None, step=None, real_macs_per_row: Optional[int] = None, want_stats: bool = True,
             xf: Optional[Tuple[torch.Tensor, bool, Sequence[int]]] = None, up2: bool = False, emit: bool = True) -> Op:
        """`xf` = (coefficients [B, Ctot, 2], silu?, per-k-block channel base or -1): fused AdaGN on the A operand.
        Returns the launch record (appended to this plan unless emit=False)."""
        d = ConvDesc()
        d.n_src = len(srcs)
        for i, s in enumerate(srcs):
            d.src[i] = s.t.data_ptr()
            d.src_rows[i] = s.t.shape[0]
            d.src_ld[i] = s.C
        d.num_kb = len(kblocks)
        for k, (si, c0, off) in enumerate(kblocks):
            d.kb_src[k], d.kb_c0[k], d.kb_rowoff[k] = si, c0, off
        assert wp.dtype == BF16 and wp.shape[1] == 64 * len(kblocks), (wp.shape, len(kblocks))
        assert wp.shape[0] % block_n == 0 and bias.numel() == wp.shape[0]
        d.weight = wp.data_ptr()
        d.cout_pad = wp.shape[0]
        d.block_n = block_n
        d.cout = cout
        d.bias = bias.data_ptr()
        d.batch, d.H, d.W = self.B, H, H
        d.epilogue = epilogue
        d.up2 = 1 if up2 else 0
        if out is not None:
            assert out.H == (2 * H if up2 else H) and out.C == cout
            d.out, d.out_ld = out.t.data_ptr(), out.C
            want_stats = want_stats and window_records_exact(H, H)     # records over the GEMM grid (up2: the input)
            if want_stats:
                # (an up2 plan writes records over the input grid's tiles, 4 parity planes wide)
                tiles_in = (self.B * (H + 1) * (H + 1) + 127) // 128
                d.stats_out = out.stats_buffer(2 * tiles_in * 4 * 4 * cout * 2 if up2 else 0).data_ptr()
                out.has_stats = True
        if residual is not None:
            assert residual.H == H and residual.C == cout
            d.residual, d.res_ld = residual.t.data_ptr(), residual.C
        d.out_f32, d.x_io, d.noise, d.coef, d.step_ptr = _ptr(out_f32), _ptr(x_io), _ptr(noise), _ptr(coef), _ptr(step)
        if xf is not None:
            ctab, xsilu, kb_xf = xf
            assert len(kb_xf) == len(kblocks) and ctab.shape[0] == self.B
            d.xf_coef, d.xf_ctot, d.xf_silu = ctab.data_ptr(), ctab.shape[1], 1 if xsilu else 0
            for k, v in enumerate(kb_xf):
                d.kb_xf[k] = v
        h = C.c_void_p()
        _lib.check(self.lib.idf_conv_plan_create(C.byref(d), C.byref(h)))
        self.conv_plans.append(h)
        self.keep.append(d)
        self.conv_tiles += int(self.lib.idf_conv_plan_tiles(h))
        if out is not None and want_stats:
            out.stats_unit = int(self.lib.idf_conv_plan_stats_unit(h))
            out.stats_planes, out.stats_rows = (4, (H + 1) * (H + 1)) if up2 else (0, 0)
        macs = real_macs_per_row if real_macs_per_row is not None else 64 * len(kblocks) * cout
        # conv_igemm_xf: the launches that also apply a fused AdaGN (+SiLU) to their A operand -- they replace a
        # stand-alone AdaGN pass and are accounted separately from the plain implicit GEMMs
        return self._emit("conv_igemm_xf" if xf is not None else "conv_igemm", self.lib.idf_conv_run, (h,),
                          flops=2 * self.B * H * H * macs,
                          nbytes=(2 * 2 * self.B * H * H * 64 * len({(si, c0) for (si, c0, _), v in zip(kblocks, xf[2]) if v >= 0})
                                  if xf is not None else 0), emit=emit)   # HBM bytes of the AdaGN pass this launch replaces

    def norm(self, src0: Act, src1: Optional[Act], gn: nn.GroupNorm, silu: bool, mod_t=None, mod_z=None, step=None,
             dropout: bool = False, mod_cols: Optional[int] = None):
        """AdaGN of one or two (channel-concatenated) activations for a following conv.  Inference plans return a
        VAct (coefficients only, applied inside the conv); otherwise the activation is materialised."""
        fuse = self.fuse_adagn or (not self.training and FUSE_ADAGN_MIN_H > 0 and src0.H >= FUSE_ADAGN_MIN_H
                                   and src0.rows >= FUSE_ADAGN_MIN_ROWS)
        if fuse and src0.has_stats and (src1 is None or src1.has_stats):
            Cc = src0.C + (src1.C if src1 is not None else 0)
            a, _, _ = self._adagn_args(src0, src1, gn, silu, mod_t, mod_z, step)
            ctab = torch.zeros(self.B, Cc, 2, dtype=torch.float32, device=self.device)
            self.keep += [a, ctab]
            self._emit("adagn_coef", self.lib.idf_adagn_coef, (C.byref(a), ctab.data_ptr()))
            return VAct([src0] if src1 is None else [src0, src1], ctab, silu, src0.H, Cc)
        out = self.ws.alloc(src0.H, src0.C + (src1.C if src1 is not None else 0))
        self.adagn(src0, src1, out, gn, silu, mod_t=mod_t, mod_z=mod_z, step=step, dropout=dropout, mod_cols=mod_cols)
        return out

    def done(self, a) -> None:
        """Release a norm() result once its consumer conv has been emitted."""
        if isinstance(a, Act):
            self.ws.free(a)

    @staticmethod
    def _operand(src, offsets: Sequence[int]):
        """(sources, k-blocks, kb_xf) of a conv over `src` (Act or VAct), K ordered (tap, concatenated channel)."""
        parts = src.srcs if isinstance(src, VAct) else [src]
        kb, kx = [], []
        for off in offsets:
            base = 0
            for si, part in enumerate(parts):
                assert part.C % 64 == 0
                for c0 in range(0, part.C, 64):
                    kb.append((si, c0, off))
                    kx.append(base + c0)
                base += part.C
        xf = (src.coef, src.silu, kx) if isinstance(src, VAct) else None
        return list(parts), kb, xf

    def _adagn_args(self, src0: Act, src1: Optional[Act], gn: nn.GroupNorm, silu: bool, mod_t, mod_z, step):
        """(AdaGNArgs, gamma, beta) shared by the stand-alone and the conv-fused AdaGN: shapes, GroupNorm affine,
        modulation, SiLU, and the sources' statistics records when their producers wrote them.  The caller sets the
        activation pointers and what only it needs."""
        a = AdaGNArgs()
        a.c0 = src0.C
        if src1 is not None:
            a.c1 = src1.C
        a.batch, a.H, a.W = self.B, src0.H, src0.H
        gamma, beta = self.f32(lambda: pv(gn.weight)), self.f32(lambda: pv(gn.bias))
        a.gamma, a.beta, a.eps = gamma.data_ptr(), beta.data_ptr(), float(gn.eps)
        if mod_t is not None:
            a.mod_t, a.mod_t_step_stride, a.mod_t_batch_stride = mod_t
        if mod_z is not None:
            a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = mod_z
        a.step_ptr = _ptr(step)
        a.apply_silu = 1 if silu else 0
        if src0.has_stats and (src1 is None or src1.has_stats):
            a.stats0, a.stats_unit0 = src0.stats.data_ptr(), src0.stats_unit
            a.stats_planes0, a.stats_rows0 = src0.stats_planes, src0.stats_rows
            if src1 is not None:
                a.stats1, a.stats_unit1 = src1.stats.data_ptr(), src1.stats_unit
                a.stats_planes1, a.stats_rows1 = src1.stats_planes, src1.stats_rows
        return a, gamma, beta

    def adagn(self, src0: Act, src1: Optional[Act], out: Act, gn: nn.GroupNorm, silu: bool, mod_t=None, mod_z=None,
              step=None, dropout: bool = False, mod_cols: Optional[int] = None) -> None:
        """Fused AdaGN.  mod_t / mod_z = (pointer, step stride, batch stride) of this block's (scale | shift)
        columns; `dropout` applies inverted dropout after the SiLU (training plans only)."""
        a, gamma, beta = self._adagn_args(src0, src1, gn, silu, mod_t, mod_z, step)
        a.src0, a.out = src0.t.data_ptr(), out.t.data_ptr()
        if src1 is not None:
            a.src1 = src1.t.data_ptr()
        if dropout and self.training and self.dropout_p > 0:
            self._drop_layers += 1
            a.dropout_p, a.dropout_seed, a.dropout_layer = self.dropout_p, self.dropout_seed.data_ptr(), self._drop_layers
        if self.training and a.stats0:
            coef = torch.zeros(self.B, out.C, 4, dtype=torch.float32, device=self.device)
            self.keep.append(coef)
            a.save_coef = coef.data_ptr()
        out.has_stats = False
        self.keep.append(a)
        self._emit("adagn", self.lib.idf_adagn_silu_fwd, (C.byref(a),), nbytes=2 * 2 * self.B * src0.H * src0.H * out.C)
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_adagn(self, a, src0, src1, out, gn, gamma, beta, mod_cols))

    def attention(self, qkv: Act, out: Act, d: int) -> None:
        S = qkv.H * qkv.H
        self._emit("attention", self.lib.idf_attn_fwd, (qkv.t.data_ptr(), out.t.data_ptr(), self.B, qkv.H, qkv.H, d,
                                                        float(d) ** -0.5), flops=self.B * 4 * S * S * d)
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_attention(self, qkv, out, d))

    def linear(self, x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], y: torch.Tensor, silu_in: bool) -> None:
        M, K = x.shape
        N = w.shape[0]
        assert w.shape[1] == K and y.shape == (M, N) and x.stride(1) == 1 and y.stride(1) == 1
        self._emit("linear", self.lib.idf_linear_f32, (x.data_ptr(), x.stride(0), w.data_ptr(), _ptr(b), y.data_ptr(),
                                                       y.stride(0), M, N, K, 1 if silu_in else 0))

    # ---- composite emitters ----------------------------------------------------------------------
    @staticmethod
    def _bn(cout: int) -> int:
        return 128 if cout % 128 == 0 else 64

    def conv3x3(self, src: Act, conv: nn.Conv2d, residual: Optional[Act] = None,
                shortcut: Optional[Tuple[nn.Conv2d, Sequence[Act]]] = None) -> Act:
        """3x3 / stride 1 / pad 1 conv (+ residual, or + 1x1 shortcut conv over raw sources as extra K-blocks)."""
        cin, cout, H = src.C, conv.out_channels, src.H
        assert conv.in_channels == cin and cout % 64 == 0
        srcs, kb, xf = self._operand(src, tap_offsets3x3(H, H))
        if shortcut is None:
            wp = lambda: pack_conv3x3(pv(conv.weight))
            bias = lambda: pv(conv.bias)
        else:
            sc_conv, raws = shortcut
            wp = lambda: torch.cat([pack_conv3x3(pv(conv.weight)), pack_conv1x1(pv(sc_conv.weight))], dim=1)
            bias = lambda: (pv(conv.bias), pv(sc_conv.bias))                      # summed by f32()
            for r in raws:
                si = next((i for i, s_ in enumerate(srcs) if s_ is r), None)   # a raw source may already be an operand
                if si is None:
                    srcs.append(r)
                    si = len(srcs) - 1
                kb += [(si, c0, 0) for c0 in range(0, r.C, 64)]
                if xf is not None:
                    xf[2].extend([-1] * (r.C // 64))
        out = self.ws.alloc(H, cout)
        self.conv(srcs, kb, self.weight(wp), self.f32(bias), H, cout, self._bn(cout), out=out, residual=residual, xf=xf)
        if self.training:
            from . import train
            parts = [train.Part(src, conv.weight, "3x3", None)]
            biases = [conv.bias]
            if shortcut is not None:
                c = 0
                for r in shortcut[1]:
                    parts.append(train.Part(r, shortcut[0].weight, "1x1", (c, c + r.C)))
                    c += r.C
                biases.append(shortcut[0].bias)
            self.tape.append(lambda: train.bwd_conv(self, parts, biases, out, residual))
        return out

    def conv1x1(self, src: Act, convs: Sequence[nn.Conv2d], residual: Optional[Act] = None,
                want_stats: bool = True) -> Act:
        """1x1 conv; several convs over the same input are stacked along N (q, k, v -> one GEMM)."""
        cout = sum(m.out_channels for m in convs)
        srcs, kb, xf = self._operand(src, [0])
        out = self.ws.alloc(src.H, cout)
        wp = lambda: _pad_cols(torch.cat([pack_conv1x1(pv(m.weight)) for m in convs], dim=0), 64 * len(kb))
        bias = lambda: torch.cat([pv(m.bias) for m in convs], dim=0)
        self.conv(srcs, kb, self.weight(wp), self.f32(bias), src.H, cout, self._bn(cout), out=out, residual=residual,
                  want_stats=want_stats, xf=xf)
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_conv1x1_stack(self, src, list(convs), out, residual))
        return out

    def downsample(self, src: Act, conv: nn.Conv2d) -> Act:
        """3x3 stride-2 conv: space-to-depth split into 4 phase maps, then 9 taps over the phases."""
        H, Ho, Cc = src.H, src.H // 2, src.C
        ph = self.ws.alloc(Ho, Cc, phases=4)
        self._emit("space_to_depth", self.lib.idf_space_to_depth, (src.t.data_ptr(), ph.t.data_ptr(), self.B, H, H, Cc))
        kb = taps_stride2(Cc, Ho, Ho, ph.rows)
        out = self.ws.alloc(Ho, conv.out_channels)
        self.conv([ph], kb, self.weight(lambda: pack_conv3x3(pv(conv.weight))), self.f32(lambda: pv(conv.bias)), Ho,
                  conv.out_channels, self._bn(conv.out_channels), out=out)
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_downsample(self, src, ph, conv, out))
        self.ws.free(ph)
        return out

    def upsample(self, src: Act, conv: nn.Conv2d) -> Act:
        """UpSample (modules.py:89-92): nearest x2 + 3x3 conv.  Inference plans fold the upsampling into the conv
        (idf_conv_desc.up2: the GEMM runs on the input grid, four taps per output parity, pre-summed weights, the
        epilogue scatters the parities: 4/9 of the FLOPs and no upsampled tensor); training plans materialise it."""
        cout = conv.out_channels
        if not self.training and cout in (64, 128) and src.C % 64 == 0:
            H = src.H
            out = self.ws.alloc(2 * H, cout)
            wp = self.weight(lambda: pack_conv3x3_up2(pv(conv.weight)))
            bias = self.f32(lambda: pv(conv.bias).repeat(4))
            # FLOP accounting stays ALGORITHMIC (SURVEY section 8d: the reference's 9 taps on each of the 4 output pixels
            # of an input pixel); the kernel executes 4/9 of these MACs
            self.conv([src], taps_up2(src.C, H, H), wp, bias, H, cout, cout, out=out, up2=True,
                      real_macs_per_row=4 * 9 * src.C * cout)
            return out
        up = self.ws.alloc(src.H * 2, src.C)
        self._emit("upsample2x", self.lib.idf_upsample2x, (src.t.data_ptr(), up.t.data_ptr(), self.B, src.H, src.H, src.C))
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_upsample(self, src, up))
        out = self.conv3x3(up, conv)
        self.ws.free(up)
        return out

    def attn_block(self, x: Act, blk: AttnBlock) -> Act:
        """GroupNorm -> fused qkv GEMM -> attention -> proj GEMM + residual (reference modules.py:145-164)."""
        Cc = x.C
        an = self.norm(x, None, blk.group_norm, silu=False)
        qkv = self.conv1x1(an, [blk.proj_q, blk.proj_k, blk.proj_v], want_stats=False)
        self.done(an)
        ao = self.ws.alloc(x.H, Cc)
        self.attention(qkv, ao, Cc)
        self.ws.free(qkv)
        out = self.conv1x1(ao, [blk.proj], residual=x)
        self.ws.free(ao)
        self.ws.free(x)
        return out

    def res_block(self, xs: Sequence[Act], blk, mod_t=None, mod_z=None, step=None, free_inputs=True,
                  mod_cols: Optional[int] = None) -> Act:
        """AuxResBlock / ResBlock / ResBlock_encoder over one or two (concatenated) inputs."""
        H = xs[0].H
        cin = sum(x.C for x in xs)
        assert cin == blk.in_ch
        cout = blk.out_ch
        x1 = xs[1] if len(xs) > 1 else None
        a1 = self.norm(xs[0], x1, blk.block1[0], silu=True)
        h = self.conv3x3(a1, blk.block1[-1])
        self.done(a1)
        a2 = self.norm(h, None, blk.block2[0], silu=True, mod_t=mod_t, mod_z=mod_z, step=step, dropout=True,
                       mod_cols=mod_cols)
        last_in, last_raw = a2, h
        has_block3 = hasattr(blk, "block3")
        if has_block3:
            h2 = self.conv3x3(a2, blk.block2[-1])
            self.done(a2)
            self.ws.free(h)                       # raw input of a2 (a VAct reads it inside the conv just emitted)
            a3 = self.norm(h2, None, blk.block3[0], silu=True, dropout=True)
            last_in, last_raw = a3, h2
        last_conv = blk.block3[-1] if has_block3 else blk.block2[-1]
        if isinstance(blk.shortcut, nn.Conv2d):
            out = self.conv3x3(last_in, last_conv, shortcut=(blk.shortcut, list(xs)))
        else:
            assert len(xs) == 1
            out = self.conv3x3(last_in, last_conv, residual=xs[0])
        self.done(last_in)
        self.ws.free(last_raw)
        if free_inputs:
            for x in xs:
                self.ws.free(x)
        if isinstance(blk.attn, AttnBlock):
            out = self.attn_block(out, blk.attn)
        return out

    def head(self, x_src: torch.Tensor, conv: nn.Conv2d, Cimg: int, H: int) -> Act:
        """head conv as im2col + K=64 GEMM (reference models.py:246,304,431)."""
        patches = self.ws.alloc(H, 64)
        self._emit("im2col_head", self.lib.idf_im2col_head, (x_src.data_ptr(), patches.t.data_ptr(), self.B, Cimg, H, H))
        cout = conv.out_channels
        h = self.ws.alloc(H, cout)
        self.conv([patches], [(0, 0, 0)], self.weight(lambda: _pad_cols(pack_conv3x3(pv(conv.weight)), 64)),
                  self.f32(lambda: pv(conv.bias)), H, cout, self._bn(cout), out=h, real_macs_per_row=9 * Cimg * cout)
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_head(self, patches, conv, h, Cimg))
        self.ws.free(patches)
        return h

    def tail(self, h: Act, gn: nn.GroupNorm, tconv: nn.Conv2d, H: int, cout: int, epilogue: int, out_f32, **extra) -> None:
        """tail: AdaGN + 3x3 conv to `cout` (<= 16) channels, fp32 NCHW out or fused sampler update."""
        ta = self.norm(h, None, gn, silu=True)
        srcs, kb, xf = self._operand(ta, tap_offsets3x3(H, H))
        self.conv(srcs, kb, self.weight(lambda: _pad_rows(pack_conv3x3(pv(tconv.weight)), 16)),
                  self.f32(lambda: _pad_rows(pv(tconv.bias), 16)), H, cout, 16, epilogue=epilogue, out_f32=out_f32,
                  xf=xf, **extra)
        if self.training:
            from . import train
            self.tape.append(lambda: train.bwd_tail(self, ta, tconv, out_f32, cout))
        self.done(ta)
        self.ws.free(h)

    def unet_body(self, net, x_src: torch.Tensor, Cimg: int, H: int, mods=None) -> Act:
        """head -> down path (every output kept as a skip) -> middle -> up path (skips popped, upsampling folded) of
        a UNet-shaped `net`; returns the activation its tail reads.  `mods(blk)`: the modulation keyword arguments of
        res_block for a conditioned block."""
        kw = mods if mods is not None else (lambda blk: {})
        h = self.head(x_src, net.head, Cimg, H)
        skips = [h]
        for layer in net.downblocks:
            if isinstance(layer, DownSample):
                h = self.downsample(h, layer.main)
            else:
                h = self.res_block([h], layer, free_inputs=False, **kw(layer))
            skips.append(h)
        for i, layer in enumerate(net.middleblocks):
            # the first middle block reads the last skip tensor, which must stay alive for the up path
            h = self.res_block([h], layer, free_inputs=i > 0, **kw(layer))
        for layer in net.upblocks:
            if isinstance(layer, UpSample):
                h2 = self.upsample(h, layer.main)
                self.ws.free(h)
                h = h2
            else:
                h = self.res_block([h, skips.pop()], layer, free_inputs=True, **kw(layer))
        assert not skips
        return h

    # modulation MLPs ------------------------------------------------------------------------------
    def _emit_time_mlp(self, net, pack: "ModulationPack", t_idx: torch.Tensor, out: torch.Tensor) -> None:
        """out[m] = concat_blocks temb_proj(SiLU(time_embedding(t_idx[m])))  (modules.py:36-38, 249, 312)."""
        te = net.time_embedding.timembedding
        M = t_idx.shape[0]
        f32 = dict(dtype=torch.float32, device=self.device)
        e0 = torch.zeros(M, te[0].weight.shape[1], **f32)
        e1 = torch.zeros(M, te[1].out_features, **f32)
        e2 = torch.zeros(M, te[3].out_features, **f32)
        self.keep += [e0, e1, e2]
        table = self.f32(te[0].weight)
        self._emit("gather_rows", self.lib.idf_gather_rows_f32, (table.data_ptr(), t_idx.data_ptr(), e0.data_ptr(), M,
                                                                 e0.shape[1]))
        self.linear(e0, self.f32(te[1].weight), self.f32(te[1].bias), e1, silu_in=False)
        self.linear(e1, self.f32(te[3].weight), self.f32(te[3].bias), e2, silu_in=True)
        self.linear(e2, pack.w_t, pack.b_t, out, silu_in=True)

    def _emit_latent_mlp(self, net, pack: "ModulationPack", a_in: torch.Tensor, out: torch.Tensor) -> None:
        """out[n] = concat_blocks aemb_proj(SiLU(fc_a(a[n])))  (models.py:298; modules.py:316)."""
        fc = net.fc_a
        pre_silu = isinstance(fc, nn.Sequential)      # BottleneckAuxUNet: fc_a = SiLU -> Linear (models.py:336-339)
        if pre_silu:
            fc = fc[1]
        aemb = torch.zeros(a_in.shape[0], fc.out_features, dtype=torch.float32, device=self.device)
        self.keep.append(aemb)
        self.linear(a_in, self.f32(fc.weight), self.f32(fc.bias), aemb, silu_in=pre_silu)
        self.linear(aemb, pack.w_z, pack.b_z, out, silu_in=True)


# ------------------------------------------------------------------------------------------------
# modulation (temb_proj / aemb_proj of every block, batched)
# ------------------------------------------------------------------------------------------------
def modulation_weights(blocks: Sequence[nn.Module]) -> Tuple[torch.Tensor, ...]:
    """(w_t, b_t, w_z, b_z): the temb_proj and aemb_proj Linears of `blocks` concatenated along their outputs in
    block order, with zero rows for a block without aemb_proj.  Not detached, so training can differentiate
    through them."""
    lin_t = [b.temb_proj[1] for b in blocks]
    lin_z = [b.aemb_proj[1] if hasattr(b, "aemb_proj") else None for b in blocks]
    w_z = [z.weight if z is not None else torch.zeros_like(t.weight) for t, z in zip(lin_t, lin_z)]
    b_z = [z.bias if z is not None else torch.zeros_like(t.bias) for t, z in zip(lin_t, lin_z)]
    return (torch.cat([t.weight for t in lin_t], 0), torch.cat([t.bias for t in lin_t], 0), torch.cat(w_z, 0),
            torch.cat(b_z, 0))


class ModulationPack:
    """Column layout of the concatenated per-block (scale | shift) projections."""

    def __init__(self, blocks: Sequence[nn.Module], device):
        self.offsets: Dict[int, int] = {}
        off = 0
        for blk in blocks:
            self.offsets[id(blk)] = off
            off += blk.temb_proj[1].out_features
        self.ncol = off
        self.w_t, self.b_t, self.w_z, self.b_z = (x.detach().to(device=device, dtype=torch.float32).contiguous()
                                                  for x in modulation_weights(blocks))


def conditioned_blocks(net) -> List[nn.Module]:
    return [b for b in list(net.downblocks) + list(net.middleblocks) + list(net.upblocks)
            if isinstance(b, (AuxResBlock, ResBlock))]


# ------------------------------------------------------------------------------------------------
# backbone plan (AuxiliaryUNet)
# ------------------------------------------------------------------------------------------------
class BackbonePlan(Plan):
    """eps = backbone(x, t, a) for a fixed batch, optionally with the sampler update fused into the tail.

    mode 'eps'     : x_in, t_idx, a_in -> eps_out; the modulation rows are computed per call.
    mode 'sampler' : x_io is updated in place, x <- cx*x + ce*eps + cn*noise with (cx,ce,cn) = coef[*step];
                     the timestep modulation is a precomputed [T, ncol] table indexed by *step, the z
                     modulation [B, ncol] is computed once per sampling call by `set_latent`.
    mode 'train'   : x_in and the modulation rows mod_t / mod_z [B, ncol] are inputs (the tiny MLPs that produce
                     them stay in torch autograd); every activation is kept, dropout is on, and the plan
                     records a backward tape (infodiffusion_b200.train).
    """

    def __init__(self, net, batch: int, device, mode: str = "eps", ws: Optional[Workspace] = None,
                 x_io: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None,
                 coef: Optional[torch.Tensor] = None, step: Optional[torch.Tensor] = None,
                 mod_t_table: Optional[torch.Tensor] = None, mod_z: Optional[torch.Tensor] = None,
                 eps_out: Optional[torch.Tensor] = None, pack: Optional[ModulationPack] = None,
                 dropout_p: float = 0.0, ordered: bool = False):
        super().__init__(batch, device, ws, training=(mode == "train"), ordered=ordered)
        assert mode in ("eps", "sampler", "train")
        self.mode = mode
        Cimg, H, W = net.shape
        assert H == W, "square images only"
        assert H in (32, 64), "the sm_100a plans support 32x32 / 64x64 inputs"
        self.net = net
        if mode == "train":
            from .train import stack_params
            self.bind_params(stack_params(net))
        B = batch
        f32 = dict(dtype=torch.float32, device=device)
        self.pack = pack if pack is not None else ModulationPack(conditioned_blocks(net), device)
        ncol = self.pack.ncol
        self.step = step
        if mode == "train":
            self.dropout_p = dropout_p
            self.dropout_seed = torch.zeros(1, dtype=torch.int64, device=device)
        if mode in ("eps", "train"):
            self.x_in = torch.zeros(B, Cimg, H, W, **f32)
            self.eps_out = torch.zeros(B, Cimg, H, W, **f32)
            self.mod_t = torch.zeros(B, ncol, **f32)
            self.mod_z = torch.zeros(B, ncol, **f32)
            if mode == "eps":
                self.t_idx = torch.zeros(B, dtype=torch.long, device=device)
                self._emit_time_mlp(net, self.pack, self.t_idx, self.mod_t)
                if hasattr(net, "fc_a"):                      # UNet (models.py:7) has no latent input
                    self.a_in = torch.zeros(B, net.a_dim, **f32)
                    self._emit_latent_mlp(net, self.pack, self.a_in, self.mod_z)
            else:
                self.d_mod_t = torch.zeros(B, ncol, **f32)
                self.d_mod_z = torch.zeros(B, ncol, **f32)
            mod_t_arg = (self.mod_t.data_ptr(), 0, ncol)
            x_src = self.x_in
        else:
            assert x_io is not None and coef is not None and step is not None and mod_t_table is not None
            self.x_in = x_io
            self.eps_out = eps_out
            self.mod_z = mod_z if mod_z is not None else torch.zeros(B, ncol, **f32)
            mod_t_arg = (mod_t_table.data_ptr(), ncol, 0)
            x_src = x_io
        mod_z_arg = (self.mod_z.data_ptr(), 0, ncol)

        def mods(blk):
            col = self.pack.offsets[id(blk)]
            off = col * 4
            mz = (mod_z_arg[0] + off, mod_z_arg[1], mod_z_arg[2]) if hasattr(blk, "aemb_proj") else None
            return dict(mod_t=(mod_t_arg[0] + off, mod_t_arg[1], mod_t_arg[2]), mod_z=mz, step=self.step, mod_cols=col)

        h = self.unet_body(net, x_src, Cimg, H, mods)
        if mode in ("eps", "train"):
            self.tail(h, net.tail[0], net.tail[-1], H, Cimg, EPI_F32_NCHW, self.eps_out)
        else:
            self.tail(h, net.tail[0], net.tail[-1], H, Cimg, EPI_SAMPLER, self.eps_out, x_io=x_io, noise=noise,
                      coef=coef, step=step)


class ModulationTables(Plan):
    """One-off plans that fill the [T, ncol] timestep table and the [B, ncol] latent rows."""

    def __init__(self, net, device, pack: ModulationPack, T: int):
        super().__init__(1, device)
        self.net, self.pack = net, pack
        self.t_all = torch.arange(T, dtype=torch.long, device=device)
        self.table = torch.zeros(T, pack.ncol, dtype=torch.float32, device=device)
        self._emit_time_mlp(net, pack, self.t_all, self.table)

    def latent_rows(self, a: torch.Tensor, out: torch.Tensor) -> None:
        if not hasattr(self.net, "fc_a"):
            return
        p = Plan(1, self.device)
        p._emit_latent_mlp(self.net, self.pack, a, out)
        p.run()
        torch.cuda.current_stream(self.device).synchronize()  # p's temporaries die with it


# ------------------------------------------------------------------------------------------------
# encoder plan
# ------------------------------------------------------------------------------------------------
class EncoderPlan(Plan):
    """(a, mu, log_var) = Encoder(x) for a fixed batch (reference models.py:488-518).  With training=True only
    the conv stack runs here (x -> 1-channel map, tape recorded); fc_a / fc_mu / fc_var stay in torch autograd.
    Given `latent_noise` [B, a_dim] (filled by the caller before each run), the plan also writes the sampled latent
    a_q = mu + latent_noise * exp(0.5 * log_var) (models.py:515) into self.a_q."""

    def __init__(self, net, batch: int, device, ws: Optional[Workspace] = None, x_in: Optional[torch.Tensor] = None,
                 training: bool = False, dropout_p: float = 0.0, latent_noise: Optional[torch.Tensor] = None,
                 ordered: bool = False):
        super().__init__(batch, device, ws, training=training, ordered=ordered)
        Cimg, H, W = net.shape
        assert H == W and H in (32, 64)
        B = batch
        f32 = dict(dtype=torch.float32, device=device)
        if training:
            self.dropout_p = dropout_p
            self.dropout_seed = torch.zeros(1, dtype=torch.int64, device=device)
        self.net = net
        if training:
            from .train import stack_params
            self.bind_params(stack_params(net))
        self.x_in = x_in if x_in is not None else torch.zeros(B, Cimg, H, W, **f32)
        self.map_out = torch.zeros(B, 1, H, W, **f32)
        self.a = torch.zeros(B, net.a_dim, **f32)
        self.mu = torch.zeros(B, net.a_dim, **f32)
        self.log_var = torch.zeros(B, net.a_dim, **f32)
        h = self.unet_body(net, self.x_in, Cimg, H)
        self.tail(h, net.tail[0], net.tail[-1], H, 1, EPI_F32_NCHW, self.map_out)
        if not training:
            flat = self.map_out.view(B, H * W)
            self.linear(flat, self.f32(net.fc_a.weight), self.f32(net.fc_a.bias), self.a, silu_in=False)
            self.linear(self.a, self.f32(net.fc_mu.weight), self.f32(net.fc_mu.bias), self.mu, silu_in=False)
            self.linear(self.a, self.f32(net.fc_var.weight), self.f32(net.fc_var.bias), self.log_var, silu_in=False)
        self.latent_noise = latent_noise
        self.a_q = None
        if latent_noise is not None:
            assert not training, "the training path samples a_q in torch autograd"
            assert latent_noise.shape == (B, net.a_dim) and latent_noise.is_contiguous()
            self.a_q = torch.zeros(B, net.a_dim, **f32)
            self._emit("reparameterize", self.lib.idf_reparameterize_f32,
                       (self.mu.data_ptr(), self.log_var.data_ptr(), latent_noise.data_ptr(), self.a_q.data_ptr(),
                        B * net.a_dim))


# ------------------------------------------------------------------------------------------------
# nn.Module entry points
# ------------------------------------------------------------------------------------------------
def _check_eval(net) -> None:
    if net.training:
        raise RuntimeError(
            "this is the inference forward (Dropout = identity): call .eval() first, or enable grad so that the "
            "training path (dropout + backward kernels, infodiffusion_b200.train) is taken.")


@torch.no_grad()
def backbone_forward(net, x: torch.Tensor, t: torch.Tensor, a: Optional[torch.Tensor]) -> torch.Tensor:
    _require_cuda(x, "x")
    _check_eval(net)
    B = x.shape[0]
    key = ("eps", B, x.device.index)
    plans = net._plans()
    if key not in plans:
        plans[key] = BackbonePlan(net, B, x.device, mode="eps")
    p: BackbonePlan = plans[key]
    p.x_in.copy_(x)
    p.t_idx.copy_(t.to(torch.long))
    if hasattr(net, "fc_a"):
        p.a_in.copy_(a)
    p.run()
    return p.eps_out.clone()


@torch.no_grad()
def encoder_forward(net, x: torch.Tensor):
    _require_cuda(x, "x")
    _check_eval(net)
    B = x.shape[0]
    key = ("enc", B, x.device.index)
    plans = net._plans()
    if key not in plans:
        plans[key] = EncoderPlan(net, B, x.device,
                                 latent_noise=torch.zeros(B, net.a_dim, dtype=torch.float32, device=x.device))
    p: EncoderPlan = plans[key]
    p.x_in.copy_(x)
    p.latent_noise.copy_(torch.randn_like(p.mu))                     # reference models.py:515
    p.run()
    return p.a.clone(), p.a_q.clone(), p.mu.clone(), p.log_var.clone()


# ------------------------------------------------------------------------------------------------
# latent eps-network (LatentUNet, reference models.py:166-234)
# ------------------------------------------------------------------------------------------------
def _emit_latent_time_chain(plan: Plan, te: nn.Sequential, e0: torch.Tensor, w_cond: torch.Tensor,
                            b_cond: torch.Tensor, out: torch.Tensor) -> None:
    """out = concat_layers linear_emb(SiLU(te[2](SiLU(te[0](e0)))))  for the rows of the sinusoid embeddings e0."""
    e1 = torch.zeros(e0.shape[0], te[0].out_features, dtype=torch.float32, device=plan.device)
    e2 = torch.zeros(e0.shape[0], te[2].out_features, dtype=torch.float32, device=plan.device)
    plan.keep += [e1, e2]
    plan.linear(e0, plan.f32(te[0].weight), plan.f32(te[0].bias), e1, silu_in=False)
    plan.linear(e1, plan.f32(te[2].weight), plan.f32(te[2].bias), e2, silu_in=True)
    plan.linear(e2, w_cond, b_cond, out, silu_in=True)                 # cond_layers = act -> linear_emb


class LatentPlan(Plan):
    """eps = LatentUNet(z, t) for a fixed batch: per layer one fp32 GEMM (idf_linear_f32) and one fused
    (1 + cond) scale -> LayerNorm -> SiLU kernel that writes straight into the [h | z] concatenation buffer the
    next layer reads (models.py:230-232).  Weight-bandwidth-bound: 13.5 M parameters for a_dim = 256.

    mode 'eps'     : z_in [B, D], t_idx [B] -> eps_out; the per-sample condition rows are computed per call.
    mode 'sampler' : z_io is updated in place by idf_sampler_update with coef[*step]; every sample shares the
                     timestep, so the condition rows come from a precomputed [T, n_cond * 4D] table."""

    def __init__(self, net, batch: int, device, mode: str = "eps", T: Optional[int] = None,
                 z_io: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None,
                 coef: Optional[torch.Tensor] = None, step: Optional[torch.Tensor] = None,
                 eps_out: Optional[torch.Tensor] = None):
        super().__init__(batch, device)
        assert mode in ("eps", "sampler")
        self.net, self.mode = net, mode
        B = batch
        f32 = dict(dtype=torch.float32, device=device)
        layers = list(net.layers)
        D = layers[0].linear.in_features
        Hd = layers[0].linear.out_features
        assert all(l.use_cond and isinstance(l.norm, nn.LayerNorm) for l in layers[:-1]) and not layers[-1].use_cond
        assert all(l.condition_bias == 1 for l in layers[:-1]), "kernel folds condition_bias = 1 (models.py:219)"
        n_cond = len(layers) - 1
        self.z_in = z_io if z_io is not None else torch.zeros(B, D, **f32)
        self.eps_out = eps_out if eps_out is not None else torch.zeros(B, D, **f32)
        self.hcat = torch.zeros(B, Hd + D, **f32)          # [h | z]: layer i >= 1 reads cat([h, z])
        self.ybuf = torch.zeros(B, Hd, **f32)
        w_cond = self.f32(torch.cat([l.linear_emb.weight for l in layers[:-1]], 0))
        b_cond = self.f32(torch.cat([l.linear_emb.bias for l in layers[:-1]], 0))
        C_t = net.num_time_emb_channels
        assert T is not None, "LatentPlan needs the number of diffusion steps for its sinusoid table"
        table = timestep_embedding(torch.arange(T, device=device), C_t).contiguous()          # modules.py:41-60
        if mode == "eps":
            self.t_idx = torch.zeros(B, dtype=torch.long, device=device)
            e0 = torch.zeros(B, C_t, **f32)
            self.cond = torch.zeros(B, n_cond * Hd, **f32)
            self.keep += [table, e0]
            self._emit("gather_rows", self.lib.idf_gather_rows_f32, (table.data_ptr(), self.t_idx.data_ptr(), e0.data_ptr(), B, C_t))
            _emit_latent_time_chain(self, net.time_embed, e0, w_cond, b_cond, self.cond)
            cond_arg = lambda i: (self.cond.data_ptr() + 4 * i * Hd, n_cond * Hd, 0, None)
        else:
            assert z_io is not None and coef is not None and step is not None
            tp = Plan(1, device)                                               # one-off: the [T, n_cond * Hd] table
            self.cond = torch.zeros(T, n_cond * Hd, **f32)
            _emit_latent_time_chain(tp, net.time_embed, table, w_cond, b_cond, self.cond)
            tp.run()
            torch.cuda.current_stream(device).synchronize()
            cond_arg = lambda i: (self.cond.data_ptr() + 4 * i * Hd, 0, n_cond * Hd, step.data_ptr())
        ld = Hd + D
        self._emit("copy2d", self.lib.idf_copy2d_f32, (self.z_in.data_ptr(), self.z_in.stride(0),
                                                       self.hcat.data_ptr() + 4 * Hd, ld, B, D))
        for i, l in enumerate(layers):
            src = self.z_in if i == 0 else self.hcat
            w, b = self.f32(l.linear.weight), self.f32(l.linear.bias)
            if i == len(layers) - 1:
                self.linear(src, w, b, self.eps_out, silu_in=False)            # plain Linear (models.py:195-200)
                break
            self.linear(src, w, b, self.ybuf, silu_in=False)
            cptr, crow, cstep, sptr = cond_arg(i)
            self._emit("scale_ln_silu", self.lib.idf_scale_layernorm_silu,
                       (self.ybuf.data_ptr(), Hd, cptr, crow, cstep, sptr, self.f32(l.norm.weight).data_ptr(),
                        self.f32(l.norm.bias).data_ptr(), float(l.norm.eps), self.hcat.data_ptr(), ld, B, Hd,
                        1 if l.activation is not None else 0))
        if mode == "sampler":
            self._emit("sampler_update", self.lib.idf_sampler_update,
                       (self.z_in.data_ptr(), self.eps_out.data_ptr(), _ptr(noise), coef.data_ptr(), step.data_ptr(), B * D))


@torch.no_grad()
def latent_forward(net, x: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, "x")
    _check_eval(net)
    B = x.shape[0]
    T = int(getattr(net, "T", 0)) or None
    key = ("latent_eps", B, x.device.index)
    plans = net._plans()
    if key not in plans:
        if T is None:
            raise RuntimeError("LatentUNet was built without T; pass T= to the constructor")
        plans[key] = LatentPlan(net, B, x.device, mode="eps", T=T)
    p: LatentPlan = plans[key]
    p.z_in.copy_(x)
    p.t_idx.copy_(t.to(torch.long))
    p.run()
    return p.eps_out.clone()


def latent_forward_autograd(net, x: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """Training-mode LatentUNet forward (reference models.py:223-234, 147-163) inside torch's autograd graph.  Every
    Linear -- the time MLP, the ten layers, their condition projections -- runs forward AND backward on the library's
    own fp32 kernels (infodiffusion_b200.linear: idf_linear_f32 / idf_gemm_f32); the elementwise glue (SiLU, the
    (1 + cond) scale, LayerNorm, dropout, cat) is ordinary torch."""
    from . import linear as L
    from .modules import timestep_embedding
    _require_cuda(x, "x")
    temb = timestep_embedding(t, net.num_time_emb_channels)
    for m in net.time_embed:
        temb = L.apply(m, temb) if isinstance(m, nn.Linear) else m(temb)
    h = x
    for i, layer in enumerate(net.layers):
        if i in net.skip_layers:
            h = torch.cat([h, x], dim=1)
        h = L.apply(layer.linear, h)
        if layer.use_cond:
            h = h * (layer.condition_bias + L.apply(layer.linear_emb, layer.act(temb)))
        h = layer.dropout(layer.act(layer.norm(h)))
    return h
