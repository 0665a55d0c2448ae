"""Training side of the engine: backward plans of AuxiliaryUNet / Encoder and their autograd bridge.

A training plan (engine.BackbonePlan(mode='train') / EncoderPlan(training=True)) keeps every activation
and records one backward emitter per forward composite.  `finalize_backward(plan)` replays the tape in
reverse and builds the backward op list once; per step only kernels run.

Gradient conventions
  * activation gradients: bf16 pad-flat buffers with the geometry of the activation (pad rows stay zero,
    which is what the conv data-gradient needs as its `padding`);
  * data gradient of a conv  = the forward implicit-GEMM kernel over dY with negated taps / transposed weights;
  * weight gradient          = idf_wgrad (tcgen05, pixels as K), fp32, one flat buffer zeroed per step;
  * bias gradient            = column sums of dY;
  * input gradient           = the head conv's data gradient into fp32 NCHW, one launch after the backward graph,
    only when the network's input requires grad (bwd_head);
  * AdaGN                    = idf_adagn_silu_bwd -> dx and (S1, S2); gamma/beta/modulation grads in closed form;
  * attention backward       = recomputed with torch matmuls for now (1 % of the FLOPs; kernel is a next step);
  * the small MLPs (time embedding, fc_a, temb/aemb projections, encoder fc heads) and the loss arithmetic stay
    in torch autograd: this module exposes the conv stacks as autograd Functions with (x, mod_t, mod_z) inputs.

Deterministic mode: a plan built while torch.are_deterministic_algorithms_enabled() is an ORDERED plan.  Its split-K
weight gradients, bias gradients and GroupNorm-affine gradients use the library's ordered variants, whose partials are
combined in a fixed index order, so the step is bitwise reproducible on one GPU model.  The plan owns their workspaces:
one scratch shared by the side-stream ops (weight / bias gradients run in stream order there) and one for the
main-stream AdaGN backward, each with its own ticket counter.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import _lib
from ._lib import EPI_F32_NCHW, AdaGNBwdArgs, WgradDesc
from .engine import (Act, BackbonePlan, EncoderPlan, Op, _require_cuda, conditioned_blocks, modulation_weights,
                     run_ops)
from .layout import pad_rows, pv, stride2_phase_dgrad, tap_offsets3x3, taps_stride2

BF16 = torch.bfloat16


def adagn_param_grads(sums: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor,
                      s_t: Optional[torch.Tensor] = None, b_t: Optional[torch.Tensor] = None,
                      s_z: Optional[torch.Tensor] = None, b_z: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """Gradients of y = silu(((xhat*gamma + beta)(1+s_t) + b_t)(1+s_z) + b_z) w.r.t. everything but x, from
    the per-(sample, channel) sums S1 = sum_hw dv, S2 = sum_hw dv*xhat the backward kernel returns
    (dv = dL/d pre-activation).  sums: [B, C, 2]; gamma/beta: [C]; modulation tensors: [B, C] or None."""
    S1, S2 = sums[..., 0], sums[..., 1]
    q = gamma[None, :] * S2 + beta[None, :] * S1          # sum_hw dv * (xhat*gamma + beta)
    T = (1 + s_t) if s_t is not None else torch.ones_like(S1)
    Z = (1 + s_z) if s_z is not None else torch.ones_like(S1)
    out = {"gamma": (T * Z * S2).sum(0), "beta": (T * Z * S1).sum(0)}
    if s_t is not None:
        out["s_t"] = Z * q
        out["b_t"] = Z * S1
    if s_z is not None:
        out["s_z"] = T * q + (b_t if b_t is not None else 0) * S1
        out["b_z"] = S1
    return out


# ------------------------------------------------------------------------------------------------
# backward-plan state attached to a training plan
# ------------------------------------------------------------------------------------------------
@dataclass
class Part:
    """One K segment of a conv: source activation, the parameter its weights come from, kernel kind and
    (for a 1x1 shortcut over concatenated sources) the input-channel slice of that parameter."""
    src: "object"
    weight: nn.Parameter
    kind: str                       # '3x3' | '1x1'
    cslice: Optional[Tuple[int, int]]


class BwdState:
    def __init__(self, plan, ordered: bool):
        self.plan = plan
        self.ops: List[Op] = []          # run in order by run_backward; callable args are resolved by finalize_backward
        self.gathers: List[Op] = []      # arena -> parameter-shaped gradients, after the side stream has joined
        self.grads: Dict[int, object] = {}               # id(Act) -> gradient Act
        self.written: Dict[int, bool] = {}
        self.flat_chunks: List[Tuple[int, int]] = []     # (offset, numel) of fp32 grad buffers in the flat arena
        self.flat_size = 0
        self.flat: Optional[torch.Tensor] = None
        self.views: List = []                            # (name, offset, shape) resolved after allocation
        self.param_grads: List[Tuple[nn.Parameter, Callable[[], torch.Tensor]]] = []
        self.keep: List = []
        self.wplans: List = []                           # (desc, handle, arena getter, op)
        self.side_stream = torch.cuda.Stream(plan.device)
        self.ordered = ordered
        self.final = False
        self.side_ws_floats = 0      # ordered: largest colsum workspace (the wgrad partials are sized once the plans exist)
        self.main_ws_floats = 0      # ordered: largest AdaGN dgamma / dbeta workspace
        self.side_ws: Optional[torch.Tensor] = None
        self.main_ws: Optional[torch.Tensor] = None
        self.tickets: Optional[torch.Tensor] = None   # [0]: side-stream ops, [1]: main-stream ops; zero between launches

    def __del__(self):
        try:
            for _, h, _, _ in self.wplans:
                if h:
                    self.plan.lib.idf_wgrad_plan_destroy(h)
        except Exception:
            pass

    # ---- fp32 arena (weight / bias gradients), zeroed once per step
    def arena(self, shape) -> Callable[[], torch.Tensor]:
        n = 1
        for d in shape:
            n *= d
        off = self.flat_size
        self.flat_size += (n + 3) // 4 * 4
        return lambda: self.flat[off:off + n].view(*shape)

    # ---- activation gradients
    def grad(self, act):
        g = self.grads.get(id(act))
        if g is None:
            t = torch.zeros_like(act.t)
            g = Act(t, act.H, act.C, act.phases, act.rows)
            self.grads[id(act)] = g
            self.written[id(act)] = False
            self.keep.append(g)
        return g

    def is_written(self, act) -> bool:
        return self.written.get(id(act), False)

    def mark(self, act) -> None:
        self.written[id(act)] = True

    def op(self, tag: str, fn, *args, kernels: int = 1, side: bool = False) -> Op:
        self.ops.append(Op(tag, fn, args, kernels, side=side))
        return self.ops[-1]


# ------------------------------------------------------------------------------------------------
# conv backward building blocks
# ------------------------------------------------------------------------------------------------
def _dgrad(plan, st: BwdState, dout, target, kblocks, wrecipe, cin: int) -> None:
    """grad(target) (+)= implicit GEMM over dout with the given (negated-tap) K-blocks and [cin, K] weights."""
    g = st.grad(target)
    acc = st.is_written(target)
    wp = plan.weight(wrecipe)
    zero_bias = torch.zeros(wp.shape[0], dtype=torch.float32, device=plan.device)
    plan.keep.append(zero_bias)
    st.ops.append(plan.conv([dout], kblocks, wp, zero_bias, target.H, cin, plan._bn(cin), out=g,
                            residual=g if acc else None, want_stats=False, emit=False))
    st.mark(target)


def _wgrad(plan, st: BwdState, dout, x, x_rows: int, cin: int, cout: int, tap_off: Sequence[int]):
    """fp32 [cout, ntaps, cin] weight-gradient buffer filled by idf_wgrad; returns its arena getter."""
    get = st.arena((cout, len(tap_off), cin))
    d = WgradDesc()
    d.dy, d.rows, d.cout = dout.t.data_ptr(), dout.rows, cout
    d.x, d.x_rows, d.cin = x.t.data_ptr(), x_rows, cin
    d.n_taps = len(tap_off)
    for i, o in enumerate(tap_off):
        d.tap_off[i] = o
    h = C.c_void_p()                         # created once the arena is allocated (needs the dw pointer)
    st.keep.append(d)
    st.wplans.append((d, h, get, st.op("wgrad", plan.lib.idf_wgrad_run, h, side=True)))
    return get


def _bias_grad(plan, st: BwdState, dout, cout: int):
    get = st.arena((cout,))
    args = (dout.t.data_ptr(), lambda: get().data_ptr(), dout.rows, cout)
    if st.ordered:
        st.side_ws_floats = max(st.side_ws_floats, int(plan.lib.idf_colsum_ws_floats(dout.rows, cout)))
        st.op("colsum", plan.lib.idf_colsum_bf16_ordered, *args, lambda: st.side_ws.data_ptr(),
              lambda: st.tickets.data_ptr(), side=True)
    else:
        st.op("colsum", plan.lib.idf_colsum_bf16, *args, side=True)
    return get


def _add_into(plan, st: BwdState, src, target) -> None:
    """grad(target) (+)= src  (identity / residual paths), plain torch elementwise on bf16 buffers."""
    g = st.grad(target)
    if st.is_written(target):
        st.op("add", g.t.add_, src.t, kernels=0)
    else:
        st.op("copy", g.t.copy_, src.t, kernels=0)
    st.mark(target)


def bwd_conv(plan, parts: Sequence[Part], biases: Sequence[nn.Parameter], out, residual) -> None:
    """conv3x3 (+ fused 1x1 shortcut parts) (+ identity residual)."""
    st = plan.bwd
    dout = st.grad(out)
    H, cout = out.H, out.C
    offs = tap_offsets3x3(H, H)
    sc_dw = []
    for prt in parts:
        src, w = prt.src, prt.weight
        if prt.kind == "3x3":
            kb = []
            for off in offs:
                kb += [(0, c0, -off) for c0 in range(0, cout, 64)]
            _dgrad(plan, st, dout, src, kb, lambda w=w: pv(w).permute(1, 2, 3, 0).reshape(w.shape[1], 9 * w.shape[0]), src.C)
            get = _wgrad(plan, st, dout, src, src.t.shape[0], src.C, cout, offs)
            st.param_grads.append((w, lambda get=get, w=w: get().view(w.shape[0], 3, 3, w.shape[1]).permute(0, 3, 1, 2)))
        else:
            c0s, c1s = prt.cslice
            kb = [(0, c0, 0) for c0 in range(0, cout, 64)]
            _dgrad(plan, st, dout, src, kb, lambda w=w, a=c0s, b=c1s: pv(w)[:, a:b, 0, 0].t(), src.C)
            sc_dw.append((prt, _wgrad(plan, st, dout, src, src.t.shape[0], src.C, cout, [0])))
    if sc_dw:
        w = sc_dw[0][0].weight
        st.param_grads.append((w, lambda: torch.cat([g()[:, 0, :] for _, g in sc_dw], dim=1)[:, :, None, None]))
    bget = _bias_grad(plan, st, dout, cout)
    for b in biases:
        st.param_grads.append((b, bget))
    if residual is not None:
        _add_into(plan, st, dout, residual)


def bwd_conv1x1_stack(plan, src, convs: Sequence[nn.Conv2d], out, residual) -> None:
    """1x1 conv(s) stacked along N (qkv / proj)."""
    st = plan.bwd
    dout = st.grad(out)
    cout, cin = out.C, src.C
    kb = [(0, c0, 0) for c0 in range(0, cout, 64)]
    _dgrad(plan, st, dout, src, kb, lambda: torch.cat([pv(m.weight)[:, :, 0, 0] for m in convs], dim=0).t(), cin)
    get = _wgrad(plan, st, dout, src, src.t.shape[0], cin, cout, [0])
    bget = _bias_grad(plan, st, dout, cout)
    o = 0
    for m in convs:
        n = m.out_channels
        st.param_grads.append((m.weight, lambda get=get, o=o, n=n: get()[o:o + n, 0, :, None, None]))
        st.param_grads.append((m.bias, lambda bget=bget, o=o, n=n: bget()[o:o + n]))
        o += n
    if residual is not None:
        _add_into(plan, st, dout, residual)


def bwd_head(plan, patches, conv: nn.Conv2d, out, Cimg: int) -> None:
    """head conv (im2col + K=64 GEMM): weight and bias gradients in the backward list.  The input gradient is a
    Cimg <- cout 3x3 conv over dY (negated taps, transposed weights, fp32 NCHW out: the tail's forward shape) whose
    conv plan is kept on the training plan as `dx_op`; _ConvStackFn.backward launches it only when the input
    requires grad, so a step without input gradient keeps its launch list."""
    st = plan.bwd
    dout = st.grad(out)
    cout, H = out.C, out.H
    get = _wgrad(plan, st, dout, patches, patches.t.shape[0], 64, cout, [0])
    st.param_grads.append((conv.weight, lambda: get()[:, 0, :9 * Cimg].view(cout, 9, Cimg).permute(0, 2, 1)
                           .reshape(cout, Cimg, 3, 3)))
    st.param_grads.append((conv.bias, _bias_grad(plan, st, dout, cout)))
    kb = [(0, c0, -off) for off in tap_offsets3x3(H, H) for c0 in range(0, cout, 64)]
    # packed with the plan's other recipes, so the re-pack before every forward keeps it on the current parameters
    wp = plan.weight(lambda: pad_rows(pv(conv.weight).permute(1, 2, 3, 0).reshape(Cimg, 9 * cout), 16))
    zero_bias = torch.zeros(wp.shape[0], dtype=torch.float32, device=plan.device)
    plan.d_x = torch.zeros(plan.B, Cimg, H, H, dtype=torch.float32, device=plan.device)
    plan.keep.append(zero_bias)
    plan.dx_op = plan.conv([dout], kb, wp, zero_bias, H, Cimg, 16, epilogue=EPI_F32_NCHW, out_f32=plan.d_x, emit=False)


def run_input_grad(plan) -> torch.Tensor:
    """d_x of the plan's input from the head output's gradient the last backward left (see bwd_head)."""
    run_ops([plan.dx_op], plan.device)
    return plan.d_x.clone()


def bwd_tail(plan, ta, tconv: nn.Conv2d, out_f32: torch.Tensor, cout: int) -> None:
    """tail conv (fp32 NCHW output): dY arrives as fp32 NCHW in plan.d_out, is re-laid out to a 64-channel
    pad-flat bf16 matrix (channels >= cout zero) and then treated like any other conv gradient."""
    st = plan.bwd
    H, cin = ta.H, ta.C
    rows = ta.rows
    dpf = Act(torch.zeros(rows, 64, dtype=BF16, device=plan.device), H, 64, 1, rows)
    st.keep.append(dpf)
    plan.d_out = torch.zeros_like(out_f32)
    st.op("nchw_to_padflat", plan.lib.idf_nchw_to_padflat_ld, plan.d_out.data_ptr(), dpf.t.data_ptr(), plan.B, cout, H, H,
          64)
    offs = tap_offsets3x3(H, H)
    kb = [(0, 0, -off) for off in offs]

    def wt():
        w = pv(tconv.weight)                                       # [cout, cin, 3, 3]
        full = torch.zeros(cin, 9, 64, dtype=w.dtype, device=w.device)
        full[:, :, :cout] = w.permute(1, 2, 3, 0).reshape(cin, 9, cout)
        return full.reshape(cin, 9 * 64)
    _dgrad(plan, st, dpf, ta, kb, wt, cin)
    get = _wgrad(plan, st, dpf, ta, rows, cin, 64, offs)
    st.param_grads.append((tconv.weight, lambda: get()[:cout].view(cout, 3, 3, cin).permute(0, 3, 1, 2)))
    bget = _bias_grad(plan, st, dpf, 64)
    st.param_grads.append((tconv.bias, lambda: bget()[:cout]))


def bwd_downsample(plan, src, ph, conv: nn.Conv2d, out) -> None:
    """stride-2 conv over space-to-depth phases: one data-gradient GEMM per phase, then depth-to-space."""
    st = plan.bwd
    dout = st.grad(out)
    Ho, Cc, cout = out.H, src.C, out.C
    rows_o = out.rows
    dph_t = torch.zeros_like(ph.t)
    st.keep.append(dph_t)
    w = conv.weight
    for phase, taps, kb in stride2_phase_dgrad(cout, Ho, Ho):
        tgt = Act(dph_t[phase * rows_o:(phase + 1) * rows_o], Ho, Cc, 1, rows_o)
        st.keep.append(tgt)
        st.grads[id(tgt)] = tgt              # the phase slice IS the gradient buffer of this pseudo-activation
        st.written[id(tgt)] = False
        _dgrad(plan, st, dout, tgt, kb,
               lambda taps=taps: torch.cat([pv(w)[:, :, ky, kx].t() for ky, kx in taps], dim=1), Cc)
    g = st.grad(src)
    st.op("depth_to_space", plan.lib.idf_depth_to_space, dph_t.data_ptr(), g.t.data_ptr(), plan.B, src.H, src.H, Cc,
          1 if st.is_written(src) else 0)
    st.mark(src)
    offs = [o for (_, _, o) in taps_stride2(64, Ho, Ho, rows_o)]      # one offset per tap (cin = 64 -> one chunk)
    get = _wgrad(plan, st, dout, ph, ph.t.shape[0], Cc, cout, offs)
    st.param_grads.append((w, lambda: get().view(cout, 3, 3, Cc).permute(0, 3, 1, 2)))
    st.param_grads.append((conv.bias, _bias_grad(plan, st, dout, cout)))


def bwd_upsample(plan, src, up) -> None:
    st = plan.bwd
    dup = st.grad(up)
    g = st.grad(src)
    st.op("upsample2x_bwd", plan.lib.idf_upsample2x_bwd, dup.t.data_ptr(), g.t.data_ptr(), plan.B, src.H, src.H, src.C,
          1 if st.is_written(src) else 0)
    st.mark(src)


def bwd_adagn(plan, a, src0, src1, out, gn: nn.GroupNorm, gamma: torch.Tensor, beta: torch.Tensor,
              mod_cols: Optional[int]) -> None:
    st = plan.bwd
    dy = st.grad(out)
    Cc = out.C
    b = AdaGNBwdArgs()
    b.f = a
    b.dy = dy.t.data_ptr()
    g0 = st.grad(src0)
    b.dx0, b.acc0 = g0.t.data_ptr(), 1 if st.is_written(src0) else 0
    st.mark(src0)
    if src1 is not None:
        g1 = st.grad(src1)
        b.dx1, b.acc1 = g1.t.data_ptr(), 1 if st.is_written(src1) else 0
        st.mark(src1)
    sums = torch.zeros(plan.B, Cc, 2, dtype=torch.float32, device=plan.device)
    ws = torch.zeros(int(plan.lib.idf_adagn_bwd_ws_floats(plan.B, Cc)), dtype=torch.float32, device=plan.device)
    b.sums, b.ws = sums.data_ptr(), ws.data_ptr()
    st.keep += [b, sums, ws]
    # gamma / beta / modulation gradients: closed forms of (S1, S2), fused into the kernel
    gget, bget = st.arena((Cc,)), st.arena((Cc,))
    if a.mod_t:
        b.d_mod_t = plan.d_mod_t.data_ptr() + 4 * mod_cols
    if a.mod_z:
        b.d_mod_z = plan.d_mod_z.data_ptr() + 4 * mod_cols
    if st.ordered:
        st.main_ws_floats = max(st.main_ws_floats, plan.B * Cc * 2)

    def args():
        b.dgamma, b.dbeta = gget().data_ptr(), bget().data_ptr()
        if st.ordered:
            b.dparam_ws, b.dparam_ticket = st.main_ws.data_ptr(), st.tickets.data_ptr() + 4
        return C.byref(b)
    st.op("adagn_bwd", plan.lib.idf_adagn_silu_bwd, args, kernels=2)       # statistics, then apply
    st.param_grads.append((gn.weight, gget))
    st.param_grads.append((gn.bias, bget))


def bwd_attention(plan, qkv, out, d: int) -> None:
    """Softmax attention backward (reference modules.py:145-164 under autograd) on the tcgen05 kernels of
    csrc/attention_bwd.cu: P and dS are recomputed from the saved q | k | v, then dQ = dS K, dK = dS^T Q, dV = P^T dO."""
    st = plan.bwd
    dout = st.grad(out)
    gq = st.grad(qkv)
    H = qkv.H
    ws = torch.empty(int(plan.lib.idf_attn_bwd_ws_bytes(plan.B, H, H)), dtype=torch.uint8, device=plan.device)
    plan.keep.append(ws)
    st.op("attention_bwd", plan.lib.idf_attn_bwd, qkv.t.data_ptr(), dout.t.data_ptr(), gq.t.data_ptr(), ws.data_ptr(),
          plan.B, H, H, d, float(d) ** -0.5, kernels=_attn_bwd_kernels(H * H, d))
    st.mark(qkv)


def _attn_bwd_kernels(S: int, d: int) -> int:
    """Kernels idf_attn_bwd launches: scores, then gradients on the tcgen05 path (d in {128, 256, 512} with S = H*W in
    {64, 256}); one small-map kernel otherwise."""
    return 2 if d in (128, 256, 512) and S in (64, 256) else 1


# ------------------------------------------------------------------------------------------------
# finalisation and execution
# ------------------------------------------------------------------------------------------------
def finalize_backward(plan) -> BwdState:
    """Replay the tape in reverse, allocate the fp32 gradient arena, create the wgrad plans and resolve the op
    arguments that point into them."""
    st = plan.bwd
    if st.final:
        return st
    for emit in reversed(plan.tape):
        emit()
    st.flat = torch.zeros(max(st.flat_size, 4), dtype=torch.float32, device=plan.device)
    for d, h, get, _ in st.wplans:
        d.dw = get().data_ptr()
        _lib.check(plan.lib.idf_wgrad_plan_create(C.byref(d), C.byref(h)))
    if st.ordered:
        # the split-K partials share the side-stream scratch; their size is known once the plans exist, and the
        # pointer is part of the plan, so the multi-slab plans are created again with it
        part = [int(plan.lib.idf_wgrad_plan_partials_floats(h)) for _, h, _, _ in st.wplans]
        st.side_ws = torch.zeros(max([st.side_ws_floats, 4] + part), dtype=torch.float32, device=plan.device)
        st.main_ws = torch.zeros(max(st.main_ws_floats, 4), dtype=torch.float32, device=plan.device)
        st.tickets = torch.zeros(2, dtype=torch.int32, device=plan.device)
        for (d, h, _, op), n in zip(st.wplans, part):
            if n:
                _lib.check(plan.lib.idf_wgrad_plan_destroy(h))
                d.partials = st.side_ws.data_ptr()
                _lib.check(plan.lib.idf_wgrad_plan_create(C.byref(d), C.byref(h)))
                op.kernels = 2                   # + the slab reduction
    for op in st.ops:
        op.args = tuple(a() if callable(a) else a for a in op.args)
    st.ops.insert(0, Op("zero_grads", st.flat.zero_, (), kernels=0))
    _build_grad_maps(plan, st)
    st.gathers = [Op("grad_gather", plan.lib.idf_gather_elems, (st.flat.data_ptr(), m.data_ptr(), None,
                                                                 st.grad_flat.data_ptr(), m.numel(), 0, 1 if k else 0))
                  for k, m in enumerate(st.grad_maps)]          # one per pass, the later passes accumulate
    st.final = True
    return st


def _build_grad_maps(plan, st: BwdState) -> None:
    """Gather maps arena -> parameter-shaped gradients.  Every entry of st.param_grads is a pure view / cat of
    arena buffers, so evaluating it over an arena of 1-based indices gives the map; pass k holds the k-th
    contribution of each parameter (a parameter used by several GEMM segments is summed over passes)."""
    pindex = plan.pindex
    values = st.flat
    st.flat = torch.arange(1, values.numel() + 1, dtype=torch.int64, device=plan.device)
    passes: List[torch.Tensor] = []
    seen: Dict[int, int] = {}
    try:
        for prm, get in st.param_grads:
            k = seen.get(id(prm), 0)
            seen[id(prm)] = k + 1
            if k == len(passes):
                passes.append(torch.zeros(pindex.total, dtype=torch.int32, device=plan.device))
            off = pindex.offset[id(prm)]
            passes[k][off:off + prm.numel()] = get().reshape(-1).to(torch.int32)
    finally:
        st.flat = values
    st.grad_maps = passes
    st.grad_flat = torch.zeros(pindex.total, dtype=torch.float32, device=plan.device)
    st.has_grad = [id(p) in seen for p in pindex.params]


def run_backward(plan) -> None:
    st = finalize_backward(plan)
    # Weight and bias gradients are leaves: each needs only dY and the saved input of its layer, nothing on the
    # data-gradient chain waits for them.  They are forked onto a second stream (inside the captured graph: parallel
    # branches), where they fill the SMs that the small-batch chain kernels leave idle; joined before the gather.
    run_ops(st.ops, plan.device, side=st.side_stream if SIDE_STREAM else None)
    run_ops(st.gathers, plan.device)


def fused_param_grads(plan) -> List[Optional[torch.Tensor]]:
    """Gradients of plan.pindex.params (None where the conv stack contributes nothing), as views of a fresh
    copy of the flat gradient buffer.  With a GradSync installed the flat buffer's all-reduce is started here,
    i.e. the backbone's gradients travel over NVLink while the encoder's backward kernels are still running."""
    st = plan.bwd
    flat = st.grad_flat.clone()
    views = plan.pindex.views(flat)
    if _grad_sync is not None:
        _grad_sync.reduce(flat, [p for p, has in zip(plan.pindex.params, st.has_grad) if has],
                          [v for v, has in zip(views, st.has_grad) if has])
    return [v if has else None for v, has in zip(views, st.has_grad)]


class GradSync:
    """Data-parallel gradient exchange overlapped with the backward pass (SURVEY section 8e, training row).

    Every conv-stack backward hands its flat fp32 gradient buffer to `reduce`, which launches one asynchronous
    all-reduce (average) on it; `finish` waits for those and all-reduces the few remaining gradients (time / latent
    MLPs, fc heads) in one more flat buffer.  Gradient clipping and the optimizer run after `finish`, so the
    global norm is identical on all ranks with no further collective."""

    def __init__(self, world: int):
        import torch.distributed as dist
        self.world = world
        self.avg = dist.get_backend() == "nccl"            # gloo has no AVG: sum, then divide
        self.pending: List = []
        self.covered: set = set()
        self.fixed_up = 0          # gradients that did not alias the reduced buffer and were copied from it (see finish)

    def reduce(self, flat: torch.Tensor, params: Sequence[nn.Parameter],
               views: Optional[Sequence[torch.Tensor]] = None) -> None:
        """Start the all-reduce of `flat`.  `views[i]` is the slice of `flat` that autograd receives as the gradient
        of `params[i]`; `finish` uses it to make sure p.grad really holds the REDUCED values."""
        import torch.distributed as dist
        op = dist.ReduceOp.AVG if self.avg else dist.ReduceOp.SUM
        # keep (offset, numel), NOT the view tensors: a second reference to a view stops AccumulateGrad from stealing
        # it (use_count check), and every gradient would then be cloned before the reduction has finished
        spans = [(p, v.storage_offset() - flat.storage_offset(), v.numel()) for p, v in zip(params, views)] if views is not None else []
        self.pending.append((dist.all_reduce(flat, op=op, async_op=True), flat, spans))
        self.covered.update(id(p) for p in params)

    def finish(self, params: Sequence[nn.Parameter]) -> None:
        allreduce_gradients([p for p in params if id(p) not in self.covered], self.world)
        for work, flat, pv_pairs in self.pending:
            work.wait()
            if not self.avg:
                flat.div_(self.world)
            # The reduction happened in `flat`.  It reaches p.grad only if AccumulateGrad STOLE the view it was
            # handed (p.grad aliases `flat`).  If p.grad already existed (zero_grad(set_to_none=False), gradient
            # accumulation, a second loss term) or autograd cloned the incoming gradient, p.grad holds local values:
            # overwrite it with the reduced slice so the ranks cannot drift apart silently.
            lo = flat.data_ptr()
            hi = lo + flat.numel() * flat.element_size()
            for prm, off, numel in pv_pairs:
                g = prm.grad
                if g is None or lo <= g.data_ptr() < hi:
                    continue
                self.fixed_up += 1
                g.copy_(flat[off:off + numel].view_as(g))
        self.pending.clear()
        self.covered.clear()


_grad_sync: Optional[GradSync] = None


def set_grad_sync(sync: Optional[GradSync]) -> None:
    global _grad_sync
    _grad_sync = sync


def collect_param_grads(plan) -> Dict[nn.Parameter, torch.Tensor]:
    """Sum the contributions per parameter (a parameter can appear in several K segments)."""
    st = plan.bwd
    out: Dict[nn.Parameter, torch.Tensor] = {}
    for prm, get in st.param_grads:
        g = get()
        if prm in out:
            out[prm] = out[prm] + g
        else:
            out[prm] = g
    return out


# ------------------------------------------------------------------------------------------------
# autograd bridge
# ------------------------------------------------------------------------------------------------
USE_GRAPHS = True
SIDE_STREAM = True      # weight / bias gradient kernels on a second stream (parallel branches of the backward graph)


def _replay(plan, slot: str, body: Callable[[], None]) -> None:
    """Run `body` (op lists over static buffers: weight re-packing + forward plan, or the backward lists).  First
    call: eager (also sets kernel attributes); second call: captured into a CUDA graph; afterwards a single graph
    replay -- the ~1000 launches of a step cost one launch on the host.  The capture counts the kernels the graph
    holds, the same declared sum as an eager run; every later replay adds that sum."""
    state = getattr(plan, slot, None)
    if not USE_GRAPHS or state is None:
        body()
        if USE_GRAPHS:
            setattr(plan, slot, "warm")
    elif state == "warm":
        torch.cuda.synchronize(plan.device)
        g = torch.cuda.CUDAGraph()
        n0 = _lib.launches()
        with torch.cuda.graph(g):
            body()
        setattr(plan, slot, (g, _lib.launches() - n0))
        g.replay()
    else:
        g, n = state
        g.replay()
        _lib.count_launch(n)


class _ConvStackFn(torch.autograd.Function):
    """out = plan(x, mod_t, mod_z); parameters are passed so that autograd routes their gradients."""

    @staticmethod
    def forward(ctx, plan, x, mod_t, mod_z, seed, *params):
        # the plan's activations live in static buffers shared by every forward at this batch size: a second
        # train-mode forward overwrites what a pending backward needs (gradient accumulation over two forwards, two
        # loss terms each calling the model).  Every forward takes a generation number; backward() of a forward
        # whose activations have since been overwritten raises instead of returning wrong gradients.
        plan._fwd_gen = getattr(plan, "_fwd_gen", 0) + 1
        ctx.gen = plan._fwd_gen
        plan.x_in.copy_(x)
        if mod_t is not None:
            plan.mod_t.copy_(mod_t)
            plan.mod_z.copy_(mod_z)
        if plan.dropout_seed is not None:
            plan.dropout_seed.fill_(int(seed))
        _replay(plan, "_g_fwd", lambda: run_ops(plan.refresh_ops() + plan.ops, plan.device))
        ctx.plan = plan
        ctx.params = params
        ctx.has_mod = mod_t is not None
        out = plan.eps_out if hasattr(plan, "eps_out") else plan.map_out
        return out.clone()

    @staticmethod
    def backward(ctx, d_out):
        plan = ctx.plan
        if ctx.gen != plan._fwd_gen:
            raise RuntimeError("infodiffusion_b200: backward of a stale forward -- the conv-stack plan keeps ONE set of "
                               "saved activations per (network, batch size) and a later training forward has "
                               "overwritten them.  Call backward() before the next forward (or run the extra forward "
                               "under torch.no_grad() / eval()).")
        finalize_backward(plan)
        plan.d_out.copy_(d_out)
        _replay(plan, "_g_bwd", lambda: run_backward(plan))
        grads = fused_param_grads(plan)            # same order as ctx.params (= plan.pindex.params)
        dmt = plan.d_mod_t.clone() if ctx.has_mod else None
        dmz = plan.d_mod_z.clone() if ctx.has_mod else None
        dx = run_input_grad(plan) if ctx.needs_input_grad[1] else None
        return (None, dx, dmt, dmz, None, *grads)


def stack_params(net) -> List[nn.Parameter]:
    """Parameters whose gradients come from the conv-stack kernels (everything spatial: convs, GroupNorms)."""
    cached = net.__dict__.get("_idf_stack_params")
    if cached is None:
        skip = ("time_embedding", "fc_a", "fc_mu", "fc_var", "temb_proj", "aemb_proj", "crossattn")
        cached = [p for n, p in net.named_parameters() if not any(s in n for s in skip)]
        net.__dict__["_idf_stack_params"] = cached
    return cached


def _train_plan(net, x: torch.Tensor, kind: str, dropout_p: float, cls, **kw):
    """The cached training plan of `net` for x's batch and device; a plan built in torch's deterministic mode is an
    ordered plan and is cached apart."""
    _require_cuda(x, "x")
    ordered = torch.are_deterministic_algorithms_enabled()
    key = (kind, x.shape[0], x.device.index, float(dropout_p), ordered)
    plans = net._plans()
    if key not in plans:
        plans[key] = cls(net, x.shape[0], x.device, dropout_p=dropout_p, ordered=ordered, **kw)
    return plans[key]


def backbone_train_forward(net, x_t: torch.Tensor, t: torch.Tensor, a: torch.Tensor, seed: int,
                           dropout_p: float) -> torch.Tensor:
    """eps = AuxiliaryUNet(x_t, t, a) with autograd through the sm_100a kernels (reference models.py:296-326)."""
    plan = _train_plan(net, x_t, "train", dropout_p, BackbonePlan, mode="train")
    # modulation rows through torch autograd (tiny GEMMs): temb -> all blocks' temb_proj, a -> fc_a -> aemb_proj
    from . import linear as L                    # fp32 Linears with autograd on the library's own kernels (no cuBLAS)
    silu = torch.nn.functional.silu
    te = net.time_embedding.timembedding
    temb = L.apply(te[3], silu(L.apply(te[1], te[0].weight[t])))
    w_t, b_t, w_z, b_z = modulation_weights(conditioned_blocks(net))
    mod_t = L.linear(silu(temb), w_t, b_t)
    if hasattr(net, "fc_a"):
        # Linear (AuxiliaryUNet) or SiLU -> Linear (BottleneckAuxUNet)
        aemb = L.apply(net.fc_a[1], silu(a)) if isinstance(net.fc_a, nn.Sequential) else L.apply(net.fc_a, a)
        mod_z = L.linear(silu(aemb), w_z, b_z)
    else:
        mod_z = torch.zeros_like(mod_t)          # UNet: no block reads it
    params = stack_params(net)
    return _ConvStackFn.apply(plan, x_t, mod_t, mod_z, seed, *params)


def encoder_train_forward(net, x: torch.Tensor, seed: int, dropout_p: float):
    """(a, a_q, mu, log_var) = Encoder(x) with autograd (reference models.py:488-518)."""
    plan = _train_plan(net, x, "train_enc", dropout_p, EncoderPlan, training=True)
    params = stack_params(net)
    fmap = _ConvStackFn.apply(plan, x, None, None, seed, *params)
    from . import linear as L
    h = torch.flatten(fmap, start_dim=1)
    a = L.apply(net.fc_a, h)
    mu = L.apply(net.fc_mu, a)
    log_var = L.apply(net.fc_var, a)
    a_q = mu + torch.randn_like(mu) * torch.exp(0.5 * log_var)
    return a, a_q, mu, log_var


def allreduce_gradients(params: Sequence[nn.Parameter], world: int) -> None:
    """Data-parallel gradient exchange: one NCCL all-reduce (average) over a flat fp32 buffer of every
    gradient that exists; parameters that never receive a gradient (dead crossattn.*, frozen table) are
    skipped exactly like the single-process optimizer skips them (SURVEY H7)."""
    import torch.distributed as dist
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch._utils._flatten_dense_tensors(grads)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat.div_(world)
    for g, f in zip(grads, torch._utils._unflatten_dense_tensors(flat, grads)):
        g.copy_(f)
