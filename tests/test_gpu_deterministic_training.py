"""Reproducible training on the B200: the ordered variants of the five order-dependent gradient reductions (split-K
weight gradient, bias gradient, AdaGN gamma / beta gradient, split-K fp32 GEMM, MMD) and whole training runs with
torch.use_deterministic_algorithms(True).

Op level: each ordered variant meets the tolerances of its default counterpart in test_gpu_ops.py, gives the same bits
on a second run (launched while another stream keeps the GPU busy) and on three CUDA-graph replays without a ticket
reset, and adds onto a prefilled output exactly as `out += result`.  Model level: three ClipAdamW steps with dropout on
and unpatched random draws, repeated on a freshly built model, give equal losses, gradients, optimizer state and
parameters, also without the side stream and without CUDA graphs."""
import contextlib
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch

from oracle import infodiff_oracle as orc
from oracle.golden_util import SEED, make_args
from tests import test_gpu_ops as ops
from tests.test_gpu_ops import lib  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = Path(__file__).resolve().parent.parent


@contextlib.contextmanager
def deterministic(on: bool = True):
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


def _ordered_and_repeatable(run, outs, accumulates=True):
    """run() launches one ordered op on the current stream into `outs` (added to them when `accumulates`).  Returns the
    result of a run on zeroed outputs after checking that it repeats bit for bit."""
    def once():
        for o in outs:
            o.zero_()
        run()
        torch.cuda.synchronize()
        return [o.clone() for o in outs]
    first = once()
    busy = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device=DEV)
    busy.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(busy):                  # other work on the GPU while the op runs
        for _ in range(12):
            a = torch.tanh(a @ a)
    for o in outs:
        o.zero_()
    run()
    torch.cuda.synchronize()
    assert all(torch.equal(o, f) for o, f in zip(outs, first)), "second run differs"
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for o in outs:
            o.zero_()
        run()
    for _ in range(3):                             # tickets come back zeroed: no reset between replays
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(o, f) for o, f in zip(outs, first)), "graph replay differs"
    base = [torch.randn(o.shape, device=DEV) for o in outs]
    for o, b in zip(outs, base):
        o.copy_(b)
    run()
    torch.cuda.synchronize()
    for o, b, f in zip(outs, base, first):
        assert torch.equal(o, b + f if accumulates else f), "prefilled output"
    return first


# ------------------------------------------------------------------------------------------------
# op level
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout,H,B", [(64, 64, 16, 3), (64, 64, 16, 8), (64, 64, 32, 4), (64, 64, 32, 8),
                                          (1024, 512, 8, 2), (768, 512, 8, 2), (768, 256, 16, 2)])
def test_ordered_weight_gradient(lib, cin, cout, H, B):
    """Split-K slabs stored to the partials buffer and added in slab order by a second launch."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import WgradDesc
    g = torch.Generator(device=DEV).manual_seed(900 + cin + cout + H + B)
    x = ops.rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    dy = ops.rbf(torch.randn(B, cout, H, H, device=DEV, generator=g))
    ref = torch.nn.grad.conv2d_weight(x.double(), (cout, cin, 3, 3), dy.double(), padding=1)
    xs, dys = ops.pf(x), ops.pf(dy)
    dw = torch.zeros(cout, 9, cin, device=DEV)
    d = WgradDesc()
    d.dy, d.rows, d.cout = dys.data_ptr(), dys.shape[0], cout
    d.x, d.x_rows, d.cin = xs.data_ptr(), xs.shape[0], cin
    d.n_taps = 9
    for t, off in enumerate(layout.tap_offsets3x3(H, H)):
        d.tap_off[t] = off
    d.dw = dw.data_ptr()
    h = C.c_void_p()
    ops.check(lib.idf_wgrad_plan_create(C.byref(d), C.byref(h)))
    n = int(lib.idf_wgrad_plan_partials_floats(h))
    lib.idf_wgrad_plan_destroy(h)
    assert n > 0 and n % (cout * 9 * cin) == 0, "expected a split-K plan"
    partials = torch.full((n,), float("nan"), device=DEV)    # every slab element is written before it is read
    d.partials = partials.data_ptr()
    ops.check(lib.idf_wgrad_plan_create(C.byref(d), C.byref(h)))
    try:
        (got,) = _ordered_and_repeatable(lambda: ops.check(lib.idf_wgrad_run(h, ops.stream())), [dw])
    finally:
        lib.idf_wgrad_plan_destroy(h)
    print(f"\n[ordered] wgrad {cin}->{cout}@{H} B={B}: {n // (cout * 9 * cin)} slabs")
    ops.assert_close(got.reshape(cout, 3, 3, cin).permute(0, 3, 1, 2), ref, rel_l2=1e-4, max_rel=1e-3,
                     what=f"ordered wgrad {cin}->{cout}@{H}")


@pytest.mark.parametrize("rows,Cc", [(1, 64), (4225 * 3, 64), (1089 * 5, 128), (289 * 2, 384), (77, 8),
                                     (81 * 32, 768), (289 * 8, 1024)])
def test_ordered_colsum(lib, rows, Cc):
    g = torch.Generator(device=DEV).manual_seed(rows + Cc + 1)
    m = torch.randn(rows, Cc, device=DEV, generator=g).to(ops.BF)
    out = torch.zeros(Cc, device=DEV)
    ws = torch.empty(int(lib.idf_colsum_ws_floats(rows, Cc)), device=DEV)
    tickets = torch.zeros(1, dtype=torch.int32, device=DEV)
    (got,) = _ordered_and_repeatable(lambda: ops.check(lib.idf_colsum_bf16_ordered(
        m.data_ptr(), out.data_ptr(), rows, Cc, ws.data_ptr(), tickets.data_ptr(), ops.stream())), [out])
    ops.assert_close(got, m.double().sum(0), rel_l2=1e-5, max_rel=1e-4, what="ordered colsum")
    assert int(tickets.item()) == 0


@pytest.mark.parametrize("B", [2, 33, 80])
@pytest.mark.parametrize("c0,c1", [(128, 128), (512, 256)])
def test_ordered_adagn_param_gradients(lib, B, c0, c1):
    """dgamma / dbeta summed over the batch in sample order; dx, the (S1, S2) sums and the modulation-gradient rows are
    bitwise those of the default path."""
    from infodiffusion_b200._lib import AdaGNArgs, AdaGNBwdArgs
    from infodiffusion_b200.train import adagn_param_grads
    H = 8
    Cc = c0 + c1
    g = torch.Generator(device=DEV).manual_seed(40 + B + Cc)
    x0 = ops.rbf(torch.randn(B, c0, H, H, device=DEV, generator=g) * 1.5 + 0.3)
    x1 = ops.rbf(torch.randn(B, c1, H, H, device=DEV, generator=g) * 0.7 - 0.2)
    gamma = 1 + 0.1 * torch.randn(Cc, device=DEV, generator=g)
    beta = 0.1 * torch.randn(Cc, device=DEV, generator=g)
    st, bt, sz, bz = (0.3 * torch.randn(B, Cc, device=DEV, generator=g) for _ in range(4))
    mt, mz = torch.cat([st, bt], 1).contiguous(), torch.cat([sz, bz], 1).contiguous()
    s0, s1 = ops.pf(x0), ops.pf(x1)
    st0, st1 = ops.tile_partials(s0, B, H, H), ops.tile_partials(s1, B, H, H)
    seed = torch.tensor([0x5eed], dtype=torch.int64, device=DEV)
    dys = ops.pf(ops.rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g)))
    a = AdaGNArgs()
    a.src0, a.c0, a.src1, a.c1 = s0.data_ptr(), c0, s1.data_ptr(), c1
    a.batch, a.H, a.W = B, H, H
    a.gamma, a.beta, a.eps = gamma.data_ptr(), beta.data_ptr(), 1e-5
    a.mod_t, a.mod_t_step_stride, a.mod_t_batch_stride = mt.data_ptr(), 0, 2 * Cc
    a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = mz.data_ptr(), 0, 2 * Cc
    a.apply_silu = 1
    a.stats0, a.stats1 = st0.data_ptr(), st1.data_ptr()
    a.dropout_p, a.dropout_seed, a.dropout_layer = 0.1, seed.data_ptr(), 3

    def launch(ordered):
        o = dict(dx0=torch.zeros_like(s0), dx1=torch.zeros_like(s1), sums=torch.zeros(B, Cc, 2, device=DEV),
                 dmt=torch.zeros(B, 2 * Cc, device=DEV), dmz=torch.zeros(B, 2 * Cc, device=DEV),
                 dgam=torch.zeros(Cc, device=DEV), dbet=torch.zeros(Cc, device=DEV))
        ws = torch.zeros(int(lib.idf_adagn_bwd_ws_floats(B, Cc)), device=DEV)
        b = AdaGNBwdArgs()
        b.f = a
        b.dy, b.dx0, b.dx1, b.sums, b.ws = dys.data_ptr(), o["dx0"].data_ptr(), o["dx1"].data_ptr(), o["sums"].data_ptr(), ws.data_ptr()
        b.d_mod_t, b.d_mod_z = o["dmt"].data_ptr(), o["dmz"].data_ptr()
        b.dgamma, b.dbeta = o["dgam"].data_ptr(), o["dbet"].data_ptr()
        keep = [ws]
        if ordered:
            pws = torch.full((B * Cc * 2,), float("nan"), device=DEV)
            ticket = torch.zeros(1, dtype=torch.int32, device=DEV)
            b.dparam_ws, b.dparam_ticket = pws.data_ptr(), ticket.data_ptr()
            keep += [pws, ticket]
        return o, b, keep

    ref, bref, _k0 = launch(False)
    ops.check(lib.idf_adagn_silu_bwd(C.byref(bref), ops.stream()))
    got, bgot, _k1 = launch(True)
    dgam, dbet = _ordered_and_repeatable(lambda: ops.check(lib.idf_adagn_silu_bwd(C.byref(bgot), ops.stream())),
                                         [got["dgam"], got["dbet"]])
    for k in ("dx0", "dx1", "sums", "dmt", "dmz"):
        assert torch.equal(got[k], ref[k]), f"{k} differs from the default path"
    want = adagn_param_grads(ref["sums"].double(), gamma.double(), beta.double(), st.double(), bt.double(), sz.double(),
                             bz.double())
    ops.assert_close(dgam, want["gamma"], rel_l2=2e-3, max_rel=1e-2, what="ordered d gamma")
    ops.assert_close(dbet, want["beta"], rel_l2=2e-3, max_rel=1e-2, what="ordered d beta")
    ops.assert_close(dgam, ref["dgam"], rel_l2=1e-5, max_rel=1e-4, what="ordered vs atomic d gamma")


@pytest.mark.parametrize("M,K,N", [(5, 4096, 32), (32, 4992, 256), (64, 1280, 1024)])
def test_ordered_gemm_f32_split_k(lib, M, K, N):
    """C (+)= A . B^T with the split-K partial tiles summed in split order (fc_a forward, a [B, 4992] x [4992, 256] data
    gradient, a LatentUNet layer)."""
    g = torch.Generator(device=DEV).manual_seed(M + K + N)
    A = torch.randn(M, K, device=DEV, generator=g)
    Bm = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5
    Cm = torch.zeros(M, N, device=DEV)
    n = int(lib.idf_gemm_f32_ws_floats(M, N, K))
    assert n > 0, "expected a split-K shape"
    ws = torch.empty(n, device=DEV)
    tickets = torch.zeros(64, dtype=torch.int32, device=DEV)

    def run(acc=1):
        ops.check(lib.idf_gemm_f32_ordered(A.data_ptr(), K, 0, Bm.data_ptr(), K, 1, Cm.data_ptr(), N, M, N, K, acc,
                                           ws.data_ptr(), tickets.data_ptr(), ops.stream()))
    (got,) = _ordered_and_repeatable(run, [Cm])
    ops.assert_close(got, A.double() @ Bm.double().t(), rel_l2=3e-6, max_rel=1e-4, what="ordered split-K gemm")
    Cm.fill_(7.0)                                  # accumulate = 0 overwrites
    run(acc=0)
    torch.cuda.synchronize()
    assert torch.equal(Cm, got)
    assert int(tickets.abs().sum()) == 0


@pytest.mark.parametrize("B", [32, 256])
@pytest.mark.parametrize("D", [32, 256])
def test_ordered_mmd(lib, B, D):
    gen = torch.Generator().manual_seed(11 + D + B)
    xs = torch.randn(B, D, generator=gen)
    ys = torch.randn(B, D, generator=gen) * 0.7 + 0.2
    yo = ys.clone().requires_grad_(True)
    vo = orc.compute_mmd(xs, yo)
    (go,) = torch.autograd.grad(vo, yo)
    x, y = xs.to(DEV), ys.to(DEV)
    loss, grad = torch.zeros((), device=DEV), torch.zeros(B, D, device=DEV)
    ws = torch.empty(int(lib.idf_mmd_ws_floats(B)), device=DEV)
    tickets = torch.zeros(1, dtype=torch.int32, device=DEV)
    v, gg = _ordered_and_repeatable(lambda: ops.check(lib.idf_mmd_fwd_bwd_ordered(
        x.data_ptr(), y.data_ptr(), loss.data_ptr(), grad.data_ptr(), B, D, ws.data_ptr(), tickets.data_ptr(),
        ops.stream())), [loss, grad], accumulates=False)
    assert abs(float(v) - float(vo)) < 5e-6, f"mmd value B={B} D={D}: {float(v)} vs {float(vo)}"
    ops.assert_close(gg.cpu(), go, rel_l2=1e-4, max_rel=1e-3, what=f"ordered mmd grad B={B} D={D}")


# ------------------------------------------------------------------------------------------------
# model level
# ------------------------------------------------------------------------------------------------
def _infodiff(**kw):
    from infodiffusion_b200.models import InfoDiff
    args = make_args(a_dim=32, diffusion_steps=1000, **kw)
    return args, InfoDiff(args, DEV, (3, 64, 64)), lambda g, B: torch.rand(B, 3, 64, 64, generator=g) * 2 - 1


def _vanilla32():
    from infodiffusion_b200.models import Diff
    args = make_args(a_dim=32, diffusion_steps=1000, model="vanilla", input_size=32, mmd_weight=0.0)
    return args, Diff(args, DEV, (3, 32, 32)), lambda g, B: torch.rand(B, 3, 32, 32, generator=g) * 2 - 1


def _latent():
    from infodiffusion_b200.models import Diff
    args = make_args(a_dim=256, diffusion_steps=1000, model="vanilla", is_latent=True, mode="train_latent_ddim",
                     mmd_weight=0.0)
    return args, Diff(args, DEV, (1, 256, 256)), lambda g, B: torch.randn(B, 256, generator=g)


MODELS = {
    "infodiff_mmd": lambda: _infodiff(),
    "infodiff_kld_C_bottleneck": lambda: _infodiff(kld_weight=1e-3, use_C=True, is_bottleneck=True),
    "vanilla_32": _vanilla32,
    "latent": _latent,
}


def _train_run(name, steps=3, B=4):
    """Build the model from the seed and take `steps` ClipAdamW steps (dropout on, torch's own random draws); returns
    everything a step leaves behind."""
    from infodiffusion_b200.optim import ClipAdamW
    torch.manual_seed(SEED)
    torch.cuda.manual_seed_all(SEED)
    args, model, data = MODELS[name]()
    g = torch.Generator().manual_seed(5)
    xs = [data(g, B).to(DEV) for _ in range(steps)]
    params = [p for p in model.parameters() if p.requires_grad]
    opt = ClipAdamW(params, lr=1e-4, weight_decay=1e-5, max_norm=1.0)
    model.train()
    losses, grads = [], []
    try:
        for s in range(steps):
            loss = model.loss_fn(args, xs[s], curr_epoch=s)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            losses.append(loss.detach().clone())
            grads.append([None if p.grad is None else p.grad.clone() for p in params])
            opt.step()
    finally:
        model.eval()
    torch.cuda.synchronize()
    state = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in opt.state[p].items()} for p in params]
    return dict(losses=losses, grads=grads, state=state, params=[p.detach().clone() for p in params])


def _assert_same(r0, r1, what):
    assert all(torch.equal(a, b) for a, b in zip(r0["losses"], r1["losses"])), f"{what}: losses differ"
    for s, (g0, g1) in enumerate(zip(r0["grads"], r1["grads"])):
        for i, (a, b) in enumerate(zip(g0, g1)):
            assert (a is None) == (b is None) and (a is None or torch.equal(a, b)), f"{what}: step {s} gradient {i} differs"
    for a, b in zip(r0["state"], r1["state"]):
        assert a.keys() == b.keys()
        for k in a:
            assert torch.equal(a[k], b[k]) if torch.is_tensor(a[k]) else a[k] == b[k], f"{what}: optimizer state {k}"
    assert all(torch.equal(a, b) for a, b in zip(r0["params"], r1["params"])), f"{what}: parameters differ"


@pytest.mark.parametrize("name", list(MODELS))
def test_training_is_bitwise_reproducible(name):
    from infodiffusion_b200 import train as T
    with deterministic():
        ref = _train_run(name)
        assert all(torch.isfinite(v) for v in ref["losses"])
        _assert_same(ref, _train_run(name), "fresh model")
        side, graphs = T.SIDE_STREAM, T.USE_GRAPHS
        try:
            T.SIDE_STREAM = False
            _assert_same(ref, _train_run(name), "SIDE_STREAM = False")
            T.SIDE_STREAM, T.USE_GRAPHS = side, False
            _assert_same(ref, _train_run(name), "USE_GRAPHS = False")
        finally:
            T.SIDE_STREAM, T.USE_GRAPHS = side, graphs
    print(f"\n[deterministic] {name}: losses {[round(float(v), 6) for v in ref['losses']]}")


def test_deterministic_gradients_match_oracle_autograd():
    """The ordered reductions keep the InfoDiff gradients within the bounds of the default path against the oracle."""
    from tests.test_gpu_network import build, test_training_step_gradients_match_oracle_autograd
    with deterministic():
        test_training_step_gradients_match_oracle_autograd(build(32, 1000))


def test_default_then_deterministic_step_on_one_model():
    """The flag is read when a training plan is built and is part of its key: a model can switch between steps."""
    from infodiffusion_b200.optim import ClipAdamW
    torch.manual_seed(SEED)
    args, model, data = _infodiff()
    opt = ClipAdamW([p for p in model.parameters() if p.requires_grad], lr=1e-4, weight_decay=1e-5, max_norm=1.0)
    x = data(torch.Generator().manual_seed(9), 4).to(DEV)
    model.train()
    try:
        for on in (False, True):
            with deterministic(on):
                loss = model.loss_fn(args, x)
                opt.zero_grad(set_to_none=True)
                loss.backward()
                opt.step()
            assert torch.isfinite(loss)
    finally:
        model.eval()
    keys = [k for k in model.backbone._plans() if k[0] == "train"]
    assert sorted(k[-1] for k in keys) == [False, True], keys


def test_run_py_deterministic_training_checkpoints_are_equal(tmp_path):
    common = ["--model", "diff", "--mode", "train", "--prior", "regular", "--dataset", "synthetic", "--a_dim", "32",
              "--batch_size", "4", "--epochs", "2", "--save_epochs", "2", "--diffusion_steps", "4", "--synthetic_size", "8",
              "--model_folder", "./models", "--deterministic_training"]
    sds = []
    for run in ("a", "b"):
        cwd = tmp_path / run
        cwd.mkdir()
        r = subprocess.run([sys.executable, str(ROOT / "run.py"), *common], cwd=cwd, capture_output=True, text=True,
                           timeout=900, env={**os.environ, "PYTHONPATH": str(ROOT)})
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        (ckpt,) = (cwd / "models").rglob("model-2.pth")
        sds.append(torch.load(ckpt, map_location="cpu"))
    assert sds[0].keys() == sds[1].keys()
    for k in sds[0]:
        assert torch.equal(sds[0][k], sds[1][k]), k
