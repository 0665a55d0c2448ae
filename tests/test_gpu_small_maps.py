"""Small maps (4x4 .. 32x32, one 64x64 case) and large batches, compared per image on the B200.

The 32x32 configurations (cifar10's InfoDiff, ch_mult [1, 2, 2, 2], and the vanilla Diff at 32x32) run GroupNorm at
4x4, where an image has R = 25 pad-flat rows and a 32-row statistics window of the conv epilogue can hold rows of
three images.  These tests follow the GroupNorm records from a real producer conv through every consumer (streaming
AdaGN, coefficient kernel, backward, fused-transform conv) and check each image against fp64 torch on the conv's
stored bf16 output, at batches that cover every phase of a 25-row image against a 32-row window (lcm(25, 32) = 800
rows = 32 images).  One norm over a whole batch would hide one wrong image among many: every bound here is per image.

Also: the backward kernels at the small shapes (weight gradient at 4x4, the stride-2 weight / data gradients through
the space-to-depth phases, small-map attention backward) and the 32x32 networks at batches >= 6."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import infodiff_oracle as orc
from oracle.golden_util import SEED, make_args, perturb_state_dict
from tests import test_gpu_ops as ops
from tests.test_gpu_network import _patched_draws
from tests.test_gpu_ops import BF, DEV, check, lib, pad_is_zero, pf, rbf, run_conv, stream, unpf  # noqa: F401

pytestmark = pytest.mark.gpu

IDF_ERR_ARG, IDF_ERR_CUDA = -1, -2

# (rel-L2, max-rel) per image, about 1.2 x the worst values measured on a B200 (1000 W power limit) over every case
# below: the outputs that pass through bf16 (AdaGN y, dx: 1.9e-3 / 3.6e-3) and the fp32 closed forms ((A, B): 1.8e-7 /
# 4.2e-7; (S1, S2) and the modulation rows: 2.1e-7 / 3.7e-7)
TOL_Y = (2.3e-3, 4.5e-3)
TOL_COEF = (2.2e-7, 5.1e-7)
TOL_SUMS = (2.6e-7, 4.5e-7)


def _last_error(lib):
    return lib.idf_last_error().decode()


def assert_per_image(got, ref, rel_l2, max_rel, what):
    """rel-L2 and max-rel (relative to the image's largest |ref|) of every image (leading dimension) on its own."""
    g, r = got.double().reshape(got.shape[0], -1), ref.double().reshape(ref.shape[0], -1)
    assert torch.isfinite(g).all(), f"{what}: non-finite output"
    err = ((g - r).norm(dim=1) / r.norm(dim=1).clamp_min(1e-30)).cpu()
    mx = ((g - r).abs().amax(dim=1) / r.abs().amax(dim=1).clamp_min(1e-30)).cpu()
    ie, im = int(err.argmax()), int(mx.argmax())
    print(f"[small-maps] {what}: worst rel-L2 {float(err[ie]):.2e} (image {ie}), worst max-rel {float(mx[im]):.2e} (image {im})")
    assert float(err[ie]) < rel_l2 and float(mx[im]) < max_rel, (
        f"{what}: image {ie} rel-L2 {float(err[ie]):.3e} (tol {rel_l2}), image {im} max-rel {float(mx[im]):.3e} (tol {max_rel})")


# ------------------------------------------------------------------------------------------------
# producer convs with GroupNorm records
# ------------------------------------------------------------------------------------------------
def _producer(lib, g, B, H, cout, cin=64, up2=False):
    """A 3x3 conv (or nearest-x2 + 3x3 folded into one, `up2`) over a random input whose images differ in mean and
    spread, so that statistics taken from the wrong image show.  Returns the pad-flat bf16 output, its records, and
    the record geometry for idf_adagn_args (unit, planes, producer rows per image)."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import ConvDesc
    n = torch.arange(B, device=DEV, dtype=torch.float32)[:, None, None, None]
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g) * (0.6 + 0.15 * (n % 5)) + 0.4 * (n % 7) - 1.0)
    w = torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5
    bias = torch.randn(cout, device=DEV, generator=g) * 0.3
    Ho = 2 * H if up2 else H
    rows_in = B * (H + 1) * (H + 1)
    out = torch.zeros(B * (Ho + 1) * (Ho + 1), cout, device=DEV, dtype=BF)
    tiles_in = (rows_in + 127) // 128
    stats = torch.full((2 * tiles_in * 4 * (4 if up2 else 1) * cout * 2,), float("nan"), device=DEV)
    xs = pf(x)
    kb = layout.taps_up2(cin, H, H) if up2 else layout.taps3x3(cin, H, H)
    wp = (layout.pack_conv3x3_up2(w) if up2 else layout.pack_conv3x3(w)).to(BF).contiguous()
    bias_p = bias.repeat(4).contiguous() if up2 else bias
    d = ConvDesc()
    d.n_src = 1
    d.src[0], d.src_rows[0], d.src_ld[0] = xs.data_ptr(), xs.shape[0], cin
    d.num_kb = len(kb)
    for k, (si, c0, off) in enumerate(kb):
        d.kb_src[k], d.kb_c0[k], d.kb_rowoff[k] = si, c0, off
    d.weight, d.cout_pad, d.cout, d.bias = wp.data_ptr(), wp.shape[0], cout, bias_p.data_ptr()
    d.block_n = cout if up2 else (128 if cout % 128 == 0 else 64)
    d.batch, d.H, d.W, d.epilogue, d.up2 = B, H, H, 0, 1 if up2 else 0
    d.out, d.out_ld, d.stats_out = out.data_ptr(), cout, stats.data_ptr()
    h = C.c_void_p()
    check(lib.idf_conv_plan_create(C.byref(d), C.byref(h)))
    check(lib.idf_conv_run(h, stream()))
    torch.cuda.synchronize()
    unit = int(lib.idf_conv_plan_stats_unit(h))
    lib.idf_conv_plan_destroy(h)
    assert pad_is_zero(out, B, Ho, Ho)
    return out, stats, (unit, 4 if up2 else 0, rows_in // B if up2 else 0)


def _reference(xin, gamma, beta, st, bt, sz, bz, silu):
    """fp64 AdaGN of the reference (GroupNorm(32) + affine, timestep and latent scale / shift, SiLU) under autograd,
    and the closed-form coefficients (A, B) with v = A*x + B."""
    B, Cc = xin.shape[:2]
    v = F.group_norm(xin, 32, gamma, beta, 1e-5)
    v = v * (1 + st)[:, :, None, None] + bt[:, :, None, None]
    v = v * (1 + sz)[:, :, None, None] + bz[:, :, None, None]
    y = F.silu(v) if silu else v
    xg = xin.detach().reshape(B, 32, -1)
    mean, var = xg.mean(-1), xg.var(-1, unbiased=False)
    rstd = (var + 1e-5).rsqrt().repeat_interleave(Cc // 32, dim=1)
    mean = mean.repeat_interleave(Cc // 32, dim=1)
    gm, bm = gamma.detach()[None], beta.detach()[None]
    s1, s2 = 1 + st.detach(), 1 + sz.detach()
    A = rstd * gm * s1 * s2
    Bc = ((bm - mean * rstd * gm) * s1 + bt.detach()) * s2 + bz.detach()
    return v, y, A, Bc


def _record_chain(lib, H, B, srcs, seed, fused_conv=True, bwd_records=True):
    """srcs: [(pad-flat bf16 map, records, (unit, planes, producer rows))] of one or two producer convs (concatenated
    along C).  Checks, per image: streaming AdaGN forward, idf_adagn_coef, the backward with save_coef and from the
    records (dx, (S1, S2), the fused modulation rows), and the fused-transform conv against AdaGN-then-conv."""
    from infodiffusion_b200._lib import IDF_CONV_MAX_KB, AdaGNArgs, AdaGNBwdArgs
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(seed)
    cs = [s[0].shape[1] for s in srcs]
    Cc = sum(cs)
    rows = B * (H + 1) * (H + 1)
    xin = torch.cat([unpf(s[0], B, H, H) for s in srcs], 1).double().requires_grad_(True)
    gamma = (1 + 0.1 * torch.randn(Cc, device=DEV, generator=g)).double().requires_grad_(True)
    beta = (0.1 * torch.randn(Cc, device=DEV, generator=g)).double().requires_grad_(True)
    st, bt, sz, bz = ((0.3 * torch.randn(B, Cc, device=DEV, generator=g)).double().requires_grad_(True) for _ in range(4))
    v, y, A, Bc = _reference(xin, gamma, beta, st, bt, sz, bz, True)

    a = AdaGNArgs()
    a.src0, a.c0 = srcs[0][0].data_ptr(), cs[0]
    a.stats0 = srcs[0][1].data_ptr()
    a.stats_unit0, a.stats_planes0, a.stats_rows0 = srcs[0][2]
    if len(srcs) > 1:
        a.src1, a.c1 = srcs[1][0].data_ptr(), cs[1]
        a.stats1 = srcs[1][1].data_ptr()
        a.stats_unit1, a.stats_planes1, a.stats_rows1 = srcs[1][2]
    out = torch.zeros(rows, Cc, device=DEV, dtype=BF)
    a.out, a.batch, a.H, a.W = out.data_ptr(), B, H, H
    gam_d, bet_d = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
    a.gamma, a.beta, a.eps = gam_d.data_ptr(), bet_d.data_ptr(), 1e-5
    mt = torch.cat([st, bt], 1).detach().float().contiguous()       # per-sample rows (scale | shift)
    mz = torch.cat([sz, bz], 1).detach().float().contiguous()
    a.mod_t, a.mod_t_step_stride, a.mod_t_batch_stride = mt.data_ptr(), 0, 2 * Cc
    a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = mz.data_ptr(), 0, 2 * Cc
    a.apply_silu = 1
    what = f"H={H} B={B} C={'+'.join(map(str, cs))} unit={srcs[0][2][0]}{' up2' if srcs[0][2][1] else ''}"

    # streaming forward (inference form) and the coefficient kernel
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    coef = torch.full((B, Cc, 2), float("nan"), device=DEV)
    check(lib.idf_adagn_coef(C.byref(a), coef.data_ptr(), stream()))
    torch.cuda.synchronize()
    assert pad_is_zero(out, B, H, H)
    assert_per_image(unpf(out, B, H, H), y.detach(), *TOL_Y, f"AdaGN forward {what}")
    assert_per_image(coef[..., 0], A, *TOL_COEF, f"AdaGN coef A {what}")
    assert_per_image(coef[..., 1], Bc, *TOL_COEF, f"AdaGN coef B {what}")

    if fused_conv:      # the consumer conv with the AdaGN folded into its A operand == AdaGN, then the conv
        cout = 64
        w = rbf(torch.randn(cout, Cc, 3, 3, device=DEV, generator=g) * (2.0 / (9 * Cc)) ** 0.5)
        wp = layout.pack_conv3x3(w).to(BF).contiguous()
        bias = torch.randn(cout, device=DEV, generator=g)
        offs = layout.tap_offsets3x3(H, H)
        kb_ref = [(0, c, off) for off in offs for c in range(0, Cc, 64)]
        kb, kx = [], []
        for off in offs:
            base = 0
            for si, c_ in enumerate(cs):
                for c in range(0, c_, 64):
                    kb.append((si, c, off)); kx.append(base + c)
                base += c_
        kbx = (C.c_int32 * IDF_CONV_MAX_KB)(*(kx + [0] * (IDF_CONV_MAX_KB - len(kx))))
        ref = run_conv(lib, [out], kb_ref, wp, bias, B, H, cout, 64)
        got = run_conv(lib, [s[0] for s in srcs], kb, wp, bias, B, H, cout, 64, xf_coef=coef, xf_ctot=Cc, xf_silu=1,
                       kb_xf=kbx)
        assert torch.equal(got, ref), f"fused-transform conv != AdaGN then conv ({what}): max diff " \
                                      f"{float((got.float() - ref.float()).abs().max())}"

    # backward: training forward with save_coef, then the backward from the saved coefficients and from the records
    dy = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    y.backward(dy.double())
    xhat = F.group_norm(xin.detach(), 32, eps=1e-5)
    sv = torch.sigmoid(v.detach())
    dv = dy.double() * sv * (1 + v.detach() * (1 - sv))
    sums_ref = torch.stack([dv.sum((2, 3)), (dv * xhat).sum((2, 3))], -1)
    save = torch.zeros(B, Cc, 4, device=DEV)
    out_t = torch.zeros_like(out)
    a.save_coef, a.out = save.data_ptr(), out_t.data_ptr()
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    torch.cuda.synchronize()
    assert_per_image(unpf(out_t, B, H, H), y.detach(), *TOL_Y, f"AdaGN training forward {what}")
    assert_per_image(save[..., 0], A, *TOL_COEF, f"saved A {what}")
    assert_per_image(save[..., 1], Bc, *TOL_COEF, f"saved B {what}")
    dys = pf(dy)
    modes = ["save_coef"] + (["records"] if bwd_records else [])
    for mode in modes:
        a.save_coef = save.data_ptr() if mode == "save_coef" else None
        b = AdaGNBwdArgs()
        b.f = a
        dxs = [torch.zeros(rows, c_, device=DEV, dtype=BF) for c_ in cs]
        sums = torch.zeros(B, Cc, 2, device=DEV)
        ws = torch.zeros(lib.idf_adagn_bwd_ws_floats(B, Cc), device=DEV)
        b.dy, b.dx0, b.sums, b.ws = dys.data_ptr(), dxs[0].data_ptr(), sums.data_ptr(), ws.data_ptr()
        if len(cs) > 1:
            b.dx1 = dxs[1].data_ptr()
        dgam, dbet = torch.zeros(Cc, device=DEV), torch.zeros(Cc, device=DEV)
        dmt, dmz = torch.zeros(B, 2 * Cc, device=DEV), torch.zeros(B, 2 * Cc, device=DEV)
        b.dgamma, b.dbeta, b.d_mod_t, b.d_mod_z = dgam.data_ptr(), dbet.data_ptr(), dmt.data_ptr(), dmz.data_ptr()
        check(lib.idf_adagn_silu_bwd(C.byref(b), stream()))
        torch.cuda.synchronize()
        dx = torch.cat([unpf(t, B, H, H) for t in dxs], 1)
        assert_per_image(dx, xin.grad, *TOL_Y, f"AdaGN dx ({mode}) {what}")
        assert_per_image(sums[..., 0], sums_ref[..., 0], *TOL_SUMS, f"AdaGN S1 ({mode}) {what}")
        assert_per_image(sums[..., 1], sums_ref[..., 1], *TOL_SUMS, f"AdaGN S2 ({mode}) {what}")
        assert_per_image(torch.cat([dmt, dmz], 1), torch.cat([st.grad, bt.grad, sz.grad, bz.grad], 1), *TOL_SUMS,
                         f"AdaGN d_mod rows ({mode}) {what}")
        ops.assert_close(dgam, gamma.grad, rel_l2=2e-3, max_rel=1e-2, what=f"fused d gamma ({mode}) {what}")
        ops.assert_close(dbet, beta.grad, rel_l2=2e-3, max_rel=1e-2, what=f"fused d beta ({mode}) {what}")
    a.save_coef = None


@pytest.mark.parametrize("H,B,C", [(4, 1, 128), (4, 5, 128), (4, 6, 128), (4, 7, 128), (4, 13, 128), (4, 33, 128),
                                   (4, 6, 1024), (8, 33, 128), (16, 13, 128), (32, 6, 128), (64, 2, 128)])
def test_groupnorm_record_chain(lib, H, B, C):
    """conv (stats_out) -> AdaGN forward / coefficients / backward / fused-transform conv, per image.  C = 1024 is the
    vanilla 32x32 model's deepest level.  Above 8x8 the producer writes work-item records, which the backward does not
    read (training saves the coefficients): there the record path of the backward must be refused."""
    g = torch.Generator(device=DEV).manual_seed(1000 + 7 * H + B + C)
    src = _producer(lib, g, B, H, C)
    unit = src[2][0]
    _record_chain(lib, H, B, [src], 2000 + H + B + C, bwd_records=unit == 32)
    if unit != 32:
        _backward_refuses_records(lib, src, B, H)


def _backward_refuses_records(lib, src, B, H):
    from infodiffusion_b200._lib import AdaGNArgs, AdaGNBwdArgs
    Cc = src[0].shape[1]
    rows = B * (H + 1) * (H + 1)
    ones, zeros = torch.ones(Cc, device=DEV), torch.zeros(Cc, device=DEV)
    b = AdaGNBwdArgs()
    b.f = AdaGNArgs()
    b.f.src0, b.f.c0, b.f.batch, b.f.H, b.f.W = src[0].data_ptr(), Cc, B, H, H
    b.f.gamma, b.f.beta, b.f.eps, b.f.apply_silu = ones.data_ptr(), zeros.data_ptr(), 1e-5, 1
    b.f.stats0 = src[1].data_ptr()
    b.f.stats_unit0, b.f.stats_planes0, b.f.stats_rows0 = src[2]
    dx = torch.full((rows, Cc), 5.0, device=DEV, dtype=BF)
    sums = torch.zeros(B, Cc, 2, device=DEV)
    ws = torch.zeros(lib.idf_adagn_bwd_ws_floats(B, Cc), device=DEV)
    b.dy, b.dx0, b.sums, b.ws = src[0].data_ptr(), dx.data_ptr(), sums.data_ptr(), ws.data_ptr()
    rc = lib.idf_adagn_silu_bwd(C.byref(b), stream())
    torch.cuda.synchronize()
    assert rc == IDF_ERR_ARG, f"backward from records of unit {src[2][0]} / planes {src[2][1]}: status {rc}"
    assert "save_coef" in _last_error(lib)
    assert bool((dx == 5.0).all())


@pytest.mark.parametrize("B", [6, 33])
def test_groupnorm_record_chain_concat_of_two_producers(lib, B):
    """torch.cat([h, skip]) then GroupNorm at 4x4 (the up path's first block): the two sources come from two different
    producer convs, each with its own records."""
    g = torch.Generator(device=DEV).manual_seed(3000 + B)
    s0 = _producer(lib, g, B, 4, 128)
    s1 = _producer(lib, g, B, 4, 64, cin=128)
    _record_chain(lib, 4, B, [s0, s1], 3100 + B)


@pytest.mark.parametrize("B", [6, 33])
def test_groupnorm_records_of_up2_conv_feed_8x8_adagn(lib, B):
    """cifar InfoDiff's 4 -> 8 upsample folded into the next conv (up2, cout 128): its records cover the 4x4 input grid
    (25 rows per image, 4 parity planes) and feed the 8x8 AdaGN (stats_planes / stats_rows).  The backward takes only
    records of its own map: from these it must refuse."""
    g = torch.Generator(device=DEV).manual_seed(4000 + B)
    src = _producer(lib, g, B, 4, 128, cin=128, up2=True)
    assert src[2] == (32, 4, 25)
    _record_chain(lib, 8, B, [src], 4100 + B, bwd_records=False)
    _backward_refuses_records(lib, src, B, 8)


@pytest.mark.parametrize("H", [1, 2, 3])
def test_groupnorm_records_refused_where_they_cannot_separate_images(lib, H):
    """At H = W <= 3 a 32-row window can hold rows of three images that are not pad rows: no two records per window
    keep them apart.  idf_conv_plan_create with stats_out and AdaGN calls with records return IDF_ERR_ARG and say
    why; the engine takes no records there (the AdaGN computes the statistics itself)."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import AdaGNArgs, ConvDesc
    assert not layout.window_records_exact(H, H) and layout.window_records_exact(4, 4)
    B, cin, cout = 8, 64, 64
    rows = B * (H + 1) * (H + 1)
    xs = torch.zeros(rows, cin, device=DEV, dtype=BF)
    wp = torch.zeros(cout, 9 * cin, device=DEV, dtype=BF)
    bias = torch.zeros(cout, device=DEV)
    out = torch.zeros(rows, cout, device=DEV, dtype=BF)
    stats = torch.zeros(2 * ((rows + 127) // 128) * 4 * cout * 2, device=DEV)
    d = ConvDesc()
    d.n_src = 1
    d.src[0], d.src_rows[0], d.src_ld[0] = xs.data_ptr(), rows, cin
    kb = layout.taps3x3(cin, H, H)
    d.num_kb = len(kb)
    for k, (si, c0, off) in enumerate(kb):
        d.kb_src[k], d.kb_c0[k], d.kb_rowoff[k] = si, c0, off
    d.weight, d.cout_pad, d.block_n, d.cout, d.bias = wp.data_ptr(), cout, 64, cout, bias.data_ptr()
    d.batch, d.H, d.W, d.epilogue = B, H, H, 0
    d.out, d.out_ld, d.stats_out = out.data_ptr(), cout, stats.data_ptr()
    h = C.c_void_p()
    assert lib.idf_conv_plan_create(C.byref(d), C.byref(h)) == IDF_ERR_ARG
    assert "stats_out" in _last_error(lib) and f"{H}x{H}" in _last_error(lib)
    d.stats_out = None
    check(lib.idf_conv_plan_create(C.byref(d), C.byref(h)))
    lib.idf_conv_plan_destroy(h)
    a = AdaGNArgs()
    ones = torch.ones(cout, device=DEV)
    a.src0, a.c0, a.out, a.batch, a.H, a.W = xs.data_ptr(), cout, out.data_ptr(), B, H, H
    a.gamma, a.beta, a.eps, a.stats0 = ones.data_ptr(), bias.data_ptr(), 1e-5, stats.data_ptr()
    coef = torch.zeros(B, cout, 2, device=DEV)
    for rc in (lib.idf_adagn_silu_fwd(C.byref(a), stream()), lib.idf_adagn_coef(C.byref(a), coef.data_ptr(), stream())):
        assert rc == IDF_ERR_ARG and "stats0" in _last_error(lib), (rc, _last_error(lib))


# ------------------------------------------------------------------------------------------------
# backward kernels at the small shapes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout", [(128, 128), (512, 256)])
def test_weight_gradient_4x4_many_images(lib, cin, cout):
    """3x3 weight gradient at 4x4 (tap clusters {-6,-5,-4}, {-1,0,1}, {4,5,6}) over 33 images."""
    ops.test_conv_weight_gradient(lib, cin, cout, 4, 33)


@pytest.mark.parametrize("Cc,H,B", [(128, 8, 33), (64, 64, 3)])
def test_stride2_weight_and_data_gradients(lib, Cc, H, B):
    """Backward of the stride-2 conv as training runs it: the weight gradient over the space-to-depth phase planes with
    the taps_stride2 offsets (8 -> 4: one tap cluster with rel = 5), and the per-phase data gradients of
    layout.stride2_phase_dgrad put back by idf_depth_to_space, against torch.nn.grad in fp64, per image (data gradient:
    worst measured on a B200 1.7e-3 / 2.7e-3)."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import WgradDesc
    g = torch.Generator(device=DEV).manual_seed(600 + Cc + H + B)
    Ho = H // 2
    rows_o = B * (Ho + 1) * (Ho + 1)
    x = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(Cc, Cc, 3, 3, device=DEV, generator=g) * (2.0 / (9 * Cc)) ** 0.5)
    dy = rbf(torch.randn(B, Cc, Ho, Ho, device=DEV, generator=g))
    dys = pf(dy)
    # weight gradient
    ph = torch.zeros(4 * rows_o, Cc, device=DEV, dtype=BF)
    check(lib.idf_space_to_depth(pf(x).data_ptr(), ph.data_ptr(), B, H, H, Cc, stream()))
    offs = [o for (_, _, o) in layout.taps_stride2(64, Ho, Ho, rows_o)]
    dw = torch.zeros(Cc, 9, Cc, device=DEV)
    d = WgradDesc()
    d.dy, d.rows, d.cout = dys.data_ptr(), rows_o, Cc
    d.x, d.x_rows, d.cin = ph.data_ptr(), ph.shape[0], Cc
    d.n_taps = 9
    for t, off in enumerate(offs):
        d.tap_off[t] = off
    d.dw = dw.data_ptr()
    h = C.c_void_p()
    check(lib.idf_wgrad_plan_create(C.byref(d), C.byref(h)))
    check(lib.idf_wgrad_run(h, stream()))
    torch.cuda.synchronize()
    lib.idf_wgrad_plan_destroy(h)
    ref_w = torch.nn.grad.conv2d_weight(x.double(), w.shape, dy.double(), stride=2, padding=1)
    ops.assert_close(dw.reshape(Cc, 3, 3, Cc).permute(0, 3, 1, 2), ref_w, rel_l2=1e-4, max_rel=1e-3,
                     what=f"stride-2 wgrad {H}->{Ho}")
    # data gradient: one implicit GEMM per phase, then depth-to-space
    dph = torch.zeros(4 * rows_o, Cc, device=DEV, dtype=BF)
    phases = layout.stride2_phase_dgrad(Cc, Ho, Ho)
    assert sorted(p for p, _, _ in phases) == [0, 1, 2, 3] and sum(len(t) for _, t, _ in phases) == 9
    for phase, taps, kb in phases:
        wp = torch.cat([w[:, :, ky, kx].t() for ky, kx in taps], dim=1).to(BF).contiguous()
        o = run_conv(lib, [dys], kb, wp, torch.zeros(Cc, device=DEV), B, Ho, Cc, 128 if Cc % 128 == 0 else 64)
        dph[phase * rows_o:(phase + 1) * rows_o] = o
    din = torch.zeros(B * (H + 1) * (H + 1), Cc, device=DEV, dtype=BF)
    check(lib.idf_depth_to_space(dph.data_ptr(), din.data_ptr(), B, H, H, Cc, 0, stream()))
    torch.cuda.synchronize()
    ref_x = torch.nn.grad.conv2d_input(x.shape, w.double(), dy.double(), stride=2, padding=1)
    assert pad_is_zero(din, B, H, H)
    assert_per_image(unpf(din, B, H, H), ref_x, 2e-3, 3.3e-3, f"stride-2 dgrad {H}->{Ho}")


def _attn_bwd(lib, H, B, d, seed, peak=None):
    """idf_attn_bwd against fp64 autograd of the reference attention; with `peak`, q and k are scaled so that every
    sample has scores of at least `peak` (as test_gpu_forward_wide._attention does)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    S = H * H

    def tok(t):
        return t.double().permute(0, 2, 3, 1).reshape(B, S, d)
    q, k, v = (torch.randn(B, d, H, H, device=DEV, generator=g) * s for s in (1.2, 1.2, 1.0))
    if peak is not None:
        f = (peak / (torch.bmm(tok(q), tok(k).transpose(1, 2)) * d ** -0.5).amax(dim=(1, 2)).min()).sqrt().float()
        q, k = q * f, k * f
    q, k, v = rbf(q), rbf(k), rbf(v)
    do = rbf(torch.randn(B, d, H, H, device=DEV, generator=g))
    qkv, dout = pf(torch.cat([q, k, v], 1)), pf(do)
    dqkv = torch.zeros(B * (H + 1) * (H + 1), 3 * d, device=DEV, dtype=BF)
    ws = torch.empty(int(lib.idf_attn_bwd_ws_bytes(B, H, H)), dtype=torch.uint8, device=DEV)
    check(lib.idf_attn_bwd(qkv.data_ptr(), dout.data_ptr(), dqkv.data_ptr(), ws.data_ptr(), B, H, H, d, d ** -0.5, stream()))
    torch.cuda.synchronize()
    qq, kk, vv = (tok(t).requires_grad_() for t in (q, k, v))
    scores = torch.bmm(qq, kk.transpose(1, 2)) * d ** -0.5
    if peak is not None:
        assert float(scores.detach().amax(dim=(1, 2)).min()) > 89.7, "a sample's scores stay below exp overflow"
    torch.bmm(torch.softmax(scores, dim=-1), vv).backward(tok(do))
    assert pad_is_zero(dqkv, B, H, H)
    got = unpf(dqkv, B, H, H)
    return [(name, got[:, sl], r.grad.reshape(B, H, H, d).permute(0, 3, 1, 2))
            for name, r, sl in (("dq", qq, slice(0, d)), ("dk", kk, slice(d, 2 * d)), ("dv", vv, slice(2 * d, 3 * d)))]


@pytest.mark.parametrize("H,B,d", [(4, 3, 512), (4, 8, 512), (4, 33, 128)])
def test_attention_backward_small_maps_per_image(lib, H, B, d):
    """The small-map attention backward at the vanilla 32x32 middle block (S = 16, d = 512) and at cifar InfoDiff's
    (S = 16, d = 128) over 33 images, per image (worst measured on a B200: 1.8e-3 / 3.6e-3)."""
    for name, got, ref in _attn_bwd(lib, H, B, d, 800 + H + B + d):
        assert_per_image(got, ref, 2.2e-3, 4.3e-3, f"attention backward {name} S={H * H} d={d} B={B}")


@pytest.mark.parametrize("H,B,d", [(16, 3, 128), (8, 3, 256), (4, 5, 128), (4, 2, 512)])
def test_attention_backward_large_logits(lib, H, B, d):
    """Scores of about +100 (exp overflows fp32): the tcgen05 backward (S = 256 / 64) and the small-map backward must
    subtract the row maximum like the forward.  Rows are nearly one-hot; the gradients are compared per image (worst
    measured on a B200: 2.5e-3 / 4.9e-3)."""
    for name, got, ref in _attn_bwd(lib, H, B, d, 900 + H + B + d, peak=100.0):
        assert_per_image(got, ref, 3e-3, 6e-3, f"attention backward, logits +100, {name} S={H * H} d={d}")


def test_attention_backward_rejects_shape_the_forward_takes(lib):
    """S = 1024, d = 256 runs forward (generic kernel) but has no backward: IDF_ERR_CUDA naming the supported
    envelopes, and dqkv untouched."""
    B, H, d = 2, 32, 256
    rows = B * (H + 1) * (H + 1)
    qkv = torch.zeros(rows, 3 * d, device=DEV, dtype=BF)
    out = torch.zeros(rows, d, device=DEV, dtype=BF)
    check(lib.idf_attn_fwd(qkv.data_ptr(), out.data_ptr(), B, H, H, d, d ** -0.5, stream()))
    dqkv = torch.full((rows, 3 * d), 3.0, device=DEV, dtype=BF)
    ws = torch.empty(max(int(lib.idf_attn_bwd_ws_bytes(B, H, H)), 1024), dtype=torch.uint8, device=DEV)
    rc = lib.idf_attn_bwd(qkv.data_ptr(), out.data_ptr(), dqkv.data_ptr(), ws.data_ptr(), B, H, H, d, d ** -0.5, stream())
    torch.cuda.synchronize()
    assert rc == IDF_ERR_CUDA, f"attention backward S={H * H} d={d}: status {rc}"
    msg = _last_error(lib)
    assert "H*W in {64,256}" in msg and "H*W*d <= 8192" in msg, msg
    assert bool((dqkv == 3.0).all()), "a rejected attention backward wrote dqkv"


# ------------------------------------------------------------------------------------------------
# the 32x32 networks at batches >= 6
# ------------------------------------------------------------------------------------------------
TOL_EPS = 2.1e-2      # tests/test_gpu_network.py


def _cifar_infodiff(T):
    from infodiffusion_b200.models import InfoDiff
    args = make_args(a_dim=32, diffusion_steps=T, input_size=32)
    torch.manual_seed(SEED)
    m = InfoDiff(args, "cpu", (3, 32, 32))
    sd = perturb_state_dict(m.state_dict())
    m.load_state_dict(sd)
    m.device = DEV
    for n in ("alpha_bars", "betas", "alphas", "alpha_prev_bars"):
        setattr(m, n, getattr(m, n).to(DEV))
    return args, m.to(DEV).eval(), sd


def test_cifar_infodiff_backbone_eps_per_sample():
    """cifar10's InfoDiff backbone (levels 32/16/8/4) at batch 8 against the oracle, every sample on its own."""
    args, m, sd = _cifar_infodiff(1000)
    g = torch.Generator().manual_seed(12)
    B = 8
    x = torch.rand(B, 3, 32, 32, generator=g) * 2 - 1
    t = torch.randint(0, 1000, (B,), generator=g)
    a = torch.randn(B, 32, generator=g)
    with torch.no_grad():
        ref = orc.aux_unet_forward(sd, x, t, a)
        got = m.backbone(x.to(DEV), t.to(DEV), a.to(DEV)).cpu()
    err = ((got.double() - ref.double()).reshape(B, -1).norm(dim=1) / ref.double().reshape(B, -1).norm(dim=1))
    print(f"\n[small-maps] cifar InfoDiff eps per-sample rel-L2: {[f'{float(e):.2e}' for e in err]}")
    assert float(err.max()) < TOL_EPS, f"sample {int(err.argmax())}: rel-L2 {float(err.max()):.3e}"


def test_cifar_infodiff_ddim_batch_independence():
    """Each sample of a batch-33 DDIM run equals the same sample run alone (to bf16 round-off: the fp32 summation order
    of the GroupNorm statistics depends on where the sample's rows fall), as test_full_size_batch_independence_and_
    chunking checks at 64x64."""
    from infodiffusion_b200.sampling import DiffusionProcess
    T, B = 3, 33
    args, m, sd = _cifar_infodiff(T)
    g = torch.Generator().manual_seed(13)
    xT = torch.randn(B, 3, 32, 32, generator=g)
    a = torch.randn(B, 32, generator=g)
    noise = {i: torch.randn(B, 3, 32, 32, generator=g) for i in range(T)}
    p = DiffusionProcess(make_args(**{**vars(args), "deterministic": True}), m, DEV, (3, 32, 32))

    def run(lo, hi):            # the process keeps one sampler (plans, graph) per batch size
        p.noise_fn = lambda idx, out: out.copy_(noise[idx][lo:hi])
        return p.sampling(hi - lo, xT=xT[lo:hi].to(DEV), a=a[lo:hi].to(DEV)).cpu()
    full = run(0, B)
    assert torch.isfinite(full).all()
    errs = []
    for n in range(B):
        alone = run(n, n + 1)
        errs.append(float((full[n] - alone[0]).double().norm() / alone[0].double().norm()))
    worst = max(range(B), key=lambda n: errs[n])
    print(f"\n[small-maps] batch-33 DDIM vs alone: worst sample {worst} rel-L2 {errs[worst]:.2e}")
    assert errs[worst] < 2e-3, f"sample {worst}: rel-L2 {errs[worst]:.3e} against the same sample alone"


def _check_grads(m, sdg, what):
    rels = []
    for name, p in m.named_parameters():
        g_ref = sdg[name].grad
        if g_ref is None or float(g_ref.abs().max()) == 0.0 or name.endswith("attn.proj_k.bias"):
            continue
        assert p.grad is not None, f"no gradient for {name}"
        g, r = p.grad.detach().cpu().double().flatten(), g_ref.double().flatten()
        rels.append((float((g - r).norm() / r.norm()), float((g @ r) / (g.norm() * r.norm())), name))
    rels.sort(reverse=True)
    med = sorted(r[0] for r in rels)[len(rels) // 2]
    print(f"\n[small-maps] {what} gradients: {len(rels)} checked, median rel-L2 {med:.3e}, worst {rels[0]}, "
          f"min cosine {min(c for _, c, _ in rels):.5f}")
    return rels, med


def test_vanilla_32x32_training_gradients_batch_8():
    """Diff(model='vanilla') at 32x32 (4x4 GroupNorms over 512 / 1024 channels), loss_fn at batch 8: loss and every
    parameter gradient against oracle autograd, as test_vanilla_training_gradients_at_native_widths does at batch 2."""
    from tests.test_gpu_train_wide import _draws, _oracle_loss, _vanilla
    args, m, sd = _vanilla(32)
    d = _draws(8, 32, torch.Generator().manual_seed(77))
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
    print(f"\n[small-maps] vanilla 32x32 B=8 loss: cuda {float(loss.detach()):.6f} vs oracle {float(loss_o.detach()):.6f}")
    assert abs(float(loss) - float(loss_o)) / abs(float(loss_o)) < 2e-2
    rels, med = _check_grads(m, sdg, "vanilla 32x32 B=8")
    assert len(rels) > 300 and med < 5e-2 and all(c > 0.98 for _, c, _ in rels), rels[:3]


def test_cifar_infodiff_training_gradients_batch_8():
    """cifar InfoDiff's loss_fn (denoising + MMD prior) at batch 8 in train() mode (dropout 0): loss and every parameter
    gradient against oracle autograd, as test_training_step_gradients_match_oracle_autograd does at 64x64."""
    args, m, sd = _cifar_infodiff(1000)
    gl = torch.Generator().manual_seed(23)
    B = 8
    xb = torch.rand(B, 3, 32, 32, generator=gl) * 2 - 1
    idx = torch.randint(0, 1000, (B,), generator=gl)
    eps = torch.randn(B, 3, 32, 32, generator=gl)
    encn = torch.randn(B, 32, generator=gl)
    prior = torch.randn(B, 32, generator=gl)
    sdg = {k: v.clone().requires_grad_(v.is_floating_point() and "timembedding.0" not in k) for k, v in sd.items()}
    sch = orc.Schedule.make(args.beta1, args.betaT, args.diffusion_steps)
    terms = orc.infodiff_loss(sdg, sch, xb, idx, eps, encn, prior, args.mmd_weight, args.kld_weight, args.diffusion_steps)
    terms["loss"].backward()
    m.train()
    m.backbone.dropout_p = 0.0
    m.encoder.dropout_p = 0.0
    m.zero_grad(set_to_none=True)
    try:
        with _patched_draws(idx.to(DEV), [eps.clone(), encn.clone(), prior.clone()]):
            loss = m.loss_fn(args, xb.to(DEV))
        loss.backward()
    finally:
        m.eval()
    print(f"\n[small-maps] cifar InfoDiff B=8 loss: cuda {float(loss):.6f} vs oracle {float(terms['loss']):.6f}")
    assert abs(float(loss) - float(terms["loss"])) / abs(float(terms["loss"])) < 2e-2
    rels, med = _check_grads(m, sdg, "cifar InfoDiff B=8")
    assert len(rels) > 500 and med < 5e-2 and all(c > 0.98 for _, c, _ in rels), rels[:3]
