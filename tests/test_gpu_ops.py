"""Per-kernel parity tests on the B200, every call going through the C ABI (ctypes).

Inputs are rounded to bf16 first, the comparator is plain fp32/fp64 torch arithmetic on those same
values (the op-level slice of the oracle), so the only admissible differences are fp32 accumulation
order and the final bf16 rounding of the output (2^-9 relative).  Tolerances are written per test.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF = torch.bfloat16


@pytest.fixture(scope="module")
def lib():
    from infodiffusion_b200 import _lib
    l = _lib.load()
    _lib.check(l.idf_init())
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return l


def stream():
    return torch.cuda.current_stream().cuda_stream


def check(rc):
    from infodiffusion_b200 import _lib
    _lib.check(rc)


def rbf(x):
    """round to bf16 and back (values exactly representable in the kernels' storage type)"""
    return x.to(BF).float()


def pf(x):
    """NCHW fp32 (cuda) -> pad-flat bf16 via plain torch ops"""
    B, Cc, H, W = x.shape
    buf = torch.zeros(B, H + 1, W + 1, Cc, device=x.device, dtype=torch.float32)
    buf[:, :H, :W, :] = x.permute(0, 2, 3, 1)
    return buf.reshape(-1, Cc).to(BF).contiguous()


def unpf(m, B, H, W):
    return m.float().reshape(B, H + 1, W + 1, -1)[:, :H, :W, :].permute(0, 3, 1, 2).contiguous()


def pad_is_zero(m, B, H, W):
    v = m.float().reshape(B, H + 1, W + 1, -1)
    return bool((v[:, H, :, :] == 0).all() and (v[:, :, W, :] == 0).all())


def assert_close(got, ref, rel_l2=3e-3, max_rel=1.6e-2, what=""):
    got, ref = got.double(), ref.double()
    err = (got - ref).norm() / ref.norm().clamp_min(1e-30)
    mx = (got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    assert err < rel_l2 and mx < max_rel, f"{what}: rel-L2 {err:.3e} (tol {rel_l2}), max-rel {mx:.3e} (tol {max_rel})"


def tile_partials(m, B, H, W):
    """GroupNorm partial sums of a pad-flat bf16 matrix, laid out as the conv epilogue writes them:
    fp32 [2, ceil(rows/128)*4, C, 2]; record A[k] sums the rows of 32-row window k that lie in the image
    of the window's first row, record B[k] the rows that already belong to the next image (plain torch)."""
    rows, Cc = m.shape
    R = (H + 1) * (W + 1)
    nwin = (rows + 127) // 128 * 4
    r = torch.arange(rows, device=m.device)
    k = r // 32
    which = (r // R) - ((k * 32) // R)              # 0 -> record A, 1 -> record B
    v = m.float()
    out = torch.zeros(2 * nwin, Cc, 2, device=m.device)
    out[:, :, 0].index_add_(0, which * nwin + k, v)
    out[:, :, 1].index_add_(0, which * nwin + k, v * v)
    return out.reshape(2, nwin, Cc, 2).contiguous()


def unit_partials(m, B, H, W, unit):
    """The same for work-item units (idf_conv_desc.stats_out, unit = 128 * MT rows): record k = item * 4 + q sums the
    rows 32q..32q+31 of each of the item's 128-row tiles, A = rows in the image the ITEM starts in, B = the rest."""
    rows, Cc = m.shape
    R = (H + 1) * (W + 1)
    nwin = (rows + 127) // 128 * 4
    r = torch.arange(rows, device=m.device)
    item = r // unit
    k = item * 4 + (r % 128) // 32
    which = (r // R) - ((item * unit) // R)
    v = m.float()
    out = torch.zeros(2 * nwin, Cc, 2, device=m.device)
    out[:, :, 0].index_add_(0, which * nwin + k, v)
    out[:, :, 1].index_add_(0, which * nwin + k, v * v)
    return out.reshape(2, nwin, Cc, 2).contiguous()


def run_conv(lib, srcs, kblocks, wp, bias, B, H, cout, block_n, residual=None, epilogue=0, info=None, **extra):
    from infodiffusion_b200._lib import ConvDesc
    d = ConvDesc()
    d.n_src = len(srcs)
    for i, s in enumerate(srcs):
        d.src[i], d.src_rows[i], d.src_ld[i] = s.data_ptr(), s.shape[0], s.shape[1]
    d.num_kb = len(kblocks)
    for k, (si, c0, off) in enumerate(kblocks):
        d.kb_src[k], d.kb_c0[k], d.kb_rowoff[k] = si, c0, off
    d.weight, d.cout_pad, d.block_n, d.cout = wp.data_ptr(), wp.shape[0], block_n, cout
    d.bias = bias.data_ptr()
    d.batch, d.H, d.W, d.epilogue = B, H, H, epilogue
    out = None
    if epilogue == 0:
        out = torch.zeros(B * (H + 1) * (H + 1), cout, device=DEV, dtype=BF)
        d.out, d.out_ld = out.data_ptr(), cout
        if residual is not None:
            d.residual, d.res_ld = residual.data_ptr(), residual.shape[1]
    for k, v in extra.items():
        setattr(d, k, v.data_ptr() if torch.is_tensor(v) else v)
    h = C.c_void_p()
    check(lib.idf_conv_plan_create(C.byref(d), C.byref(h)))
    check(lib.idf_conv_run(h, stream()))
    torch.cuda.synchronize()
    if info is not None:
        info["stats_unit"] = int(lib.idf_conv_plan_stats_unit(h))
    lib.idf_conv_plan_destroy(h)
    return out


# ------------------------------------------------------------------------------------------------
def test_layout_kernels(lib):
    g = torch.Generator(device=DEV).manual_seed(0)
    for (B, Cc, H) in [(2, 64, 8), (3, 128, 16), (1, 192, 32)]:
        x = torch.randn(B, Cc, H, H, device=DEV, generator=g)
        out = torch.zeros(B * (H + 1) * (H + 1), Cc, device=DEV, dtype=BF)
        check(lib.idf_nchw_to_padflat(x.data_ptr(), out.data_ptr(), B, Cc, H, H, stream()))
        assert torch.equal(out, pf(x))
        back = torch.zeros_like(x)
        check(lib.idf_padflat_to_nchw(out.data_ptr(), back.data_ptr(), B, Cc, H, H, stream()))
        assert torch.equal(back, rbf(x))


@pytest.mark.parametrize("cin,cout,H,B,res", [
    (64, 64, 16, 2, False), (64, 64, 16, 2, True), (128, 128, 8, 3, True), (256, 128, 16, 2, False),
    (192, 64, 8, 2, False), (64, 128, 32, 1, False), (128, 128, 64, 1, True), (128, 128, 8, 37, False)])
def test_conv3x3(lib, cin, cout, H, B, res):
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(cin + cout + H)
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    r = rbf(torch.randn(B, cout, H, H, device=DEV, generator=g)) if res else None
    ref = F.conv2d(x.double(), w.double(), b.double(), padding=1)
    if res:
        ref = ref + r.double()
    out = run_conv(lib, [pf(x)], layout.taps3x3(cin, H, H), layout.pack_conv3x3(w).to(BF).contiguous(), b, B, H, cout,
                   128 if cout % 128 == 0 else 64, residual=pf(r) if res else None)
    assert pad_is_zero(out, B, H, H), "kernel wrote a pad row"
    assert_close(unpf(out, B, H, H), ref, what=f"conv3x3 {cin}->{cout}@{H} B={B} res={res}")


@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("cin,cout,H,B,mt", [(64, 64, 16, 3, 2), (64, 64, 16, 3, 4), (128, 128, 16, 3, 2),
                                              (128, 64, 8, 5, 4), (256, 128, 8, 4, 2), (128, 128, 8, 37, 1)])
def test_conv3x3_forced_tiles_per_cta(lib, cin, cout, H, B, mt, pair):
    """Every (BN, MT) instantiation of the halo kernel, as CTA pairs (cta_group::2, odd numbers of super tiles leave the
    peer CTA's rows out of range) and as single CTAs, including partially filled work units; both give the same bits."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(100 + cin + cout + H + mt)
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    ref = F.conv2d(x.double(), w.double(), b.double(), padding=1)
    check(lib.idf_set_option(b"conv_force_mt", mt))
    check(lib.idf_set_option(b"conv_pair", pair))
    try:
        out = run_conv(lib, [pf(x)], layout.taps3x3(cin, H, H), layout.pack_conv3x3(w).to(BF).contiguous(), b, B, H,
                       cout, 128 if cout % 128 == 0 else 64)
        check(lib.idf_set_option(b"conv_pair", 1 - pair))
        out2 = run_conv(lib, [pf(x)], layout.taps3x3(cin, H, H), layout.pack_conv3x3(w).to(BF).contiguous(), b, B, H,
                        cout, 128 if cout % 128 == 0 else 64)
    finally:
        check(lib.idf_set_option(b"conv_force_mt", 0))
        check(lib.idf_set_option(b"conv_pair", 1))
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, what=f"conv3x3 {cin}->{cout}@{H} MT={mt} pair={pair}")
    assert torch.equal(out, out2), "CTA pairs and single CTAs must produce identical bits"


def test_conv3x3_large_auto_tiles(lib):
    """Sizes at which the planner itself picks MT = 4 (BN = 64) and MT = 2 (BN = 128)."""
    from infodiffusion_b200 import layout
    for (cin, cout, H, B) in [(64, 64, 64, 40), (128, 128, 32, 80)]:
        g = torch.Generator(device=DEV).manual_seed(7 + cin)
        x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
        w = rbf(torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5)
        b = torch.randn(cout, device=DEV, generator=g)
        ref = F.conv2d(x, w, b, padding=1)          # fp32 (TF32 disabled by the fixture)
        out = run_conv(lib, [pf(x)], layout.taps3x3(cin, H, H), layout.pack_conv3x3(w).to(BF).contiguous(), b, B, H,
                       cout, 128 if cout % 128 == 0 else 64)
        assert_close(unpf(out, B, H, H), ref, what=f"conv3x3 {cin}->{cout}@{H} B={B}")


@pytest.mark.parametrize("cin,cout,H,B,mt", [(64, 64, 16, 3, 0), (128, 128, 8, 7, 0), (64, 128, 8, 5, 2), (64, 64, 32, 2, 4),
                                             (64, 64, 16, 5, 2), (128, 128, 32, 3, 2), (64, 64, 64, 2, 4), (128, 128, 16, 9, 1)])
def test_conv_epilogue_groupnorm_partials(lib, cin, cout, H, B, mt):
    """stats_out of the conv epilogue == (sum, sumsq) of the bf16 output it stored, per 32-row window or -- when an
    image has at least as many rows as a work item -- per (work item, lane quarter)."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(300 + cin + cout + H)
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    rows = B * (H + 1) * (H + 1)
    nwin = (rows + 127) // 128 * 4
    stats = torch.zeros(2, nwin, cout, 2, device=DEV)
    stats[0] = float("nan")                        # every A record must be written; B records only when straddling
    info = {}
    check(lib.idf_set_option(b"conv_force_mt", mt))
    try:
        out = run_conv(lib, [pf(x)], layout.taps3x3(cin, H, H), layout.pack_conv3x3(w).to(BF).contiguous(), b, B, H,
                       cout, 128 if cout % 128 == 0 else 64, stats_out=stats, info=info)
    finally:
        check(lib.idf_set_option(b"conv_force_mt", 0))
    unit = info["stats_unit"]
    assert unit == 32 or (unit % 128 == 0 and unit <= (H + 1) * (H + 1))
    # the cases reach both record kinds: an 8x8 image (81 rows) is smaller than any work item, the larger ones are not
    assert (unit == 32) == (H == 8), f"unexpected statistics unit {unit} at H={H}"
    if unit == 32:
        ref = tile_partials(out, B, H, H)
        assert torch.isfinite(stats).all(), "a window record was not written"
    else:
        ref = unit_partials(out, B, H, H, unit)
        n_rec = (rows + unit - 1) // unit * 4
        assert torch.isfinite(stats[0, :n_rec]).all(), "an item record was not written"
        stats[0, n_rec:] = 0.0                     # capacity beyond the item records is not touched
    assert_close(stats, ref, rel_l2=1e-5, max_rel=1e-5, what=f"conv epilogue GroupNorm partials (unit {unit})")


@pytest.mark.parametrize("cin,cout,H,B", [(64, 64, 16, 3), (128, 128, 8, 5), (64, 128, 16, 2), (256, 128, 8, 3),
                                           (128, 64, 32, 2)])
def test_conv_data_gradient_through_forward_kernel(lib, cin, cout, H, B):
    """dX = conv2d_input(dY, W): the forward implicit GEMM over dY with negated taps and transposed weights."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(400 + cin + cout + H)
    dy = rbf(torch.randn(B, cout, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5)
    ref = torch.nn.grad.conv2d_input((B, cin, H, H), w.double(), dy.double(), padding=1)
    out = run_conv(lib, [pf(dy)], layout.taps3x3_dgrad(cout, H, H), layout.pack_conv3x3_dgrad(w).to(BF).contiguous(),
                   torch.zeros(cin, device=DEV), B, H, cin, 128 if cin % 128 == 0 else 64)
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, what=f"dgrad {cin}<-{cout}@{H}")


@pytest.mark.parametrize("cin,cout,H,B", [(64, 64, 16, 3), (128, 128, 8, 5), (64, 128, 16, 2), (256, 128, 8, 3),
                                           (128, 64, 32, 2), (192, 64, 8, 2)])
def test_conv_weight_gradient(lib, cin, cout, H, B):
    """dW = conv2d_weight(X, dY) on tcgen05 (pixels as K, MN-major operands, row-shifted tap views)."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import WgradDesc
    g = torch.Generator(device=DEV).manual_seed(500 + cin + cout + H)
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    dy = rbf(torch.randn(B, cout, H, H, device=DEV, generator=g))
    ref = torch.nn.grad.conv2d_weight(x.double(), (cout, cin, 3, 3), dy.double(), padding=1)
    xs, dys = pf(x), pf(dy)
    dw = torch.zeros(cout, 9, cin, device=DEV)
    d = WgradDesc()
    d.dy, d.rows, d.cout = dys.data_ptr(), dys.shape[0], cout
    d.x, d.x_rows, d.cin = xs.data_ptr(), xs.shape[0], cin
    d.n_taps = 9
    for t, off in enumerate(layout.tap_offsets3x3(H, H)):
        d.tap_off[t] = off
    d.dw = dw.data_ptr()
    h = C.c_void_p()
    check(lib.idf_wgrad_plan_create(C.byref(d), C.byref(h)))
    check(lib.idf_wgrad_run(h, stream()))
    torch.cuda.synchronize()
    lib.idf_wgrad_plan_destroy(h)
    got = dw.reshape(cout, 3, 3, cin).permute(0, 3, 1, 2)
    assert_close(got, ref, rel_l2=1e-4, max_rel=1e-3, what=f"wgrad {cin}->{cout}@{H}")   # fp32 accumulation only


def test_conv1x1_qkv(lib):
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(5)
    B, H, cin, cout = 3, 16, 128, 384
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, cin, 1, 1, device=DEV, generator=g) * cin ** -0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    ref = F.conv2d(x.double(), w.double(), b.double())
    out = run_conv(lib, [pf(x)], layout.taps1x1(cin), layout.pack_conv1x1(w).to(BF).contiguous(), b, B, H, cout, 128)
    assert_close(unpf(out, B, H, H), ref, what="conv1x1 qkv")


def test_conv3x3_fused_shortcut(lib):
    """conv3(act) + shortcut1x1(cat(h, skip)): three A sources in one K loop."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(6)
    B, H, ch, cs, cout = 2, 16, 128, 64, 128
    act = rbf(torch.randn(B, cout, H, H, device=DEV, generator=g))
    h = rbf(torch.randn(B, ch, H, H, device=DEV, generator=g))
    s = rbf(torch.randn(B, cs, H, H, device=DEV, generator=g))
    w3 = rbf(torch.randn(cout, cout, 3, 3, device=DEV, generator=g) * 0.03)
    wsc = rbf(torch.randn(cout, ch + cs, 1, 1, device=DEV, generator=g) * 0.07)
    b = torch.randn(cout, device=DEV, generator=g)
    ref = F.conv2d(act.double(), w3.double(), b.double(), padding=1) + F.conv2d(torch.cat([h, s], 1).double(), wsc.double())
    kb = layout.taps3x3(cout, H, H, 0) + layout.taps1x1(ch, 1) + layout.taps1x1(cs, 2)
    wp = torch.cat([layout.pack_conv3x3(w3), layout.pack_conv1x1(wsc)], 1).to(BF).contiguous()
    out = run_conv(lib, [pf(act), pf(h), pf(s)], kb, wp, b, B, H, cout, 128)
    assert_close(unpf(out, B, H, H), ref, what="conv3 + fused shortcut")


@pytest.mark.parametrize("Cc,H,B", [(64, 16, 2), (128, 32, 3)])
def test_downsample_stride2(lib, Cc, H, B):
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(7)
    x = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(Cc, Cc, 3, 3, device=DEV, generator=g) * (2.0 / (9 * Cc)) ** 0.5)
    b = torch.randn(Cc, device=DEV, generator=g)
    ref = F.conv2d(x.double(), w.double(), b.double(), stride=2, padding=1)
    Ho = H // 2
    rows_o = B * (Ho + 1) * (Ho + 1)
    ph = torch.zeros(4 * rows_o, Cc, device=DEV, dtype=BF)
    check(lib.idf_space_to_depth(pf(x).data_ptr(), ph.data_ptr(), B, H, H, Cc, stream()))
    out = run_conv(lib, [ph], layout.taps_stride2(Cc, Ho, Ho, rows_o), layout.pack_conv3x3(w).to(BF).contiguous(), b, B,
                   Ho, Cc, 128 if Cc % 128 == 0 else 64)
    assert_close(unpf(out, B, Ho, Ho), ref, what="stride-2 conv")


def test_upsample2x(lib):
    g = torch.Generator(device=DEV).manual_seed(8)
    B, Cc, H = 3, 128, 8
    x = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    out = torch.zeros(B * (2 * H + 1) * (2 * H + 1), Cc, device=DEV, dtype=BF)
    check(lib.idf_upsample2x(pf(x).data_ptr(), out.data_ptr(), B, H, H, Cc, stream()))
    assert torch.equal(unpf(out, B, 2 * H, 2 * H), F.interpolate(x, scale_factor=2.0, mode="nearest"))
    assert pad_is_zero(out, B, 2 * H, 2 * H)


@pytest.mark.parametrize("cin,cout,H,B", [(128, 128, 8, 3), (128, 128, 16, 5), (64, 64, 16, 2), (128, 128, 32, 2), (192, 128, 8, 7)])
def test_upsample_folded_into_conv(lib, cin, cout, H, B):
    """idf_conv_desc.up2: conv3x3(nearest_x2(x)) computed on the input grid with four pre-summed taps per output
    parity (UpSample, modules.py:89-92) -- output, zero pads, and the GroupNorm statistics (4 parity planes over the
    input grid) consumed by the AdaGN kernel, against F.interpolate + F.conv2d."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import AdaGNArgs, ConvDesc
    g = torch.Generator(device=DEV).manual_seed(900 + cin + H)
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * (2.0 / (9 * cin)) ** 0.5
    b = torch.randn(cout, device=DEV, generator=g)
    wp = layout.pack_conv3x3_up2(w).to(BF).contiguous()
    # reference with the SAME (pre-summed, bf16-rounded) weights: undo the packing per parity
    up = F.interpolate(x, scale_factor=2.0, mode="nearest")
    ref_exact = F.conv2d(up.double(), w.double(), b.double(), padding=1)
    rows_in, rows_up = B * (H + 1) * (H + 1), B * (2 * H + 1) * (2 * H + 1)
    out = torch.zeros(rows_up, cout, device=DEV, dtype=BF)
    tiles_in = (rows_in + 127) // 128
    stats = torch.zeros(2 * tiles_in * 4 * 4 * cout * 2, device=DEV)
    xs = pf(x)
    d = ConvDesc()
    d.n_src = 1
    d.src[0], d.src_rows[0], d.src_ld[0] = xs.data_ptr(), xs.shape[0], cin
    kb = layout.taps_up2(cin, H, H)
    d.num_kb = len(kb)
    for k, (si, c0, off) in enumerate(kb):
        d.kb_src[k], d.kb_c0[k], d.kb_rowoff[k] = si, c0, off
    bias4 = b.repeat(4).contiguous()
    d.weight, d.cout_pad, d.block_n, d.cout, d.bias = wp.data_ptr(), 4 * cout, cout, cout, bias4.data_ptr()
    d.batch, d.H, d.W, d.epilogue, d.up2 = B, H, H, 0, 1
    d.out, d.out_ld, d.stats_out = out.data_ptr(), cout, stats.data_ptr()
    h = C.c_void_p()
    check(lib.idf_conv_plan_create(C.byref(d), C.byref(h)))
    check(lib.idf_conv_run(h, stream()))
    torch.cuda.synchronize()
    unit = int(lib.idf_conv_plan_stats_unit(h))
    lib.idf_conv_plan_destroy(h)
    assert pad_is_zero(out, B, 2 * H, 2 * H)
    # bf16 rounding of the pre-summed weights differs from rounding each 3x3 tap: compare against both
    assert_close(unpf(out, B, 2 * H, 2 * H), ref_exact, rel_l2=6e-3, max_rel=3e-2, what=f"up2 conv {cin}->{cout}@{H}")
    wq = wp.float().reshape(4, cout, 4, cin)
    refq = torch.zeros_like(ref_exact)
    xp = F.pad(x.double(), (1, 1, 1, 1))
    for py in (0, 1):
        for px in (0, 1):
            acc = b.double()[None, :, None, None].expand(B, cout, H, H).clone()
            for ty in (0, 1):
                for tx in (0, 1):
                    patch = xp[:, :, py + ty:py + ty + H, px + tx:px + tx + H]
                    acc += torch.einsum("oc,bchw->bohw", wq[py * 2 + px, :, ty * 2 + tx, :].double(), patch)
            refq[:, :, py::2, px::2] = acc
    assert_close(unpf(out, B, 2 * H, 2 * H), refq, what=f"up2 conv (same packed weights) {cin}->{cout}@{H}")
    # the statistics feed an AdaGN of the upsampled map
    a = AdaGNArgs()
    gamma, beta = torch.rand(cout, device=DEV, generator=g) + 0.5, torch.randn(cout, device=DEV, generator=g)
    o1, o2 = torch.zeros_like(out), torch.zeros_like(out)
    a.src0, a.c0, a.batch, a.H, a.W = out.data_ptr(), cout, B, 2 * H, 2 * H
    a.gamma, a.beta, a.eps, a.apply_silu = gamma.data_ptr(), beta.data_ptr(), 1e-5, 1
    a.out = o1.data_ptr()
    st_ref = tile_partials(out, B, 2 * H, 2 * H)
    a.stats0 = st_ref.data_ptr()
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    a.out, a.stats0, a.stats_unit0, a.stats_planes0, a.stats_rows0 = o2.data_ptr(), stats.data_ptr(), unit, 4, (H + 1) * (H + 1)
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    torch.cuda.synchronize()
    assert_close(o2.float(), o1.float(), rel_l2=1e-3, max_rel=2e-2, what="AdaGN from up2 statistics vs window statistics")


def test_im2col_head_and_gemm(lib):
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(9)
    B, H = 3, 64
    x = torch.rand(B, 3, H, H, device=DEV, generator=g) * 2 - 1
    w = rbf(torch.randn(64, 3, 3, 3, device=DEV, generator=g) * 0.2)
    b = torch.randn(64, device=DEV, generator=g)
    patches = torch.zeros(B * (H + 1) * (H + 1), 64, device=DEV, dtype=BF)
    check(lib.idf_im2col_head(x.data_ptr(), patches.data_ptr(), B, 3, H, H, stream()))
    ref = F.conv2d(rbf(x).double(), w.double(), b.double(), padding=1)
    wp = layout.pad_cols(layout.pack_conv3x3(w), 64).to(BF).contiguous()
    out = run_conv(lib, [patches], [(0, 0, 0)], wp, b, B, H, 64, 64)
    assert_close(unpf(out, B, H, H), ref, what="head conv (im2col + K=64 GEMM)")


def test_tail_fp32_and_sampler_epilogue(lib):
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(10)
    B, H, cin = 3, 16, 64
    a = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(3, cin, 3, 3, device=DEV, generator=g) * 0.05)
    b = torch.randn(3, device=DEV, generator=g)
    eps_ref = F.conv2d(a.double(), w.double(), b.double(), padding=1)
    wp = layout.pad_rows(layout.pack_conv3x3(w), 16).to(BF).contiguous()
    bias = layout.pad_rows(b, 16).contiguous()
    kb = layout.taps3x3(cin, H, H)
    eps = torch.zeros(B, 3, H, H, device=DEV)
    run_conv(lib, [pf(a)], kb, wp, bias, B, H, 3, 16, epilogue=1, out_f32=eps)
    assert_close(eps, eps_ref, rel_l2=1e-5, max_rel=1e-5, what="tail fp32 NCHW")   # fp32 out: accumulation order only
    # fused sampler update, step-indexed coefficients
    coef = torch.tensor([[9., 9., 9.], [0.7, -0.3, 0.05], [1., 1., 1.]], device=DEV)
    step = torch.tensor([1], dtype=torch.int32, device=DEV)
    x = torch.randn(B, 3, H, H, device=DEV, generator=g)
    nz = torch.randn(B, 3, H, H, device=DEV, generator=g)
    x_ref = 0.7 * x.double() - 0.3 * eps_ref + 0.05 * nz.double()
    x_io, eps2 = x.clone(), torch.zeros_like(eps)
    run_conv(lib, [pf(a)], kb, wp, bias, B, H, 3, 16, epilogue=2, out_f32=eps2, x_io=x_io, noise=nz, coef=coef,
             step_ptr=step)
    assert torch.equal(eps2, eps)
    assert_close(x_io, x_ref, rel_l2=1e-5, max_rel=1e-5, what="fused sampler update")


@pytest.mark.parametrize("c0,c1,H,B,mod,silu", [
    (64, 0, 64, 2, False, True), (128, 0, 32, 3, True, True), (128, 64, 32, 2, False, True),
    (128, 128, 16, 3, True, True), (128, 0, 8, 5, False, False), (64, 64, 64, 1, True, True)])
def test_adagn(lib, c0, c1, H, B, mod, silu):
    from infodiffusion_b200._lib import AdaGNArgs
    g = torch.Generator(device=DEV).manual_seed(c0 + c1 + H)
    Cc = c0 + c1
    x0 = rbf(torch.randn(B, c0, H, H, device=DEV, generator=g) * 1.5 + 0.3)
    x1 = rbf(torch.randn(B, c1, H, H, device=DEV, generator=g) * 0.7 - 0.2) if c1 else None
    gamma = 1 + 0.1 * torch.randn(Cc, device=DEV, generator=g)
    beta = 0.1 * torch.randn(Cc, device=DEV, generator=g)
    xin = torch.cat([x0, x1], 1) if c1 else x0
    ref = F.group_norm(xin.double(), 32, gamma.double(), beta.double(), 1e-5)
    a = AdaGNArgs()
    s0 = pf(x0)
    a.src0, a.c0 = s0.data_ptr(), c0
    if c1:
        s1 = pf(x1)
        a.src1, a.c1 = s1.data_ptr(), c1
    out = torch.zeros(B * (H + 1) * (H + 1), Cc, device=DEV, dtype=BF)
    a.out, a.batch, a.H, a.W = out.data_ptr(), B, H, H
    a.gamma, a.beta, a.eps = gamma.data_ptr(), beta.data_ptr(), 1e-5
    if mod:
        nsteps, ncol, off = 4, 3 * 2 * Cc, 2 * Cc          # a wider table: this block's columns start at `off`
        tt = 0.3 * torch.randn(nsteps, ncol, device=DEV, generator=g)   # step-indexed, shared by the batch
        zz = 0.3 * torch.randn(B, ncol, device=DEV, generator=g)        # per-sample
        step = torch.tensor([2], dtype=torch.int32, device=DEV)
        a.mod_t, a.mod_t_step_stride, a.mod_t_batch_stride = tt.data_ptr() + off * 4, ncol, 0
        a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = zz.data_ptr() + off * 4, 0, ncol
        a.step_ptr = step.data_ptr()
        st, bt = tt[2, off:off + Cc].double(), tt[2, off + Cc:off + 2 * Cc].double()
        sz, bz = zz[:, off:off + Cc].double(), zz[:, off + Cc:off + 2 * Cc].double()
        ref = ref * (1 + st)[None, :, None, None] + bt[None, :, None, None]
        ref = ref * (1 + sz)[:, :, None, None] + bz[:, :, None, None]
    a.apply_silu = 1 if silu else 0
    if silu:
        ref = F.silu(ref)
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    torch.cuda.synchronize()
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, rel_l2=3e-3, max_rel=8e-3, what=f"adagn C={c0}+{c1}@{H}")
    # streaming variant: statistics supplied as per-tile partial sums (what the conv epilogue writes)
    out2 = torch.zeros_like(out)
    st0 = tile_partials(s0, B, H, H)
    a.stats0, a.out = st0.data_ptr(), out2.data_ptr()
    if c1:
        st1 = tile_partials(s1, B, H, H)
        a.stats1 = st1.data_ptr()
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    torch.cuda.synchronize()
    assert pad_is_zero(out2, B, H, H)
    assert_close(unpf(out2, B, H, H), ref, rel_l2=3e-3, max_rel=8e-3, what=f"adagn (streaming) C={c0}+{c1}@{H}")
    # the same with work-item statistics units (128 * MT rows, four records each); the two sources of a concatenation
    # may come from producers with different units
    R = (H + 1) * (H + 1)
    units = [u for u in (512, 256, 128) if u <= R]
    if units:
        out3 = torch.zeros_like(out)
        u0, u1 = units[0], units[-1]
        st0u = unit_partials(s0, B, H, H, u0)
        a.stats0, a.stats_unit0, a.out = st0u.data_ptr(), u0, out3.data_ptr()
        if c1:
            st1u = unit_partials(s1, B, H, H, u1)
            a.stats1, a.stats_unit1 = st1u.data_ptr(), u1
        check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
        torch.cuda.synchronize()
        assert_close(out3.float(), out2.float(), rel_l2=1e-3, max_rel=2e-2, what=f"adagn (item units {u0}/{u1}) vs window units")


@pytest.mark.parametrize("save", [False, True])
@pytest.mark.parametrize("c0,c1,H,B,mod,silu,drop", [
    (64, 0, 32, 2, False, True, 0.0), (128, 0, 16, 3, True, True, 0.0), (128, 64, 16, 2, False, True, 0.0),
    (128, 128, 8, 3, True, True, 0.0), (128, 0, 8, 4, False, False, 0.0), (128, 0, 16, 3, True, True, 0.1)])
def test_adagn_backward(lib, c0, c1, H, B, mod, silu, drop, save):
    """dx and the (S1, S2) sums of idf_adagn_silu_bwd against torch autograd of the same expression
    (with dropout: the keep-mask is read off the forward output, the hash is the kernel's own)."""
    from infodiffusion_b200._lib import AdaGNArgs, AdaGNBwdArgs
    from infodiffusion_b200.train import adagn_param_grads
    g = torch.Generator(device=DEV).manual_seed(700 + c0 + c1 + H)
    Cc = c0 + c1
    x0 = rbf(torch.randn(B, c0, H, H, device=DEV, generator=g) * 1.5 + 0.3)
    x1 = rbf(torch.randn(B, c1, H, H, device=DEV, generator=g) * 0.7 - 0.2) if c1 else None
    gamma = (1 + 0.1 * torch.randn(Cc, device=DEV, generator=g)).requires_grad_(True)
    beta = (0.1 * torch.randn(Cc, device=DEV, generator=g)).requires_grad_(True)
    dy = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    xin = (torch.cat([x0, x1], 1) if c1 else x0).clone().requires_grad_(True)
    st = bt = sz = bz = None
    if mod:
        st, bt, sz, bz = (0.3 * torch.randn(B, Cc, device=DEV, generator=g) for _ in range(4))
        for v in (st, bt, sz, bz):
            v.requires_grad_(True)
    s0 = pf(x0)
    s1 = pf(x1) if c1 else None
    a = AdaGNArgs()
    a.src0, a.c0 = s0.data_ptr(), c0
    if c1:
        a.src1, a.c1 = s1.data_ptr(), c1
    out = torch.zeros(B * (H + 1) * (H + 1), Cc, device=DEV, dtype=BF)
    a.out, a.batch, a.H, a.W = out.data_ptr(), B, H, H
    gam_d, bet_d = gamma.detach().clone(), beta.detach().clone()
    a.gamma, a.beta, a.eps = gam_d.data_ptr(), bet_d.data_ptr(), 1e-5
    if mod:
        mt = torch.cat([st, bt], 1).detach().contiguous()      # per-sample rows (scale | shift)
        mz = torch.cat([sz, bz], 1).detach().contiguous()
        a.mod_t, a.mod_t_step_stride, a.mod_t_batch_stride = mt.data_ptr(), 0, 2 * Cc
        a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = mz.data_ptr(), 0, 2 * Cc
    a.apply_silu = 1 if silu else 0
    st0 = tile_partials(s0, B, H, H)
    a.stats0 = st0.data_ptr()
    if c1:
        st1 = tile_partials(s1, B, H, H)
        a.stats1 = st1.data_ptr()
    seed = torch.tensor([0x1234567], dtype=torch.int64, device=DEV)
    if drop > 0:
        a.dropout_p, a.dropout_seed, a.dropout_layer = drop, seed.data_ptr(), 7
    coef = torch.zeros(B, Cc, 4, device=DEV)
    if save:
        a.save_coef = coef.data_ptr()       # backward reads the forward's coefficients instead of the records
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    torch.cuda.synchronize()
    # reference expression under autograd (fp64)
    v = F.group_norm(xin.double(), 32, gamma.double(), beta.double(), 1e-5)
    if mod:
        v = v * (1 + st.double())[:, :, None, None] + bt.double()[:, :, None, None]
        v = v * (1 + sz.double())[:, :, None, None] + bz.double()[:, :, None, None]
    y = F.silu(v) if silu else v
    got_y = unpf(out, B, H, H).double()
    if drop > 0:
        keep = (got_y != 0)
        frac = 1.0 - keep.double().mean().item()
        assert abs(frac - drop) < 0.01, f"dropped fraction {frac}"
        thr = round(drop * 65536)
        y = y * keep * (65536.0 / (65536 - thr))
    assert_close(got_y, y.detach(), rel_l2=4e-3, max_rel=1e-2, what="adagn forward (train)")
    y.backward(dy.double())
    # kernel backward
    b = AdaGNBwdArgs()
    b.f = a
    dys = pf(dy)
    dx0 = torch.zeros_like(s0)
    dx1 = torch.zeros_like(s1) if c1 else None
    sums = torch.zeros(B, Cc, 2, device=DEV)
    ws = torch.zeros(lib.idf_adagn_bwd_ws_floats(B, Cc), device=DEV)
    b.dy, b.dx0, b.sums, b.ws = dys.data_ptr(), dx0.data_ptr(), sums.data_ptr(), ws.data_ptr()
    if c1:
        b.dx1 = dx1.data_ptr()
    # fused closed forms: gamma / beta accumulate over samples, modulation rows are written per sample
    dgam, dbet = torch.zeros(Cc, device=DEV), torch.zeros(Cc, device=DEV)
    b.dgamma, b.dbeta = dgam.data_ptr(), dbet.data_ptr()
    if mod:
        dmt, dmz = torch.zeros(B, 2 * Cc, device=DEV), torch.zeros(B, 2 * Cc, device=DEV)
        b.d_mod_t, b.d_mod_z = dmt.data_ptr(), dmz.data_ptr()
    check(lib.idf_adagn_silu_bwd(C.byref(b), stream()))
    torch.cuda.synchronize()
    assert_close(dgam, gamma.grad, rel_l2=2e-3, max_rel=1e-2, what="fused d gamma")
    assert_close(dbet, beta.grad, rel_l2=2e-3, max_rel=1e-2, what="fused d beta")
    if mod:
        for name, got, t in (("s_t", dmt[:, :Cc], st), ("b_t", dmt[:, Cc:], bt), ("s_z", dmz[:, :Cc], sz), ("b_z", dmz[:, Cc:], bz)):
            assert_close(got, t.grad, rel_l2=2e-3, max_rel=1e-2, what="fused d " + name)
    dx_ref = xin.grad
    assert_close(unpf(dx0, B, H, H), dx_ref[:, :c0], rel_l2=6e-3, max_rel=2e-2, what="adagn dx0")
    if c1:
        assert_close(unpf(dx1, B, H, H), dx_ref[:, c0:], rel_l2=6e-3, max_rel=2e-2, what="adagn dx1")
    gr = adagn_param_grads(sums, gam_d, bet_d, *(t.detach() if t is not None else None for t in (st, bt, sz, bz)))
    assert_close(gr["gamma"], gamma.grad, rel_l2=2e-3, max_rel=1e-2, what="d gamma")
    assert_close(gr["beta"], beta.grad, rel_l2=2e-3, max_rel=1e-2, what="d beta")
    if mod:
        for name, t in (("s_t", st), ("b_t", bt), ("s_z", sz), ("b_z", bz)):
            assert_close(gr[name], t.grad, rel_l2=2e-3, max_rel=1e-2, what="d " + name)
    # accumulation flag: running again with acc0 adds the same gradient on top
    b.acc0 = 1
    if c1:
        b.acc1 = 1
    check(lib.idf_adagn_silu_bwd(C.byref(b), stream()))
    torch.cuda.synchronize()
    assert_close(unpf(dx0, B, H, H), 2 * dx_ref[:, :c0], rel_l2=8e-3, max_rel=3e-2, what="adagn dx0 accumulate")


@pytest.mark.parametrize("H,B", [(16, 3), (8, 5)])
def test_attention(lib, H, B):
    g = torch.Generator(device=DEV).manual_seed(11 + H)
    d, S = 128, H * H
    q, k, v = (rbf(torch.randn(B, d, H, H, device=DEV, generator=g) * s) for s in (1.2, 1.2, 1.0))
    qkv = pf(torch.cat([q, k, v], 1))
    out = torch.zeros(B * (H + 1) * (H + 1), d, device=DEV, dtype=BF)
    check(lib.idf_attn_fwd(qkv.data_ptr(), out.data_ptr(), B, H, H, d, d ** -0.5, stream()))
    torch.cuda.synchronize()
    qq = q.double().permute(0, 2, 3, 1).reshape(B, S, d)
    kk = k.double().reshape(B, d, S)
    vv = v.double().permute(0, 2, 3, 1).reshape(B, S, d)
    w = torch.softmax(torch.bmm(qq, kk) * d ** -0.5, dim=-1)
    ref = torch.bmm(w, vv).reshape(B, H, H, d).permute(0, 3, 1, 2)
    assert pad_is_zero(out, B, H, H)
    # P is rounded to bf16 before the PV product: 2^-9 per probability, averaged over S keys
    assert_close(unpf(out, B, H, H), ref, rel_l2=6e-3, max_rel=2e-2, what=f"attention S={S}")


def test_linear_and_gather(lib):
    g = torch.Generator(device=DEV).manual_seed(12)
    for (M, N, K, silu) in [(100, 4992, 256, True), (37, 256, 64, False), (2, 32, 4096, False)]:
        x = torch.randn(M, K, device=DEV, generator=g)
        w = torch.randn(N, K, device=DEV, generator=g) * K ** -0.5
        b = torch.randn(N, device=DEV, generator=g)
        y = torch.zeros(M, N, device=DEV)
        check(lib.idf_linear_f32(x.data_ptr(), K, w.data_ptr(), b.data_ptr(), y.data_ptr(), N, M, N, K, int(silu), stream()))
        xin = F.silu(x.double()) if silu else x.double()
        assert_close(y, xin @ w.double().t() + b.double(), rel_l2=2e-6, max_rel=2e-5, what=f"linear {M}x{N}x{K}")
    table = torch.randn(50, 64, device=DEV, generator=g)
    idx = torch.randint(0, 50, (17,), device=DEV, generator=g)
    y = torch.zeros(17, 64, device=DEV)
    check(lib.idf_gather_rows_f32(table.data_ptr(), idx.data_ptr(), y.data_ptr(), 17, 64, stream()))
    assert torch.equal(y, table[idx])


def test_sampler_update(lib):
    g = torch.Generator(device=DEV).manual_seed(13)
    n = 2 * 3 * 64 * 64 + 4
    x, e, z = (torch.randn(n, device=DEV, generator=g) for _ in range(3))
    coef = torch.tensor([[1., 2., 3.], [0.9, -0.2, 0.01]], device=DEV)
    step = torch.tensor([1], dtype=torch.int32, device=DEV)
    ref = 0.9 * x.double() - 0.2 * e.double() + 0.01 * z.double()
    check(lib.idf_sampler_update(x.data_ptr(), e.data_ptr(), z.data_ptr(), coef.data_ptr(), step.data_ptr(), n, stream()))
    assert_close(x, ref, rel_l2=1e-6, max_rel=1e-6, what="sampler update")


def test_mmd_against_oracle_and_golden(lib, golden_dir):
    from infodiffusion_b200.utils import compute_mmd
    from oracle import infodiff_oracle as orc
    gold = np.load(golden_dir / "mmd.npz")
    for D in (32, 256):
        gen = torch.Generator().manual_seed(11 + D)
        xs = torch.randn(32, D, generator=gen)
        ys = torch.randn(32, D, generator=gen) * 0.7 + 0.2
        yo = ys.clone().requires_grad_(True)
        vo = orc.compute_mmd(xs, yo)
        (go,) = torch.autograd.grad(vo, yo)
        yg = ys.to(DEV).requires_grad_(True)
        vg = compute_mmd(xs.to(DEV), yg)
        (gg,) = torch.autograd.grad(vg, yg)
        # the loss is a small difference of O(1) means: compare on the scale of the terms (fp32 sum order)
        assert abs(float(vg) - float(vo)) < 5e-6, f"mmd value D={D}: {float(vg)} vs {float(vo)}"
        assert_close(gg.cpu(), go, rel_l2=1e-4, max_rel=1e-3, what=f"mmd grad D={D}")
        assert abs(float(vg) - float(gold[f"v{D}"])) < 5e-6, "mmd vs golden"


@pytest.mark.parametrize("rows,Cc", [(1, 64), (4225 * 3, 64), (1089 * 5, 128), (289 * 2, 384), (77, 8)])
def test_colsum_bias_gradient(lib, rows, Cc):
    """idf_colsum_bf16 accumulates the column sums of a bf16 matrix into an fp32 vector (conv bias gradient)."""
    g = torch.Generator(device=DEV).manual_seed(rows + Cc)
    mth = (torch.randn(rows, Cc, device=DEV, generator=g)).to(BF)
    out = torch.full((Cc,), 0.5, device=DEV)
    check(lib.idf_colsum_bf16(mth.data_ptr(), out.data_ptr(), rows, Cc, stream()))
    torch.cuda.synchronize()
    want = mth.double().sum(0) + 0.5
    assert_close(out, want, rel_l2=1e-5, max_rel=1e-4, what="colsum")


@pytest.mark.parametrize("M,N,bcast,silu,affine", [(5, 128, False, True, True), (70, 1024, True, True, True),
                                                   (3, 1000, False, False, False), (1, 32, False, True, True)])
def test_scale_layernorm_silu(lib, M, N, bcast, silu, affine):
    """LatentUNet layer tail (reference models.py:147-163): SiLU(LayerNorm(y * (1 + cond)))."""
    g = torch.Generator(device=DEV).manual_seed(M * 7 + N)
    ld = N + 8
    ybuf = torch.randn(M, ld, device=DEV, generator=g)
    cond = torch.randn(1 if bcast else M, N, device=DEV, generator=g) * 0.3
    gamma = 1 + 0.1 * torch.randn(N, device=DEV, generator=g)
    beta = 0.1 * torch.randn(N, device=DEV, generator=g)
    out = torch.zeros(M, ld, device=DEV)
    check(lib.idf_scale_layernorm_silu(ybuf.data_ptr(), ld, cond.data_ptr(), 0 if bcast else N, 0, None,
                                       gamma.data_ptr() if affine else None, beta.data_ptr() if affine else None, 1e-5,
                                       out.data_ptr(), ld, M, N, int(silu), stream()))
    torch.cuda.synchronize()
    v = ybuf[:, :N].double() * (1 + cond.double())
    v = F.layer_norm(v, (N,), gamma.double() if affine else None, beta.double() if affine else None, 1e-5)
    want = F.silu(v) if silu else v
    assert_close(out[:, :N], want, rel_l2=2e-6, max_rel=2e-4, what="scale_layernorm_silu")
    assert float(out[:, N:].abs().max()) == 0.0


def test_clip_adamw_matches_torch():
    """ClipAdamW.step() == clip_grad_norm_(params, 1.) + torch.optim.AdamW.step() (reference run.py:199-200, 177),
    over several steps, ragged tensor sizes, a parameter without gradient and a gradient view with an odd offset."""
    from infodiffusion_b200.optim import ClipAdamW
    g = torch.Generator(device=DEV).manual_seed(5)
    shapes = [(64, 64, 3, 3), (4097,), (3,), (128, 9), (5000, 3), (7,)]
    ref = [torch.nn.Parameter(torch.randn(s, device=DEV, generator=g)) for s in shapes]
    mine = [torch.nn.Parameter(p.detach().clone()) for p in ref]
    o_ref = torch.optim.AdamW(ref, lr=3e-3, weight_decay=1e-2)
    o_mine = ClipAdamW(mine, lr=3e-3, weight_decay=1e-2, max_norm=1.0)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(o_mine, T_max=5)
    sched_ref = torch.optim.lr_scheduler.CosineAnnealingLR(o_ref, T_max=5)
    for it in range(4):
        scale = 10.0 if it % 2 == 0 else 0.01          # clipping active / inactive
        flat = torch.randn(sum(p.numel() for p in ref) + 1, device=DEV, generator=g) * scale
        off = 1                                        # odd offset: unaligned gradient views
        for i, (pr, pm) in enumerate(zip(ref, mine)):
            if i == 2 and it == 0:
                pr.grad = pm.grad = None               # skipped like torch skips it
                continue
            gv = flat[off:off + pr.numel()].view(pr.shape)
            off += pr.numel()
            pr.grad = gv.clone()
            pm.grad = gv
        want_norm = torch.nn.utils.clip_grad_norm_([p for p in ref if p.grad is not None], 1.0)
        o_ref.step()
        o_mine.step()
        sched.step(); sched_ref.step()
        torch.cuda.synchronize()
        assert abs(float(o_mine.total_norm) - float(want_norm)) <= 1e-5 * float(want_norm)
        for pr, pm in zip(ref, mine):
            assert_close(pm.detach(), pr.detach(), rel_l2=1e-6, max_rel=1e-4, what=f"adamw step {it}")


@pytest.mark.parametrize("c0,c1,cout,H,B,k,silu,mt,sc", [
    (64, 0, 64, 16, 3, 3, True, 0, False), (128, 0, 128, 8, 5, 3, True, 0, False), (128, 64, 64, 16, 2, 3, True, 0, True),
    (128, 128, 128, 8, 3, 3, True, 0, True), (128, 0, 384, 16, 2, 1, False, 0, False), (64, 0, 64, 32, 6, 3, True, 4, False),
    (128, 0, 128, 16, 9, 3, True, 2, False), (64, 0, 3, 16, 3, 3, True, 0, False), (64, 0, 64, 64, 3, 3, True, 0, False),
    # several work items per CTA (persistent loop, both halo stages recycled), plain and with raw shortcut groups
    (64, 0, 64, 32, 160, 3, True, 0, False), (128, 64, 64, 16, 300, 3, True, 0, True), (128, 0, 128, 32, 90, 3, True, 0, False)])
def test_conv_with_fused_adagn_equals_adagn_then_conv(lib, c0, c1, cout, H, B, k, silu, mt, sc):
    """idf_conv with xf_coef (AdaGN + SiLU applied to the A operand in shared memory) against the two-kernel path
    idf_adagn_silu_fwd -> idf_conv on the same inputs.  Covers concatenated sources, an untransformed 1x1
    shortcut over the raw sources, 1x1 convs, the narrow fp32 epilogue and MT > 1 work units."""
    from infodiffusion_b200 import layout
    from infodiffusion_b200._lib import AdaGNArgs
    g = torch.Generator(device=DEV).manual_seed(c0 + c1 + cout + H + k)
    Cc = c0 + c1
    x0 = rbf(torch.randn(B, c0, H, H, device=DEV, generator=g) * 1.5 + 0.3)
    x1 = rbf(torch.randn(B, c1, H, H, device=DEV, generator=g) * 0.7 - 0.2) if c1 else None
    s0, s1 = pf(x0), (pf(x1) if c1 else None)
    gamma = 1 + 0.1 * torch.randn(Cc, device=DEV, generator=g)
    beta = 0.1 * torch.randn(Cc, device=DEV, generator=g)
    zz = 0.3 * torch.randn(B, 2 * Cc, device=DEV, generator=g)
    a = AdaGNArgs()
    a.src0, a.c0 = s0.data_ptr(), c0
    st0 = tile_partials(s0, B, H, H)
    a.stats0 = st0.data_ptr()
    if c1:
        a.src1, a.c1 = s1.data_ptr(), c1
        st1 = tile_partials(s1, B, H, H)
        a.stats1 = st1.data_ptr()
    normed = torch.zeros(B * (H + 1) * (H + 1), Cc, device=DEV, dtype=BF)
    a.out, a.batch, a.H, a.W = normed.data_ptr(), B, H, H
    a.gamma, a.beta, a.eps = gamma.data_ptr(), beta.data_ptr(), 1e-5
    a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = zz.data_ptr(), 0, 2 * Cc
    a.apply_silu = 1 if silu else 0
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    coef = torch.zeros(B, Cc, 2, device=DEV)
    check(lib.idf_adagn_coef(C.byref(a), coef.data_ptr(), stream()))
    torch.cuda.synchronize()
    # weights
    cpad = 16 if cout < 64 else cout
    w = rbf(torch.randn(cout, Cc, k, k, device=DEV, generator=g) * (2.0 / (k * k * Cc)) ** 0.5)
    wp = layout.pack_conv3x3(w) if k == 3 else layout.pack_conv1x1(w)
    offs = layout.tap_offsets3x3(H, H) if k == 3 else [0]
    bias = torch.randn(cpad, device=DEV, generator=g)
    # unfused: one materialised source
    kb_ref = [(0, c, off) for off in offs for c in range(0, Cc, 64)]
    srcs_ref = [normed]
    # fused: raw sources + coefficient bases
    srcs, kb, kx = [s0] + ([s1] if c1 else []), [], []
    for off in offs:
        for c in range(0, c0, 64):
            kb.append((0, c, off)); kx.append(c)
        for c in range(0, c1, 64):
            kb.append((1, c, off)); kx.append(c0 + c)
    if sc:                                   # fused 1x1 shortcut over the RAW sources: no transform on those k-blocks
        wsc = rbf(torch.randn(cout, Cc, 1, 1, device=DEV, generator=g) * (1.0 / Cc) ** 0.5)
        wp = torch.cat([wp, layout.pack_conv1x1(wsc)], dim=1)
        srcs_ref = [normed, s0] + ([s1] if c1 else [])
        for c in range(0, c0, 64):
            kb_ref.append((1, c, 0)); kb.append((0, c, 0)); kx.append(-1)
        for c in range(0, c1, 64):
            kb_ref.append((2, c, 0)); kb.append((1, c, 0)); kx.append(-1)
    wp = layout.pad_rows(wp, cpad).to(BF).contiguous()
    bn = 16 if cout < 64 else (128 if cout % 128 == 0 else 64)
    extra = {}
    if cout < 64:
        out_ref, out_fused = torch.zeros(B, cout, H, H, device=DEV), torch.zeros(B, cout, H, H, device=DEV)
        epi = 1
    else:
        epi = 0
    from infodiffusion_b200._lib import IDF_CONV_MAX_KB
    kbx = (C.c_int32 * IDF_CONV_MAX_KB)(*(kx + [0] * (IDF_CONV_MAX_KB - len(kx))))
    if mt:
        check(lib.idf_set_option(b"conv_force_mt", mt))
    try:
        if epi == 0:
            ref = run_conv(lib, srcs_ref, kb_ref, wp, bias, B, H, cout, bn)
            got = run_conv(lib, srcs, kb, wp, bias, B, H, cout, bn, xf_coef=coef, xf_ctot=Cc, xf_silu=int(silu), kb_xf=kbx)
            assert pad_is_zero(got, B, H, H)
        else:
            run_conv(lib, srcs_ref, kb_ref, wp, bias, B, H, cout, bn, epilogue=1, out_f32=out_ref)
            run_conv(lib, srcs, kb, wp, bias, B, H, cout, bn, epilogue=1, out_f32=out_fused, xf_coef=coef, xf_ctot=Cc,
                     xf_silu=int(silu), kb_xf=kbx)
            ref, got = out_ref, out_fused
    finally:
        if mt:
            check(lib.idf_set_option(b"conv_force_mt", 0))
    assert float(ref.float().abs().max()) > 0.1
    if sc:      # raw and transformed k-blocks interleave differently: fp32 accumulation order differs, 1 bf16 ulp at most
        assert_close(got.float(), ref.double(), rel_l2=1e-3, max_rel=1.6e-2, what="fused conv + shortcut")
    else:       # same fp32 arithmetic, same bf16 rounding of the operand: bitwise identical
        assert torch.equal(got, ref), f"fused != unfused: max diff {float((got.float() - ref.float()).abs().max())}"
    # the raw sources must be untouched (the transform happens in shared memory only)
    assert torch.equal(s0, pf(x0))


@pytest.mark.parametrize("H,B,d", [(4, 5, 128), (2, 3, 128), (8, 2, 64)])
def test_attention_small_maps(lib, H, B, d):
    """Maps below the tensor-core kernel's shapes (e.g. the 4x4 middle block of a 32x32 model): plain-FMA kernel."""
    g = torch.Generator(device=DEV).manual_seed(31 + H + d)
    S = H * H
    q, k, v = (rbf(torch.randn(B, d, H, H, device=DEV, generator=g) * s) for s in (1.2, 1.2, 1.0))
    qkv = pf(torch.cat([q, k, v], 1))
    out = torch.zeros(B * (H + 1) * (H + 1), d, device=DEV, dtype=BF)
    check(lib.idf_attn_fwd(qkv.data_ptr(), out.data_ptr(), B, H, H, d, d ** -0.5, stream()))
    torch.cuda.synchronize()
    qq = q.double().permute(0, 2, 3, 1).reshape(B, S, d)
    kk = k.double().reshape(B, d, S)
    vv = v.double().permute(0, 2, 3, 1).reshape(B, S, d)
    ref = torch.bmm(torch.softmax(torch.bmm(qq, kk) * d ** -0.5, dim=-1), vv).reshape(B, H, H, d).permute(0, 3, 1, 2)
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, rel_l2=3e-3, max_rel=1e-2, what=f"small attention S={S} d={d}")


@pytest.mark.parametrize("M,K,N,bias", [(2, 64, 256, True), (32, 256, 4992, True), (5, 4096, 32, True), (70, 1280, 1024, False),
                                         (1, 33, 7, True)])
def test_linear_autograd_on_own_kernels(lib, M, K, N, bias):
    """infodiffusion_b200.linear (idf_linear_f32 forward, idf_gemm_f32 for dX / dW / db) against torch's F.linear in
    fp64: the Linears of the time / latent MLPs and fc heads under autograd (modules.py:24-27, models.py:147-163, 470-472)."""
    from infodiffusion_b200 import linear as L
    g = torch.Generator(device=DEV).manual_seed(M * 7 + K + N)
    x = torch.randn(M, K, device=DEV, generator=g, requires_grad=True)
    w = (torch.randn(N, K, device=DEV, generator=g) / K ** 0.5).requires_grad_()
    b = torch.randn(N, device=DEV, generator=g).requires_grad_() if bias else None
    dy = torch.randn(M, N, device=DEV, generator=g)
    y = L.linear(x, w, b)
    y.backward(dy)
    xr, wr = x.detach().double().requires_grad_(), w.detach().double().requires_grad_()
    br = b.detach().double().requires_grad_() if bias else None
    yr = torch.nn.functional.linear(xr, wr, br)
    yr.backward(dy.double())
    # fp32 accumulation over up to 4992 terms in a fixed order
    assert_close(y.detach(), yr.detach(), rel_l2=3e-6, max_rel=1e-4, what="linear y")
    assert_close(x.grad, xr.grad, rel_l2=3e-6, max_rel=1e-4, what="linear dx")
    assert_close(w.grad, wr.grad, rel_l2=3e-6, max_rel=1e-4, what="linear dw")
    if bias:
        assert_close(b.grad, br.grad, rel_l2=3e-6, max_rel=1e-4, what="linear db")


@pytest.mark.parametrize("H,B,d", [(16, 3, 128), (8, 5, 128), (16, 33, 128), (4, 3, 128), (2, 2, 128)])
def test_attention_backward(lib, H, B, d):
    """idf_attn_bwd (tcgen05: S and dP recomputed, P / dS rows through a workspace, then dQ = dS K, dK = dS^T Q,
    dV = P^T dO; plain-FMA kernel for the small maps) against torch autograd of the reference's attention
    (modules.py:152-161) in fp64."""
    g = torch.Generator(device=DEV).manual_seed(41 + H + B)
    S = H * H
    q, k, v = (rbf(torch.randn(B, d, H, H, device=DEV, generator=g) * s) for s in (1.2, 1.2, 1.0))
    do = rbf(torch.randn(B, d, H, H, device=DEV, generator=g))
    qkv = pf(torch.cat([q, k, v], 1))
    dout = pf(do)
    dqkv = torch.zeros(B * (H + 1) * (H + 1), 3 * d, device=DEV, dtype=BF)
    ws = torch.empty(int(lib.idf_attn_bwd_ws_bytes(B, H, H)), dtype=torch.uint8, device=DEV)
    check(lib.idf_attn_bwd(qkv.data_ptr(), dout.data_ptr(), dqkv.data_ptr(), ws.data_ptr(), B, H, H, d, d ** -0.5, stream()))
    torch.cuda.synchronize()
    qq = q.double().permute(0, 2, 3, 1).reshape(B, S, d).requires_grad_()
    kk = k.double().permute(0, 2, 3, 1).reshape(B, S, d).requires_grad_()
    vv = v.double().permute(0, 2, 3, 1).reshape(B, S, d).requires_grad_()
    w = torch.softmax(torch.bmm(qq, kk.transpose(1, 2)) * d ** -0.5, dim=-1)
    o = torch.bmm(w, vv)
    o.backward(do.double().permute(0, 2, 3, 1).reshape(B, S, d))
    got = unpf(dqkv, B, H, H)                                   # [B, 3d, H, W]
    assert pad_is_zero(dqkv, B, H, H)
    for name, ref, sl in (("dq", qq.grad, slice(0, d)), ("dk", kk.grad, slice(d, 2 * d)), ("dv", vv.grad, slice(2 * d, 3 * d))):
        ref = ref.reshape(B, H, H, d).permute(0, 3, 1, 2)
        # P and dS pass through bf16 (2^-9 relative per entry) before the second set of GEMMs
        assert_close(got[:, sl], ref, rel_l2=8e-3, max_rel=3e-2, what=f"attention backward {name} S={S}")
