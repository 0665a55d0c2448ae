"""Forward kernels of the vanilla Diff model at the widths it hard-wires (UNet ch_mult [1, 2, 4, 8]: 512-channel levels,
GroupNorms over concatenations of up to 1024 channels, a 1536-wide qkv projection, attention heads of 256 and 512
channels), op by op on the B200.

The network-level check of this model compares one eps output and would pass a local error (one bad block of 16
queries, the last granule of a 1024-channel GroupNorm).  Here every kernel of idf_attn_fwd, the conv forward at the
wide shapes (3x3 over 1024 channels, the 1536-wide qkv projection, fused shortcuts up to IDF_CONV_MAX_KB k-blocks, the
data gradient, GroupNorm epilogue records) and the inference form of the wide AdaGN are compared with plain fp64 torch
on the same bf16-rounded inputs, with the tolerances of their narrow counterparts in test_gpu_ops.py.  Shapes outside
the documented envelope are tested for their rejection: IDF_ERR_ARG from the host before any launch."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests import test_gpu_ops as ops
from tests.test_gpu_ops import (BF, DEV, assert_close, check, lib, pad_is_zero, pf, rbf, run_conv,  # noqa: F401
                                stream, tile_partials, unit_partials, unpf)

pytestmark = pytest.mark.gpu

IDF_ERR_ARG, IDF_ERR_CUDA = -1, -2


def _last_error(lib):
    return lib.idf_last_error().decode()


# ------------------------------------------------------------------------------------------------
# attention: tcgen05 (d = 128, S in {64, 256}), small maps (S <= 64, S*d <= 8192), generic CUDA-core kernel (the rest)
# ------------------------------------------------------------------------------------------------
LN_FLT_MAX = 88.72      # exp(x) overflows fp32 above this


def _attention(lib, H, B, d, seed, peak=None):
    """idf_attn_fwd on random q, k, v and the fp64 reference of test_attention_small_maps.  With `peak`, q and k are
    scaled so that the largest score (scale d^-0.5 included) of the least peaked sample is `peak`: with peak above
    ln(FLT_MAX), exp of a raw score overflows fp32 in every sample, so only a softmax that subtracts the row maximum
    before the exponential stays finite."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    S = H * H

    def tokens(t):                                  # [B, d, H, W] -> [B, S, d]
        return t.double().permute(0, 2, 3, 1).reshape(B, S, d)

    def scores_of(q, k):
        return torch.bmm(tokens(q), tokens(k).transpose(1, 2)) * d ** -0.5

    q, k, v = (torch.randn(B, d, H, H, device=DEV, generator=g) * s for s in (1.2, 1.2, 1.0))
    if peak is not None:
        f = (peak / scores_of(q, k).amax(dim=(1, 2)).min()).sqrt().float()
        q, k = q * f, k * f
    q, k, v = rbf(q), rbf(k), rbf(v)
    qkv = pf(torch.cat([q, k, v], 1))
    out = torch.zeros(B * (H + 1) * (H + 1), d, device=DEV, dtype=BF)
    check(lib.idf_attn_fwd(qkv.data_ptr(), out.data_ptr(), B, H, H, d, d ** -0.5, stream()))
    torch.cuda.synchronize()
    scores = scores_of(q, k)
    if peak is not None:
        assert float(scores.amax(dim=(1, 2)).min()) > LN_FLT_MAX + 1, "a sample's scores stay below exp overflow"
    ref = torch.bmm(torch.softmax(scores, dim=-1), tokens(v)).reshape(B, H, H, d).permute(0, 3, 1, 2)
    assert pad_is_zero(out, B, H, H), "attention wrote a pad row"
    return unpf(out, B, H, H), ref


@pytest.mark.parametrize("H,B,d", [
    (16, 3, 256), (8, 4, 512),     # the 64x64 vanilla model: d = 256 at S = 256, d = 512 at S = 64
    (16, 40, 256),                 # 16 query blocks x 40 images: a grid larger than the machine
    (8, 3, 256),                   # the 32x32 vanilla model
    (5, 3, 512),                   # S = 25: the second 16-query block has 9 valid rows, the masked ones must not be written
    (32, 2, 128)])                 # S = 1024, the documented maximum
def test_attention_generic_kernel(lib, H, B, d):
    """The CUDA-core kernel (fp32 scores, softmax and P, like the small-map kernel): its tolerance."""
    got, ref = _attention(lib, H, B, d, 51 + H + d)
    assert_close(got, ref, rel_l2=3e-3, max_rel=1e-2, what=f"generic attention S={H * H} d={d} B={B}")


def test_attention_small_kernel_at_its_limit(lib):
    """S * d == 8192 (d = 512 on the 4x4 middle block of the 32x32 vanilla model): the largest small-map case."""
    got, ref = _attention(lib, 4, 3, 512, 61)
    assert_close(got, ref, rel_l2=3e-3, max_rel=1e-2, what="small attention S=16 d=512")


@pytest.mark.parametrize("H,B,d,rel_l2,max_rel", [
    (16, 3, 128, 6e-3, 2e-2),      # tcgen05 (P in bf16: the tolerance of test_attention)
    (4, 3, 128, 3e-3, 1e-2),       # small-map kernel
    (16, 3, 256, 3e-3, 1e-2),      # generic kernel
    (5, 2, 512, 3e-3, 1e-2)])      # generic kernel, partial last query block
def test_attention_large_logits(lib, H, B, d, rel_l2, max_rel):
    """Scores of about +100 in every sample (exp(100) is not an fp32 number): the softmax must subtract the row maximum
    before the exponential, otherwise the rows holding such scores come out inf / NaN.  The rows are nearly one-hot,
    which the tolerances of the ordinary cases cover."""
    got, ref = _attention(lib, H, B, d, 71 + H + d, peak=100.0)
    assert_close(got, ref, rel_l2=rel_l2, max_rel=max_rel, what=f"attention with logits of +100, S={H * H} d={d}")


@pytest.mark.parametrize("H,d", [(16, 12), (33, 64), (8, 1032)])
def test_attention_rejects_unsupported_shapes(lib, H, d):
    """d % 8 != 0, S = 1089 > 1024 and d = 1032 > 1024 (none of them a small map): IDF_ERR_CUDA with the supported
    envelopes in idf_last_error(), nothing launched, the output untouched."""
    B = 2
    rows = B * (H + 1) * (H + 1)
    qkv = torch.zeros(rows, 3 * d, device=DEV, dtype=BF)
    out = torch.full((rows, d), 3.0, device=DEV, dtype=BF)
    rc = lib.idf_attn_fwd(qkv.data_ptr(), out.data_ptr(), B, H, H, d, d ** -0.5, stream())
    torch.cuda.synchronize()
    assert rc == IDF_ERR_CUDA, f"attention S={H * H} d={d}: status {rc}"
    msg = _last_error(lib)
    assert "H*W*d <= 8192" in msg and "d <= 1024" in msg and "H*W <= 1024" in msg, msg
    assert bool((out == 3.0).all()), "a rejected attention call wrote its output"


# ------------------------------------------------------------------------------------------------
# conv forward at the wide shapes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout,H,B,res", [(1024, 512, 8, 2, False), (768, 512, 8, 2, False), (768, 256, 16, 2, False),
                                              (512, 512, 8, 3, True)])
def test_conv3x3_wide(lib, cin, cout, H, B, res):
    """3x3 convs of the up path (144, 108 and 108 k-blocks) and the 512-wide residual conv, as test_conv3x3."""
    ops.test_conv3x3(lib, cin, cout, H, B, res)


@pytest.mark.parametrize("cin,H,B", [(512, 8, 3), (256, 16, 2)])
def test_conv1x1_qkv_wide(lib, cin, H, B):
    """qkv projections of the 512- and 256-wide attention layers: cout_pad = 1536 is the bias-staging limit."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(81 + cin)
    cout = 3 * cin
    x = rbf(torch.randn(B, cin, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, cin, 1, 1, device=DEV, generator=g) * cin ** -0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    ref = F.conv2d(x.double(), w.double(), b.double())
    out = run_conv(lib, [pf(x)], layout.taps1x1(cin), layout.pack_conv1x1(w).to(BF).contiguous(), b, B, H, cout, 128)
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, what=f"conv1x1 qkv {cin}->{cout}@{H}")


def _shortcut_case(ca, ch, cs, cout, H, B, seed):
    """conv3x3 over `act` (ca channels) + 1x1 shortcut over cat(h, skip) (ch + cs): sources, k-blocks, packed weights,
    bias and the fp64 reference."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(seed)
    act = rbf(torch.randn(B, ca, H, H, device=DEV, generator=g))
    h = rbf(torch.randn(B, ch, H, H, device=DEV, generator=g))
    s = rbf(torch.randn(B, cs, H, H, device=DEV, generator=g))
    w3 = rbf(torch.randn(cout, ca, 3, 3, device=DEV, generator=g) * (1.0 / (9 * ca)) ** 0.5)
    wsc = rbf(torch.randn(cout, ch + cs, 1, 1, device=DEV, generator=g) * (1.0 / (ch + cs)) ** 0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    ref = F.conv2d(act.double(), w3.double(), b.double(), padding=1) + F.conv2d(torch.cat([h, s], 1).double(), wsc.double())
    kb = layout.taps3x3(ca, H, H, 0) + layout.taps1x1(ch, 1) + layout.taps1x1(cs, 2)
    wp = torch.cat([layout.pack_conv3x3(w3), layout.pack_conv1x1(wsc)], 1).to(BF).contiguous()
    return [pf(act), pf(h), pf(s)], kb, wp, b, ref


@pytest.mark.parametrize("ca,ch,cs,cout,H,B,nkb", [
    (512, 512, 512, 512, 8, 2, 88),       # the model's up-path ResBlock: 3x3 over 512 + 1x1 over a 512 + 512 concatenation
    (1024, 512, 512, 128, 8, 2, 160)])    # exactly IDF_CONV_MAX_KB
def test_conv3x3_fused_shortcut_wide(lib, ca, ch, cs, cout, H, B, nkb):
    """Three A sources in one K loop, as test_conv3x3_fused_shortcut, up to the largest k-block table."""
    from infodiffusion_b200._lib import IDF_CONV_MAX_KB
    srcs, kb, wp, b, ref = _shortcut_case(ca, ch, cs, cout, H, B, 91 + ca + cout)
    assert len(kb) == nkb <= IDF_CONV_MAX_KB
    out = run_conv(lib, srcs, kb, wp, b, B, H, cout, 128)
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, what=f"conv3 + fused shortcut, {nkb} k-blocks")


def _create_plan_rc(lib, srcs, kblocks, wp, bias, B, H, cout, block_n, out):
    """idf_conv_plan_create on a descriptor like run_conv's; returns (status, plan handle) without running anything."""
    from infodiffusion_b200._lib import ConvDesc
    d = ConvDesc()
    d.n_src = len(srcs)
    for i, s in enumerate(srcs):
        d.src[i], d.src_rows[i], d.src_ld[i] = s.data_ptr(), s.shape[0], s.shape[1]
    d.num_kb = len(kblocks)
    for k, (si, c0, off) in enumerate(kblocks[:len(d.kb_src)]):
        d.kb_src[k], d.kb_c0[k], d.kb_rowoff[k] = si, c0, off
    d.weight, d.cout_pad, d.block_n, d.cout, d.bias = wp.data_ptr(), wp.shape[0], block_n, cout, bias.data_ptr()
    d.batch, d.H, d.W, d.epilogue = B, H, H, 0
    d.out, d.out_ld = out.data_ptr(), cout
    h = C.c_void_p()
    return lib.idf_conv_plan_create(C.byref(d), C.byref(h)), h


def test_conv_plan_rejects_beyond_the_envelope(lib):
    """161 k-blocks and cout_pad = 1664 (bias staging holds 1536 columns): IDF_ERR_ARG from plan creation, no plan."""
    from infodiffusion_b200 import layout
    srcs, kb, wp, b, _ = _shortcut_case(1024, 512, 512, 128, 8, 2, 95)
    out = torch.zeros(srcs[0].shape[0], 128, device=DEV, dtype=BF)
    rc, h = _create_plan_rc(lib, srcs, kb, wp, b, 2, 8, 128, 128, out)       # 160 k-blocks: accepted
    check(rc)
    lib.idf_conv_plan_destroy(h)
    wp161 = torch.cat([wp, wp[:, :64]], 1).contiguous()
    rc, h = _create_plan_rc(lib, srcs, kb + [(0, 0, 0)], wp161, b, 2, 8, 128, 128, out)
    assert rc == IDF_ERR_ARG and h.value is None, f"161 k-blocks: status {rc}"
    assert "num_kb" in _last_error(lib)
    x = pf(torch.zeros(2, 64, 8, 8, device=DEV))
    wide = torch.zeros(1664, 64, device=DEV, dtype=BF)
    out = torch.zeros(x.shape[0], 1664, device=DEV, dtype=BF)
    rc, h = _create_plan_rc(lib, [x], layout.taps1x1(64), wide, torch.zeros(1664, device=DEV), 2, 8, 1664, 128, out)
    assert rc == IDF_ERR_ARG and h.value is None, f"cout_pad 1664: status {rc}"
    assert "1536" in _last_error(lib)


def test_conv_data_gradient_wide(lib):
    """dX of the 1024 -> 512 up-path conv through the forward kernel (72 k-blocks, 1024 output columns)."""
    ops.test_conv_data_gradient_through_forward_kernel(lib, 1024, 512, 8, 2)


@pytest.mark.parametrize("cin,H,B,mt", [(512, 8, 3, 0), (256, 8, 5, 1), (256, 16, 2, 1), (512, 16, 3, 2)])
def test_conv_epilogue_groupnorm_partials_wide(lib, cin, H, B, mt):
    """GroupNorm records of a 512-wide output: 32-row windows at 8x8, work-item records at 16x16."""
    ops.test_conv_epilogue_groupnorm_partials(lib, cin, 512, H, B, mt)


@pytest.mark.parametrize("Cc,H,B", [(256, 32, 2), (512, 16, 4)])
def test_downsample_stride2_wide(lib, Cc, H, B):
    ops.test_downsample_stride2(lib, Cc, H, B)


def test_upsample2x_then_wide_conv(lib):
    """Up-sampling of a 512-wide map (up2 folding needs cout <= 128, so these widths upsample explicitly) followed by
    the 3x3 512 -> 256 conv, against F.interpolate + F.conv2d."""
    from infodiffusion_b200 import layout
    g = torch.Generator(device=DEV).manual_seed(101)
    B, Cc, H, cout = 3, 512, 8, 256
    x = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    w = rbf(torch.randn(cout, Cc, 3, 3, device=DEV, generator=g) * (2.0 / (9 * Cc)) ** 0.5)
    b = torch.randn(cout, device=DEV, generator=g)
    up = torch.zeros(B * (2 * H + 1) * (2 * H + 1), Cc, device=DEV, dtype=BF)
    check(lib.idf_upsample2x(pf(x).data_ptr(), up.data_ptr(), B, H, H, Cc, stream()))
    torch.cuda.synchronize()
    x_up = F.interpolate(x, scale_factor=2.0, mode="nearest")
    assert torch.equal(unpf(up, B, 2 * H, 2 * H), x_up)
    assert pad_is_zero(up, B, 2 * H, 2 * H)
    out = run_conv(lib, [up], layout.taps3x3(Cc, 2 * H, 2 * H), layout.pack_conv3x3(w).to(BF).contiguous(), b, B, 2 * H,
                   cout, 128)
    assert pad_is_zero(out, B, 2 * H, 2 * H)
    assert_close(unpf(out, B, 2 * H, 2 * H), F.conv2d(x_up.double(), w.double(), b.double(), padding=1),
                 what="upsample2x 512 + conv3x3 512->256")


@pytest.mark.parametrize("pair", [1, 0])
def test_conv3x3_wide_forced_tiles_per_cta(lib, pair):
    """1024 -> 512 with two tiles per work unit, as CTA pairs and as single CTAs: identical bits."""
    ops.test_conv3x3_forced_tiles_per_cta(lib, 1024, 512, 8, 3, 2, pair)


@pytest.mark.parametrize("cin,cout,block_n,H,B", [(64, 64, 64, 8, 5), (512, 1536, 128, 8, 3), (256, 512, 128, 16, 2),
                                                  (64, 128, 64, 32, 1)])
def test_conv_plan_tiles(lib, cin, cout, block_n, H, B):
    """idf_conv_plan_tiles = ceil(rows / 128) * cout_pad / block_n for plain plans."""
    from infodiffusion_b200 import layout
    x = torch.zeros(B * (H + 1) * (H + 1), cin, device=DEV, dtype=BF)
    out = torch.zeros(x.shape[0], cout, device=DEV, dtype=BF)
    wp = torch.zeros(cout, cin, device=DEV, dtype=BF)
    rc, h = _create_plan_rc(lib, [x], layout.taps1x1(cin), wp, torch.zeros(cout, device=DEV), B, H, cout, block_n, out)
    check(rc)
    try:
        assert int(lib.idf_conv_plan_tiles(h)) == (x.shape[0] + 127) // 128 * (cout // block_n)
    finally:
        lib.idf_conv_plan_destroy(h)


# ------------------------------------------------------------------------------------------------
# AdaGN forward, inference form, C = 512, 768 (512 + 256), 1024 (512 + 512)
# ------------------------------------------------------------------------------------------------
def _adagn_inference_case(c0, c1, H, B, silu, seed):
    """Sources, parameters, a step-indexed timestep table (this block's columns at an offset inside a wider table,
    shared by the batch) and per-sample latent rows, with the fp64 GroupNorm expression and its (A, B) closed form."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    Cc = c0 + c1
    x0 = rbf(torch.randn(B, c0, H, H, device=DEV, generator=g) * 1.5 + 0.3)
    x1 = rbf(torch.randn(B, c1, H, H, device=DEV, generator=g) * 0.7 - 0.2) if c1 else None
    gamma = 1 + 0.1 * torch.randn(Cc, device=DEV, generator=g)
    beta = 0.1 * torch.randn(Cc, device=DEV, generator=g)
    nsteps, ncol, off, step = 4, 3 * 2 * Cc, 2 * Cc, 2
    tt = 0.3 * torch.randn(nsteps, ncol, device=DEV, generator=g)
    zz = 0.3 * torch.randn(B, ncol, device=DEV, generator=g)
    xin = (torch.cat([x0, x1], 1) if c1 else x0).double()
    st, bt = tt[step, off:off + Cc].double()[None], tt[step, off + Cc:off + 2 * Cc].double()[None]
    sz, bz = zz[:, off:off + Cc].double(), zz[:, off + Cc:off + 2 * Cc].double()
    v = F.group_norm(xin, 32, gamma.double(), beta.double(), 1e-5)
    v = v * (1 + st)[:, :, None, None] + bt[:, :, None, None]
    v = v * (1 + sz)[:, :, None, None] + bz[:, :, None, None]
    xg = xin.reshape(B, 32, -1)
    mean, var = xg.mean(-1), xg.var(-1, unbiased=False)
    cpg = Cc // 32
    rstd = (var + 1e-5).rsqrt().repeat_interleave(cpg, 1)
    mean = mean.repeat_interleave(cpg, 1)
    A = rstd * gamma.double() * (1 + st) * (1 + sz)
    Bc = ((beta.double() - mean * rstd * gamma.double()) * (1 + st) + bt) * (1 + sz) + bz
    from infodiffusion_b200._lib import AdaGNArgs
    a = AdaGNArgs()
    s0 = pf(x0)
    s1 = pf(x1) if c1 else None
    a.src0, a.c0 = s0.data_ptr(), c0
    if c1:
        a.src1, a.c1 = s1.data_ptr(), c1
    a.batch, a.H, a.W = B, H, H
    a.gamma, a.beta, a.eps = gamma.data_ptr(), beta.data_ptr(), 1e-5
    stp = torch.tensor([step], dtype=torch.int32, device=DEV)
    a.mod_t, a.mod_t_step_stride, a.mod_t_batch_stride = tt.data_ptr() + off * 4, ncol, 0
    a.mod_z, a.mod_z_step_stride, a.mod_z_batch_stride = zz.data_ptr() + off * 4, 0, ncol
    a.step_ptr = stp.data_ptr()
    a.apply_silu = 1 if silu else 0
    keep = (x0, x1, gamma, beta, tt, zz, stp)       # buffers the args point at
    return a, s0, s1, (F.silu(v) if silu else v), A, Bc, keep


@pytest.mark.parametrize("silu", [True, False])
@pytest.mark.parametrize("H,B", [(8, 5), (16, 3)])
@pytest.mark.parametrize("c0,c1", [(512, 0), (512, 256), (512, 512)])
def test_adagn_inference_wide(lib, c0, c1, H, B, silu):
    """Streaming AdaGN (the only variant above 256 channels) with 32-row window records and, where an image has enough
    rows, work-item records of different units for the two sources; tolerances of test_adagn."""
    a, s0, s1, ref, _, _, keep = _adagn_inference_case(c0, c1, H, B, silu, 111 + c0 + c1 + H)
    Cc = c0 + c1
    rows = B * (H + 1) * (H + 1)
    out = torch.zeros(rows, Cc, device=DEV, dtype=BF)
    st0 = tile_partials(s0, B, H, H)
    st1 = tile_partials(s1, B, H, H) if c1 else None
    a.out, a.stats0 = out.data_ptr(), st0.data_ptr()
    if c1:
        a.stats1 = st1.data_ptr()
    check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
    torch.cuda.synchronize()
    assert pad_is_zero(out, B, H, H)
    assert_close(unpf(out, B, H, H), ref, rel_l2=3e-3, max_rel=8e-3, what=f"adagn C={c0}+{c1}@{H} B={B} silu={silu}")
    R = (H + 1) * (H + 1)
    if R >= 256:
        out2 = torch.zeros_like(out)
        st0u = unit_partials(s0, B, H, H, 256)
        a.out, a.stats0, a.stats_unit0 = out2.data_ptr(), st0u.data_ptr(), 256
        if c1:
            st1u = unit_partials(s1, B, H, H, 128)
            a.stats1, a.stats_unit1 = st1u.data_ptr(), 128
        check(lib.idf_adagn_silu_fwd(C.byref(a), stream()))
        torch.cuda.synchronize()
        assert pad_is_zero(out2, B, H, H)
        assert_close(unpf(out2, B, H, H), ref, rel_l2=3e-3, max_rel=8e-3, what=f"adagn (item units 256/128) C={c0}+{c1}@{H}")


@pytest.mark.parametrize("H,B", [(8, 5), (16, 3)])
@pytest.mark.parametrize("c0,c1", [(512, 0), (512, 256), (512, 512)])
def test_adagn_coef_wide(lib, c0, c1, H, B):
    """idf_adagn_coef (the 1024-channel instantiation above 256) against the fp64 closed form of (A, B).  fp32 sums of up
    to 8192 elements per group and E[x^2] - mean^2: about 1e-5 relative."""
    a, s0, s1, _, A, Bc, keep = _adagn_inference_case(c0, c1, H, B, True, 121 + c0 + c1 + H)
    st0 = tile_partials(s0, B, H, H)
    st1 = tile_partials(s1, B, H, H) if c1 else None
    a.stats0 = st0.data_ptr()
    if c1:
        a.stats1 = st1.data_ptr()
    coef = torch.full((B, c0 + c1, 2), float("nan"), device=DEV)
    check(lib.idf_adagn_coef(C.byref(a), coef.data_ptr(), stream()))
    torch.cuda.synchronize()
    assert_close(coef[..., 0], A, rel_l2=1e-4, max_rel=1e-4, what=f"adagn coef A C={c0}+{c1}@{H}")
    assert_close(coef[..., 1], Bc, rel_l2=1e-4, max_rel=1e-4, what=f"adagn coef B C={c0}+{c1}@{H}")


@pytest.mark.parametrize("c0,c1", [(512, 0), (512, 256), (512, 512), (256, 64)])
def test_adagn_without_statistics_rejects_wide(lib, c0, c1):
    """The two-sweep variant (no producer statistics) serves <= 256 channels: a wider call, or one with statistics for
    the first source only, returns IDF_ERR_CUDA (as include/idf_b200.h documents) and leaves the output untouched."""
    H, B = 8, 3
    a, s0, s1, _, _, _, keep = _adagn_inference_case(c0, c1, H, B, True, 131 + c0 + c1)
    st0 = tile_partials(s0, B, H, H)
    a.stats0 = st0.data_ptr() if c1 else None
    g = torch.Generator(device=DEV).manual_seed(7)
    out = torch.randn(B * (H + 1) * (H + 1), c0 + c1, device=DEV, generator=g).to(BF)
    before = out.clone()
    a.out = out.data_ptr()
    rc = lib.idf_adagn_silu_fwd(C.byref(a), stream())
    torch.cuda.synchronize()
    assert rc == IDF_ERR_CUDA, f"AdaGN over {c0}+{c1} channels without statistics: status {rc}"
    assert "adagn" in _last_error(lib)
    assert torch.equal(out, before), "a rejected AdaGN call wrote its output"


@pytest.mark.parametrize("c0,c1,cout,H,B,silu,sc", [
    (512, 512, 128, 8, 3, True, False),    # xf_ctot = 1024, 144 transformed k-blocks
    (512, 256, 256, 16, 2, False, False),  # xf_ctot = 768
    (512, 512, 128, 8, 3, True, True)])    # + a raw 1x1 shortcut over both sources: 160 k-blocks
def test_conv_with_fused_adagn_wide(lib, c0, c1, cout, H, B, silu, sc):
    """The fused-transform conv at the vanilla model's concatenation widths against AdaGN-then-conv, as
    test_conv_with_fused_adagn_equals_adagn_then_conv requires (bitwise without the shortcut)."""
    ops.test_conv_with_fused_adagn_equals_adagn_then_conv(lib, c0, c1, cout, H, B, 3, silu, 0, sc)
