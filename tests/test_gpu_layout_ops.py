"""Layout and data-movement kernels of the training step and the latent sampler, bit for bit on the B200.

These kernels only move, sum or round values, so each has an exact reference in plain torch: the same fp32 additions
in the kernel's order, rounded to bf16 where the kernel stores bf16.  Destinations are pre-filled with sentinels so that
a write outside the intended block (a pad row, the channels beyond C of a wider row, the bytes around a 2-D block)
shows up as a changed value.  Rejections are host-side: IDF_ERR_ARG before any launch, with idf_last_error() naming
the cause."""
import ctypes as C

import pytest
import torch

from tests.test_gpu_ops import BF, DEV, check, lib, pf, rbf, stream, unpf  # noqa: F401

pytestmark = pytest.mark.gpu

IDF_ERR_ARG = -1
SENTINEL = -77.0          # exactly representable in bf16


def _pad_mask(B, H, W, device=DEV):
    """[rows] bool: the pad rows (y == H or x == W) of a pad-flat B x H x W map."""
    m = torch.zeros(B, H + 1, W + 1, dtype=torch.bool, device=device)
    m[:, H, :] = True
    m[:, :, W] = True
    return m.reshape(-1)


def _with_pad_sentinel(m, B, H, W):
    m = m.clone()
    m[_pad_mask(B, H, W)] = SENTINEL
    return m


def _assert_pads_kept(m, before, B, H, W, what):
    pad = _pad_mask(B, H, W)
    assert torch.equal(m[pad], before[pad]), f"{what}: a pad row was written"


@pytest.mark.parametrize("acc", [0, 1])
@pytest.mark.parametrize("H", [4, 8, 16])
@pytest.mark.parametrize("Cc", [64, 256, 512])
def test_upsample2x_bwd(lib, Cc, H, acc):
    """d(nearest x2): din[n, y, x] = bf16 of the fp32 sum of the four taps (0,0), (0,1), (1,0), (1,1) in that order;
    with accumulate, bf16(din + that).  The gradient's own pad rows carry a sentinel the kernel must not read."""
    B = 3
    g = torch.Generator(device=DEV).manual_seed(Cc + H + acc)
    dout = _with_pad_sentinel(pf(torch.randn(B, Cc, 2 * H, 2 * H, device=DEV, generator=g)), B, 2 * H, 2 * H)
    din0 = pf(torch.randn(B, Cc, H, H, device=DEV, generator=g)) if acc else torch.zeros(B * (H + 1) ** 2, Cc, device=DEV, dtype=BF)
    din = _with_pad_sentinel(din0, B, H, H)
    before = din.clone()
    check(lib.idf_upsample2x_bwd(dout.data_ptr(), din.data_ptr(), B, H, H, Cc, acc, stream()))
    torch.cuda.synchronize()
    t = unpf(dout, B, 2 * H, 2 * H)
    s = ((t[:, :, 0::2, 0::2] + t[:, :, 0::2, 1::2]) + t[:, :, 1::2, 0::2]) + t[:, :, 1::2, 1::2]
    want = rbf(s)
    if acc:
        want = rbf(unpf(before, B, H, H) + want)
    assert torch.equal(unpf(din, B, H, H), want), f"upsample2x_bwd C={Cc} H={H} acc={acc}"
    _assert_pads_kept(din, before, B, H, H, "upsample2x_bwd")


@pytest.mark.parametrize("acc", [0, 1])
@pytest.mark.parametrize("Cc,H,B", [(64, 8, 3), (256, 16, 2), (512, 16, 3), (128, 32, 1)])
def test_depth_to_space(lib, Cc, H, B, acc):
    """idf_depth_to_space is the exact inverse of idf_space_to_depth (H, W: full resolution); with accumulate it adds
    in fp32 and rounds to bf16.  The phase maps' pad rows carry a sentinel the kernel must not read."""
    g = torch.Generator(device=DEV).manual_seed(200 + Cc + H + acc)
    x = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    Ho = H // 2
    rows_o = B * (Ho + 1) * (Ho + 1)
    ph = torch.full((4 * rows_o, Cc), SENTINEL, device=DEV, dtype=BF)
    check(lib.idf_space_to_depth(pf(x).data_ptr(), ph.data_ptr(), B, H, H, Cc, stream()))
    y = rbf(torch.randn(B, Cc, H, H, device=DEV, generator=g))
    din = _with_pad_sentinel(pf(y) if acc else torch.zeros(B * (H + 1) ** 2, Cc, device=DEV, dtype=BF), B, H, H)
    before = din.clone()
    check(lib.idf_depth_to_space(ph.data_ptr(), din.data_ptr(), B, H, H, Cc, acc, stream()))
    torch.cuda.synchronize()
    assert torch.equal(unpf(din, B, H, H), rbf(y + x) if acc else x), f"depth_to_space C={Cc} H={H} acc={acc}"
    _assert_pads_kept(din, before, B, H, H, "depth_to_space")


@pytest.mark.parametrize("B,Cc,H,ld", [(2, 3, 16, 64), (3, 40, 8, 64), (2, 96, 8, 128), (1, 64, 32, 192), (3, 3, 5, 64),
                                       (2, 40, 7, 64)])
def test_nchw_to_padflat_ld(lib, B, Cc, H, ld):
    """NCHW fp32 -> pad-flat bf16 rows of ld >= C channels: channels C..ld-1 and the pad rows keep what they held.  The
    5x5 and 7x7 maps end in a partial 32-pixel tile."""
    g = torch.Generator(device=DEV).manual_seed(300 + Cc + H)
    x = torch.randn(B, Cc, H, H, device=DEV, generator=g)
    out = torch.full((B * (H + 1) * (H + 1), ld), SENTINEL, device=DEV, dtype=BF)
    check(lib.idf_nchw_to_padflat_ld(x.data_ptr(), out.data_ptr(), B, Cc, H, H, ld, stream()))
    torch.cuda.synchronize()
    assert torch.equal(unpf(out[:, :Cc].contiguous(), B, H, H), rbf(x))
    assert bool((out[:, Cc:] == SENTINEL).all()), "channels beyond C were written"
    assert bool((out[_pad_mask(B, H, H)] == SENTINEL).all()), "a pad row was written"


@pytest.mark.parametrize("M,N,lds,ldd,r0,c0", [(37, 50, 61, 83, 1, 7), (700, 700, 701, 720, 2, 9), (1, 1, 1, 5, 0, 3)])
def test_copy2d_f32(lib, M, N, lds, ldd, r0, c0):
    """An M x N fp32 block between distinct row pitches: exact, and every other element of the destination is untouched.
    The 700 x 700 case has more elements (490,000) than the capped grid of 1184 x 256 threads, so it runs the
    grid-stride loop."""
    g = torch.Generator(device=DEV).manual_seed(400 + M + N)
    src = torch.randn(M, lds, device=DEV, generator=g)
    dst = torch.full((r0 + M + 1, ldd), SENTINEL, device=DEV)
    ptr = dst.data_ptr() + (r0 * ldd + c0) * 4
    check(lib.idf_copy2d_f32(src.data_ptr(), lds, ptr, ldd, M, N, stream()))
    torch.cuda.synchronize()
    want = torch.full_like(dst, SENTINEL)
    want[r0:r0 + M, c0:c0 + N] = src[:, :N]
    assert torch.equal(dst, want)


@pytest.mark.parametrize("bf16,use_idx2,acc", [(0, 0, 0), (0, 1, 0), (0, 0, 1), (0, 1, 1), (1, 0, 0), (1, 1, 0)])
def test_gather_elems(lib, bf16, use_idx2, acc):
    """dst[i] (+)= src[idx[i] - 1] (+ src[idx2[i] - 1]) with index 0 read as literal zero, in fp32 in that order; a bf16
    destination gets the rounded sum.  n is large enough for the grid-stride loop; the elements after n are untouched."""
    g = torch.Generator(device=DEV).manual_seed(500 + 4 * bf16 + 2 * use_idx2 + acc)
    n, nsrc = 4 * 400_000, 5000
    src = torch.randn(nsrc, device=DEV, generator=g)
    table = torch.cat([torch.zeros(1, device=DEV), src])                # table[0] = the literal zero
    idx = torch.randint(0, nsrc + 1, (n,), device=DEV, generator=g, dtype=torch.int32)
    idx[::7] = 0
    idx2 = torch.randint(0, nsrc + 1, (n,), device=DEV, generator=g, dtype=torch.int32)
    idx2[::5] = 0
    want = table[idx.long()]
    if use_idx2:
        want = want + table[idx2.long()]
    tail = 8
    if bf16:
        dst = torch.full((n + tail,), SENTINEL, device=DEV, dtype=BF)
        want = want.to(BF)
    else:
        dst = torch.full((n + tail,), SENTINEL, device=DEV)
        if acc:
            dst[:n] = torch.randn(n, device=DEV, generator=g)
            want = want + dst[:n]
    check(lib.idf_gather_elems(src.data_ptr(), idx.data_ptr(), idx2.data_ptr() if use_idx2 else None, dst.data_ptr(), n,
                               bf16, acc, stream()))
    torch.cuda.synchronize()
    assert torch.equal(dst[:n], want)
    assert bool((dst[n:].float() == SENTINEL).all()), "elements after n were written"


def test_gather_elems_host_rejections(lib):
    """n % 4 != 0, a bf16 destination with accumulate and a misaligned idx: IDF_ERR_ARG, named by idf_last_error(), the
    destination untouched."""
    src = torch.randn(64, device=DEV)
    idx = torch.arange(1, 65, device=DEV, dtype=torch.int32)
    dst = torch.full((64,), SENTINEL, device=DEV)
    dst_bf = torch.full((64,), SENTINEL, device=DEV, dtype=BF)
    cases = [("n = 6", (src.data_ptr(), idx.data_ptr(), None, dst.data_ptr(), 6, 0, 0), "multiple of 4"),
             ("bf16 + accumulate", (src.data_ptr(), idx.data_ptr(), None, dst_bf.data_ptr(), 64, 1, 1), "fp32 destination"),
             ("misaligned idx", (src.data_ptr(), idx.data_ptr() + 4, None, dst.data_ptr(), 32, 0, 0), "aligned")]
    for what, args, cause in cases:
        rc = lib.idf_gather_elems(*args, stream())
        assert rc == IDF_ERR_ARG, f"{what}: status {rc}"
        msg = lib.idf_last_error().decode()
        assert cause in msg, f"{what}: idf_last_error() = {msg!r}"
    torch.cuda.synchronize()
    assert bool((dst == SENTINEL).all()) and bool((dst_bf.float() == SENTINEL).all())
