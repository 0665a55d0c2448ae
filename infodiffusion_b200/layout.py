"""Pure host-side layout logic (no CUDA): pad-flat geometry, K-block tables, weight packing.

Pad-flat NHWC: image n, pixel (y, x) of an H x W x C map is row (n*(H+1) + y)*(W+1) + x of a
[rows, C] matrix; row y == H and column x == W of every image are zero and double as the
top / left border of the next row / image, so a 3x3 tap (dy, dx) is the constant row offset
dy*(W+1) + dx and TMA's out-of-bounds zero fill covers the very first / last image.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch

KBlock = Tuple[int, int, int]   # (source index, first channel of the 64-wide slice, signed row offset)


def padflat_rows(batch: int, H: int, W: int) -> int:
    return batch * (H + 1) * (W + 1)


def taps3x3(cin: int, H: int, W: int, src: int = 0) -> List[KBlock]:
    """K-blocks of a 3x3 / stride 1 / pad 1 conv: tap-major, then 64-channel slices."""
    kb: List[KBlock] = []
    for tap in range(9):
        ky, kx = divmod(tap, 3)
        off = (ky - 1) * (W + 1) + (kx - 1)
        kb += [(src, c0, off) for c0 in range(0, cin, 64)]
    return kb


def taps_stride2(cin: int, Ho: int, Wo: int, phase_rows: int, src: int = 0) -> List[KBlock]:
    """K-blocks of a 3x3 / stride 2 / pad 1 conv over a space-to-depth source holding the four phase
    maps phase[py*2+px][n, y, x] = in[n, 2y+py, 2x+px] stacked along rows (each pad-flat Ho x Wo).
    Input row 2*oy + ky - 1:  ky=0 -> odd phase, previous half-res row;  ky=1 -> even phase, same row;
    ky=2 -> odd phase, same row (likewise for columns)."""
    sel = {0: (1, -1), 1: (0, 0), 2: (1, 0)}
    kb: List[KBlock] = []
    for tap in range(9):
        ky, kx = divmod(tap, 3)
        (py, dy), (px, dx) = sel[ky], sel[kx]
        off = (py * 2 + px) * phase_rows + dy * (Wo + 1) + dx
        kb += [(src, c0, off) for c0 in range(0, cin, 64)]
    return kb


def stride2_phase_dgrad(cout: int, Ho: int, Wo: int, src: int = 0) -> List[Tuple[int, List[Tuple[int, int]], List[KBlock]]]:
    """Data gradient of the stride-2 conv above, one implicit GEMM per space-to-depth phase (py, px): the taps (ky, kx)
    that read that phase and their K-blocks over dY (negated row offsets, K ordered (tap, cout)).  Returns
    [(phase = py*2 + px, taps, k-blocks)]; the weights of phase p are cat([W[:, :, ky, kx]^T for (ky, kx) in taps], 1)."""
    sel = {0: (1, -1), 1: (0, 0), 2: (1, 0)}
    out = []
    for py in (0, 1):
        for px in (0, 1):
            taps = [(ky, kx) for ky in range(3) for kx in range(3) if sel[ky][0] == py and sel[kx][0] == px]
            kb: List[KBlock] = []
            for ky, kx in taps:
                off = sel[ky][1] * (Wo + 1) + sel[kx][1]
                kb += [(src, c0, -off) for c0 in range(0, cout, 64)]
            out.append((py * 2 + px, taps, kb))
    return out


def window_records_exact(H: int, W: int) -> bool:
    """Whether the conv epilogue's 32-row GroupNorm records (idf_conv_desc.stats_out) keep the images of an H x W
    pad-flat grid apart (mirror of window_records_exact in csrc/kernels.cuh): false for H = W <= 3, where
    idf_conv_plan_create rejects stats_out."""
    R = (H + 1) * (W + 1)
    return R >= 32 or 31 - R <= W + 2


def taps1x1(cin: int, src: int = 0) -> List[KBlock]:
    return [(src, c0, 0) for c0 in range(0, cin, 64)]


def pack_conv3x3(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> [Cout, 9*Cin] with k = (ky*3+kx)*Cin + c."""
    co, ci = w.shape[0], w.shape[1]
    return w.detach().permute(0, 2, 3, 1).reshape(co, 9 * ci)


def taps_up2(cin: int, H: int, W: int, src: int = 0) -> List[KBlock]:
    """K-blocks of a nearest-x2-upsample + 3x3 conv folded onto the INPUT grid (idf_conv_desc.up2): the four taps of
    output parity (0, 0) -- input rows {y-1, y} x columns {x-1, x} -- tap-major, then 64-channel slices; parity
    (py, px) uses the same taps shifted by py rows and px pixels (done by the kernel per column tile)."""
    kb: List[KBlock] = []
    for dy in (-1, 0):
        for dx in (-1, 0):
            kb += [(src, c0, dy * (W + 1) + dx) for c0 in range(0, cin, 64)]
    return kb


def pack_conv3x3_up2(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> [4*Cout, 4*Cin]: row block p = 2*py + px holds the weights of output parity (py, px), k =
    (ty*2 + tx)*Cin + c for the 2x2 input neighbourhood (ty, tx); the 3x3 taps that read the same input pixel after
    nearest upsampling are summed (ky -> ty: parity 0: {0} | {1, 2}; parity 1: {0, 1} | {2})."""
    grp = {0: ((0,), (1, 2)), 1: ((0, 1), (2,))}
    co, ci = w.shape[0], w.shape[1]
    w = w.detach()
    blocks = []
    for py in (0, 1):
        for px in (0, 1):
            taps = []
            for ty in (0, 1):
                for tx in (0, 1):
                    acc = None
                    for ky in grp[py][ty]:
                        for kx in grp[px][tx]:
                            acc = w[:, :, ky, kx] if acc is None else acc + w[:, :, ky, kx]
                    taps.append(acc)                                # [Cout, Cin]
            blocks.append(torch.stack(taps, dim=1).reshape(co, 4 * ci))
    return torch.cat(blocks, dim=0)


def tap_offsets3x3(H: int, W: int) -> List[int]:
    """Row offset of each of the 9 taps (tap = ky*3 + kx) in the pad-flat layout."""
    return [(t // 3 - 1) * (W + 1) + (t % 3 - 1) for t in range(9)]


def taps3x3_dgrad(cout: int, H: int, W: int, src: int = 0) -> List[KBlock]:
    """K-blocks of the DATA gradient of a 3x3 / stride 1 / pad 1 conv: the same implicit GEMM run over dY
    with negated tap offsets (dX[r] = sum_t dY[r - off_t] . W_t^T), K ordered (tap, cout)."""
    kb: List[KBlock] = []
    for off in tap_offsets3x3(H, W):
        kb += [(src, c0, -off) for c0 in range(0, cout, 64)]
    return kb


def pack_conv3x3_dgrad(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> [Cin, 9*Cout] with k = (ky*3+kx)*Cout + co (weights of the data-gradient GEMM)."""
    co, ci = w.shape[0], w.shape[1]
    return w.detach().permute(1, 2, 3, 0).reshape(ci, 9 * co)


def pack_conv1x1(w: torch.Tensor) -> torch.Tensor:
    return w.detach().reshape(w.shape[0], w.shape[1])


def pad_rows(m: torch.Tensor, rows: int) -> torch.Tensor:
    if m.shape[0] == rows:
        return m
    out = torch.zeros(rows, *m.shape[1:], dtype=m.dtype, device=m.device)
    out[: m.shape[0]] = m
    return out


def pad_cols(m: torch.Tensor, cols: int) -> torch.Tensor:
    if m.shape[1] == cols:
        return m
    out = torch.zeros(m.shape[0], cols, dtype=m.dtype, device=m.device)
    out[:, : m.shape[1]] = m
    return out


# ------------------------------------------------------------------------------------------------
# parameter index probing (training): packing recipes are pure re-orderings (permute / reshape / cat / zero
# pad), so running one over "1 + flat index" tensors instead of values yields the gather map of the packing.
# ------------------------------------------------------------------------------------------------
class ParamIndex:
    """Flat fp32 layout of a parameter list: parameter i occupies [offset[i], offset[i] + numel), densely packed in
    list order (what torch's flatten / unflatten helpers assume); `total` is rounded up to a multiple of 4."""

    def __init__(self, params: Sequence[torch.Tensor], device):
        self.params = list(params)
        self.device = device
        self.offset = {}
        off = 0
        for p in self.params:
            self.offset[id(p)] = off
            off += p.numel()
        self.dense = off
        self.total = max((off + 3) // 4 * 4, 4)

    def index_of(self, p) -> torch.Tensor:
        off = self.offset[id(p)]
        return torch.arange(off + 1, off + 1 + p.numel(), dtype=torch.int64, device=self.device).view(p.shape)

    def views(self, flat: torch.Tensor) -> List[torch.Tensor]:
        """Parameter-shaped views of a flat buffer in this layout (one C++ call, not a Python loop over ~400 tensors)."""
        return list(torch._utils._unflatten_dense_tensors(flat[: self.dense], self.params))


_probe: List[ParamIndex] = []


def pv(p):
    """Value of parameter `p` inside a packing recipe: the tensor itself, or -- while probing -- the int64
    tensor of its 1-based flat indices."""
    return _probe[-1].index_of(p) if _probe else p


class probing:
    def __init__(self, pindex: ParamIndex):
        self.pindex = pindex

    def __enter__(self):
        _probe.append(self.pindex)

    def __exit__(self, *exc):
        _probe.pop()


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous batch shard of `total` independent samples for `rank` (sampling / encoding are
    per-sample independent: GroupNorm and attention never mix samples)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)
