"""AdaGN apply kernel against a plain device copy of the same bytes (what the measured HBM peak is made of)."""
import ctypes as C
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from infodiffusion_b200 import _lib  # noqa: E402
from infodiffusion_b200._lib import AdaGNArgs  # noqa: E402

lib = _lib.load()
_lib.check(lib.idf_init())
dev = "cuda:0"
BF = torch.bfloat16


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3     # us


SHAPES = [(256, 64, 64), (256, 32, 128), (256, 16, 128), (256, 8, 128), (256, 16, 256), (256, 8, 256), (32, 64, 64), (32, 32, 128)]
for (B, H, Cc) in SHAPES:
    rows = B * (H + 1) * (H + 1)
    x = torch.randn(rows, Cc, device=dev).to(BF)
    out = torch.zeros_like(x)
    tiles = (rows + 127) // 128
    stats = torch.rand(2 * tiles * 4 * Cc * 2, device=dev) + 1.0
    gamma, beta = torch.ones(Cc, device=dev), torch.zeros(Cc, device=dev)
    a = AdaGNArgs()
    a.src0, a.c0, a.out = x.data_ptr(), Cc, out.data_ptr()
    a.batch, a.H, a.W = B, H, H
    a.gamma, a.beta, a.eps, a.apply_silu = gamma.data_ptr(), beta.data_ptr(), 1e-5, 1
    a.stats0 = stats.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    # two buffers alternating so that nothing stays in L2 between repetitions
    x2, out2 = x.clone(), torch.zeros_like(x)
    b = AdaGNArgs.from_buffer_copy(a)
    b.src0, b.out = x2.data_ptr(), out2.data_ptr()
    flip = [0]

    def run_adagn():
        flip[0] ^= 1
        _lib.check(lib.idf_adagn_silu_fwd(C.byref(a if flip[0] else b), st))

    def run_copy():
        flip[0] ^= 1
        (out if flip[0] else out2).copy_(x if flip[0] else x2)

    mb = 2 * rows * Cc * 2 / 1e6
    t_a, t_c = timeit(run_adagn), timeit(run_copy)
    print(f"B={B} H={H} C={Cc}: {mb:7.1f} MB  adagn {t_a:7.1f} us = {mb / t_a * 1e3 / 1e3:6.2f} TB/s   "
          f"torch copy {t_c:7.1f} us = {mb / t_c * 1e3 / 1e3:6.2f} TB/s")
