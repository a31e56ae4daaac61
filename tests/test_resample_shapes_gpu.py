"""GPU: the x2 time resamplers (net_ops.resample2: eight outputs per thread, rows addressed by a 2-D block) at
the row lengths and row counts of the network's octaves and at short / non-power-of-two rows, forward and
gradient, against an fp64 evaluation of UpDownResample (networks/cqtdiff+.py:522-580) on the device."""
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

pytestmark = pytest.mark.gpu


def _reference64(x, up):
    from babe_b200 import denoiser
    c = x.shape[1]
    k = torch.tensor(denoiser._CUBIC, dtype=torch.float64, device=x.device)
    w = k[None, None, None, :].expand(c, 1, 1, -1)
    pad = len(denoiser._CUBIC) // 2 - 1
    if not up:
        return F.conv2d(F.pad(x, (pad, pad, 0, 0), "reflect"), w, stride=(1, 2), groups=c)
    p = (pad + 1) // 2
    return F.conv_transpose2d(F.pad(x, (p, p, 0, 0), "reflect"), w, stride=(1, 2), padding=(0, pad * 2 + 1), groups=c)


# (N, C, F, T): the octave layers' (T = 2048 ... 32, up to 917504 rows) and short or odd-length rows
SHAPES = [(8, 64, 64, 2048), (8, 96, 128, 1024), (8, 256, 448, 32), (2, 3, 5, 10), (2, 3, 5, 24), (3, 5, 7, 100),
          (1, 2, 3, 66)]


@pytest.mark.parametrize("up", [False, True])
@pytest.mark.parametrize("shape", SHAPES)
def test_resample_matches_fp64(shape, up):
    from babe_b200 import build, denoiser, net_ops
    build.build()
    g = torch.Generator(device="cuda").manual_seed(shape[-1])
    x = torch.randn(shape, device="cuda", generator=g).requires_grad_(True)
    y = net_ops.resample2(x, denoiser._CUBIC, up)
    x64 = x.detach().double().requires_grad_(True)
    ref = _reference64(x64, up)
    assert y.shape == ref.shape
    assert rel_l2(y.detach(), ref.detach()) < 1e-6
    gy = torch.randn(ref.shape, device="cuda", generator=g)
    gx, = torch.autograd.grad(y, x, gy)
    gref, = torch.autograd.grad(ref, x64, gy.double())
    assert rel_l2(gx, gref) < 1e-6
