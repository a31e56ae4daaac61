"""GPU: one ResnetBlock's dilated layers as one chain (net_ops.res_chain: statistics from the producing
gate_residual, the preceding layer's g_v from gn_film_gelu_bwd) against the same layers one by one
(net_ops.res_layer) and against an fp64 evaluation of networks/cqtdiff+.py:470-482 on the device,
forward and gradient wrt the activations; the fused by-products against the standalone kernels; bitwise
repeatability, eagerly and replayed from a CUDA graph."""
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

pytestmark = pytest.mark.gpu

G, EPS = 8, 1e-7

# (N, C, F, T), dilations: the largest octave layer of the network, and tails -- P = F*T not a multiple
# of 4 (scalar paths), an odd number of planes per group, P a multiple of 4 but not of the 4096 elements
# of one CTA (vector path with a partial last chunk)
CASES = [((8, 96, 128, 1024), 4), ((3, 24, 7, 9), 3), ((2, 16, 33, 1025), 2), ((1, 64, 20, 37), 3),
         ((2, 16, 32, 100), 2), ((2, 16, 33, 1028), 3)]


@pytest.fixture(scope="module")
def net_ops():
    from babe_b200 import build, net_ops
    build.build()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return net_ops


def _layers(shape, n_dils, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n, c = shape[:2]
    out = []
    for i in range(n_dils):
        gamma = 1 + 0.2 * torch.randn(1, c, 1, 1, device="cuda", generator=g)
        aff = 0.5 * torch.randn(n, c, device="cuda", generator=g)
        gate = torch.randn(n, c, device="cuda", generator=g)
        w = torch.randn(c, c, 5, 3, device="cuda", generator=g) / (c * 15) ** 0.5
        out.append((gamma, aff, gate, w, (2 ** i, 1)))
    return out, g


def _input(shape, g, misaligned=False):
    x = torch.randn(shape, device="cuda", generator=g) * 1.7 + 0.3
    if misaligned:                       # contiguous, but 4 bytes past a 16-byte boundary
        base = torch.empty(x.numel() + 1, device="cuda")
        base[1:].copy_(x.reshape(-1))
        x = base[1:].view(shape).detach()
    return x.requires_grad_(True)


def _reference64(x, layers):
    for gamma, aff, gate, w, dil in layers:
        n, c, f, t = x.shape
        xg = x.reshape(n, G, -1)
        h = (xg / (xg.std(-1, keepdim=True) + EPS)).reshape(n, c, f, t) * gamma.double()
        h = F.gelu(h * (aff.double()[:, :, None, None] + 1))
        x = (x + F.conv2d(h, w.double(), padding="same", dilation=dil) * gate.double()[:, :, None, None]) / 2 ** 0.5
    return x


@pytest.mark.parametrize("misaligned", [False, True])
@pytest.mark.parametrize("shape,n_dils", CASES)
def test_chain_matches_layers_and_fp64(net_ops, shape, n_dils, misaligned):
    if misaligned and shape[0] * shape[1] * shape[2] * shape[3] > 1 << 24:
        pytest.skip("alignment tail: small shapes only")
    layers, g = _layers(shape, n_dils, 1)
    x = _input(shape, g, misaligned)
    gy = torch.randn(shape, device="cuda", generator=g)
    y = net_ops.res_chain(x, layers, G, EPS)
    gx, = torch.autograd.grad(y, x, gy)
    yl = x
    for gamma, aff, gate, w, dil in layers:
        yl = net_ops.res_layer(yl, gamma, aff, gate, w, dil, G, EPS)
    gxl, = torch.autograd.grad(yl, x, gy)
    assert rel_l2(y, yl) <= 1e-6 and rel_l2(gx, gxl) <= 1e-6
    x64 = x.detach().double().requires_grad_(True)
    y64 = _reference64(x64, layers)
    gx64, = torch.autograd.grad(y64, x64, gy.double())
    assert rel_l2(y.double(), y64) <= 1e-5
    assert rel_l2(gx.double(), gx64) <= 1e-5


@pytest.mark.parametrize("shape", [(8, 96, 128, 1024), (3, 24, 7, 9), (2, 16, 33, 1025), (2, 16, 32, 100),
                                   (2, 16, 33, 1028)])
def test_fused_byproducts_match_standalone(net_ops, shape):
    g = torch.Generator(device="cuda").manual_seed(2)
    n, c = shape[:2]
    x0, v, gh, gy = (torch.randn(shape, device="cuda", generator=g) for _ in range(4))
    gate, gate_prev = torch.randn(n, c, device="cuda", generator=g), torch.randn(n, c, device="cuda", generator=g)
    gamma = 1 + 0.2 * torch.randn(c, device="cuda", generator=g)
    aff = 0.5 * torch.randn(n, c, device="cuda", generator=g)
    # epilogue statistics of gate_residual == gn_stats of the same output (fp64 sums in another partition)
    y, (st, _) = net_ops.gate_residual(x0, v, gate, groups=G)
    assert torch.equal(y, net_ops.gate_residual(x0, v, gate))
    ref, _ = net_ops.gn_stats(y, G)
    std = ref[:, 1]
    assert (st[:, 1] - std).abs().max() <= 1e-6 * std.min()
    assert ((st[:, 0] - ref[:, 0]).abs() <= 1e-6 * std).all()
    y64 = y.double().reshape(n, G, -1)
    assert torch.allclose(st[:, 0].double(), y64.mean(-1).reshape(-1), rtol=0, atol=1e-6 * std.min().item())
    assert torch.allclose(st[:, 1].double(), y64.std(-1).reshape(-1), rtol=1e-6, atol=0)
    # g_v written by the backward kernel == the standalone gate pass on its g_x, bit for bit
    rec = net_ops.gn_stats(x0, G)
    gx, gv = net_ops.gn_film_gelu_bwd(gh, x0, gy, *rec, gamma, aff, G, EPS, gate_prev=gate_prev)
    assert torch.equal(gx, net_ops.gn_film_gelu_bwd(gh, x0, gy, *rec, gamma, aff, G, EPS))
    assert torch.equal(gv, net_ops.gate_residual(None, gx, gate_prev))
    assert all(c.count_nonzero().item() == 0 for c in net_ops._COUNTERS.values())


def test_chain_bitwise_repeatable_and_graph_replay(net_ops):
    shape = (4, 64, 64, 512)
    layers, g = _layers(shape, 3, 3)
    x = _input(shape, g)
    gy = torch.randn(shape, device="cuda", generator=g)
    prev = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        def run():
            y = net_ops.res_chain(x, layers, G, EPS)
            gx, = torch.autograd.grad(y, x, gy)
            return y.detach(), gx

        y1, g1 = run()
        y2, g2 = run()
        assert torch.equal(y1, y2) and torch.equal(g1, g2)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            yg, gg = run()
        for _ in range(2):
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(yg, y1) and torch.equal(gg, g1)
    finally:
        torch.backends.cudnn.deterministic = prev
    assert all(c.count_nonzero().item() == 0 for c in net_ops._COUNTERS.values())
