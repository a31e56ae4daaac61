"""CQTDiff+ denoiser body (PyTorch) around the CUDA constant-Q transform.

The convolutional U-Net is OUT OF SCOPE of the hand-written kernels ("the
denoiser's convolutions stay in PyTorch", BASELINE.json); it is restated here
only because the sampler benchmark needs the named model on machines where the
reference tree does not exist.  Architecture, constructor order (hence the
random initialisation under a fixed seed) and state-dict keys follow
``networks/cqtdiff+.py`` (Unet_CQT_oct_with_attention, :583-845), so a reference
state dict LOADS key for key (tests/test_denoiser_cpu.py, tests/test_integration_*.py).  Whether pretrained
weights then BEHAVE as trained depends on the constant-Q transform around the body: upstream's
``cqt_nsgt_pytorch`` is not available offline and the in-repo transform follows its own specification
(oracle/nsgt.py, parity unpinned) -- validate a checkpoint before relying on it.  Attention layers (all
disabled in conf/network/cqtdiff+.yaml:27) are not implemented.

Execution differences that do not change the mathematics: the x2 time
resamplers run as single-channel FIR convolutions instead of rebuilding a dense
diagonal CxCx8 weight per call (networks/cqtdiff+.py:564-570).
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import net_ops


def _init(shape, mode, fan_in, fan_out):
    """networks/cqtdiff+.py:21-26."""
    if mode == 'xavier_uniform':
        return np.sqrt(6 / (fan_in + fan_out)) * (torch.rand(*shape) * 2 - 1)
    if mode == 'xavier_normal':
        return np.sqrt(2 / (fan_in + fan_out)) * torch.randn(*shape)
    if mode == 'kaiming_uniform':
        return np.sqrt(3 / fan_in) * (torch.rand(*shape) * 2 - 1)
    if mode == 'kaiming_normal':
        return np.sqrt(1 / fan_in) * torch.randn(*shape)
    raise ValueError(f'Invalid init mode "{mode}"')


FUSED = True          # use the fused CUDA glue (net_ops) when the parameters are frozen


def _add_scale(a, b):
    """(a + b) / sqrt(2)"""
    if FUSED and a.shape == b.shape and net_ops.usable(a) and b.is_cuda and b.dtype == torch.float32:
        return net_ops.add_scale(a, b)
    return (a + b) / (2 ** 0.5)


class Linear(nn.Module):
    """networks/cqtdiff+.py:28-42."""

    def __init__(self, in_features, out_features, bias=True, init_mode='kaiming_normal',
                 init_weight=1, init_bias=0):
        super().__init__()
        kw = dict(mode=init_mode, fan_in=in_features, fan_out=out_features)
        self.weight = nn.Parameter(_init([out_features, in_features], **kw) * init_weight)
        self.bias = nn.Parameter(_init([out_features], **kw) * init_bias) if bias else None

    def forward(self, x):
        return F.linear(x, self.weight, self.bias)


class Conv2d(nn.Module):
    """networks/cqtdiff+.py:66-88: bias-free 'same' convolution, dilated in frequency."""

    def __init__(self, in_channels, out_channels, kernel=(1, 1), bias=False, dilation=1,
                 init_mode='kaiming_normal', init_weight=1, init_bias=0):
        super().__init__()
        self.dilation = dilation
        kw = dict(mode=init_mode, fan_in=in_channels * kernel[0] * kernel[1],
                  fan_out=out_channels * kernel[0] * kernel[1])
        self.weight = nn.Parameter(_init([out_channels, in_channels, kernel[0], kernel[1]], **kw) * init_weight)
        self.bias = nn.Parameter(_init([out_channels], **kw) * init_bias) if bias else None

    def forward(self, x):
        if FUSED and self.bias is None and net_ops.usable(x, self.weight) and x.requires_grad \
                and self.weight.shape[2] % 2 == 1 and self.weight.shape[3] % 2 == 1:
            return net_ops.conv_frozen(x, self.weight, self.dilation)
        return F.conv2d(x, self.weight, self.bias, padding="same", dilation=self.dilation)


class BiasFreeGroupNorm(nn.Module):
    """networks/cqtdiff+.py:137-163: divide by the group's (unbiased) standard
    deviation, no mean removal, learned per-channel gain."""

    def __init__(self, num_features, num_groups=32, eps=1e-7):
        super().__init__()
        self.gamma = nn.Parameter(torch.ones(1, num_features, 1, 1))
        self.num_groups, self.eps = num_groups, eps

    def forward(self, x):
        n, c, f, t = x.shape
        xg = x.reshape(n, self.num_groups, -1)
        xg = xg / (xg.std(-1, keepdim=True) + self.eps)
        return xg.reshape(n, c, f, t) * self.gamma


class RFF_MLP_Block(nn.Module):
    """networks/cqtdiff+.py:167-209: random Fourier features of the noise level + MLP."""

    def __init__(self, emb_dim=512, rff_dim=32, init=None):
        super().__init__()
        self.RFF_freq = nn.Parameter(16 * torch.randn([1, rff_dim]), requires_grad=False)
        self.MLP = nn.ModuleList([Linear(2 * rff_dim, 128, **init), Linear(128, 256, **init),
                                  Linear(256, emb_dim, **init)])

    def forward(self, sigma):
        table = 2 * np.pi * sigma * self.RFF_freq
        x = torch.cat([torch.sin(table), torch.cos(table)], dim=1)
        for layer in self.MLP:
            x = F.relu(layer(x))
        return x


class ResnetBlock(nn.Module):
    """networks/cqtdiff+.py:382-487 without the attention branch."""

    def __init__(self, dim, dim_out, use_norm=True, num_dils=6, bias=False, kernel_size=(5, 3),
                 emb_dim=512, proj_place='before', init=None, init_zero=None, attention_dict=None,
                 Fdim=128):
        super().__init__()
        if attention_dict is not None:
            raise NotImplementedError("time attention is disabled in conf/network/cqtdiff+.yaml:27 "
                                      "and not implemented here")
        if not use_norm:
            raise NotImplementedError("use_norm=False breaks the reference's forward (zip over self.norm)")
        self.proj_place = proj_place
        N = dim_out if proj_place == 'before' else dim
        if proj_place != 'before':
            self.proj_out = Conv2d(N, dim_out, bias=bias, **init) if N != dim_out else nn.Identity()
        self.res_conv = Conv2d(dim, dim_out, bias=bias, **init) if dim != dim_out else nn.Identity()
        self.proj_in = Conv2d(dim, N, bias=bias, **init) if dim != N else nn.Identity()
        self.H, self.affine, self.gate, self.norm = nn.ModuleList(), nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        for i in range(num_dils):
            self.norm.append(BiasFreeGroupNorm(N, 8))
            self.affine.append(Linear(emb_dim, N, **init))
            self.gate.append(Linear(emb_dim, N, **init_zero))
            self.H.append(Conv2d(N, N, kernel=kernel_size, dilation=(2 ** i, 1), bias=bias, **init))

    def forward(self, input_x, sigma):
        x = self.proj_in(input_x)
        layers = list(zip(self.norm, self.affine, self.gate, self.H))
        norm0 = self.norm[0]
        if FUSED and all(n.num_groups == norm0.num_groups and n.eps == norm0.eps for n in self.norm) and \
                all(net_ops.usable(x, norm.gamma, conv.weight, affine.weight, gate.weight, sigma)
                    for norm, affine, gate, conv in layers):
            # csrc/net_ops.cu: at most 3 launches around each convolution instead of ~8 PyTorch kernels
            x = net_ops.res_chain(x, [(norm.gamma, affine(sigma), gate(sigma), conv.weight, conv.dilation)
                                      for norm, affine, gate, conv in layers], norm0.num_groups, norm0.eps)
        else:
            for norm, affine, gate, conv in layers:
                x0 = x
                x = norm(x) * (affine(sigma)[:, :, None, None] + 1)
                x = (x0 + conv(F.gelu(x)) * gate(sigma)[:, :, None, None]) / (2 ** 0.5)
        if self.proj_place == 'after':
            x = self.proj_out(x)
        return _add_scale(x, self.res_conv(input_x))


_CUBIC = [-0.01171875, -0.03515625, 0.11328125, 0.43359375,
          0.43359375, 0.11328125, -0.03515625, -0.01171875]     # networks/cqtdiff+.py:505-507


class UpDownResample(nn.Module):
    """networks/cqtdiff+.py:522-580 (mode 'T', cubic filter, reflect padding): anti-aliased x2
    resampling along time, every (channel, frequency) row filtered independently."""

    def __init__(self, up=False, down=False):
        super().__init__()
        assert up != down
        self.up, self.down = up, down
        self.register_buffer('kernel', torch.tensor(_CUBIC, dtype=torch.float32))
        self.pad = len(_CUBIC) // 2 - 1

    def forward(self, x):
        c = x.shape[1]
        if FUSED and x.is_cuda and x.dtype == torch.float32 and x.shape[-1] % 2 == 0 \
                and x.shape[-1] >= len(_CUBIC):
            return net_ops.resample2(x, _CUBIC, self.up)    # csrc/net_ops.cu: pad + FIR in one pass
        # depthwise (1 x 8) convolution along time: one FIR per (channel, frequency) row
        w = self.kernel.to(x.dtype)[None, None, None, :].expand(c, 1, 1, -1)
        if self.down:
            return F.conv2d(F.pad(x, (self.pad, self.pad, 0, 0), 'reflect'), w, stride=(1, 2), groups=c)
        p = (self.pad + 1) // 2
        return F.conv_transpose2d(F.pad(x, (p, p, 0, 0), 'reflect'), w, stride=(1, 2),
                                  padding=(0, self.pad * 2 + 1), groups=c)


class CQTDiffPlus(nn.Module):
    """networks/cqtdiff+.py:583-845.  ``forward(inputs[B,T], sigma[B,1]) -> [B,T]``; the attribute
    ``CQTransform`` is used directly by the samplers (testing/blind_bwe_sampler.py:156)."""

    def __init__(self, args, device, cqt=None):
        super().__init__()
        net = args.network
        self.args = args
        self.depth = self.num_octs = net.cqt.num_octs
        self.bins_per_oct = net.cqt.bins_per_oct
        init = dict(init_mode='kaiming_uniform', init_weight=np.sqrt(1 / 3))
        init_zero = dict(init_mode='kaiming_uniform', init_weight=1e-7)
        self.emb_dim = net.emb_dim
        self.embedding = RFF_MLP_Block(emb_dim=net.emb_dim, init=init)
        self.use_norm = net.use_norm
        if net.use_fencoding:
            raise NotImplementedError("use_fencoding is False in conf/network/cqtdiff+.yaml:8")
        win = ("kaiser", net.cqt.beta) if net.cqt.window == "kaiser" else net.cqt.window
        if cqt is None:
            from cqt_nsgt_pytorch import CQT_nsgt
            cqt = CQT_nsgt(self.num_octs, self.bins_per_oct, mode="oct", window=win,
                           fs=args.exp.sample_rate, audio_len=args.exp.audio_len,
                           dtype=torch.float32, device=device)
        self.CQTransform = cqt
        Ns, dils = net.Ns, net.num_dils
        if any(net.attention_layers):
            raise NotImplementedError("attention layers")
        self.downsamplerT = UpDownResample(down=True)
        self.upsamplerT = UpDownResample(up=True)
        self.downs, self.middle, self.ups = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        common = dict(emb_dim=self.emb_dim, init=init, init_zero=init_zero, bias=False)
        for i in range(self.num_octs):
            dim_in = Ns[0] if i == 0 else Ns[i - 1]
            dim_out = Ns[i]
            self.downs.append(nn.ModuleList([
                ResnetBlock(2, dim_in, self.use_norm, num_dils=1, kernel_size=(1, 1), **common),
                Conv2d(2, dim_out, kernel=(5, 3), bias=False, **init),
                ResnetBlock(dim_in, dim_out, self.use_norm, num_dils=dils[i],
                            Fdim=(i + 1) * self.bins_per_oct, **common)]))
        if net.bottleneck_type != "res_dil_convs":
            raise NotImplementedError("bottleneck type not implemented")
        for i in range(net.num_bottleneck_layers):
            self.middle.append(nn.ModuleList([
                ResnetBlock(Ns[-1], 2, use_norm=self.use_norm, num_dils=1, kernel_size=(1, 1),
                            proj_place="after", **common),
                ResnetBlock(Ns[-1], Ns[-1], self.use_norm, num_dils=dils[-1],
                            Fdim=self.num_octs * self.bins_per_oct, **common)]))
        for i in range(self.num_octs - 1, -1, -1):
            dim_in = Ns[i] * 2
            dim_out = Ns[0] if i == 0 else Ns[i - 1]
            self.ups.append(nn.ModuleList([
                ResnetBlock(dim_out, 2, use_norm=self.use_norm, num_dils=1, kernel_size=(1, 1),
                            proj_place="after", **common),
                ResnetBlock(dim_in, dim_out, use_norm=self.use_norm, num_dils=dils[i],
                            Fdim=(i + 1) * self.bins_per_oct, **common)]))

    def forward(self, inputs, sigma):
        emb = self.embedding(sigma)
        # the CUDA transform emits / consumes the planar (B,2,F,T) layout directly, which removes the
        # 14 transposing copies per evaluation of networks/cqtdiff+.py:750-753 and :826-830
        planar = hasattr(self.CQTransform, "fwd_planar")
        if planar:
            octaves = self.CQTransform.fwd_planar(inputs)            # lowest octave first
        else:
            octaves = self.CQTransform.fwd(inputs.unsqueeze(1))
        out_octaves = [None] * self.num_octs
        hs = []
        X = pyr = None
        last = self.num_octs - 1
        for i, (init_block, pyr_proj, res_block) in enumerate(self.downs):
            # octave consumed from the top: complex (B,1,F,T) -> planar (B,2,F,T)
            if planar:
                C = octaves[-1 - i]
            else:
                C = torch.view_as_real(octaves[-1 - i].squeeze(1)).permute(0, 3, 1, 2).contiguous()
            C2 = init_block(C, emb)
            if i == 0:
                X, pyr = C2, self.downsamplerT(C)
            elif i < last:
                pyr = torch.cat((self.downsamplerT(C), self.downsamplerT(pyr)), dim=2)
                X = torch.cat((C2, X), dim=2)
            else:
                pyr = torch.cat((C, pyr), dim=2)
                X = torch.cat((C2, X), dim=2)
            X = res_block(X, emb)
            hs.append(X)
            if i < last:
                X = self.downsamplerT(X)
            X = _add_scale(X, pyr_proj(pyr))
        for out_block, res_block in self.middle:
            X = res_block(X, emb)
            Xout = out_block(X, emb)
        for i, (out_block, res_block) in enumerate(self.ups):
            j = len(self.ups) - i - 1
            X = res_block(torch.cat((X, hs.pop()), dim=1), emb)
            Xout = _add_scale(Xout, out_block(X, emb))
            X = X[:, :, self.bins_per_oct:, :]
            Out, Xout = Xout[:, :, :self.bins_per_oct, :], Xout[:, :, self.bins_per_oct:, :]
            if planar:
                out_octaves[i] = Out.contiguous()
            else:
                out_octaves[i] = torch.view_as_complex(Out.permute(0, 2, 3, 1).contiguous()).unsqueeze(1)
            if j > 0:
                X = self.upsamplerT(X)
                Xout = self.upsamplerT(Xout)
        if planar:
            pred = self.CQTransform.bwd_planar(out_octaves)[:, :inputs.shape[-1]]
        else:
            pred = self.CQTransform.bwd(out_octaves).squeeze(1)[:, :inputs.shape[-1]]
        assert pred.shape == inputs.shape, "bad shapes"
        return pred


# name used by conf/network/cqtdiff+.yaml:5
Unet_CQT_oct_with_attention = CQTDiffPlus
