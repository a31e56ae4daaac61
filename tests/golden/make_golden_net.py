#!/usr/bin/env python
"""Golden vectors for the denoiser layer glue, produced by the UNMODIFIED reference modules
(networks/cqtdiff+.py: ResnetBlock :382-487 with BiasFreeGroupNorm :137-163, UpDownResample
:522-580).  Needs BABE_REFERENCE set to a checkout of eloimoliner/BABE:

    python tests/golden/make_golden_net.py        ->  tests/golden/net_glue.npz

The file imports the reference network module with a stub for the absent third-party
``cqt_nsgt_pytorch`` (only the classes named above are used; no transform is constructed).
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("BABE_REFERENCE") or sys.exit("set BABE_REFERENCE to a checkout of eloimoliner/BABE")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)
stub = types.ModuleType("cqt_nsgt_pytorch")
stub.CQT_nsgt = object
sys.modules.setdefault("cqt_nsgt_pytorch", stub)
ref = importlib.import_module("networks.cqtdiff+")


def main():
    torch.manual_seed(20260117)
    out = {}
    # --- one ResnetBlock with dim == dim_out (identity projections), two dilated layers -------------
    N, C, Fd, T, E = 2, 16, 12, 10, 8
    init = dict(init_mode='kaiming_uniform', init_weight=np.sqrt(1 / 3))
    blk = ref.ResnetBlock(C, C, use_norm=True, num_dils=2, bias=False, kernel_size=(5, 3), emb_dim=E,
                          proj_place='before', init=init, init_zero=init, attention_dict=None, Fdim=Fd)
    with torch.no_grad():
        for i in range(2):
            blk.norm[i].gamma.copy_(1 + 0.3 * torch.randn(1, C, 1, 1))
    x = (torch.randn(N, C, Fd, T) * 1.5 + 0.2).requires_grad_(True)
    emb = torch.randn(N, E)
    gy = torch.randn(N, C, Fd, T)
    y = blk(x, emb)
    gx, = torch.autograd.grad(y, x, gy)
    out.update(blk_x=x.detach(), blk_emb=emb, blk_gy=gy, blk_y=y.detach(), blk_gx=gx)
    for i in range(2):
        out[f"blk_gamma{i}"] = blk.norm[i].gamma.detach().reshape(-1)
        out[f"blk_aff{i}"] = blk.affine[i](emb).detach()
        out[f"blk_gate{i}"] = blk.gate[i](emb).detach()
        out[f"blk_w{i}"] = blk.H[i].weight.detach()
    # --- the norm alone ---------------------------------------------------------------------------
    out["norm_y"] = blk.norm[0](x).detach()
    # --- x2 resamplers ----------------------------------------------------------------------------
    for name, kw in (("down", dict(down=True)), ("up", dict(up=True))):
        rs = ref.UpDownResample(**kw)
        xr = torch.randn(2, 3, 4, 16, requires_grad=True)
        yr = rs(xr)
        g = torch.randn_like(yr)
        gxr, = torch.autograd.grad(yr, xr, g)
        out.update({f"rs_{name}_x": xr.detach(), f"rs_{name}_y": yr.detach(), f"rs_{name}_gy": g,
                    f"rs_{name}_gx": gxr})
    np.savez_compressed(os.path.join(HERE, "net_glue.npz"), **{k: v.numpy() for k, v in out.items()})
    print("wrote net_glue.npz:", {k: tuple(v.shape) for k, v in out.items()})


if __name__ == "__main__":
    main()
