import sys
sys.path.insert(0, ".")
import torch
from cqt_nsgt_pytorch import CQT_nsgt
from babe_b200._lib import lib
dev = torch.device("cuda")
cq = CQT_nsgt(7, 64, mode="oct", window=("kaiser", 1), fs=22050, audio_len=184184, device=dev)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
if len(sys.argv) > 2:
    assert lib().babe_set_cqt_band_variant(int(sys.argv[2])) == 0, "band variant: 1 (default) or 2"
xc = torch.randn(B, 184184, device=dev) * 0.063
for _ in range(2):
    cs = cq.fwd(xc.unsqueeze(1))
    y = cq.bwd(cs)
    z = cq.apply_hpf_DC(xc)
    cp = cq.fwd_planar(xc)
    yp = cq.bwd_planar(cp)
torch.cuda.synchronize()
print("ok")
