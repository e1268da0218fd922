import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from unidefense_b200 import ops
g = torch.Generator().manual_seed(0)
x = (torch.rand(32, 3, 380, 380, generator=g) * 2 - 1).cuda()
st = x.flip(0).contiguous()
lm = (torch.rand(32, generator=g) / 2 + 0.5).cuda()
mk = torch.rand(32, 380, 191, generator=g).cuda()
for _ in range(2):
    y = ops.spatial_style_transfer(x, st, lm)
    z = ops.spectral_mask_filter(x, mk)
torch.cuda.synchronize()
print("ok", float(y.mean()), float(z.mean()))
