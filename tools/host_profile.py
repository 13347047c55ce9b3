import cProfile, pstats, sys, io, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vit_adapter_b200 as vab
from vit_adapter_b200.adapter import InteractionBlock, deform_inputs
dev = torch.device('cuda', 0)
blk = InteractionBlock(768, 12, 4, deform_ratio=0.5, cffn_ratio=0.25, init_values=0.0, extra_extractor=False).to(dev)
vab.set_amp_value_dtype(torch.bfloat16)
img = torch.zeros(2, 3, 512, 512, device=dev)
di1, di2 = deform_inputs(img)
h = 32
x = torch.randn(2, h * h, 768, device=dev, requires_grad=True)
c = torch.randn(2, 21 * (h // 2) ** 2, 768, device=dev, requires_grad=True)
def step():
    with torch.autocast('cuda', dtype=torch.bfloat16):
        xo, co = blk(x, c, [], di1, di2, h, h)
    (xo.float().square().sum() + co.float().square().sum()).backward()
for _ in range(5): step()
torch.cuda.synchronize()
import time
t0 = time.perf_counter()
for _ in range(50): step()
torch.cuda.synchronize()
print('wall per step ms', (time.perf_counter() - t0) / 50 * 1e3)
pr = cProfile.Profile(); pr.enable()
for _ in range(50): step()
torch.cuda.synchronize()
pr.disable()
s = io.StringIO(); pstats.Stats(pr, stream=s).sort_stats('tottime').print_stats(28); print(s.getvalue()[:6000])
