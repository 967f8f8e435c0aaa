import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, numpy as np
import bench
from torch.profiler import profile, ProfilerActivity
dev = torch.device('cuda:0')
from deeprecommendation_b200 import ops
ops.set_gemm_engine('tf32x3')
w = bench.build_attention(dev, 0, n_batches=2)
model = w['model']
res = [tuple(t.to(dev) for t in b) for b in w['host']]
model.train()
opt = torch.optim.Adam(model.parameters(), lr=1e-4)
y = torch.rand(512, 1, device=dev)
def step(i):
    opt.zero_grad(set_to_none=True)
    (model(*res[i % 2]) - y).square().sum().backward()
    opt.step()
for i in range(3): step(i)
torch.cuda.synchronize()
t0 = time.perf_counter()
for i in range(5): step(i)
torch.cuda.synchronize()
print('ms/step', (time.perf_counter() - t0) / 5 * 1e3)
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    for i in range(3): step(i)
    torch.cuda.synchronize()
print(prof.key_averages().table(sort_by='cuda_time_total', row_limit=25, max_name_column_width=70))
print(prof.key_averages().table(sort_by='self_cpu_time_total', row_limit=15, max_name_column_width=70))
