import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from distributed_rl_b200 import replay as R
N = 1 << 20
rep = R.DeviceReplay(N, fields=(R.Field("a", torch.int32, ()),), device="cuda:0")
rep.build(torch.rand(N, device="cuda") + 0.01)
ui = torch.randint(0, N, (512,), device="cuda"); uv = torch.rand(512, device="cuda") + 0.01
for _ in range(4):
    rep.update(ui, uv)
x = torch.zeros(512, dtype=torch.int32, device="cuda")
for _ in range(3):
    rep.push([x], uv)
