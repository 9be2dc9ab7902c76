import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tools'))
from pointnet12_b200 import ops, synthetic as syn
from microbench import time_ms
dev = torch.device('cuda', 0)
B, N, S = 8, 24000, 1024
pts = torch.from_numpy(syn.kitti_batch(B, N, config=2)).to(dev)
xyz = pts.permute(0, 2, 1)[:, :, :3]
start = torch.zeros(B, dtype=torch.long, device=dev)
x1 = ops.index_points(xyz, ops.fps(xyz, S, start))
grid = ops.ball_grid(xyz, 0.1)
print("scan   ms", time_ms(lambda: ops.three_nn(xyz, x1, method="scan")))
print("blocks ms (ordered, incl. build)", time_ms(lambda: ops.three_nn(xyz, x1, order=grid, method="blocks")))
print("blocks ms (raw order, incl. build)", time_ms(lambda: ops.three_nn(xyz, x1, method="blocks")))
