import os, sys, json, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from pointnet12_b200 import ops, synthetic as syn
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from microbench import time_ms
dev = torch.device('cuda', 0)
B, npoint = 8, 1024
for cl, th, ex in [(8, 128, 2), (8, 128, 3), (4, 128, 2), (4, 256, 2), (8, 256, 2), (16, 128, 2)]:
    for N in [2048, 8192, 16384, 24000]:
        if N / cl / th > 32: continue
        pts = torch.from_numpy(syn.kitti_batch(B, N, config=2)).to(dev)
        xyz = pts.permute(0, 2, 1)[:, :, :3]
        start = torch.zeros(B, dtype=torch.long, device=dev)
        try:
            ops.fps_set_config(cl, th, ex)
            t = time_ms(lambda: ops.fps(xyz, npoint, start))
            print(json.dumps(dict(cl=cl, th=th, ex=ex, N=N, pts_per_thread=N / cl / th, us_per_iter=round(t * 1000 / npoint, 3))), flush=True)
        except RuntimeError as e:
            print(cl, th, N, str(e)[:80])
        finally:
            ops.fps_set_config(0, 0, 0)
