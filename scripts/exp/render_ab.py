"""C4 render frame (1920x1080, 64 + 64 samples, 131072-ray chunks); prints ms/frame.
Usage: python scripts/exp/render_ab.py"""
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from nerfpp_b200.pipeline import HashNeRF  # noqa: E402

BBOX = [-1.5, -1.5, -1.5, 1.5, 1.5, 1.5]
m = HashNeRF(BBOX, seed=42)
H, W = 1080, 1920
focal = 0.5 * W / math.tan(0.5 * 0.6911)
K = [[focal, 0, 0.5 * W], [0, focal, 0.5 * H], [0, 0, 1]]
c2w = torch.eye(4)
c2w[2, 3] = 4.0
m.render_image(H, W, K, c2w, chunk=131072, n_importance=64)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(3):
    m.render_image(H, W, K, c2w, chunk=131072, n_importance=64)
e1.record()
torch.cuda.synchronize()
print(json.dumps({"env": {k: v for k, v in os.environ.items() if k.startswith("NRF_")}, "ms_per_frame": e0.elapsed_time(e1) / 3}))
