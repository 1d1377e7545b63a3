"""Crop-layer backward under compute-sanitizer (memcheck / racecheck): gather form (tile-row CTAs), two and three crops per
image, a whole-image box and a short focal length.
    compute-sanitizer --tool racecheck python scripts/sanitize_pcl_bwd.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hands_b200 import _lib
from hands_b200.pcl import perspective_crop
from hands_b200.synthetic import synthetic_pcl_inputs
dev = torch.device("cuda:0")
lib = _lib.load()
for cpi in (2, 3):
    B = 2
    n = B * cpi
    img, bbox, K = synthetic_pcl_inputs(n, seed=cpi, img_res=224, smin=40, smax=200)
    img = img[:B].contiguous()
    bbox[0] = torch.tensor([0, 0, 223, 223])
    K[1, 0, 0] = 120.0; K[1, 1, 1] = 130.0
    x = img.to(dev).requires_grad_(True)
    crop, rot = perspective_crop(x, bbox.to(dev), K.to(dev), img_res=224, crops_per_img=cpi)
    crop.sum().backward()
torch.cuda.synchronize()
print("done")
