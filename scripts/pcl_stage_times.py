"""Per-kernel times of the PCL path on one B200: forward, backward-mid, backward-img, each timed alone over one
1024-image launch (2 crops per image), CUDA events.  Development aid; not the bench line."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hands_b200.step import GeometryStep  # noqa: E402


def cuda_time(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    st = GeometryStep(n, torch.device("cuda:0"), with_mano=False)
    st.pcl_setup()
    st.pcl_forward()
    st.pcl_backward()
    out = {"images": n,
           "fwd_us": cuda_time(st.pcl_forward),
           "mid_us": cuda_time(lambda: st.pcl_backward_stage(1)),
           "img_us": cuda_time(lambda: st.pcl_backward_stage(2))}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
