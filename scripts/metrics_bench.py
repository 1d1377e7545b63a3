"""Time hb_procrustes_metrics (PA / RA point errors as device partial sums) against a batched torch implementation on the
GPU (torch.linalg.svd) and the reference's way, a numpy SVD per sample on the host.

    python scripts/metrics_bench.py [--sizes 8192,65536] [--points 21,778] [--host-sample 512]

Kernel time: CUDA events around back-to-back launches on preallocated buffers, after a warm-up, over a window of at least
0.5 s.  Algorithmic bytes: the two (B,N,3) fp32 inputs (B*N*24) plus per-hand results, the (B,8) partial rows written
and read once, and the 8 sums.  The HBM share divides the achieved rate by a device-to-device copy measured in the same
run.  At N = 21 the inputs (4 MB at B = 8192) stay in the 126 MB L2 across launches, so that rate is not an HBM rate; at
N = 778 and B = 8192 they are 153 MB, larger than L2.  The host loop is timed on a bounded sample and scaled to B.
Prints one JSON object with the GPU name and power limit beside the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hands_b200 import _lib  # noqa: E402
from hands_b200.functional import _ptr, _stream  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power, clock = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers are still printed; the card is then named by torch only
        return {"name": torch.cuda.get_device_name(), "power_limit": None, "query_error": str(e)}


def timed(fn, min_window=0.5):
    """Seconds per call: warm-up, then back-to-back calls between two CUDA events over >= min_window seconds."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    reps = 1
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        dt = e0.elapsed_time(e1) * 1e-3
        if dt >= min_window:
            return dt / reps
        reps = max(reps * 2, int(reps * min_window * 1.2 / max(dt, 1e-6)))


def copy_bandwidth(dev):
    n = 1 << 30   # 4 GiB of fp32 each way
    a = torch.empty(n, device=dev).normal_()
    b = torch.empty_like(a)
    t = timed(lambda: b.copy_(a))
    del a, b
    torch.cuda.empty_cache()
    return 8 * n / t


def inputs(B, N, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    centre = torch.tensor([0.05, -0.1, 0.8], device=dev) + 0.2 * torch.randn(B, 1, 3, device=dev, generator=g)
    gt = centre + 0.04 * torch.randn(B, N, 3, device=dev, generator=g)
    pred = gt + 0.01 * torch.randn(B, N, 3, device=dev, generator=g)
    return pred.contiguous(), gt.contiguous()


def torch_batched(pred, gt):
    """compute_similarity_transform batched with torch on the GPU: PA and RA per hand (root = point 0)."""
    mu_p, mu_q = pred.mean(1, keepdim=True), gt.mean(1, keepdim=True)
    X, Y = pred - mu_p, gt - mu_q
    var = (X * X).sum((1, 2))
    C = X.transpose(1, 2) @ Y
    U, _, Vh = torch.linalg.svd(C)
    V = Vh.transpose(1, 2)
    Z = torch.eye(3, device=pred.device, dtype=pred.dtype).repeat(pred.shape[0], 1, 1)
    Z[:, 2, 2] = torch.sign(torch.det(U @ Vh))
    R = V @ Z @ U.transpose(1, 2)
    s = torch.diagonal(R @ C, dim1=1, dim2=2).sum(1) / var
    aligned = s[:, None, None] * X @ R.transpose(1, 2) + mu_q
    pa = (aligned - gt).norm(dim=2).mean(1)
    ra = ((pred - pred[:, :1]) - (gt - gt[:, :1])).norm(dim=2).mean(1)
    return pa, ra


def host_loop(pred, gt):
    """The reference's way: per sample on the host, one numpy SVD each (compute_similarity_transform)."""
    out = np.empty(len(pred))
    for b in range(len(pred)):
        p, q = pred[b], gt[b]
        mu_p, mu_q = p.mean(0), q.mean(0)
        X, Y = p - mu_p, q - mu_q
        U, _, Vt = np.linalg.svd(X.T @ Y)
        Z = np.eye(3)
        Z[2, 2] = np.sign(np.linalg.det(U @ Vt))
        R = Vt.T @ Z @ U.T
        s = np.trace(R @ X.T @ Y) / (X * X).sum()
        out[b] = np.linalg.norm(s * p @ R.T + (mu_q - s * R @ mu_p) - q, axis=1).mean()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="8192,65536")
    ap.add_argument("--points", default="21,778")
    ap.add_argument("--host-sample", type=int, default=512)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    res = {"gpu": gpu_info(), "copy_GBs": copy_bandwidth(dev) / 1e9, "runs": []}
    for N in [int(x) for x in args.points.split(",")]:
        for B in [int(x) for x in args.sizes.split(",")]:
            pred, gt = inputs(B, N, dev)
            partial = torch.empty(B, _lib.KP_SUMS, device=dev)
            sums = torch.empty(_lib.KP_SUMS, device=dev)
            per_hand = torch.empty(B, 2, device=dev)

            def kernel():
                _lib.check(lib.hb_procrustes_metrics(_ptr(pred), _ptr(gt), B, N, None, None, None, _ptr(per_hand), None, _ptr(partial), _ptr(sums),
                                                     _stream()), "hb_procrustes_metrics")

            t_k = timed(kernel)
            nbytes = B * N * 24 + B * 8 + 2 * B * _lib.KP_SUMS * 4 + _lib.KP_SUMS * 4
            t_t = timed(lambda: torch_batched(pred, gt))
            pa_t, _ = torch_batched(pred, gt)
            kernel()
            agree = float(((per_hand[:, 0] - pa_t).abs() / pa_t).max())
            n = min(args.host_sample, B)
            p_h, g_h = pred[:n].double().cpu().numpy(), gt[:n].double().cpu().numpy()
            t0 = time.perf_counter()
            host_loop(p_h, g_h)
            t_h = (time.perf_counter() - t0) / n * B
            rate = nbytes / t_k
            res["runs"].append({"B": B, "N": N, "kernel_us": t_k * 1e6, "alg_bytes": nbytes, "GBs": rate / 1e9,
                                "share_of_copy_bw": rate / (res["copy_GBs"] * 1e9), "inputs_exceed_L2": B * N * 24 > 126e6,
                                "torch_svd_us": t_t * 1e6, "speedup_vs_torch": t_t / t_k,
                                "host_numpy_loop_s_scaled": t_h, "host_sample": n, "max_rel_diff_pa_vs_torch_fp32": agree})
            del pred, gt, partial, per_hand
            torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
