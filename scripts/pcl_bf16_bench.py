"""Time the crop layer with bf16 crop planes against the fp32 crop layer and against the cast a bf16 consumer would
otherwise run, at the benchmark's size (8192 source images x 2 crops of 3x224x224, boxes as in GeometryStep).

    python scripts/pcl_bf16_bench.py [--samples 8192] [--rounds 3] [--window 0.5] [--out FILE]

1. crop forward:  fp32 | fp32 + cast to bf16 | bf16 (fp32 source) | fp32 (uint8 source) | bf16 (uint8 source)
2. crop backward: fp32 on an fp32 gradient | cast bf16 -> fp32 + fp32 | bf16
3. the fused GeometryStep as a CUDA-graph replay, fp32 crops vs bf16 crops, and the peak memory of each step

Each number is CUDA events around back-to-back calls on preallocated buffers over a window of >= --window seconds, after a
warm-up; the variants of a group alternate round by round and the median over the rounds is reported.  The working set
(several GB per buffer) is far larger than the 126 MB L2.  The cast is `dst.copy_(src)` into a preallocated buffer, the
same elementwise kernel autocast's `_to_copy` runs, without the allocation.  Prints one JSON object with the GPU name and
its power limit beside the numbers."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hands_b200 import _lib  # noqa: E402
from hands_b200.functional import _ptr, _stream  # noqa: E402
from hands_b200.synthetic import synthetic_pcl_inputs  # noqa: E402

R, C, CPI = 224, 3, 2
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power, clock = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers are still printed; the card is then named by torch only
        return {"name": torch.cuda.get_device_name(), "power_limit": None, "query_error": str(e)}


def timed(fn, min_window):
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


def alternate(variants, rounds, window):
    """variants: {name: fn}; every round times each variant once, in order; returns {name: (median us, [us per round])}"""
    runs = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            runs[k].append(timed(fn, window) * 1e6)
    return {k: {"us": round(statistics.median(v), 1), "rounds_us": [round(x, 1) for x in v]} for k, v in runs.items()}


def kernels(S, rounds, window, dev):
    lib = _lib.load()
    n = S * CPI
    _, bbox, K = synthetic_pcl_inputs(n, seed=0, img_res=R, smin=R // 4, smax=3 * R // 4)   # GeometryStep's boxes
    bbox, K = bbox.to(dev), K.to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    img = torch.randn(S, C, R, R, generator=g, device=dev)
    img8 = torch.randint(0, 256, (S, C, R, R), generator=g, device=dev, dtype=torch.uint8)
    params = torch.empty(n, _lib.PCL_PARAM_FLOATS, device=dev)
    rot = torch.empty(n, 3, 3, device=dev)
    _lib.check(lib.hb_pcl_setup(_ptr(bbox), _ptr(K), n, R, _ptr(params), _ptr(rot), _stream()), "hb_pcl_setup")
    crop32 = torch.empty(n, C, R, R, device=dev)
    crop16 = torch.empty(n, C, R, R, dtype=torch.bfloat16, device=dev)
    m = ctypes.cast((ctypes.c_float * 3)(*MEAN), ctypes.c_void_p)
    s = ctypes.cast((ctypes.c_float * 3)(*STD), ctypes.c_void_p)

    def chk(rc, what):
        if rc:
            _lib.check(rc, what)

    fwd = {
        "fp32": lambda: chk(lib.hb_pcl_fwd(_ptr(img), _ptr(params), n, CPI, C, R, _ptr(crop32), _stream()), "hb_pcl_fwd"),
        "fp32+cast_to_bf16": lambda: (chk(lib.hb_pcl_fwd(_ptr(img), _ptr(params), n, CPI, C, R, _ptr(crop32), _stream()), "hb_pcl_fwd"), crop16.copy_(crop32)),
        "bf16": lambda: chk(lib.hb_pcl_fwd_bf16(_ptr(img), _ptr(params), n, CPI, C, R, _ptr(crop16), _stream()), "hb_pcl_fwd_bf16"),
        "u8_fp32": lambda: chk(lib.hb_pcl_fwd_u8(_ptr(img8), m, s, _ptr(params), n, CPI, C, R, _ptr(crop32), _stream()), "hb_pcl_fwd_u8"),
        "u8_bf16": lambda: chk(lib.hb_pcl_fwd_u8_bf16(_ptr(img8), m, s, _ptr(params), n, CPI, C, R, _ptr(crop16), _stream()), "hb_pcl_fwd_u8_bf16"),
    }
    res = {"forward": alternate(fwd, rounds, window)}
    # the bf16 crop is the rounded fp32 crop (checked on the timed buffers)
    lib.hb_pcl_fwd(_ptr(img), _ptr(params), n, CPI, C, R, _ptr(crop32), _stream())
    lib.hb_pcl_fwd_bf16(_ptr(img), _ptr(params), n, CPI, C, R, _ptr(crop16), _stream())
    res["forward_bf16_equals_rounded_fp32"] = bool(torch.equal(crop16.view(torch.int16), crop32.to(torch.bfloat16).view(torch.int16)))
    del crop32, img8
    g16 = crop16.normal_(generator=g)   # the crop buffer is reused as the bf16 gradient
    g32 = torch.empty(n, C, R, R, device=dev)
    g32.copy_(g16)
    g_img = torch.empty(S, C, R, R, device=dev)
    ws_bytes = lib.hb_pcl_bwd_workspace_bytes(n, CPI, C, R)
    ws = torch.empty((ws_bytes + 3) // 4, device=dev)
    g32c = torch.empty_like(g32)
    bwd = {
        "fp32": lambda: chk(lib.hb_pcl_bwd(_ptr(g32), _ptr(params), n, CPI, C, R, _ptr(g_img), _ptr(ws), ws_bytes, _stream()), "hb_pcl_bwd"),
        "cast_to_fp32+fp32": lambda: (g32c.copy_(g16), chk(lib.hb_pcl_bwd(_ptr(g32c), _ptr(params), n, CPI, C, R, _ptr(g_img), _ptr(ws), ws_bytes, _stream()), "hb_pcl_bwd")),
        "bf16": lambda: chk(lib.hb_pcl_bwd_bf16(_ptr(g16), _ptr(params), n, CPI, C, R, _ptr(g_img), _ptr(ws), ws_bytes, _stream()), "hb_pcl_bwd_bf16"),
    }
    res["backward"] = alternate(bwd, rounds, window)
    ref = g_img.clone()
    lib.hb_pcl_bwd(_ptr(g32), _ptr(params), n, CPI, C, R, _ptr(ref), _ptr(ws), ws_bytes, _stream())
    lib.hb_pcl_bwd_bf16(_ptr(g16), _ptr(params), n, CPI, C, R, _ptr(g_img), _ptr(ws), ws_bytes, _stream())
    res["backward_bf16_equals_fp32_on_widened"] = bool(torch.equal(ref, g_img))
    plane = n * C * R * R
    res["cast_bytes_per_pass"] = plane * 6   # read 4 + write 2 (or read 2 + write 4) per element
    return res


def step(S, rounds, window, dev):
    from hands_b200.step import GeometryStep

    out, steps = {}, {}
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        st = GeometryStep(S, dev, seed=0, crop_dtype=dt)
        launches = st.capture()
        st.replay()
        torch.cuda.synchronize()
        out[name] = {"launches_per_replay": launches, "peak_bytes": torch.cuda.max_memory_allocated(dev) - base,
                     "bytes_per_sample": st.bytes_per_sample()}
        steps[name] = st
    t = alternate({k: st.replay for k, st in steps.items()}, rounds, window)
    for k in out:
        out[k].update(t[k])
        out[k]["ms"] = round(out[k]["us"] / 1e3, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=8192)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--window", type=float, default=0.5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pcl_bf16_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "samples": a.samples, "crops": a.samples * CPI, "img_res": R, "rounds": a.rounds, "window_s": a.window}
    res.update(kernels(a.samples, a.rounds, a.window, dev))
    torch.cuda.empty_cache()
    res["step_graph"] = step(a.samples, a.rounds, a.window, dev)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
