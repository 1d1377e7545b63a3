#!/usr/bin/env python
"""bench.py -- hands/s of the fused geometry step (MANO + LBS + PCL + projection, fwd+bwd) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--samples S] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], the one the metric is quoted on, as one GPU's shard):
two hands (left+right MANO constants) + 2 PCL crops per sample sharing one source image + projection,
8192 samples per GPU (65,536 samples at 8 GPUs, weak scaling), synthetic inputs, random-init
MANO-shaped constants.  One step = one forward+backward pass over the GPU's shard.

Prints ONE JSON line (rank 0).  `value` = hands/s with inputs resident in HBM; `e2e` = the same step
with host buffers (pinned H2D of the step's inputs, D2H of the per-hand gradients) in the timed region;
`roofline` = the dominant kernel timed alone; `cpu_baseline` = the oracle (reference torch CPU path)
on the host cores for a bounded sample.  `--impl reference` times only that CPU path.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "hands/sec MANO+LBS+PCL fwd+bwd"
UNIT = "hands/s"
IMG_RES = 224
HANDS_PER_SAMPLE = 2
A_MANO = 31068.0            # algorithmic bytes per hand, MANO head fwd+bwd (SURVEY.md §8(d))


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference CPU path (the oracle), one bounded step
WORKLOAD = "C4 two-hand (left+right MANO) + 2 PCL crops/sample sharing one source image + projection, fwd+bwd"


# ------------------------------------------------------------------------------------------------
def cpu_baseline_variants(samples, steps, warmup, want_pool=True):
    """The reference torch CPU path (oracle) on the host cores, several ways (scripts/bench_legs.py):
      per_sample_loop_all_threads   the reference's per-sample crop loop + batched MANO heads, torch intra-op threads = all cores
      per_sample_loop_1_thread      the same on one thread (bounded to a quarter of the sample)
      worker_pool                   one single-threaded process per core for the crops (the reference's DataLoader-worker
                                    parallelism) while the parent runs the MANO heads on all threads
      batched_fixed_s               ONE grid_sample + ONE interpolate for the batch (only possible at a single box size:
                                    an upper bound for a batched CPU rewrite, not the reference's code)
    Returns (best hands/s among the first three, dict)."""
    from scripts import bench_legs as L

    cores = os.cpu_count() or 1
    out = {}
    v, dt = L.cpu_loop_all_threads(samples, steps, warmup)
    out["per_sample_loop_all_threads"] = {"value": v, "ms_per_step": dt * 1e3, "cores": cores, "samples": samples}
    s1 = max(2, samples // 4)
    v1, dt1 = L.cpu_loop_one_thread(s1)
    out["per_sample_loop_1_thread"] = {"value": v1, "ms_per_step": dt1 * 1e3, "cores": 1, "samples": s1}
    if want_pool:
        r = L.cpu_worker_pool(samples, steps, warmup)
        if r is not None:
            out["worker_pool"] = {"value": r[0], "ms_per_step": r[1] * 1e3, "cores": cores, "workers": r[2], "samples": samples}
    vb, dtb = L.cpu_batched(samples, steps, warmup)
    out["batched_fixed_s"] = {"value": vb, "ms_per_step": dtb * 1e3, "cores": cores, "samples": samples, "s": 112}
    best = max((k for k in out if k != "batched_fixed_s"), key=lambda k: out[k]["value"] if k != "per_sample_loop_1_thread" else -1.0)
    return best, out


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's threads (and therefore the first touch of its pinned host buffers) to the NUMA node its GPU hangs off:
    with 8 ranks copying 1.2 GB/step each, host buffers on the wrong socket halve the aggregate H2D rate.  Best effort: a
    box that hides its topology (node -1, one node) is left alone.  Returns what was done, for the JSON line."""
    info = {"gpu_numa_node": None, "bound": False}
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        info["gpu_numa_node"] = node
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        info["host_numa_nodes"] = len(nodes)
        if node < 0 or len(nodes) < 2:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info["bound"], info["cpus"] = True, len(cpus)
    except Exception as exc:   # topology not readable: leave the scheduler alone
        info["error"] = str(exc)[:80]
    return info


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    samples = args.ref_samples
    best, var = cpu_baseline_variants(samples, max(1, args.steps), max(1, args.warmup))
    hps, dt = var[best]["value"], var[best]["ms_per_step"] * 1e-3
    cores = os.cpu_count() or 1
    line = {
        "impl": "reference", "metric": METRIC, "value": hps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "arm": "reference torch ops on the host CPU (oracle), bounded sample of the same workload; best of the "
                   "all-thread per-sample loop and the one-process-per-core crop workers",
                   "samples_per_step": samples, "hands_per_sample": HANDS_PER_SAMPLE, "img_res": IMG_RES, "bbox_side": "U{56..168}",
                   "grads_on": ["v3d.cam", "j3d.cam", "j2d.norm", "crops"]},
        "cpu_baseline": {"value": hps, "unit": UNIT, "cores": cores, "kind": "port", "cpu": cpu_model(), "variant": best, "variants": var,
                         "sample": f"{samples} samples ({samples * HANDS_PER_SAMPLE} hands + crops) per step; oracle/geometry_oracle.py = reference torch ops on CPU"},
        "e2e": {"value": hps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cuda_time(fn, steps, warmup, dev):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) * 1e-3 / steps


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist

    from hands_b200 import _lib
    from hands_b200.step import GeometryStep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU baseline)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else {"bound": False, "note": "single rank: not bound (the CPU baseline leg uses every core)"}
    S = args.samples
    step = GeometryStep(S, dev, img_res=IMG_RES, seed=rank)
    streams_desc = "one + a forked branch for the left-hand MANO side" if step.mano_side_stream is not None else "single"
    metrics_vec = torch.zeros(64, device=dev)

    graph_launches = 0
    if not args.no_graph:
        graph_launches = step.capture()       # the launches of a step replayed from one CUDA graph

    def one_step():
        if graph_launches:
            step.replay()
        else:
            step.run()
        if world > 1:
            dist.all_reduce(metrics_vec)   # packed metric scalars (north_star); no data-path collective

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        one_step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        one_step()
    e1.record()
    barrier()
    launches = _lib.launch_count() - l0 + graph_launches * args.steps   # replays launch the captured kernels without host calls
    elapsed = e0.elapsed_time(e1) * 1e-3
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # before the legs below reuse the step's buffers
        dump_outputs(step, args.dump_outputs)
    if world > 1:
        t = torch.tensor([elapsed], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed = float(t.item())
    hands_per_step = S * HANDS_PER_SAMPLE * world
    value = hands_per_step * args.steps / elapsed
    bytes_per_sample = step.bytes_per_sample()

    # ---- per-family and per-kernel timing (each alone on the current stream, CUDA events) for the roofline ------------
    # A 1024-image batch (2048 crops) for the kernels, so one call == one launch of the kernel in question (the timed step
    # runs the same kernels over 4096-image chunks).  Every leg re-reads inputs far larger than L2.
    from scripts import bench_legs as L

    peak, peak_src = peaks()
    fam, kern, overlap, tf32_peak = {}, {}, {}, None
    if rank == 0:
        n = step.n
        plane = 3 * IMG_RES * IMG_RES * 4
        reps = max(5, args.steps)
        step.pcl_setup()
        t_fwd = cuda_time(step.pcl_forward, reps, 2, dev)
        t_bwd = cuda_time(step.pcl_backward, reps, 2, dev)
        t_mf = cuda_time(lambda: [step.mano_forward(0), step.mano_forward(1)], reps, 2, dev)
        t_mb = cuda_time(lambda: [step.mano_backward(0), step.mano_backward(1)], reps, 2, dev)
        b_fwd = n * (plane + 12.0 * step.mean_s2)
        b_bwd = n * plane + S * plane
        fam = {
            "pcl_fwd": {"ms": t_fwd * 1e3, "alg_bytes": b_fwd, "gbs": b_fwd / t_fwd / 1e9, "frac": b_fwd / t_fwd / 1e9 / peak},
            "pcl_bwd (scan + mid + img kernels, all chunks)": {"ms": t_bwd * 1e3, "alg_bytes": b_bwd, "gbs": b_bwd / t_bwd / 1e9, "frac": b_bwd / t_bwd / 1e9 / peak},
            "mano_fwd r+l (pose + blend_tc + skin)": {"ms": t_mf * 1e3, "alg_bytes": 2 * S * 20020.0, "gbs": 2 * S * 20020.0 / t_mf / 1e9,
                                                      "frac": 2 * S * 20020.0 / t_mf / 1e9 / peak, "hands_per_s": 2 * S / t_mf},
            "mano_bwd r+l (pose + blend_tc + skin + gfeat_tc + pose)": {"ms": t_mb * 1e3, "alg_bytes": 2 * S * 11048.0, "gbs": 2 * S * 11048.0 / t_mb / 1e9,
                                                                        "frac": 2 * S * 11048.0 / t_mb / 1e9 / peak, "hands_per_s": 2 * S / t_mb},
        }
        fused_ms = elapsed / args.steps * 1e3
        overlap = {"fused_ms": fused_ms, "sum_of_families_ms": (t_fwd + t_bwd + t_mf + t_mb) * 1e3,
                   "pcl_alone_ms": (t_fwd + t_bwd) * 1e3, "mano_alone_ms": (t_mf + t_mb) * 1e3,
                   "note": "PCL and MANO on one stream (the PCL kernels fill the register file, no MANO CTA can be co-resident); the right and left MANO sides run as two forked branches (hands_b200/step.py)"}
        Sk = min(S, 1024)
        ks = step if S == Sk else GeometryStep(Sk, dev, img_res=IMG_RES, seed=7)
        ks.pcl_setup()
        ks.pcl_forward()
        ks.pcl_backward()
        tk_fwd = cuda_time(ks.pcl_forward, reps, 2, dev)
        tk_mid = cuda_time(lambda: ks.pcl_backward_stage(1), reps, 2, dev)
        tk_img = cuda_time(lambda: ks.pcl_backward_stage(2), reps, 2, dev)
        traffic, traffic_src = {}, None
        for name in ("traffic_r2.json", "traffic_r1.json"):   # dram bytes per launch from the committed `ncu --set full` captures
            try:
                with open(os.path.join(ROOT, "profiles", name)) as fh:
                    traffic, traffic_src = json.load(fh), "profiles/" + name
                break
            except Exception:
                pass
        ab = {"pcl_fwd_kernel": ks.n * (plane + 12.0 * ks.mean_s2), "pcl_bwd_mid_kernel": ks.n * plane, "pcl_bwd_img_kernel": Sk * plane}
        tt = {"pcl_fwd_kernel": tk_fwd, "pcl_bwd_mid_kernel": tk_mid, "pcl_bwd_img_kernel": tk_img}
        for name in ab:
            kern[name] = {"us_per_launch": tt[name] * 1e6, "alg_bytes_per_launch": ab[name], "achieved": ab[name] / tt[name] / 1e9,
                          "frac": ab[name] / tt[name] / 1e9 / peak, "traffic": next((v for k, v in traffic.items() if k.startswith(name[:-len("_kernel")])), None),
                          "crops_per_launch": ks.n}
        del ks
        if not args.quick:   # (kept out of the profiling command's launch list)
            try:
                tf32_peak = L.measure_tf32_peak(dev)
            except Exception:
                tf32_peak = None

    # ---- e2e: host buffers, copies inside the timed region ---------------------------------------------
    e2e = e2e_f32 = None
    if not args.no_e2e:
        e2e = run_e2e(step, args, dev, world, barrier, src_u8=True)
        if world == 1 and not args.quick:
            e2e_f32 = run_e2e(step, args, dev, world, barrier, src_u8=False, steps=2)

    # ---- the other BASELINE.json configs + the autograd-API path (sub-results, not the headline) ---------
    configs = {}
    if not args.quick:
        if world > 1:
            configs["C5"] = L_c5(dev, world, rank, args)
            if S * world != 65536 and 65536 % world == 0 and 65536 // world <= 32768:
                configs["C4_true_shard"] = c4_true_shard(dev, world, rank, 65536 // world, barrier, args)
        if rank == 0 and world == 1:
            del step
            torch.cuda.empty_cache()
            step = None
            configs["C1"] = L.config_c1()
            configs["C2"] = L.config_c2(dev, peak, tf32_peak)
            configs["C3"] = L.config_c3(dev, peak)
            configs["api_autograd"] = L.autograd_api(dev)
            configs["silhouette"] = L.silhouette_consumer(dev)

    if rank != 0:
        return
    # share of the step: the per-1024-image launch times scaled to the step's images
    chunks = max(1, (S + 1023) // 1024)
    share = {"pcl_fwd_kernel": fam["pcl_fwd"]["ms"], "pcl_bwd_mid_kernel": kern["pcl_bwd_mid_kernel"]["us_per_launch"] * 1e-3 * chunks,
             "pcl_bwd_img_kernel": kern["pcl_bwd_img_kernel"]["us_per_launch"] * 1e-3 * chunks}
    dom = max(share, key=share.get)
    bps = bytes_per_sample
    step_bytes = bps * S
    step_gbs = value / world / HANDS_PER_SAMPLE * bps / 1e9
    # DRAM traffic of one step, from the committed per-launch ncu captures (1024-image launches) scaled to this step's
    # launches; MANO kernels from the same capture file (8192-hand launches would be ~8x the 1024-hand figures)
    step_traffic = None
    try:
        per1024 = sum(kern[k]["traffic"] for k in kern)
        mano_names = ("mano_pose_fwd_kernel", "mano_blend_tc_kernel", "mano_skin_fwd_kernel", "mano_skin_bwd_kernel", "mano_gfeat_tc_kernel", "mano_pose_bwd_kernel")
        mano1024 = sum(traffic.get(k, 0.0) for k in mano_names)
        step_traffic = (per1024 + HANDS_PER_SAMPLE * mano1024) * (S / 1024.0)
    except Exception:
        pass
    mano_hps = 2 * S / ((fam["mano_fwd r+l (pose + blend_tc + skin)"]["ms"] + fam["mano_bwd r+l (pose + blend_tc + skin + gfeat_tc + pose)"]["ms"]) * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "samples_per_gpu": S, "global_samples": S * world, "hands_per_sample": HANDS_PER_SAMPLE, "img_res": IMG_RES,
                   "bbox_side": "U{56..168}", "grads_on": ["v3d.cam", "j3d.cam", "j2d.norm", "crops"], "parallelism": f"dp{world} (batch sharded, no data-path collective)",
                   "l2": "inputs larger than L2 (%.1f GB working set per GPU), no flush needed" % (step_bytes / 1e9),
                   "streams": streams_desc, "cuda_graph": bool(graph_launches),
                   "pcl_forward": "exact (torch op order)" if os.environ.get("HB_PCL_EXACT", "0") == "1" else "default (reference sample positions, separable resize)",
                   "mano_contractions": "tcgen05 3xTF32" if os.environ.get("HB_MANO_TC", "1") != "0" else "ffma"},
        "clocks": clocks,
        "numa": numa,
        "gpu_launches": int(launches),
        "e2e": e2e,
        "e2e_fp32_source": e2e_f32,
        "roofline": {"bound": "hbm", "kernel": "fused C4 step (all kernels of one fwd+bwd pass)", "achieved": step_gbs, "peak": peak, "unit": "GB/s",
                     "frac": step_gbs / peak, "traffic": step_traffic, "peak_source": peak_src,
                     "note": "achieved = algorithmic bytes of the whole step (SURVEY.md 8(d): %.0f B/sample) / device time of the timed region; "
                             "per-kernel fractions (each kernel timed alone, one launch over %d crops) are under `kernels`; `traffic` = dram bytes "
                             "of one step = the per-launch `ncu --set full` captures of %s scaled to this step's launches (vs %.1f GB algorithmic)"
                             % (bps, kern[dom]["crops_per_launch"], traffic_src, bps * S / 1e9),
                     "alg_bytes_per_sample": bps,
                     "tensor_peak_tf32_tflops": tf32_peak, "tensor_peak_source": "measured here: torch.matmul fp32 with allow_tf32, 8192^3, best of 10",
                     "tensor_frac": (mano_hps * L.F_GEMM / (tf32_peak * 1e12)) if tf32_peak else None,
                     "tensor_note": "MANO head r+l alone (fwd+bwd families above): hands/s x %.0f algorithmic contraction FLOP/hand / measured TF32 peak; "
                                    "MMA passes actually issued (3xTF32) are not credited" % L.F_GEMM,
                     "dominant_kernel": dom, "step_share_ms": share, "overlap": overlap, "kernels": kern, "families": fam},
        "configs": configs,
    }
    if world == 1 and not args.no_cpu_baseline:
        best, var = cpu_baseline_variants(args.ref_samples, 2, 1, want_pool=not args.quick)
        line["cpu_baseline"] = {"value": var[best]["value"], "unit": UNIT, "cores": var[best]["cores"], "kind": "port", "cpu": cpu_model(), "variant": best,
                                "variants": var,
                                "sample": f"{args.ref_samples} samples ({args.ref_samples * HANDS_PER_SAMPLE} hands + crops) x 2 timed steps of the same workload; oracle = reference torch ops on CPU"}
    print(json.dumps(line), flush=True)


DUMP_HAND_SAMPLES = 512    # samples whose per-hand outputs are written (40 KB per sample)
DUMP_IMAGE_SAMPLES = 16    # samples whose crops and source-image gradient are written (1.8 MB per sample)
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(step, out_dir):
    """Write what the last step left in its output buffers, i.e. what a caller of the step receives, as `out_dir/<name>.npy`
    (float32), so that two builds can be compared output for output.  The whole output of an 8192-sample step is ~15 GB,
    so a fixed sample of it is written, ~50 MB: the per-hand outputs of 512 samples and the crops and image gradients of
    16 samples, both drawn by a seeded permutation of the sample index.  Crop rows are [sample][right, left]."""
    import numpy as np

    perm = torch.randperm(step.S, generator=torch.Generator().manual_seed(0))
    hand_idx = perm[:DUMP_HAND_SAMPLES].sort().values.to(step.dev)
    img_idx = perm[:DUMP_IMAGE_SAMPLES].sort().values.to(step.dev)
    crop_idx = (img_idx[:, None] * step.hps + torch.arange(step.hps, device=step.dev)).flatten()
    out = {
        "crops": step.crops[crop_idx],
        "g_img": step.g_img[img_idx],
        "rot": step.rot.view(step.S, step.hps, 3, 3)[hand_idx],
    }
    for side, h in zip(("right", "left"), step.hands):
        for key in ("vertices", "v3d", "joints3d", "j3d", "j2d", "cam_t", "g_rotmat", "g_betas", "g_cam"):
            out[f"{side}_{key}"] = h[key][hand_idx]
    out = {k: v.float().cpu().numpy() for k, v in out.items()}
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def L_c5(dev, world, rank, args):
    """C5: HaMeR-light MANO head training step with the parameter-gradient all-reduce (scripts/c5_hamer_head.py), both the
    read-out-sized (894 KB) and the decoder-head-sized (158 MB) gradient."""
    from scripts import c5_hamer_head as C5

    out = {}
    for full in (False, True):
        try:
            out["full_head_158MB" if full else "readouts_894KB"] = C5.run(dev, world, rank, batch=8192, steps=10, warmup=3, full_head=full)
        except Exception as exc:  # keep the headline line even if a side leg fails
            out["error"] = str(exc)[:200]
    return out


def c4_true_shard(dev, world, rank, S, barrier, args):
    """C4 at its stated shard size (65,536 samples / world per GPU), device-timed like the headline (max over ranks)."""
    import torch.distributed as dist

    from hands_b200.step import GeometryStep

    st = GeometryStep(S, dev, img_res=IMG_RES, seed=1000 + rank)
    for _ in range(2):
        st.run()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k = 3
    e0.record()
    for _ in range(k):
        st.run()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) * 1e-3], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del st
    torch.cuda.empty_cache()
    el = float(t.item())
    return {"samples_per_gpu": S, "global_samples": S * world, "ms_per_step": el / k * 1e3, "value": S * HANDS_PER_SAMPLE * world * k / el, "unit": UNIT}


def run_e2e(step, args, dev, world, barrier, src_u8=True, steps=None):
    """Same workload with HOST buffers: per step, pinned H2D of the samples' inputs (source images, boxes,
    intrinsics, poses, shapes, cameras) and D2H of the per-hand gradients + one metric scalar, all inside the
    timed region.  The batch is processed in chunks of `--e2e-chunk` samples through two device buffer sets so the
    copy of chunk c+1 (copy stream) overlaps the kernels of chunk c; the step is PCIe-bound (0.6 MB per sample)."""
    import torch.distributed as dist

    from hands_b200.step import GeometryStep

    S = step.S
    CH = min(args.e2e_chunk, S)
    nch = S // CH
    if nch * CH != S:
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": "samples not divisible by e2e chunk"}
    sets = [GeometryStep(CH, dev, img_res=IMG_RES, seed=100 + k, src_u8=src_u8) for k in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)

    def dev_inputs(gs):
        t = [gs.img, gs.bbox, gs.Kcrop]
        for h in gs.hands:
            t += [h["rotmat"], h["betas"], h["cam"], h["K"]]
        return t

    def dev_outputs(gs):
        t = []
        for h in gs.hands:
            t += [h["g_rotmat"], h["g_betas"], h["g_cam"]]
        return t

    try:
        # host side: the full batch in pinned memory (inputs) and pinned result buffers
        host_in = [torch.empty((nch,) + tuple(t.shape), dtype=t.dtype, pin_memory=True) for t in dev_inputs(sets[0])]
        for hb, t in zip(host_in, dev_inputs(step)):
            if hb.dtype == t.dtype:
                hb.view((S * (t.shape[0] // S),) + tuple(t.shape[1:])).copy_(t)
            else:   # 8-bit source images: synthetic bytes (the main step holds the fp32 form)
                hb.random_(0, 256)
        host_out = [torch.empty((nch,) + tuple(t.shape), dtype=t.dtype, pin_memory=True) for t in dev_outputs(sets[0])]
        metric_host = torch.empty(nch, dtype=torch.float32, pin_memory=True)
    except RuntimeError as exc:  # pinned allocation refused
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": str(exc)[:120]}
    h2d = sum(t.numel() * t.element_size() for t in host_in)
    d2h = sum(t.numel() * t.element_size() for t in host_out) + 4 * nch
    ready = [torch.cuda.Event() for _ in range(2)]     # inputs of set k are on the device
    consumed = [torch.cuda.Event() for _ in range(2)]  # kernels of set k have read their inputs

    def one():
        cur = torch.cuda.current_stream(dev)
        for c in range(nch):
            k = c & 1
            gs = sets[k]
            with torch.cuda.stream(copy_stream):
                if c >= 2:
                    copy_stream.wait_event(consumed[k])
                for hb, d in zip(host_in, dev_inputs(gs)):
                    d.copy_(hb[c], non_blocking=True)
                ready[k].record(copy_stream)
            cur.wait_event(ready[k])
            gs.run()
            consumed[k].record(cur)
            for hb, o in zip(host_out, dev_outputs(gs)):
                hb[c].copy_(o, non_blocking=True)
            metric_host[c : c + 1].copy_(gs.hands[0]["j2d"][0, 0, :1], non_blocking=True)

    k = steps or max(2, min(args.steps, 5))
    for _ in range(2):
        one()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(k):
        one()
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    el = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        t = torch.tensor([el], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        el = float(t.item())
    return {"value": S * HANDS_PER_SAMPLE * world * k / el, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "steps": k, "ms_per_step": el / k * 1e3, "wall_ms_per_step": wall / k * 1e3, "chunk_samples": CH,
            "source_image_dtype": "uint8 (normalisation fused into the crop forward, hb_pcl_fwd_u8)" if src_u8 else "float32 (normalised on the host)",
            "h2d_gbs": h2d * k / el / 1e9,
            "d2h": "per-hand gradients (g_rotmat, g_betas, g_cam) + one metric scalar per chunk; crops and g_img stay on the device for the backbone",
            "pipeline": "H2D of chunk c+1 overlaps kernels of chunk c (2 device buffer sets)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=8192, help="samples per GPU per step (C4: 65536 / 8)")
    ap.add_argument("--ref-samples", type=int, default=256, help="samples per CPU-reference step (bounded sample)")
    ap.add_argument("--e2e-chunk", type=int, default=1024, help="samples per pipelined e2e chunk")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step kernel by kernel instead of replaying its CUDA graph")
    ap.add_argument("--quick", action="store_true", help="skip the side legs (other configs, fp32-source e2e, CPU worker pool)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
