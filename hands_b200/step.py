"""Pre-allocated geometry step: the fast path a training loop (and bench.py) drives.

One `GeometryStep` owns every buffer of a two-hand sample batch on one GPU and runs

    PCL setup -> PCL forward (2 crops / sample, one shared source image)
    MANO head forward right + left  (global orientation pre-rotated by R_virt2orig,
        hands_light/model.py:330-334, fused as `pre_rot`)
    MANO head backward right + left
    PCL backward

through the C ABI on the current stream, with no allocation and no autograd bookkeeping inside the step.  The autograd
drop-ins in `hands_b200.functional` call the same entry points; this class only removes the per-call allocations.
"""
import ctypes

import torch

from . import _lib
from .functional import ManoHandle, _ptr, check_crop_dtype
from .synthetic import synthetic_head_inputs, synthetic_mano_buffers, synthetic_pcl_inputs

NV, NJ, NOJ, NB = 778, 16, 21, 10


class GeometryStep:
    IMG_MEAN = (0.485, 0.456, 0.406)   # the reference's img_norm_mean / img_norm_std (src/parsers/parser.py:45-46)
    IMG_STD = (0.229, 0.224, 0.225)

    def __init__(self, samples, device, img_res=224, with_pcl=True, with_mano=True, hands_per_sample=2, seed=0, grads_on=("v3d", "j3d", "j2d"),
                 src_u8=False, crop_dtype=torch.float32):
        """crop_dtype torch.bfloat16: `crops` and `g_crops` are bf16 (what a backbone under bf16 autocast reads and returns) and
        the step runs the bf16 crop-layer entry points; the image, its gradient and everything MANO stay fp32."""
        self.lib = _lib.load()
        self.crop_dtype = check_crop_dtype(crop_dtype)
        self.crop_bf16 = crop_dtype == torch.bfloat16
        self.S, self.dev, self.R = int(samples), torch.device(device), int(img_res)
        self.with_pcl, self.with_mano, self.hps = with_pcl, with_mano, hands_per_sample
        self.grads_on = grads_on
        S, R, dev = self.S, self.R, self.dev
        f32 = dict(dtype=torch.float32, device=dev)
        n = S * hands_per_sample  # crops == hands
        self.n = n
        gen = torch.Generator(device=dev).manual_seed(seed)
        if with_pcl:
            _, bbox, Kc = synthetic_pcl_inputs(n, seed=seed, img_res=R, smin=R // 4, smax=3 * R // 4)
            self.bbox = bbox.to(dev)
            self.Kcrop = Kc.to(dev)
            self.src_u8 = bool(src_u8)
            if self.src_u8:   # the data loader's 8-bit image; normalisation fused into the crop forward (hb_pcl_fwd_u8)
                self.img = torch.randint(0, 256, (S, 3, R, R), generator=gen, device=dev, dtype=torch.uint8)
                self._mean = (ctypes.c_float * 3)(*self.IMG_MEAN)
                self._std = (ctypes.c_float * 3)(*self.IMG_STD)
            else:
                self.img = torch.randn(S, 3, R, R, generator=gen, **f32)
            self.crops = torch.empty(n, 3, R, R, dtype=crop_dtype, device=dev)
            # drawn in fp32 either way, so the generator's later draws (the MANO gradients) do not depend on crop_dtype
            self.g_crops = torch.randn(n, 3, R, R, generator=gen, **f32).to(crop_dtype)
            self.g_img = torch.empty(S, 3, R, R, **f32)
            self.params = torch.empty(n, _lib.PCL_PARAM_FLOATS, **f32)
            self.rot = torch.empty(n, 3, 3, **f32)
            self.pcl_ws_bytes = self.lib.hb_pcl_bwd_workspace_bytes(n, hands_per_sample, 3, R)
            self.pcl_ws = torch.empty((self.pcl_ws_bytes + 3) // 4, **f32)
            self.mean_s2 = float(((self.bbox[:, 2:] - self.bbox[:, :2]).max(dim=1).values.float() ** 2).mean())
        if with_mano:
            self.hands = []
            for side in range(hands_per_sample):
                is_rhand = side == 0
                handle = ManoHandle(synthetic_mano_buffers(is_rhand), dev)
                rotmat, betas, cam, K = [t.to(dev) for t in synthetic_head_inputs(S, seed=seed + 10 * side)]
                h = dict(handle=handle, rotmat=rotmat, betas=betas, cam=cam, K=K)
                h["vertices"] = torch.empty(S, NV, 3, **f32)
                h["v3d"] = torch.empty(S, NV, 3, **f32)
                h["joints3d"] = torch.empty(S, NOJ, 3, **f32)
                h["j3d"] = torch.empty(S, NOJ, 3, **f32)
                h["j2d"] = torch.empty(S, NOJ, 2, **f32)
                h["cam_t"] = torch.empty(S, 3, **f32)
                h["g_v3d"] = torch.randn(S, NV, 3, generator=gen, **f32) if "v3d" in grads_on else None
                h["g_j3d"] = torch.randn(S, NOJ, 3, generator=gen, **f32) if "j3d" in grads_on else None
                h["g_j2d"] = torch.randn(S, NOJ, 2, generator=gen, **f32) if "j2d" in grads_on else None
                h["g_rotmat"] = torch.empty(S, NJ, 3, 3, **f32)
                h["g_betas"] = torch.empty(S, NB, **f32)
                h["g_cam"] = torch.empty(S, 3, **f32)
                h["pre_rot"] = torch.empty(S, 3, 3, **f32) if with_pcl else None
                self.hands.append(h)
            # one backward-sized workspace per hand side: the backward picks up the forward's intermediates (hb_mano_head_bwd_reuse)
            self.mano_ws_bytes = self.lib.hb_mano_workspace_bytes(S, 1)
            self.mano_ws = [torch.empty((self.mano_ws_bytes + 3) // 4, **f32) for _ in range(hands_per_sample)]
            self.mano_fwd_valid = [False] * hands_per_sample
        # second stream for the left hand side of the fused step
        self.mano_side_stream = None
        if with_mano and hands_per_sample == 2:
            self.mano_side_stream = torch.cuda.Stream(device=self.dev)

    # ---- pieces (each enqueues on the CURRENT torch stream) ------------------------------------
    def _st(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def pcl_setup(self):
        _lib.check(self.lib.hb_pcl_setup(_ptr(self.bbox), _ptr(self.Kcrop), self.n, self.R, _ptr(self.params), _ptr(self.rot), self._st()), "hb_pcl_setup")

    def pcl_forward(self):
        sfx = "_bf16" if self.crop_bf16 else ""
        if self.src_u8:
            fn = "hb_pcl_fwd_u8" + sfx
            _lib.check(getattr(self.lib, fn)(_ptr(self.img), ctypes.cast(self._mean, ctypes.c_void_p), ctypes.cast(self._std, ctypes.c_void_p), _ptr(self.params),
                                             self.n, self.hps, 3, self.R, _ptr(self.crops), self._st()), fn)
            return
        fn = "hb_pcl_fwd" + sfx
        _lib.check(getattr(self.lib, fn)(_ptr(self.img), _ptr(self.params), self.n, self.hps, 3, self.R, _ptr(self.crops), self._st()), fn)

    def pcl_backward(self):
        fn = "hb_pcl_bwd_bf16" if self.crop_bf16 else "hb_pcl_bwd"
        _lib.check(getattr(self.lib, fn)(_ptr(self.g_crops), _ptr(self.params), self.n, self.hps, 3, self.R, _ptr(self.g_img), _ptr(self.pcl_ws),
                                         self.pcl_ws_bytes, self._st()), fn)

    def pcl_backward_stage(self, stages):
        """stages 1 = transposed resize, 2 = transposed gather (single-chunk batches only; used by bench.py's roofline leg)."""
        if self.crop_bf16:
            raise NotImplementedError("pcl_backward_stage: the stage-by-stage entry point (hb_pcl_bwd_stages) takes fp32 crop gradients only")
        _lib.check(self.lib.hb_pcl_bwd_stages(_ptr(self.g_crops), _ptr(self.params), self.n, self.hps, 3, self.R, _ptr(self.g_img), _ptr(self.pcl_ws),
                                              self.pcl_ws_bytes, int(stages), self._st()), "hb_pcl_bwd_stages")

    def gather_pre_rot(self):
        # rot is (S*hps,3,3) interleaved [sample][side]; each hand side takes its strided view (one small copy kernel)
        for side, h in enumerate(self.hands):
            h["pre_rot"].copy_(self.rot.view(self.S, self.hps, 3, 3)[:, side])

    def mano_forward(self, side):
        h = self.hands[side]
        _lib.check(self.lib.hb_mano_head_fwd(h["handle"].handle, _ptr(h["rotmat"]), 1, _ptr(h["pre_rot"]), _ptr(h["betas"]), _ptr(h["cam"]), _ptr(h["K"]),
                                             None, self.S, float(self.R), 0.1, _ptr(h["vertices"]), _ptr(h["v3d"]), _ptr(h["joints3d"]), _ptr(h["j3d"]),
                                             _ptr(h["j2d"]), _ptr(h["cam_t"]), _ptr(self.mano_ws[side]), self.mano_ws_bytes, self._st()), "hb_mano_head_fwd")
        self.mano_fwd_valid[side] = True

    def mano_backward(self, side):
        h = self.hands[side]
        # the backward leaves the forward's part of the workspace intact: it stays valid until the inputs change
        fn = self.lib.hb_mano_head_bwd_reuse if self.mano_fwd_valid[side] else self.lib.hb_mano_head_bwd
        _lib.check(fn(h["handle"].handle, _ptr(h["rotmat"]), 1, _ptr(h["pre_rot"]), _ptr(h["betas"]), _ptr(h["cam"]), _ptr(h["K"]),
                                             None, self.S, float(self.R), 0.1, None, _ptr(h["g_v3d"]), None, _ptr(h["g_j3d"]), _ptr(h["g_j2d"]), None,
                      _ptr(h["g_rotmat"]), _ptr(h["g_betas"]), _ptr(h["g_cam"]), None, None, _ptr(self.mano_ws[side]),
                      self.mano_ws_bytes, self._st()), "hb_mano_head_bwd")

    # ---- the fused step ----------------------------------------------------------------------------
    def run(self):
        """Enqueue one full fwd+bwd step on the current stream.

        The crop layer and MANO share one stream on purpose.  Round 1 ran MANO on a second stream "overlapped" with the crop
        layer; measured, the fused step took exactly the sum of its families (10.84 vs 10.87 ms): every PCL kernel fills the
        register file (5 x 256 x 48, 3 x 256 x 80, 4 x 256 x 62 registers per SM), so no MANO CTA can become resident beside
        one, whatever the stream priorities -- the second stream only queued.  What does overlap is MANO with itself: the
        right and the left hand side run on two forked streams (10.31 -> 10.19 ms per 8192-sample step)."""
        with torch.cuda.device(self.dev):   # launches and cudaFuncSetAttribute target self.dev whatever the caller's device
            if self.with_pcl:
                self.pcl_setup()
                self.pcl_forward()
            if self.with_mano:
                if self.with_pcl:
                    self.gather_pre_rot()
                if self.mano_side_stream is not None:
                    # the two hand sides are independent (own constants, inputs, workspace): the left side runs on a forked
                    # stream, so its latency-bound kernels (pose, the tcgen05 contractions: at most one CTA per SM) share the
                    # GPU with the right side's skinning kernels; joined before the crop layer's backward.  Inside a capture
                    # this becomes two parallel branches of the graph.
                    cur = torch.cuda.current_stream(self.dev)
                    self.mano_side_stream.wait_stream(cur)
                    with torch.cuda.stream(self.mano_side_stream):
                        self.mano_forward(1)
                        self.mano_backward(1)
                    self.mano_forward(0)
                    self.mano_backward(0)
                    cur.wait_stream(self.mano_side_stream)
                else:
                    for side in range(self.hps):
                        self.mano_forward(side)
                    for side in range(self.hps):
                        self.mano_backward(side)
            if self.with_pcl:
                self.pcl_backward()

    # ---- the same step as one CUDA graph -------------------------------------------------------------
    def capture(self):
        """Capture one `run()` (19 library launches at the recommended workspace size: 7 PCL, 12 MANO; plus 2 strided copies) into a CUDA graph.  Every buffer is
        pre-allocated and every argument is a fixed device pointer, so the step replays verbatim; `replay()` then costs one
        host call and removes the launch gaps between the kernels.  Returns the number of library launches per replay."""
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            self.run()                                   # warm-up outside the capture (function attributes, lazy module loads)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        n0 = _lib.launch_count()
        self.graph = torch.cuda.CUDAGraph()
        # thread_local: other threads of the process (NCCL's watchdog under torchrun) keep making CUDA calls during the capture
        with torch.cuda.graph(self.graph, stream=side, capture_error_mode="thread_local"):
            self.run()
        self.launches_per_replay = _lib.launch_count() - n0
        return self.launches_per_replay

    def replay(self):
        self.graph.replay()

    # ---- algorithmic bytes (SURVEY.md §8(d)) -----------------------------------------------------
    def mano_bytes_per_hand(self):
        return 31068.0

    def crop_elem_bytes(self):
        return 2 if self.crop_bf16 else 4

    def pcl_bytes_per_crop(self):
        # out write + g_out read (crop dtype) + g_img write (fp32) + src footprint
        return 3 * self.R * self.R * (2 * self.crop_elem_bytes() + 4) + 12.0 * self.mean_s2

    def bytes_per_sample(self):
        b = 0.0
        if self.with_mano:
            b += self.hps * self.mano_bytes_per_hand()
        if self.with_pcl:
            plane = 3 * self.R * self.R * self.crop_elem_bytes()   # the crop and its gradient, in the crop dtype
            # SURVEY.md §8(d) convention for crops sharing one source image: 2*hps planes + the source footprints
            # (4 x 602,112 + 2 x 12 s^2 for two hands; the shared g_img write is not counted, so the figure is
            # conservative -- real traffic is one plane higher)
            b += plane * (2 * self.hps) + self.hps * 12.0 * self.mean_s2
        return b
