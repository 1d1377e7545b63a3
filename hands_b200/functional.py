"""torch.autograd.Function drop-ins over the C ABI (include/hands_b200.h).

PyTorch is plumbing here: it owns device memory and streams and supplies autograd's graph; all
arithmetic of the path runs in libhands_b200.so.  Forward saves INPUTS only; backward recomputes.
There is no CPU path: CPU tensors raise.
"""
import ctypes

import torch

from . import _lib

NV, NJ, NOJ, NB = 778, 16, 21, 10


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name, shape=None):
    """Mirror of the reference's asserts (common/transforms.py:322-326): real fp32 CUDA tensors."""
    if t is None:
        return None
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: hands_b200 has no CPU path; expected a CUDA tensor (got {t.device})")
    if t.dtype != torch.float32:
        raise TypeError(f"{name}: expected torch.float32, got {t.dtype}")
    if shape is not None:
        if t.dim() != len(shape) or any(s is not None and s != d for s, d in zip(shape, t.shape)):
            raise ValueError(f"{name}: expected shape {tuple('B' if s is None else s for s in shape)}, got {tuple(t.shape)}")
    return t.contiguous()


class ManoHandle:
    """Owns one hb_mano* (MANO constants of one hand side on one CUDA device)."""

    def __init__(self, buffers, device):
        lib = _lib.load()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("ManoHandle needs a CUDA device")
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        f = lambda k: buffers[k].detach().to("cpu", torch.float32).contiguous()  # noqa: E731
        i = lambda k: buffers[k].detach().to("cpu", torch.int32).contiguous()  # noqa: E731
        host = [f("v_template"), f("shapedirs"), f("posedirs"), f("J_regressor"), f("lbs_weights"), i("parents"), f("pose_mean"), i("tip_ids")]
        assert host[0].shape == (NV, 3) and host[1].shape == (NV, 3, NB) and host[2].shape == (135, NV * 3)
        assert host[3].shape == (NJ, NV) and host[4].shape == (NV, NJ) and host[5].shape == (NJ,) and host[6].shape == (48,) and host[7].shape == (5,)
        out = ctypes.c_void_p()
        rc = lib.hb_mano_create(*[ctypes.c_void_p(t.data_ptr()) for t in host], idx, ctypes.byref(out))
        _lib.check(rc, "hb_mano_create")
        self.handle = out
        self.device = torch.device("cuda", idx)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().hb_mano_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def _workspace(nbytes, device):
    return torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=device)


class ManoHeadFunction(torch.autograd.Function):
    """MANO layer (+ optional camera head).  Returns
    (vertices, v3d_cam, joints3d, j3d_cam, j2d_norm, cam_t); the camera outputs are None without cam/K.

    Reference: src/nets/hand_heads/mano_head.py:21-65 and smplx.MANO.forward (SURVEY.md Appendix A)."""

    @staticmethod
    def forward(ctx, handle, pose, betas, cam, K, transl, pre_rot, img_res, min_s, rot6d_layout=None, materialise=None):
        lib = _lib.load()
        B = betas.shape[0]
        if rot6d_layout is not None:   # (B,16,6) 6D rotations, conversion fused in front of the log map
            is_rotmat = _lib.POSE_ROT6D + _lib.ROT6D_LAYOUTS[rot6d_layout]
            pose = _f32c(pose, "pose", (B, NJ, 6))
        else:
            is_rotmat = int(pose.dim() == 4)
            pose = _f32c(pose, "pose", (B, NJ, 3, 3) if is_rotmat else (B, 48))
        betas = _f32c(betas, "betas", (B, NB))
        cam = _f32c(cam, "cam", (B, 3))
        K = _f32c(K, "K", (B, 3, 3))
        transl = _f32c(transl, "transl", (B, 3))
        pre_rot = _f32c(pre_rot, "pre_rot", (B, 3, 3))
        dev = betas.device
        if dev != handle.device:
            raise RuntimeError(f"inputs on {dev} but MANO constants on {handle.device}")
        has_cam = cam is not None
        new = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731
        # `materialise`: names of the outputs to write (None = all).  The C ABI skips NULL outputs, so a consumer that only
        # reads j3d.cam / j2d.norm (the key-point losses) never pays the 18.7 KB/hand of vertex stores.
        want = lambda k: materialise is None or k in materialise  # noqa: E731
        vertices = new(B, NV, 3) if want("vertices") else None
        joints3d = new(B, NOJ, 3) if want("joints3d") else None
        v3d = new(B, NV, 3) if has_cam and want("v3d.cam") else None
        j3d = new(B, NOJ, 3) if has_cam and want("j3d.cam") else None
        j2d = new(B, NOJ, 2) if has_cam and want("j2d.norm") else None
        cam_t = new(B, 3) if has_cam and want("cam_t") else None
        # When a gradient will be asked for, the forward runs in a backward-sized workspace that the backward then picks up
        # (hb_mano_head_bwd_reuse: no second log-map / Rodrigues / chain / blendshape pass).  Inputs are still what is saved
        # for autograd's purposes; the workspace is scratch the backward may or may not find (double backward recomputes).
        keep = any(ctx.needs_input_grad)
        nbytes = lib.hb_mano_workspace_bytes(B, 1 if keep else 0)
        ws = _workspace(nbytes, dev)
        with torch.cuda.device(dev):
            rc = lib.hb_mano_head_fwd(handle.handle, _ptr(pose), int(is_rotmat), _ptr(pre_rot), _ptr(betas), _ptr(cam), _ptr(K), _ptr(transl),
                                      B, float(img_res), float(min_s), _ptr(vertices), _ptr(v3d), _ptr(joints3d), _ptr(j3d), _ptr(j2d),
                                      _ptr(cam_t), _ptr(ws), nbytes, _stream())
        _lib.check(rc, "hb_mano_head_fwd")
        ctx.handle, ctx.is_rotmat, ctx.img_res, ctx.min_s = handle, is_rotmat, float(img_res), float(min_s)
        ctx.ws = ws if keep else None
        ctx.save_for_backward(pose, betas, cam, K, transl, pre_rot)
        ctx.set_materialize_grads(False)
        return vertices, v3d, joints3d, j3d, j2d, cam_t

    @staticmethod
    def backward(ctx, g_vertices, g_v3d, g_joints3d, g_j3d, g_j2d, g_cam_t):
        lib = _lib.load()
        pose, betas, cam, K, transl, pre_rot = ctx.saved_tensors
        B, dev = betas.shape[0], betas.device
        cg = lambda g: None if g is None else g.contiguous().float()  # noqa: E731
        g_vertices, g_v3d, g_joints3d, g_j3d, g_j2d, g_cam_t = map(cg, (g_vertices, g_v3d, g_joints3d, g_j3d, g_j2d, g_cam_t))
        g_pose = torch.empty_like(pose)
        g_betas = torch.empty_like(betas)
        g_cam = torch.empty_like(cam) if cam is not None else None
        g_transl = torch.empty_like(transl) if transl is not None else None
        g_pre = torch.empty_like(pre_rot) if pre_rot is not None else None
        nbytes = lib.hb_mano_workspace_bytes(B, 1)
        ws, ctx.ws = ctx.ws, None   # used once: a second backward through the same node recomputes
        bwd = lib.hb_mano_head_bwd_reuse if ws is not None else lib.hb_mano_head_bwd
        if ws is None:
            ws = _workspace(nbytes, dev)
        with torch.cuda.device(dev):
            rc = bwd(ctx.handle.handle, _ptr(pose), int(ctx.is_rotmat), _ptr(pre_rot), _ptr(betas), _ptr(cam), _ptr(K),
                                      _ptr(transl), B, ctx.img_res, ctx.min_s, _ptr(g_vertices), _ptr(g_v3d), _ptr(g_joints3d), _ptr(g_j3d),
                                      _ptr(g_j2d), _ptr(g_cam_t), _ptr(g_pose), _ptr(g_betas), _ptr(g_cam), _ptr(g_transl), _ptr(g_pre),
                                      _ptr(ws), nbytes, _stream())
        _lib.check(rc, "hb_mano_head_bwd")
        # inputs: handle, pose, betas, cam, K, transl, pre_rot, img_res, min_s, rot6d_layout, materialise
        return None, g_pose, g_betas, g_cam, None, g_transl, g_pre, None, None, None, None


class Rot6dToRotmatFunction(torch.autograd.Function):
    """6D rotation representation -> rotation matrix in one of the reference's three layouts:
    "rows" (pytorch3d rotation_6d_to_matrix, hand_hmr.py:85-87), "cols" (hamer_light/geometry.py:47-62,
    handoccnet_light/mano_head.py:132-141), "cols_paired" (common/rot.py:367-381)."""

    @staticmethod
    def forward(ctx, x6, layout):
        lay = _lib.ROT6D_LAYOUTS[layout]
        x = _f32c(x6, "x6", (None, 6))
        R = torch.empty(x.shape[0], 3, 3, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().hb_rot6d_to_rotmat_fwd(_ptr(x), x.shape[0], lay, _ptr(R), _stream()), "hb_rot6d_to_rotmat_fwd")
        ctx.save_for_backward(x)
        ctx.lay = lay
        return R

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        g = g.contiguous().float()
        gx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().hb_rot6d_to_rotmat_bwd(_ptr(x), _ptr(g), x.shape[0], ctx.lay, _ptr(gx), _stream()), "hb_rot6d_to_rotmat_bwd")
        return gx, None


class MatrixToAxisAngleFunction(torch.autograd.Function):
    """common/rot.py:180-193."""

    @staticmethod
    def forward(ctx, R):
        lead = R.shape[:-2]
        Rc = _f32c(R.reshape(-1, 3, 3), "matrix", (None, 3, 3))
        aa = torch.empty(Rc.shape[0], 3, dtype=torch.float32, device=Rc.device)
        with torch.cuda.device(Rc.device):
            _lib.check(_lib.load().hb_matrix_to_axis_angle_fwd(_ptr(Rc), Rc.shape[0], _ptr(aa), _stream()), "hb_matrix_to_axis_angle_fwd")
        ctx.save_for_backward(Rc)
        ctx.lead = lead
        return aa.reshape(lead + (3,))

    @staticmethod
    def backward(ctx, g):
        (Rc,) = ctx.saved_tensors
        g = g.reshape(-1, 3).contiguous().float()
        gR = torch.empty_like(Rc)
        with torch.cuda.device(Rc.device):
            _lib.check(_lib.load().hb_matrix_to_axis_angle_bwd(_ptr(Rc), _ptr(g), Rc.shape[0], _ptr(gR), _stream()), "hb_matrix_to_axis_angle_bwd")
        return gR.reshape(ctx.lead + (3, 3))


class Project2DFunction(torch.autograd.Function):
    """common/transforms.py:316-329 (+ normalize_kp2d when img_res > 0).  K gets no gradient."""

    @staticmethod
    def forward(ctx, K, pts, img_res):
        K = _f32c(K, "K", (None, 3, 3))
        pts = _f32c(pts, "pts_cam", (K.shape[0], None, 3))
        B, N = pts.shape[:2]
        out = torch.empty(B, N, 2, dtype=torch.float32, device=pts.device)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().hb_project2d_fwd(_ptr(K), _ptr(pts), B, N, float(img_res), _ptr(out), _stream()), "hb_project2d_fwd")
        ctx.save_for_backward(K, pts)
        ctx.img_res = float(img_res)
        return out

    @staticmethod
    def backward(ctx, g):
        K, pts = ctx.saved_tensors
        B, N = pts.shape[:2]
        g = g.contiguous().float()
        gp = torch.empty_like(pts)
        with torch.cuda.device(pts.device):
            _lib.check(_lib.load().hb_project2d_bwd(_ptr(K), _ptr(pts), _ptr(g), B, N, ctx.img_res, _ptr(gp), _stream()), "hb_project2d_bwd")
        return None, gp, None


class WeakToPerspFunction(torch.autograd.Function):
    """common/camera.py:456-474."""

    @staticmethod
    def forward(ctx, cam, focal, img_res, min_s):
        cam = _f32c(cam, "weak_perspective_camera", (None, 3))
        B = cam.shape[0]
        if not isinstance(focal, torch.Tensor):
            focal = torch.full((B,), float(focal), dtype=torch.float32, device=cam.device)
        focal = _f32c(focal.expand(B) if focal.dim() == 0 else focal, "focal_length", (B,))
        out = torch.empty(B, 3, dtype=torch.float32, device=cam.device)
        with torch.cuda.device(cam.device):
            _lib.check(_lib.load().hb_weak_to_persp_fwd(_ptr(cam), _ptr(focal), B, float(img_res), float(min_s), _ptr(out), _stream()), "hb_weak_to_persp_fwd")
        ctx.save_for_backward(cam, focal)
        ctx.img_res, ctx.min_s = float(img_res), float(min_s)
        return out

    @staticmethod
    def backward(ctx, g):
        cam, focal = ctx.saved_tensors
        g = g.contiguous().float()
        gc = torch.empty_like(cam)
        with torch.cuda.device(cam.device):
            _lib.check(_lib.load().hb_weak_to_persp_bwd(_ptr(cam), _ptr(focal), _ptr(g), cam.shape[0], ctx.img_res, ctx.min_s, _ptr(gc), _stream()), "hb_weak_to_persp_bwd")
        return gc, None, None, None


def persp_to_weak(cam_t, focal, img_res):
    """common/camera.py:10-29 (GT side, no gradient in the reference: process_arctic.py:59-65)."""
    cam_t = _f32c(cam_t.detach(), "perspective_camera", (None, 3))
    B = cam_t.shape[0]
    if not isinstance(focal, torch.Tensor):
        focal = torch.full((B,), float(focal), dtype=torch.float32, device=cam_t.device)
    focal = _f32c(focal.expand(B) if focal.dim() == 0 else focal, "focal_length", (B,))
    out = torch.empty(B, 3, dtype=torch.float32, device=cam_t.device)
    with torch.cuda.device(cam_t.device):
        _lib.check(_lib.load().hb_persp_to_weak_fwd(_ptr(cam_t), _ptr(focal), B, float(img_res), _ptr(out), _stream()), "hb_persp_to_weak_fwd")
    return out


class RotApplyFunction(torch.autograd.Function):
    """out[b] = R[b] @ M[b]  (src/models/hands_light/model.py:330-334).  Gradients: g_M = R^T g, and g_R = g M^T when R
    requires grad (the crop layer's R_virt2orig does not; a `pre_rot` that is itself a prediction does, and the reference's
    torch product would give it this gradient through the returned `pose`)."""

    @staticmethod
    def forward(ctx, R, M):
        R = _f32c(R, "R_virt2orig", (None, 3, 3))
        M = _f32c(M, "global_orient", (R.shape[0], 3, 3))
        out = torch.empty_like(M)
        with torch.cuda.device(M.device):
            _lib.check(_lib.load().hb_rot_apply(_ptr(R), _ptr(M), M.shape[0], 0, _ptr(out), _stream()), "hb_rot_apply")
        ctx.save_for_backward(R, M if ctx.needs_input_grad[0] else None)
        return out

    @staticmethod
    def backward(ctx, g):
        R, M = ctx.saved_tensors
        g = g.contiguous().float()
        gr = gm = None
        lib = _lib.load()
        with torch.cuda.device(g.device):
            if ctx.needs_input_grad[0]:
                gr = torch.empty_like(g)
                # g M^T = (M g^T)^T: the same kernel on transposed operands
                gt = g.transpose(1, 2).contiguous()
                _lib.check(lib.hb_rot_apply(_ptr(M), _ptr(gt), g.shape[0], 0, _ptr(gr), _stream()), "hb_rot_apply")
                gr = gr.transpose(1, 2)
            if ctx.needs_input_grad[1]:
                gm = torch.empty_like(g)
                _lib.check(lib.hb_rot_apply(_ptr(R), _ptr(g), g.shape[0], 1, _ptr(gm), _stream()), "hb_rot_apply")
        return gr, gm


CROP_DTYPES = (torch.float32, torch.bfloat16)


def check_crop_dtype(dtype):
    """The crop layer writes fp32 or bf16 crop planes (hb_pcl_fwd*, hb_pcl_fwd*_bf16); anything else is an error."""
    if dtype not in CROP_DTYPES:
        raise TypeError(f"out_dtype: expected torch.float32 or torch.bfloat16, got {dtype}")
    return dtype


class PerspectiveCropFunction(torch.autograd.Function):
    """Batched Perspective Crop Layer (src/datasets/hands_light_dataset.py:354-467).
    img (Bi,C,R,R); bbox (Bi*n,4) int32; K (Bi*n,3,3) -> crop (Bi*n,C,R,R), R_virt2orig (Bi*n,3,3).
    Gradient w.r.t. img only (the sampling grid is data).
    out_dtype torch.bfloat16: the crop is written as bf16 (the RNE rounding of the fp32 crop) and its gradient is read as
    bf16; R_virt2orig and the image gradient stay fp32."""

    @staticmethod
    def forward(ctx, img, bbox, K, crops_per_img, mean=None, std=None, out_dtype=torch.float32):
        lib = _lib.load()
        bf16 = check_crop_dtype(out_dtype) == torch.bfloat16
        needs_grad = bool(img.requires_grad)   # read before _f32c: .contiguous() of a strided image is a new tensor
        u8 = isinstance(img, torch.Tensor) and img.dtype == torch.uint8
        if u8:
            # the data loader's 8-bit image: (u/255 - mean)/std (hands_light_dataset.py:177-184) is fused into the gather
            if not img.is_cuda:
                raise RuntimeError(f"img: hands_b200 has no CPU path; expected a CUDA tensor (got {img.device})")
            if mean is None or std is None:
                raise ValueError("a uint8 image needs mean= and std= (the reference's img_norm_mean / img_norm_std)")
            img = img.contiguous()
        else:
            img = _f32c(img, "img")
        if img.dim() != 4 or img.shape[2] != img.shape[3]:
            raise ValueError(f"img: expected (B,C,R,R), got {tuple(img.shape)}")
        Bi, C, R, _ = img.shape
        n = Bi * crops_per_img
        dev = img.device
        if bbox.dtype not in (torch.int16, torch.int32, torch.int64):
            raise TypeError(f"bbox: expected an integer tensor, got {bbox.dtype}")
        if tuple(bbox.shape) != (n, 4):
            raise ValueError(f"bbox: expected ({n},4), got {tuple(bbox.shape)}")
        if n > 0 and (needs_grad or not bbox.is_cuda):
            # Checked on the tensor as given: free for boxes that arrive on the host (the data loader's), one sync for
            # device boxes (only paid when a gradient is requested).
            wh = bbox[:, 2:] - bbox[:, :2]
            side, low = int(wh.max()), int(wh.min())
            if low < 0:
                # the reference raises in torch.linspace(0, 1, s) for s < 0 (hands_light_dataset.py:390-391)
                raise ValueError(f"perspective_crop: inverted box (x1 < x0 or y1 < y0, extent {low})")
            # The backward packs an s x s intermediate per crop into a workspace sized for s <= R, which the reference
            # guarantees by clipping boxes to the image (common/data_utils.py:508).  Fail loudly otherwise.
            if needs_grad and side > R:
                raise ValueError(f"perspective_crop backward needs boxes no larger than the image (side {side} > {R}); "
                                 "clip the boxes or call under torch.no_grad()")
        bbox = bbox.to(device=dev, dtype=torch.int32).contiguous()
        K = _f32c(K.to(dev) if isinstance(K, torch.Tensor) else K, "K", (n, 3, 3))
        params = torch.empty(n, _lib.PCL_PARAM_FLOATS, dtype=torch.float32, device=dev)
        rot = torch.empty(n, 3, 3, dtype=torch.float32, device=dev)
        out = torch.empty(n, C, R, R, dtype=out_dtype, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.hb_pcl_setup(_ptr(bbox), _ptr(K), n, R, _ptr(params), _ptr(rot), _stream()), "hb_pcl_setup")
            if u8:
                m = (ctypes.c_float * C)(*[float(v) for v in mean])
                sd = (ctypes.c_float * C)(*[float(v) for v in std])
                name = "hb_pcl_fwd_u8_bf16" if bf16 else "hb_pcl_fwd_u8"
                _lib.check(getattr(lib, name)(_ptr(img), ctypes.cast(m, ctypes.c_void_p), ctypes.cast(sd, ctypes.c_void_p), _ptr(params), n,
                                              crops_per_img, C, R, _ptr(out), _stream()), name)
            else:
                name = "hb_pcl_fwd_bf16" if bf16 else "hb_pcl_fwd"
                _lib.check(getattr(lib, name)(_ptr(img), _ptr(params), n, crops_per_img, C, R, _ptr(out), _stream()), name)
        ctx.save_for_backward(params)
        ctx.dims = (Bi, C, R, crops_per_img)
        ctx.bf16 = bf16
        ctx.mark_non_differentiable(rot)
        return out, rot

    @staticmethod
    def backward(ctx, g_out, _g_rot):
        lib = _lib.load()
        (params,) = ctx.saved_tensors
        Bi, C, R, cpi = ctx.dims
        n = Bi * cpi
        dev = params.device
        # a bf16 crop takes its gradient as bf16 (what the consumer's backward produces under autocast), read by the kernel as is
        g_dtype, name = (torch.bfloat16, "hb_pcl_bwd_bf16") if ctx.bf16 else (torch.float32, "hb_pcl_bwd")
        g_out = g_out.contiguous().to(g_dtype)
        g_img = torch.empty(Bi, C, R, R, dtype=torch.float32, device=dev)
        nbytes = lib.hb_pcl_bwd_workspace_bytes(n, cpi, C, R)
        ws = _workspace(nbytes, dev)
        with torch.cuda.device(dev):
            _lib.check(getattr(lib, name)(_ptr(g_out), _ptr(params), n, cpi, C, R, _ptr(g_img), _ptr(ws), nbytes, _stream()), name)
        return g_img, None, None, None, None, None, None


class SilhouetteHandle:
    """Owns one hb_sil* (face table + vertex->corner adjacency of one mesh topology on one CUDA device)."""

    def __init__(self, faces, n_verts, device):
        lib = _lib.load()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("SilhouetteHandle needs a CUDA device")
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        f = torch.as_tensor(faces).detach().to("cpu", torch.int32).contiguous()
        if f.dim() != 2 or f.shape[1] != 3:
            raise ValueError(f"faces: expected (F,3), got {tuple(f.shape)}")
        out = ctypes.c_void_p()
        _lib.check(lib.hb_sil_create(ctypes.c_void_p(f.data_ptr()), f.shape[0], int(n_verts), idx, ctypes.byref(out)), "hb_sil_create")
        self.handle = out
        self.n_faces, self.n_verts = f.shape[0], int(n_verts)
        self.device = torch.device("cuda", idx)

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            try:
                _lib.load().hb_sil_destroy(h)
            except Exception:
                pass


class SoftSilhouetteFunction(torch.autograd.Function):
    """pytorch3d MeshRasterizer + SoftSilhouetteShader as the reference configures them
    (src/models/hands_light/renderer.py:124-199).  verts_cam (B,V,3), K (B,3,3) -> mask (B,1,S,S).
    Gradient w.r.t. verts_cam only (intrinsics are data); the backward reads the forward's scratch
    (face records, per-pixel alpha and depth threshold), so a forward that needs a gradient keeps it."""

    @staticmethod
    def forward(ctx, handle, verts_cam, K, img_res, sigma, blur_radius):
        lib = _lib.load()
        needs_grad = bool(verts_cam.requires_grad)
        verts_cam = _f32c(verts_cam, "verts_cam", (None, handle.n_verts, 3))
        B = verts_cam.shape[0]
        K = _f32c(K, "K", (B, 3, 3))
        dev = verts_cam.device
        if dev != handle.device:
            raise RuntimeError(f"verts_cam is on {dev}, the silhouette handle on {handle.device}")
        S = int(img_res)
        mask = torch.empty(B, 1, S, S, dtype=torch.float32, device=dev)
        nbytes = lib.hb_sil_workspace_bytes(handle.handle, B, S)
        ws = _workspace(nbytes, dev)
        with torch.cuda.device(dev):
            _lib.check(lib.hb_sil_fwd(handle.handle, _ptr(verts_cam), _ptr(K), B, S, float(sigma), float(blur_radius), _ptr(mask),
                                      _ptr(ws), nbytes, _stream()), "hb_sil_fwd")
        if needs_grad:
            ctx.save_for_backward(verts_cam, K)
            ctx.ws, ctx.nbytes, ctx.handle, ctx.cfg = ws, nbytes, handle, (B, S, float(sigma), float(blur_radius))
        return mask

    @staticmethod
    def backward(ctx, g_mask):
        lib = _lib.load()
        verts_cam, K = ctx.saved_tensors
        B, S, sigma, blur = ctx.cfg
        g_mask = g_mask.contiguous().float()
        g_verts = torch.empty_like(verts_cam)
        with torch.cuda.device(verts_cam.device):
            _lib.check(lib.hb_sil_bwd(ctx.handle.handle, _ptr(verts_cam), _ptr(K), _ptr(g_mask), B, S, sigma, blur, _ptr(ctx.ws), ctx.nbytes,
                                      _ptr(g_verts), _stream()), "hb_sil_bwd")
        return None, g_verts, None, None, None, None
