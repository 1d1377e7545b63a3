"""Key-point loss terms and metric partial sums computed straight from the head's outputs (SURVEY.md 8(f) f2).

Drop-in for the terms of the reference's loss that read the geometry path's outputs
(`src/callbacks/loss/loss_arctic_sf.py:70-92,131-136`: `hand_kp3d_loss` on `mano.j3d.cam.*`, `joints_loss` on
`mano.j2d.norm.*`, MSE, masked by `joints_valid_*`, gated by `meta_info['is_j3d_loss'|'is_j2d_loss']`, `.mean()`),
and for the evaluation metrics on the same tensors (`common/metrics.py:23-55` as called from
`src/utils/eval_modules.py:95-118,373,407-421`): instead of per-metric `.cpu()` round trips the kernels leave
partial sums + counts on the device, ready for `hands_b200.distributed.PackedMetrics`.
"""
import torch

from . import _lib
from .functional import _f32c, _ptr, _stream

NOJ = 21


class KeypointLossFunction(torch.autograd.Function):
    """(j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, hand_valid, gate_j3d, gate_j2d, img_res)
    -> (loss_kp3d, loss_kp2d, sums[8]); gradients flow to j3d_cam and j2d_norm only (the targets are data)."""

    @staticmethod
    def forward(ctx, j3d, j2d, gt3, gt2, jv, hv, gate3, gate2, img_res):
        lib = _lib.load()
        B = j3d.shape[0]
        j3d, gt3 = _f32c(j3d, "j3d_cam", (B, NOJ, 3)), _f32c(gt3, "gt_j3d_cam", (B, NOJ, 3))
        j2d, gt2 = _f32c(j2d, "j2d_norm", (B, NOJ, 2)), _f32c(gt2, "gt_j2d_norm", (B, NOJ, 2))
        jv = _f32c(jv, "joints_valid", (B, NOJ))
        hv, gate3, gate2 = _f32c(hv, "hand_valid", (B,)), _f32c(gate3, "gate_j3d", (B,)), _f32c(gate2, "gate_j2d", (B,))
        dev = j3d.device
        partial = torch.empty(max(B, 1), _lib.KP_SUMS, dtype=torch.float32, device=dev)
        sums = torch.empty(_lib.KP_SUMS, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = lib.hb_kp_loss_fwd(_ptr(j3d), _ptr(j2d), _ptr(gt3), _ptr(gt2), _ptr(jv), _ptr(hv), _ptr(gate3), _ptr(gate2), B, float(img_res),
                                    _ptr(partial), _ptr(sums), _stream())
        _lib.check(rc, "hb_kp_loss_fwd")
        ctx.save_for_backward(j3d, j2d, gt3, gt2, jv, gate3, gate2)
        ctx.set_materialize_grads(False)
        n = max(B, 1) * NOJ
        ctx.mark_non_differentiable(sums)
        return sums[0] / (n * 3), sums[1] / (n * 2), sums

    @staticmethod
    def backward(ctx, g3, g2, _g_sums):
        lib = _lib.load()
        j3d, j2d, gt3, gt2, jv, gate3, gate2 = ctx.saved_tensors
        B = j3d.shape[0]
        g3 = None if g3 is None else g3.reshape(1).contiguous().float()
        g2 = None if g2 is None else g2.reshape(1).contiguous().float()
        g_j3d = torch.empty_like(j3d) if ctx.needs_input_grad[0] else None
        g_j2d = torch.empty_like(j2d) if ctx.needs_input_grad[1] else None
        with torch.cuda.device(j3d.device):
            rc = lib.hb_kp_loss_bwd(_ptr(j3d), _ptr(j2d), _ptr(gt3), _ptr(gt2), _ptr(jv), _ptr(gate3), _ptr(gate2), B, _ptr(g3), _ptr(g2),
                                    _ptr(g_j3d), _ptr(g_j2d), _stream())
        _lib.check(rc, "hb_kp_loss_bwd")
        return g_j3d, g_j2d, None, None, None, None, None, None, None


def keypoint_losses(j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, hand_valid=None, gate_j3d=None, gate_j2d=None, img_res=224):
    """Returns (loss_kp3d, loss_kp2d, sums) for one hand side; `sums` is the 8-float device vector described in
    include/hands_b200.h (MPJPE-RA and pixel-error numerators / counts in [2..5])."""
    return KeypointLossFunction.apply(j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, hand_valid, gate_j3d, gate_j2d, float(img_res))


def mrrpe_sums(j3d_cam_r, j3d_cam_l, gt_j3d_cam_r, gt_j3d_cam_l, valid=None):
    """common/metrics.py:47-55 as partial sums: tensor([sum of valid distances, number of valid samples, 0...])."""
    lib = _lib.load()
    B = j3d_cam_r.shape[0]
    args = [_f32c(t, n, (B, NOJ, 3)) for t, n in ((j3d_cam_r, "j3d_cam_r"), (j3d_cam_l, "j3d_cam_l"), (gt_j3d_cam_r, "gt_j3d_cam_r"), (gt_j3d_cam_l, "gt_j3d_cam_l"))]
    valid = _f32c(valid, "valid", (B,))
    dev = args[0].device
    partial = torch.empty(max(B, 1), _lib.KP_SUMS, dtype=torch.float32, device=dev)
    sums = torch.empty(_lib.KP_SUMS, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.hb_mrrpe(*[_ptr(t) for t in args], _ptr(valid), B, _ptr(partial), _ptr(sums), _stream())
    _lib.check(rc, "hb_mrrpe")
    return sums


def procrustes_metrics(pred, gt, hand_valid=None, root_pred=None, root_gt=None, return_aligned=False):
    """Procrustes-aligned and root-relative point errors of one hand side, as device partial sums (hb_procrustes_metrics):
    the similarity fit of the HMR / ARCTIC `compute_similarity_transform` (src/utils/eval_modules.py:136-219, a numpy SVD
    per sample there) solved per hand on the GPU, then the mean point distance after alignment (PA) and after subtracting
    the root points (RA).  pred, gt (B,N,3) fp32 CUDA; root_pred, root_gt (B,3) or None (= point 0); hand_valid (B,) or
    None.  On joints (N = 21) PA is PA-MPJPE and RA is MPJPE-RA; on `v3d.cam` vertices pass joint 0 of `j3d.cam` as the
    roots and RA is the root-relative MPVPE.  A metric: inputs are detached, there is no gradient.

    Returns (sums, per_hand[, aligned]): sums (8,) = [PA sum over valid non-degenerate hands, their count, RA sum over valid
    hands, their count, valid hands left out as degenerate (var == 0, e.g. N = 1), 0, 0, 0]; per_hand (B,2) = [PA, RA],
    NaN for invalid hands and PA NaN for degenerate ones; aligned (B,N,3) = s R pred + t.  With
    `hands_b200.distributed.PackedMetrics`:

        sums, _ = procrustes_metrics(pred["mano.j3d.cam.r"], gt["mano.j3d.cam.r"], gt["right_valid"])
        pm.add("pa_mpjpe/r", sums[0], sums[1])
        pm.add("mpjpe_ra/r", sums[2], sums[3])
    """
    lib = _lib.load()
    d = lambda t: t.detach() if isinstance(t, torch.Tensor) else t  # noqa: E731
    pred = _f32c(d(pred), "pred", (None, None, 3))
    B, N = pred.shape[:2]
    if N < 1:
        raise ValueError("pred: expected at least one point per hand (N >= 1)")
    gt = _f32c(d(gt), "gt", (B, N, 3))
    root_pred, root_gt = _f32c(d(root_pred), "root_pred", (B, 3)), _f32c(d(root_gt), "root_gt", (B, 3))
    hand_valid = _f32c(d(hand_valid), "hand_valid", (B,))
    dev = pred.device
    partial = torch.empty(max(B, 1), _lib.KP_SUMS, dtype=torch.float32, device=dev)
    sums = torch.empty(_lib.KP_SUMS, dtype=torch.float32, device=dev)
    per_hand = torch.empty(B, 2, dtype=torch.float32, device=dev)
    aligned = torch.empty(B, N, 3, dtype=torch.float32, device=dev) if return_aligned else None
    with torch.cuda.device(dev):
        rc = lib.hb_procrustes_metrics(_ptr(pred), _ptr(gt), B, N, _ptr(root_pred), _ptr(root_gt), _ptr(hand_valid), _ptr(per_hand),
                                       _ptr(aligned), _ptr(partial), _ptr(sums), _stream())
    _lib.check(rc, "hb_procrustes_metrics")
    return (sums, per_hand, aligned) if return_aligned else (sums, per_hand)


class VectorLossFunction(torch.autograd.Function):
    """loss = mean_b,e [ valid*valid2*gate * ( ((pred - pred_minus) - (gt - gt_minus))^2 + (pred2 - (gt - gt_minus))^2 ) ].
    Gradients flow to pred, pred_minus and pred2; targets and masks are data.  (hb_vec_loss_fwd/bwd)"""

    @staticmethod
    def forward(ctx, pred, pred_minus, pred2, gt, gt_minus, valid, valid2, gate):
        lib = _lib.load()
        B, D = pred.shape   # (B, D) views are made by the caller, so autograd sees the gradient in the shape it gave
        f = lambda t, n: None if t is None else _f32c(t, n, (B, D))  # noqa: E731
        pred, pred_minus, pred2, gt, gt_minus = f(pred, "pred"), f(pred_minus, "pred_minus"), f(pred2, "pred2"), f(gt, "gt"), f(gt_minus, "gt_minus")
        valid, valid2, gate = _f32c(valid, "valid", (B,)), _f32c(valid2, "valid2", (B,)), _f32c(gate, "gate", (B,))
        dev = pred.device
        partial = torch.empty(max(B, 1), dtype=torch.float32, device=dev)
        out = torch.empty(1, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = lib.hb_vec_loss_fwd(_ptr(pred), _ptr(pred_minus), _ptr(gt), _ptr(gt_minus), _ptr(pred2), _ptr(valid), _ptr(valid2), _ptr(gate), B, D,
                                     _ptr(partial), _ptr(out), _stream())
        _lib.check(rc, "hb_vec_loss_fwd")
        ctx.save_for_backward(pred, pred_minus, pred2, gt, gt_minus, valid, valid2, gate)
        ctx.dims = (B, D)
        return out[0] / float(max(B, 1) * D)

    @staticmethod
    def backward(ctx, g):
        lib = _lib.load()
        pred, pred_minus, pred2, gt, gt_minus, valid, valid2, gate = ctx.saved_tensors
        B, D = ctx.dims
        g = g.reshape(1).contiguous().float()
        need = ctx.needs_input_grad
        g_pred = torch.empty_like(pred) if need[0] else None
        g_minus = torch.empty_like(pred_minus) if (pred_minus is not None and need[1]) else None
        g_pred2 = torch.empty_like(pred2) if (pred2 is not None and need[2]) else None
        with torch.cuda.device(pred.device):
            rc = lib.hb_vec_loss_bwd(_ptr(pred), _ptr(pred_minus), _ptr(gt), _ptr(gt_minus), _ptr(pred2), _ptr(valid), _ptr(valid2), _ptr(gate), B, D,
                                     _ptr(g), _ptr(g_pred), _ptr(g_minus), _ptr(g_pred2), _stream())
        _lib.check(rc, "hb_vec_loss_bwd")
        return g_pred, g_minus, g_pred2, None, None, None, None, None


def vector_loss(pred, gt, valid=None, gate=None, pred2=None, pred_minus=None, gt_minus=None, valid2=None):
    """One masked, gated vector MSE term of `compute_loss_light` (src/callbacks/loss/loss_arctic_sf.py:52-69, 94-158 with
    src/utils/loss_modules.py:99-113): returns the scalar the reference calls `loss_*.mean()`.  Shapes (B, ...) with equal
    trailing sizes; `pred2` is a second prediction scored against the same target (cam_t.wp.init); `pred_minus`/`gt_minus`
    are subtracted first (the relative translation l - r); valid/valid2/gate are (B,) masks."""
    B = pred.shape[0]
    v = lambda t: None if t is None else t.reshape(B, -1)  # noqa: E731
    return VectorLossFunction.apply(v(pred), v(pred_minus), v(pred2), v(gt), v(gt_minus), valid, valid2, gate)


def axis_angle_to_matrix(aa):
    """pytorch3d.transforms.axis_angle_to_matrix as the reference applies it to the GT pose (loss_arctic_sf.py:48-49):
    (...,3) -> (...,3,3); no gradient (GT side)."""
    lead = aa.shape[:-1]
    x = _f32c(aa.detach().reshape(-1, 3), "axis_angle", (None, 3))
    R = torch.empty(x.shape[0], 3, 3, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().hb_axis_angle_to_matrix(_ptr(x), x.shape[0], _ptr(R), _stream()), "hb_axis_angle_to_matrix")
    return R.reshape(lead + (3, 3))


class MaskL1LossFunction(torch.autograd.Function):
    """mean over (B, n) of |pred - gt| * valid[b] * gate[b]; gradient w.r.t. pred only."""

    @staticmethod
    def forward(ctx, pred, gt, valid, gate):
        B = pred.shape[0]          # (B, n) views: the caller flattens (autograd must see the same shape come back)
        pred = _f32c(pred, "pred_mask", (None, None))
        n = pred.shape[1]
        gt = _f32c(gt.detach().reshape(B, -1).float(), "gt_mask", (B, n))
        valid = None if valid is None else _f32c(valid.detach().float().reshape(-1), "valid", (B,))
        gate = None if gate is None else _f32c(gate.detach().float().reshape(-1), "gate", (B,))
        partial = torch.empty(max(B, 1), dtype=torch.float32, device=pred.device)
        loss = torch.empty(1, dtype=torch.float32, device=pred.device)
        with torch.cuda.device(pred.device):
            _lib.check(_lib.load().hb_mask_l1_loss_fwd(_ptr(pred), _ptr(gt), _ptr(valid), _ptr(gate), B, n, _ptr(partial), _ptr(loss), _stream()),
                       "hb_mask_l1_loss_fwd")
        ctx.save_for_backward(pred, gt, valid, gate)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        pred, gt, valid, gate = ctx.saved_tensors
        B, n = pred.shape
        g = g.reshape(1).contiguous().float()
        g_pred = torch.empty_like(pred)
        with torch.cuda.device(pred.device):
            _lib.check(_lib.load().hb_mask_l1_loss_bwd(_ptr(pred), _ptr(gt), _ptr(valid), _ptr(gate), _ptr(g), B, n, _ptr(g_pred), _stream()),
                       "hb_mask_l1_loss_bwd")
        return g_pred, None, None, None


def render_loss(pred_mask, gt_mask, is_valid, gate=None):
    """`render_loss(...).mean()` of the reference (src/utils/loss_modules.py:146-152 as used at
    src/callbacks/loss/loss_arctic_sf.py:177-183, `gate` = meta_info['is_mask_loss']): one fused L1 + reduction."""
    B = pred_mask.shape[0]
    return MaskL1LossFunction.apply(pred_mask.reshape(B, -1), gt_mask, is_valid, gate)


def compute_loss_light(pred, gt, meta_info, img_res=224):
    """Drop-in for the MANO terms of the reference's `compute_loss_light` (src/callbacks/loss/loss_arctic_sf.py:20-158): same
    dictionary of (loss, weight) pairs under the same keys, every term one fused launch (+ one fixed-order reduction) on the
    path's outputs.  `pred` / `gt` / `meta_info` use the reference's key names; masks are float tensors like the reference's.
    (The optional grasp term, :160-171, is a cross-entropy on a classifier head -- not on the geometry path.)"""
    out = {}
    rv, lv = gt["right_valid"], gt["left_valid"]
    gates = {k: meta_info[k].float() for k in ("is_cam_loss", "is_j2d_loss", "is_j3d_loss", "is_pose_loss", "is_beta_loss")}
    for side, valid, jv in (("r", rv, gt["joints_valid_r"]), ("l", lv, gt["joints_valid_l"])):
        gt_pose = axis_angle_to_matrix(gt[f"mano.pose.{side}"].reshape(-1, 3)).reshape(-1, 16, 3, 3)
        out[f"loss/mano/cam_t/{side}"] = (vector_loss(pred[f"mano.cam_t.wp.{side}"], gt[f"mano.cam_t.wp.{side}"], valid, gates["is_cam_loss"],
                                                      pred2=pred[f"mano.cam_t.wp.init.{side}"]).view(-1), 1.0)
        l3, l2, _ = keypoint_losses(pred[f"mano.j3d.cam.{side}"], pred[f"mano.j2d.norm.{side}"], gt[f"mano.j3d.cam.{side}"], gt[f"mano.j2d.norm.{side}"],
                                    jv, None, gates["is_j3d_loss"], gates["is_j2d_loss"], img_res)
        out[f"loss/mano/kp2d/{side}"] = (l2.view(-1), 5.0)
        out[f"loss/mano/kp3d/{side}"] = (l3.view(-1), 5.0)
        out[f"loss/mano/pose/{side}"] = (vector_loss(pred[f"mano.pose.{side}"], gt_pose, valid, gates["is_pose_loss"]).view(-1), 10.0)
        out[f"loss/mano/beta/{side}"] = (vector_loss(pred[f"mano.beta.{side}"], gt[f"mano.beta.{side}"], valid, gates["is_beta_loss"]).view(-1), 0.001)
    out["loss/mano/transl/l"] = (vector_loss(pred["mano.cam_t.wp.l"], gt["mano.cam_t.wp.l"], rv, gates["is_cam_loss"], pred_minus=pred["mano.cam_t.wp.r"],
                                             gt_minus=gt["mano.cam_t.wp.r"], valid2=lv).view(-1), 1.0)
    if "render.r" in pred and "render.r" in gt:   # args.use_render_seg_loss (loss_arctic_sf.py:172-183)
        gate = meta_info["is_mask_loss"].float() if "is_mask_loss" in meta_info else None
        for side in ("r", "l"):
            out[f"loss/mask/{side}"] = (render_loss(pred[f"render.{side}"], gt[f"render.{side}"], gt[f"render_valid_{side}"], gate).view(-1), 10.0)
    return out
