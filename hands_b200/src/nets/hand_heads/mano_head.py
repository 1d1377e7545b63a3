"""Drop-in for the reference's src/nets/hand_heads/mano_head.py:12-65 (`MANOHead`).

Same constructor, same `forward(rotmat, shape, cam, K)`, same nine `xdict` keys with the `.r`/`.l`
postfix; the whole chain (log map -> MANO -> weak-persp camera -> cam-space add -> projection ->
normalisation) is two CUDA launches forward and three backward instead of ~150 torch ops.
"""
import torch.nn as nn

from ....common.body_models import build_mano_aa
from ....common.xdict import xdict
from ....functional import ManoHeadFunction


class MANOHead(nn.Module):
    OUTPUTS = ("vertices", "joints3d", "v3d.cam", "j3d.cam", "j2d.norm", "cam_t")

    def __init__(self, is_rhand, focal_length, img_res, synthetic=False, materialise=None):
        """materialise (extension, default None = all six): the subset of OUTPUTS to compute into memory; the other keys are
        absent from the result (reading one raises KeyError).  E.g. ("j3d.cam", "j2d.norm") for a step whose loss reads only
        the key-points (loss_arctic_sf.py:70-92): the 778-vertex tensors are then never written."""
        super().__init__()
        if materialise is not None and not set(materialise) <= set(self.OUTPUTS):
            raise ValueError(f"materialise: unknown output(s) {sorted(set(materialise) - set(self.OUTPUTS))}")
        self.materialise = None if materialise is None else frozenset(materialise)
        self.mano = build_mano_aa(is_rhand, synthetic=synthetic)
        self.focal_length = focal_length
        self.img_res = img_res
        self.is_rhand = is_rhand

    def forward(self, rotmat, shape, cam, K, pre_rot=None):
        """
        rotmat: (B,16,3,3) rotation matrices, or (B,48) axis-angle
        shape:  (B,10) betas;  cam: (B,3) weak-perspective [s,tx,ty];  K: (B,3,3) intrinsics
        pre_rot (extension, default None): (B,3,3) R_virt2orig fused onto the global orientation
                (the PCL fix-up of hands_light/model.py:330-334) instead of a separate in-place bmm.  A pre_rot
                that requires grad receives it through every output, the returned `pose` included.
        """
        pose = rotmat if rotmat.shape[-1] == 48 else rotmat.reshape(-1, 16, 3, 3)
        if pre_rot is not None:
            # the reference rotates hmr_output["pose"][:,0] in place BEFORE this head (hands_light/model.py:330-334), so the
            # `pose` it returns (mano_head.py:30,61), which feeds the pose loss (loss_arctic_sf.py:23-27), is the ROTATED one
            from ....pcl import apply_virtual_rotation

            rotmat_original = apply_virtual_rotation(pre_rot, pose)
        else:
            rotmat_original = rotmat.clone()
        handle = self.mano.handle(shape.device)
        vertices, v3d_cam, joints3d, j3d_cam, j2d_norm, cam_t = ManoHeadFunction.apply(
            handle, pose, shape, cam, K, None, pre_rot, float(self.img_res), 0.1, None, self.materialise
        )
        return self._pack(cam, cam_t, joints3d, vertices, j3d_cam, v3d_cam, j2d_norm, shape, rotmat_original)

    def _pack(self, cam, cam_t, joints3d, vertices, j3d_cam, v3d_cam, j2d_norm, shape, pose):
        output = xdict()
        output["cam_t.wp"] = cam
        for key, val in (("cam_t", cam_t), ("joints3d", joints3d), ("vertices", vertices), ("j3d.cam", j3d_cam), ("v3d.cam", v3d_cam), ("j2d.norm", j2d_norm)):
            if val is not None:
                output[key] = val
        output["beta"] = shape
        output["pose"] = pose
        return output.postfix(".r" if self.is_rhand else ".l")

    def forward_rot6d(self, pose6d, shape, cam, K, layout="rows", pre_rot=None):
        """Same outputs from the network's 6D pose read-out (B,96) / (B,16,6): the 6D -> rotation-matrix
        conversion the reference runs just before this head (hand_hmr.py:85-87 "rows"; hamer_light/mano_head.py:98-105
        and handoccnet_light/mano_head.py:194 "cols"; common/rot.py:367-381 "cols_paired") is fused into the pose
        kernel.  `pose` in the result is the rotation matrices (one extra small launch), as the reference returns."""
        from ....functional import Rot6dToRotmatFunction

        B = shape.shape[0]
        x6 = pose6d.reshape(B, 16, 6)
        handle = self.mano.handle(shape.device)
        vertices, v3d_cam, joints3d, j3d_cam, j2d_norm, cam_t = ManoHeadFunction.apply(
            handle, x6, shape, cam, K, None, pre_rot, float(self.img_res), 0.1, layout, self.materialise
        )
        pose_mats = Rot6dToRotmatFunction.apply(x6.reshape(-1, 6), layout).reshape(B, 16, 3, 3)
        if pre_rot is not None:   # as in forward(): the returned pose carries the rotated global orientation
            from ....pcl import apply_virtual_rotation

            pose_mats = apply_virtual_rotation(pre_rot, pose_mats)
        return self._pack(cam, cam_t, joints3d, vertices, j3d_cam, v3d_cam, j2d_norm, shape, pose_mats)
