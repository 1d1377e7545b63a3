"""Batched Perspective Crop Layer (seam 4 of SURVEY.md §8(b); no batched function exists in the
reference, where the closure at src/datasets/hands_light_dataset.py:354-467 runs per sample on the
CPU inside the data loader)."""
import torch

from .functional import PerspectiveCropFunction, RotApplyFunction, check_crop_dtype


def perspective_crop(img, bbox_xyxy, K, img_res=224, crops_per_img=1, mean=None, std=None, out_dtype=torch.float32):
    """img (Bi,3,img_res,img_res) fp32 CUDA; bbox_xyxy (Bi*crops_per_img,4) int [x0,y0,x1,y1] inside the
    image; K (Bi*crops_per_img,3,3).  Crop c samples image c // crops_per_img.
    Returns crop (Bi*crops_per_img,3,img_res,img_res) and R_virt2orig (Bi*crops_per_img,3,3).
    Semantics = lines 425-467 of the reference closure; gradient flows to img.

    Extension: `img` may be the data loader's uint8 image with `mean`/`std` (the reference's img_norm_mean/std, C floats):
    the normalisation (u/255 - mean)/std the reference applies before the crop (hands_light_dataset.py:177-184) is fused
    into the gather -- same crops, a quarter of the bytes over PCIe.  No gradient flows to a uint8 image.

    out_dtype=torch.bfloat16 (for a backbone trained under bf16 autocast): the crop is returned as bf16, bit-identical to
    the fp32 crop rounded to nearest even, and its gradient is consumed as bf16 -- no cast kernel on either side.
    R_virt2orig and the gradient w.r.t. an fp32 `img` stay fp32.  Any other dtype raises TypeError."""
    check_crop_dtype(out_dtype)
    if img.shape[-1] != img_res or img.shape[-2] != img_res:
        raise ValueError(f"img must be {img_res}x{img_res} (the reference crops from the resized full image)")
    return PerspectiveCropFunction.apply(img, bbox_xyxy, K, int(crops_per_img), mean, std, out_dtype)


def apply_virtual_rotation(R_virt2orig, pose):
    """pose (B,16,3,3): returns a copy with pose[:,0] <- R_virt2orig @ pose[:,0]
    (src/models/hands_light/model.py:330-334, written out-of-place so autograd stays valid)."""
    rotated = RotApplyFunction.apply(R_virt2orig, pose[:, 0])
    return torch.cat([rotated[:, None], pose[:, 1:]], dim=1)


def kpe_features(bbox_xyxy, K, n_freq):
    """KPE angles of the crop boxes and their sinusoidal encodings, batched on the GPU (the reference computes the angles per
    sample on the CPU, src/datasets/hands_light_dataset.py:259-279, and the encodings in the model,
    src/models/hands_light/model.py:444-460).  bbox_xyxy (n,4) int, K (n,3,3) ->
    dict(center_angle (n,2), corner_angle (n,8), center_pos_enc (n, n_freq*4), corner_pos_enc (n, n_freq*16))."""
    import torch

    from . import _lib
    from .functional import _f32c, _ptr, _stream

    K = _f32c(K, "K", (None, 3, 3))
    n = K.shape[0]
    bbox = bbox_xyxy.to(device=K.device, dtype=torch.int32).contiguous()
    if bbox.shape != (n, 4):
        raise ValueError(f"bbox_xyxy: expected shape ({n}, 4), got {tuple(bbox.shape)}")
    new = lambda c: torch.empty(n, c, dtype=torch.float32, device=K.device)  # noqa: E731
    out = {"center_angle": new(2), "corner_angle": new(8), "center_pos_enc": new(n_freq * 4), "corner_pos_enc": new(n_freq * 16)}
    with torch.cuda.device(K.device):
        rc = _lib.load().hb_kpe_features(_ptr(bbox), _ptr(K), n, int(n_freq), _ptr(out["center_angle"]), _ptr(out["corner_angle"]),
                                         _ptr(out["center_pos_enc"]), _ptr(out["corner_pos_enc"]), _stream())
    _lib.check(rc, "hb_kpe_features")
    return out
