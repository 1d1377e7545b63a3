"""bf16 crop planes of the Perspective Crop Layer (hb_pcl_fwd_bf16, hb_pcl_fwd_u8_bf16, hb_pcl_bwd_bf16) against their fp32
twins: the bf16 crop is the fp32 crop rounded to nearest even, bit for bit, and the image gradient from a bf16 crop gradient
is the fp32 backward's on the exactly widened gradient, bit for bit.  "Equal" below compares bit patterns."""
import ctypes

import pytest
import torch

from hands_b200 import _lib
from hands_b200.functional import _ptr, _stream
from hands_b200.synthetic import synthetic_pcl_inputs
from oracle import geometry_oracle as O

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
MEAN, STD = (0.485, 0.456, 0.406, 0.5), (0.229, 0.224, 0.225, 0.25)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture
def lib():
    return _lib.load()


@pytest.fixture(params=[0, 1], ids=["fast", "exact"])
def mode(request, lib):
    prev = lib.hb_pcl_set_exact(request.param)
    yield request.param
    lib.hb_pcl_set_exact(prev)


def bits_equal(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    if a.dtype == BF16:
        return torch.equal(a.view(torch.int16), b.view(torch.int16))
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def boxes(n, res, seed):
    """synthetic boxes inside the image, the first three replaced by one touching the top-left corner, one touching the
    bottom-right corner and an empty box (s = img_res)"""
    _, bbox, K = synthetic_pcl_inputs(n, seed=seed, img_res=res, smin=res // 4, smax=3 * res // 4)
    if n >= 3:
        bbox[0] = torch.tensor([0, 0, min(30, res - 1), min(40, res - 1)])
        bbox[1] = torch.tensor([max(res - 41, 0), max(res - 31, 0), res - 1, res - 1])
        bbox[2] = torch.tensor([7, 9, 7, 9])
    return bbox, K


def setup_params(lib, bbox, K, res):
    n = bbox.shape[0]
    params = torch.empty(n, _lib.PCL_PARAM_FLOATS, dtype=torch.float32, device=bbox.device)
    rot = torch.empty(n, 3, 3, dtype=torch.float32, device=bbox.device)
    _lib.check(lib.hb_pcl_setup(_ptr(bbox), _ptr(K), n, res, _ptr(params), _ptr(rot), _stream()), "hb_pcl_setup")
    return params


def forward(lib, src, params, cpi, out):
    """one crop-layer forward into `out` (fp32 or bf16, any element offset) from an fp32 or uint8 source"""
    n, C, R = out.shape[0], out.shape[1], out.shape[2]
    bf = out.dtype == BF16
    if src.dtype == torch.uint8:
        m = (ctypes.c_float * C)(*MEAN[:C])
        s = (ctypes.c_float * C)(*STD[:C])
        fn = lib.hb_pcl_fwd_u8_bf16 if bf else lib.hb_pcl_fwd_u8
        rc = fn(_ptr(src), ctypes.cast(m, ctypes.c_void_p), ctypes.cast(s, ctypes.c_void_p), _ptr(params), n, cpi, C, R, _ptr(out), _stream())
    else:
        fn = lib.hb_pcl_fwd_bf16 if bf else lib.hb_pcl_fwd
        rc = fn(_ptr(src), _ptr(params), n, cpi, C, R, _ptr(out), _stream())
    _lib.check(rc, "crop forward")
    return out


def backward(lib, g_out, params, cpi, ws_bytes=None):
    n, C, R = g_out.shape[0], g_out.shape[1], g_out.shape[2]
    if ws_bytes is None:
        ws_bytes = lib.hb_pcl_bwd_workspace_bytes(n, cpi, C, R)
    ws = torch.empty((ws_bytes + 3) // 4, dtype=torch.float32, device=g_out.device)
    g_img = torch.empty(n // cpi, C, R, R, dtype=torch.float32, device=g_out.device)
    fn = lib.hb_pcl_bwd_bf16 if g_out.dtype == BF16 else lib.hb_pcl_bwd
    _lib.check(fn(_ptr(g_out), _ptr(params), n, cpi, C, R, _ptr(g_img), _ptr(ws), ws_bytes, _stream()), "crop backward")
    return g_img


def offset_view(n, C, R, dtype, dev):
    """(n,C,R,R) view one element into its allocation: no two-element alignment, so no vector stores / four-column loads"""
    buf = torch.zeros(n * C * R * R + 1, dtype=dtype, device=dev)
    return buf[1:].view(n, C, R, R)


def source(B, C, res, seed, u8, dev):
    g = torch.Generator().manual_seed(seed)
    if u8:
        return torch.randint(0, 256, (B, C, res, res), generator=g, dtype=torch.uint8).to(dev)
    return torch.randn(B, C, res, res, generator=g).to(dev)


# ---- forward ---------------------------------------------------------------------------------------------------------
FWD_SHAPES = [(224, 3, 1, 6), (224, 3, 2, 4), (224, 3, 5, 2), (50, 3, 1, 4), (96, 1, 1, 4), (64, 4, 2, 3)]


@pytest.mark.parametrize("src_u8", [False, True], ids=["fp32src", "u8src"])
@pytest.mark.parametrize("res,C,cpi,B", FWD_SHAPES)
def test_forward_is_rounded_fp32_forward(dev, lib, mode, res, C, cpi, B, src_u8):
    """R = 224 with 1, 2 and 5 (> PCL_RECS) crops per image and the generic paths (R, C) = (50, 3), (96, 1), (64, 4), in both
    arithmetic modes, from an fp32 and from an 8-bit source; boxes touching the image corners and an empty box (s = R)."""
    n = B * cpi
    bbox, K = boxes(n, res, seed=res + cpi)
    params = setup_params(lib, bbox.to(dev), K.to(dev), res)
    src = source(B, C, res, seed=res * 7 + C, u8=src_u8, dev=dev)
    ref = forward(lib, src, params, cpi, torch.empty(n, C, res, res, device=dev))
    got = forward(lib, src, params, cpi, torch.empty(n, C, res, res, dtype=BF16, device=dev))
    torch.cuda.synchronize()
    assert float(ref.abs().max()) > 0
    assert bits_equal(got, ref.to(BF16))
    # an output one element into its allocation (scalar 2-byte stores instead of the paired stores)
    got_off = forward(lib, src, params, cpi, offset_view(n, C, res, BF16, dev))
    assert bits_equal(got_off, ref.to(BF16))


def test_forward_box_larger_than_image(dev, lib, mode):
    """s > img_res (down-sampling) takes the forward's generic in-kernel path; forward only."""
    res = 64
    src = source(2, 3, res, seed=3, u8=False, dev=dev)
    bbox = torch.tensor([[-10, -5, 90, 80], [5, -20, 60, 75]], dtype=torch.int32, device=dev)
    K = torch.tensor([[[80.0, 0, 32], [0, 80.0, 32], [0, 0, 1]], [[120.0, 0, 30], [0, 110.0, 33], [0, 0, 1]]], device=dev)
    params = setup_params(lib, bbox, K, res)
    ref = forward(lib, src, params, 1, torch.empty(2, 3, res, res, device=dev))
    got = forward(lib, src, params, 1, torch.empty(2, 3, res, res, dtype=BF16, device=dev))
    assert bits_equal(got, ref.to(BF16))


def test_forward_against_oracle_within_bf16_rounding(dev):
    from hands_b200.pcl import perspective_crop

    B, cpi, res = 3, 2, 96
    n = B * cpi
    img, bbox, K = synthetic_pcl_inputs(n, seed=B, img_res=res, smin=res // 4, smax=3 * res // 4)
    img = img[:B].contiguous()
    with torch.no_grad():
        crop, _ = perspective_crop(img.to(dev), bbox.to(dev), K.to(dev), img_res=res, crops_per_img=cpi, out_dtype=BF16)
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        ref, _ = O.perspective_crop(img.repeat_interleave(cpi, dim=0), bbox, K, res)
    finally:
        torch.set_num_threads(nt)
    err = (crop.float().cpu() - ref).abs()
    assert bool((err <= 2.0 ** -8 * ref.abs() + 5e-5).all()), float((err - 2.0 ** -8 * ref.abs()).max())


# ---- backward --------------------------------------------------------------------------------------------------------
BWD_SHAPES = [(224, 3, 1, 6), (224, 3, 2, 4), (224, 3, 5, 2), (50, 3, 1, 4), (96, 1, 1, 4), (64, 4, 2, 3)]


@pytest.mark.parametrize("res,C,cpi,B", BWD_SHAPES)
def test_backward_is_fp32_backward_on_widened_gradient(dev, lib, res, C, cpi, B):
    n = B * cpi
    bbox, K = boxes(n, res, seed=res + 11 * cpi)
    params = setup_params(lib, bbox.to(dev), K.to(dev), res)
    g16 = torch.randn(n, C, res, res, generator=torch.Generator(device=dev).manual_seed(res + C), device=dev).to(BF16)
    ref = backward(lib, g16.float(), params, cpi)
    got = backward(lib, g16, params, cpi)
    torch.cuda.synchronize()
    assert float(ref.abs().max()) > 0
    assert bits_equal(got, ref)
    # a gradient one element into its allocation (scalar-column transposed resize), against an fp32 gradient offset alike
    g16o, g32o = offset_view(n, C, res, BF16, dev), offset_view(n, C, res, torch.float32, dev)
    g16o.copy_(g16)
    g32o.copy_(g16.float())
    ref_o = backward(lib, g32o, params, cpi)
    got_o = backward(lib, g16o, params, cpi)
    assert bits_equal(got_o, ref_o)
    # bit-reproducible run to run
    assert bits_equal(backward(lib, g16, params, cpi), got)


@pytest.mark.parametrize("fmin,fmax,cpi", [(300.0, 1500.0, 2), (110.0, 200.0, 2), (60.0, 110.0, 3), (2000.0, 9000.0, 1)])
def test_backward_perspective_regimes(dev, lib, fmin, fmax, cpi):
    """The four perspective regimes of the fp32 gather-form test (mild to extreme foreshortening, region-scan fallback)."""
    B = 12
    n = B * cpi
    _, bbox, K = synthetic_pcl_inputs(n, seed=int(fmin), img_res=224, smin=40, smax=224)
    g = torch.Generator().manual_seed(int(fmax))
    f = fmin + (fmax - fmin) * torch.rand(n, generator=g)
    K[:, 0, 0] = f
    K[:, 1, 1] = f * (0.9 + 0.2 * torch.rand(n, generator=g))
    K[:, 0, 2] += 30 * torch.randn(n, generator=g)
    bbox[0] = torch.tensor([0, 0, 223, 223])
    bbox[1] = torch.tensor([150, 160, 223, 223])
    bbox[2] = torch.tensor([0, 0, 40, 223])
    params = setup_params(lib, bbox.to(dev), K.to(dev), 224)
    g16 = torch.randn(n, 3, 224, 224, generator=g).to(BF16).to(dev)
    got = backward(lib, g16, params, cpi)
    assert bits_equal(got, backward(lib, g16.float(), params, cpi))
    assert bits_equal(got, backward(lib, g16, params, cpi))


def test_backward_several_workspace_chunks(dev, lib):
    """A workspace of three images' worth for 8 images: the backward runs in three chunks; same chunking for both dtypes."""
    B, cpi, res = 8, 2, 224
    n = B * cpi
    bbox, K = boxes(n, res, seed=17)
    params = setup_params(lib, bbox.to(dev), K.to(dev), res)
    ws3 = 3 * lib.hb_pcl_bwd_workspace_bytes(cpi, cpi, 3, res)
    g16 = torch.randn(n, 3, res, res, generator=torch.Generator(device=dev).manual_seed(8), device=dev).to(BF16)
    got = backward(lib, g16, params, cpi, ws_bytes=ws3)
    assert bits_equal(got, backward(lib, g16.float(), params, cpi, ws_bytes=ws3))
    assert float(got[-1].abs().max()) > 0


def test_more_than_65535_crops(dev):
    """66,000 crops: the forward's launch split at 65,535 crops and the backward's image chunks step through bf16 buffers in
    bf16 elements; a slice recomputed on its own matches bit for bit, forward and backward."""
    from hands_b200.pcl import perspective_crop

    res, n = 32, 66000
    g = torch.Generator().manual_seed(9)
    img = torch.randn(n, 1, res, res, generator=g).to(dev)
    side = torch.randint(8, 25, (n,), generator=g)
    x0 = torch.randint(0, res - 25, (n,), generator=g)
    y0 = torch.randint(0, res - 25, (n,), generator=g)
    bbox = torch.stack([x0, y0, x0 + side, y0 + side], dim=1).int().to(dev)
    K = torch.tensor([[60.0, 0, 16], [0, 60.0, 16], [0, 0, 1]]).expand(n, 3, 3).contiguous().to(dev)
    w = torch.randn(n, 1, res, res, generator=g).to(BF16).to(dev)
    x = img.clone().requires_grad_(True)
    crop, _ = perspective_crop(x, bbox, K, img_res=res, out_dtype=BF16)
    (gx,) = torch.autograd.grad(crop, x, grad_outputs=w)
    sl = slice(65500, 65900)
    xs = img[sl].clone().requires_grad_(True)
    cs, _ = perspective_crop(xs, bbox[sl], K[sl], img_res=res, out_dtype=BF16)
    (gs,) = torch.autograd.grad(cs, xs, grad_outputs=w[sl])
    assert bits_equal(cs, crop[sl].detach()) and bits_equal(gs, gx[sl])
    assert float(crop[-1].float().abs().max()) > 0
    x32 = img.clone().requires_grad_(True)
    c32, _ = perspective_crop(x32, bbox, K, img_res=res)
    (g32,) = torch.autograd.grad(c32, x32, grad_outputs=w.float())
    assert bits_equal(crop.detach(), c32.detach().to(BF16)) and bits_equal(gx, g32)


# ---- autograd --------------------------------------------------------------------------------------------------------
def test_autograd_bf16_crop(dev):
    from hands_b200.pcl import perspective_crop

    B, cpi, res = 4, 2, 224
    n = B * cpi
    img, bbox, K = synthetic_pcl_inputs(n, seed=5, img_res=res)
    img, bbox, K = img[:B].contiguous().to(dev), bbox.to(dev), K.to(dev)
    x16 = img.clone().requires_grad_(True)
    crop16, rot16 = perspective_crop(x16, bbox, K, img_res=res, crops_per_img=cpi, out_dtype=BF16)
    assert crop16.dtype == BF16 and rot16.dtype == torch.float32 and crop16.requires_grad
    x32 = img.clone().requires_grad_(True)
    crop32, rot32 = perspective_crop(x32, bbox, K, img_res=res, crops_per_img=cpi)
    assert bits_equal(crop16.detach(), crop32.detach().to(BF16)) and bits_equal(rot16, rot32)
    w = torch.randn(n, 3, res, res, generator=torch.Generator(device=dev).manual_seed(1), device=dev).to(BF16)
    (g16,) = torch.autograd.grad(crop16, x16, grad_outputs=w)
    (g32,) = torch.autograd.grad(crop32, x32, grad_outputs=w.float())
    assert g16.dtype == torch.float32 and bits_equal(g16, g32)
    # a uint8 source: bf16 crops, no gradient
    u8 = torch.randint(0, 256, (B, 3, res, res), generator=torch.Generator().manual_seed(2), dtype=torch.uint8).to(dev)
    c8, _ = perspective_crop(u8, bbox, K, img_res=res, crops_per_img=cpi, mean=MEAN[:3], std=STD[:3], out_dtype=BF16)
    c8f, _ = perspective_crop(u8, bbox, K, img_res=res, crops_per_img=cpi, mean=MEAN[:3], std=STD[:3])
    assert c8.dtype == BF16 and not c8.requires_grad and bits_equal(c8, c8f.to(BF16))
    for bad in (torch.float16, torch.float64):
        with pytest.raises(TypeError, match="out_dtype"):
            perspective_crop(x16, bbox, K, img_res=res, crops_per_img=cpi, out_dtype=bad)


def test_autocast_conv_consumes_bf16_crop(dev):
    """A bf16 conv under torch.autocast reads the crop as is and back-propagates into the fp32 image through
    hb_pcl_bwd_bf16: the image gradient equals the fp32 backward of the (widened) gradient the conv returned."""
    from hands_b200.pcl import perspective_crop

    B, res = 3, 224
    img, bbox, K = synthetic_pcl_inputs(B, seed=6, img_res=res)
    img, bbox, K = img.to(dev), bbox.to(dev), K.to(dev)
    conv = torch.nn.Conv2d(3, 8, 3, padding=1).to(dev)
    x = img.clone().requires_grad_(True)
    seen = {}
    with torch.autocast("cuda", dtype=torch.bfloat16):
        crop, _ = perspective_crop(x, bbox, K, img_res=res, out_dtype=BF16)
        crop.register_hook(lambda g: seen.setdefault("g", g))
        y = conv(crop)
        assert y.dtype == BF16
        loss = y.float().square().mean()
    loss.backward()
    g = seen["g"]
    assert g.dtype == BF16 and x.grad.dtype == torch.float32
    assert torch.isfinite(x.grad).all() and float(x.grad.abs().max()) > 0
    x32 = img.clone().requires_grad_(True)
    c32, _ = perspective_crop(x32, bbox, K, img_res=res)
    (g32,) = torch.autograd.grad(c32, x32, grad_outputs=g.float())
    assert bits_equal(x.grad, g32)


# ---- the fused step --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src_u8", [False, True], ids=["fp32src", "u8src"])
def test_geometry_step_bf16_crops(dev, src_u8):
    from hands_b200.step import GeometryStep

    S, R = 96, 224
    s32 = GeometryStep(S, dev, seed=4, src_u8=src_u8)
    s16 = GeometryStep(S, dev, seed=4, src_u8=src_u8, crop_dtype=BF16)
    assert s16.crops.dtype == BF16 and s16.g_crops.dtype == BF16 and s16.g_img.dtype == torch.float32
    assert bits_equal(s16.g_crops, s32.g_crops.to(BF16))
    # the fp32 step reads the widened bf16 gradient
    s32.g_crops.copy_(s16.g_crops.float())
    s32.run()
    s16.run()
    torch.cuda.synchronize()
    assert bits_equal(s16.crops, s32.crops.to(BF16))
    assert bits_equal(s16.g_img, s32.g_img) and float(s16.g_img.abs().max()) > 0
    for h16, h32 in zip(s16.hands, s32.hands):
        for k in ("g_rotmat", "g_betas", "g_cam", "vertices", "j2d"):
            assert bits_equal(h16[k], h32[k]), k
    # the same step as one CUDA graph: same launch count, same results on replay
    n32, n16 = s32.capture(), s16.capture()
    assert n16 == n32 > 0
    s16.crops.zero_()
    s16.g_img.zero_()
    s32.replay()
    s16.replay()
    torch.cuda.synchronize()
    assert bits_equal(s16.crops, s32.crops.to(BF16))
    assert bits_equal(s16.g_img, s32.g_img)
    # byte accounting: 2-byte crop and crop-gradient planes
    plane = 3 * R * R
    assert s32.pcl_bytes_per_crop() - s16.pcl_bytes_per_crop() == pytest.approx(plane * 4, abs=1e-3)
    assert s32.bytes_per_sample() - s16.bytes_per_sample() == pytest.approx(2 * s16.hps * plane * 2, abs=1e-3)
    with pytest.raises(NotImplementedError):
        s16.pcl_backward_stage(1)
