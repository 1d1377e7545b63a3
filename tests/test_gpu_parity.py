"""GPU parity: the CUDA path (through the C ABI, via the drop-in modules) against the CPU oracle.

Tolerances are the ones BASELINE.json states: vertices/joints 1e-5 relative, key-points 1e-3 px,
gradients 1e-4 relative, indices bit-exact.  "Relative" is max|got-ref| / max|ref| per tensor.
Where fp32 conditioning itself limits the reference (angles near pi), the bound is widened to
3x the fp32 oracle's own distance from the fp64 oracle.
"""
import os

import numpy as np
import pytest
import torch

from hands_b200.synthetic import synthetic_head_inputs, synthetic_mano_buffers, synthetic_pcl_inputs
from oracle import geometry_oracle as O
from _tol import tol_check

pytestmark = pytest.mark.gpu

IMG_RES = 224.0


def rel(got, ref):
    ref = ref.double()
    return float((got.double().cpu() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def heads(dev):
    from hands_b200.src.nets.hand_heads.mano_head import MANOHead

    return {
        True: MANOHead(True, 1000.0, IMG_RES, synthetic=True).to(dev),
        False: MANOHead(False, 1000.0, IMG_RES, synthetic=True).to(dev),
    }


def oracle_head(is_rhand, rotmat, betas, cam, K, dtype):
    buf = synthetic_mano_buffers(is_rhand)
    return O.mano_head_forward(buf, rotmat.to(dtype), betas.to(dtype), cam.to(dtype), K.to(dtype), IMG_RES, 0.1)


@pytest.mark.parametrize("B,is_rhand,edge", [(64, True, None), (17, False, None), (1, True, None), (33, True, "identity"), (16, False, "near_pi")])
def test_head_forward(heads, dev, B, is_rhand, edge):
    rotmat, betas, cam, K = synthetic_head_inputs(B, seed=B, edge=edge, small_s_frac=0.25)
    out = heads[is_rhand](rotmat.to(dev), betas.to(dev), cam.to(dev), K.to(dev))
    pf = ".r" if is_rhand else ".l"
    assert sorted(out.keys()) == sorted(k + pf for k in ["cam_t.wp", "cam_t", "joints3d", "vertices", "j3d.cam", "v3d.cam", "j2d.norm", "beta", "pose"])
    ref64 = oracle_head(is_rhand, rotmat, betas, cam, K, torch.float64)
    ref32 = oracle_head(is_rhand, rotmat, betas, cam, K, torch.float32)
    for key in ["vertices", "joints3d", "v3d.cam", "j3d.cam", "cam_t"]:
        own = rel(ref32[key], ref64[key])
        r = rel(out[key + pf], ref64[key])
        tol_check(f"head_fwd[{B},{edge}].{key}", r, 1e-5, own)
    px = (out["j2d.norm" + pf].double().cpu() - ref64["j2d.norm"]).abs().max() * IMG_RES / 2
    own_px = (ref32["j2d.norm"].double() - ref64["j2d.norm"]).abs().max() * IMG_RES / 2
    tol_check(f"head_fwd[{B},{edge}].j2d_px", px, 1e-3, own_px)
    assert torch.equal(out["pose" + pf].cpu(), rotmat) and torch.equal(out["beta" + pf].cpu(), betas)
    assert out["vertices" + pf].shape == (B, 778, 3) and out["joints3d" + pf].shape == (B, 21, 3) and out["j2d.norm" + pf].shape == (B, 21, 2)
    # fingertip gather is indexing: bit-exact against our own vertices
    tips = out["vertices" + pf][:, list(O.TIP_IDS)]
    assert torch.equal(out["joints3d" + pf][:, 16:], tips)


def _head_grads(fn, rotmat, betas, cam, K, weights, keys):
    rotmat, betas, cam = rotmat.clone().requires_grad_(True), betas.clone().requires_grad_(True), cam.clone().requires_grad_(True)
    out = fn(rotmat, betas, cam, K)
    loss = sum((out[k] * weights[k].to(out[k].device, out[k].dtype)).sum() for k in keys)
    return torch.autograd.grad(loss, (rotmat, betas, cam))


@pytest.mark.parametrize("B,is_rhand,edge,keys", [
    (48, True, None, ("v3d.cam", "j3d.cam", "j2d.norm")),
    (19, False, None, ("v3d.cam", "j3d.cam", "j2d.norm", "vertices", "joints3d", "cam_t")),
    (16, True, "identity", ("v3d.cam", "j3d.cam", "j2d.norm")),
    (16, True, "near_pi", ("j3d.cam", "j2d.norm")),
    (5, False, None, ("j2d.norm",)),
])
def test_head_backward(heads, dev, B, is_rhand, edge, keys):
    rotmat, betas, cam, K = synthetic_head_inputs(B, seed=100 + B, edge=edge, small_s_frac=0.2)
    g = torch.Generator().manual_seed(B)
    shapes = {"v3d.cam": (B, 778, 3), "vertices": (B, 778, 3), "j3d.cam": (B, 21, 3), "joints3d": (B, 21, 3), "j2d.norm": (B, 21, 2), "cam_t": (B, 3)}
    weights = {k: torch.randn(shapes[k], generator=g) for k in keys}
    pf = ".r" if is_rhand else ".l"

    def ours(r, b, c, k):
        o = heads[is_rhand](r, b, c, k)
        return {key: o[key + pf] for key in keys}

    got = _head_grads(ours, rotmat.to(dev), betas.to(dev), cam.to(dev), K.to(dev), weights, keys)
    ref64 = _head_grads(lambda r, b, c, k: oracle_head(is_rhand, r, b, c, k, torch.float64), rotmat.double(), betas.double(), cam.double(), K.double(), weights, keys)
    ref32 = _head_grads(lambda r, b, c, k: oracle_head(is_rhand, r, b, c, k, torch.float32), rotmat, betas, cam, K, weights, keys)
    for name, a, r64, r32 in zip(("rotmat", "betas", "cam"), got, ref64, ref32):
        own = rel(r32, r64)
        r = rel(a, r64)
        tol_check(f"head_bwd[{B},{edge}].g_{name}", r, 1e-4, own)
    # clamp: zero gradient for s < min_s (camera.py:463)
    small = cam[:, 0] < 0.1
    assert (got[2].cpu()[small, 0] == 0).all()


@pytest.mark.parametrize("layout,ofn,gkey", [("cols_paired", O.rot6d_to_rotmat_paired, "paired"), ("cols", O.rot6d_to_rotmat_cols, "cols"), ("rows", O.rotation_6d_to_matrix, None)])
def test_rot6d_free_functions(dev, golden_dir, layout, ofn, gkey):
    """6D -> rotation matrix, the reference's three layouts, forward and backward, against the reference's own
    outputs (golden) and the oracle."""
    from hands_b200.common import rot

    fn = {"cols_paired": rot.rot6d_to_rotmat, "cols": rot.rot6d_to_rotmat_hamer, "rows": rot.rotation_6d_to_matrix}[layout]
    d = np.load(os.path.join(golden_dir, "rot6d.npz"))
    x = torch.from_numpy(d["x"])
    g = torch.Generator().manual_seed(3)
    w = torch.from_numpy(d[f"w_{gkey}"]) if gkey else torch.randn(64, 3, 3, generator=g)
    xi = x.to(dev).requires_grad_(True)
    R = fn(xi)
    (gx,) = torch.autograd.grad((R * w.to(dev)).sum(), xi)
    xo = x.double().requires_grad_(True)
    Ro = ofn(xo)
    (gxo,) = torch.autograd.grad((Ro * w.double()).sum(), xo)
    well = slice(0, 56)   # rows 56..59 are nearly parallel pairs in the contiguous layouts: fp32 itself is ill-conditioned there
    own = rel(ofn(x), Ro.detach())   # the fp32 reference's own distance from fp64
    assert R.shape == (64, 3, 3) and rel(R[well], Ro.detach()[well]) <= 1e-5
    tol_check(f"rot6d[{layout}].R_all_rows", rel(R, Ro.detach()), 1e-5, own)
    assert rel(gx[well], gxo[well]) <= 1e-4
    if gkey:
        assert rel(R[well], torch.from_numpy(d[f"R_{gkey}"])[well]) <= 1e-6
        assert rel(gx[well], torch.from_numpy(d[f"gx_{gkey}"])[well]) <= 1e-4
    z = fn(torch.zeros(2, 6, device=dev))   # F.normalize eps: zero input gives the zero matrix, not NaN
    assert torch.isfinite(z).all() and float(z.abs().max()) == 0.0


@pytest.mark.parametrize("layout,ofn", [("rows", O.rotation_6d_to_matrix), ("cols", O.rot6d_to_rotmat_cols), ("cols_paired", O.rot6d_to_rotmat_paired)])
def test_head_from_rot6d(heads, dev, layout, ofn):
    """The 6D prologue fused into the head (SURVEY.md 8(f) f1): outputs and gradients equal the reference's chain
    rot6d -> MANOHead."""
    B = 24
    _, betas, cam, K = synthetic_head_inputs(B, seed=5, small_s_frac=0.2)
    g = torch.Generator().manual_seed(9)
    x6 = torch.randn(B, 96, generator=g)
    keys = ("v3d.cam", "j3d.cam", "j2d.norm")
    weights = {"v3d.cam": torch.randn(B, 778, 3, generator=g), "j3d.cam": torch.randn(B, 21, 3, generator=g), "j2d.norm": torch.randn(B, 21, 2, generator=g)}
    xi, bi, ci = x6.to(dev).requires_grad_(True), betas.to(dev).requires_grad_(True), cam.to(dev).requires_grad_(True)
    out = heads[True].forward_rot6d(xi, bi, ci, K.to(dev), layout=layout)
    loss = sum((out[k + ".r"] * weights[k].to(dev)).sum() for k in keys)
    got = torch.autograd.grad(loss, (xi, bi, ci))

    def chain(dtype):
        xo, bo, co = x6.to(dtype).requires_grad_(True), betas.to(dtype).requires_grad_(True), cam.to(dtype).requires_grad_(True)
        rotmat = ofn(xo.reshape(-1, 6)).reshape(B, 16, 3, 3)
        o = oracle_head(True, rotmat, bo, co, K, dtype)
        lo = sum((o[k] * weights[k].to(dtype)).sum() for k in keys)
        return o, rotmat, torch.autograd.grad(lo, (xo, bo, co))

    o64, rot64, g64 = chain(torch.float64)
    o32, _, g32 = chain(torch.float32)
    for k in ("vertices", "joints3d", "v3d.cam", "j3d.cam"):
        assert rel(out[k + ".r"], o64[k]) <= max(1e-5, 3 * rel(o32[k], o64[k])), k
    assert rel(out["pose.r"], rot64.detach()) <= 1e-5
    for name, a, r64, r32 in zip(("x6", "betas", "cam"), got, g64, g32):
        assert rel(a, r64) <= max(1e-4, 3 * rel(r32, r64)), name


def test_keypoint_losses_and_metric_sums(dev, golden_dir):
    """SURVEY.md 8(f) f2: loss terms + metric partial sums straight from the head's outputs, against the reference's own
    functions (golden) -- values, gradients, and the partial sums the packed all-reduce carries."""
    from hands_b200.losses import keypoint_losses, mrrpe_sums

    d = {k: torch.from_numpy(np.asarray(v)) for k, v in np.load(os.path.join(golden_dir, "kp_loss.npz")).items()}
    c = {k: v.to(dev) for k, v in d.items()}
    j3d, j2d = c["j3d"].clone().requires_grad_(True), c["j2d"].clone().requires_grad_(True)
    l3, l2, sums = keypoint_losses(j3d, j2d, c["gt3"], c["gt2"], c["jv"], c["hv"], c["gate3"], c["gate2"], img_res=224)
    assert abs(float(l3.detach()) - float(d["loss3"])) <= 1e-5 * float(d["loss3"]) and abs(float(l2.detach()) - float(d["loss2"])) <= 1e-5 * float(d["loss2"])
    g3, g2 = torch.autograd.grad(5.0 * l3 + 3.0 * l2, (j3d, j2d))
    assert rel(g3, d["g3"]) <= 1e-4 and rel(g2, d["g2"]) <= 1e-4
    s = sums.cpu().double()
    mp, pix = d["mpjpe"].numpy(), d["pix"].numpy()
    assert int(s[3]) == int(np.isfinite(mp).sum()) and int(s[5]) == int(np.isfinite(pix).sum())          # counts: bit-exact
    assert abs(float(s[2] / s[3]) - float(np.nanmean(mp))) <= 1e-5 * float(np.nanmean(mp))
    assert abs(float(s[4] / s[5]) - float(np.nanmean(pix))) <= 1e-5 * float(np.nanmean(pix))           # well inside 1e-3 px
    m = mrrpe_sums(c["j3d"], c["j3d_l"], c["gt3"], c["gt3_l"], c["hv"]).cpu().double()
    ref = d["mrrpe"].numpy()
    assert int(m[1]) == int(np.isfinite(ref).sum()) and abs(float(m[0] / m[1]) - float(np.nanmean(ref))) <= 1e-5 * float(np.nanmean(ref))
    # reproducible: the reduction order is fixed
    _, _, sums2 = keypoint_losses(c["j3d"], c["j2d"], c["gt3"], c["gt2"], c["jv"], c["hv"], c["gate3"], c["gate2"], img_res=224)
    assert torch.equal(sums, sums2)
    # no gates / masks given, larger ragged batch, against the oracle
    g = torch.Generator().manual_seed(2)
    B = 1031
    a3, b3 = torch.randn(B, 21, 3, generator=g), torch.randn(B, 21, 3, generator=g)
    a2, b2 = torch.randn(B, 21, 2, generator=g), torch.randn(B, 21, 2, generator=g)
    ones = torch.ones(B, 21)
    l3, l2, _ = keypoint_losses(a3.to(dev), a2.to(dev), b3.to(dev), b2.to(dev), ones.to(dev))
    o3, o2 = O.keypoint_losses(a3.double(), a2.double(), b3.double(), b2.double(), ones.double())
    assert abs(float(l3) - float(o3)) <= 1e-5 * float(o3) and abs(float(l2) - float(o2)) <= 1e-5 * float(o2)


def test_process_data_light_gt_side(dev, golden_dir):
    """SURVEY.md 8(f) f3: the drop-in process_data_light against the reference's own function (golden)."""
    from types import SimpleNamespace

    from hands_b200.common.body_models import build_mano_aa
    from hands_b200.src.callbacks.process.process_arctic import process_data_light

    d = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(golden_dir, "process_gt.npz")).items()}
    models = {"mano_r": build_mano_aa(True, synthetic=True).to(dev), "mano_l": build_mano_aa(False, synthetic=True).to(dev)}
    targets = {k[3:]: v.to(dev) for k, v in d.items() if k.startswith("in_")}
    _, out, _ = process_data_light(models, {}, targets, {"intrinsics": d["K"].to(dev)}, "train", SimpleNamespace(img_res=224))
    for k, ref in d.items():
        if not k.startswith("out_"):
            continue
        got = out[k[4:]]
        assert got.shape == ref.shape, k
        tol = 1e-5 if "wp" not in k else 2e-6
        assert rel(got, ref) <= tol, (k, rel(got, ref))
    assert out["mano.j3d.cam.r"] is targets["mano.j3d.full.r"]
    assert not out["mano.v3d.cam.r"].requires_grad


def test_kpe_features(dev, golden_dir):
    """SURVEY.md 8(f) f4: KPE angles + encodings, batched on the GPU, against the reference's own lines (golden)."""
    from hands_b200.pcl import kpe_features

    d = np.load(os.path.join(golden_dir, "kpe.npz"))
    L = int(d["L"])
    out = kpe_features(torch.from_numpy(d["bbox"]).to(dev), torch.from_numpy(d["K"]).to(dev), L)
    assert (out["center_angle"].cpu() - torch.from_numpy(d["center"])).abs().max() <= 1.2e-7
    assert (out["corner_angle"].cpu() - torch.from_numpy(d["corner"])).abs().max() <= 1.2e-7
    assert out["center_pos_enc"].shape == (12, L * 4) and out["corner_pos_enc"].shape == (12, L * 16)
    assert (out["center_pos_enc"].cpu() - torch.from_numpy(d["center_enc"])).abs().max() <= 2e-6
    assert (out["corner_pos_enc"].cpu() - torch.from_numpy(d["corner_enc"])).abs().max() <= 2e-6


@pytest.mark.parametrize("B", [8, 300])
def test_tensor_core_blendshapes_partial_tiles(heads, dev, B):
    """The blendshape contraction and its transpose run on tcgen05/TMEM (3xTF32) in tiles of 128 hands.  B = 8 leaves
    one tile mostly empty; B = 300 spans three tiles, the last one partial.  Vertices, joints and the gradients that flow
    through the feature rows (rotmat, betas) are checked against the fp64 oracle."""
    rotmat, betas, cam, K = synthetic_head_inputs(B, seed=4242 + B, small_s_frac=0.1)
    w = torch.randn(B, 778, 3, generator=torch.Generator().manual_seed(7))
    r = rotmat.to(dev).requires_grad_(True)
    bb = betas.to(dev).requires_grad_(True)
    o = heads[True](r, bb, cam.to(dev), K.to(dev))
    got = torch.autograd.grad((o["v3d.cam.r"] * w.to(dev)).sum() + o["j2d.norm.r"].sum(), (r, bb))
    ref64 = oracle_head(True, rotmat, betas, cam, K, torch.float64)
    assert rel(o["vertices.r"], ref64["vertices"]) <= 1e-5
    assert rel(o["joints3d.r"], ref64["joints3d"]) <= 1e-5

    def oracle_grads(dtype):
        ro, bo = rotmat.to(dtype).requires_grad_(True), betas.to(dtype).requires_grad_(True)
        ref = oracle_head(True, ro, bo, cam, K, dtype)
        return torch.autograd.grad((ref["v3d.cam"] * w.to(dtype)).sum() + ref["j2d.norm"].sum(), (ro, bo))

    g64, g32 = oracle_grads(torch.float64), oracle_grads(torch.float32)
    for name, a, r64, r32 in zip(("rotmat", "betas"), got, g64, g32):
        tol_check(f"tc_blend[{B}].g_{name}", rel(a, r64), 1e-4, rel(r32, r64))


def test_mano_layer_axis_angle_and_transl(dev):
    from hands_b200.common.body_models import build_mano_aa

    layer = build_mano_aa(True, synthetic=True).to(dev)
    buf = synthetic_mano_buffers(True)
    g = torch.Generator().manual_seed(3)
    B = 21
    pose = torch.randn(B, 48, generator=g) * 0.3
    betas = torch.randn(B, 10, generator=g)
    transl = torch.randn(B, 3, generator=g)
    for t in (None, transl):
        p, b = pose.to(dev).requires_grad_(True), betas.to(dev).requires_grad_(True)
        tt = None if t is None else t.to(dev).requires_grad_(True)
        out = layer(betas=b, global_orient=p[:, :3], hand_pose=p[:, 3:], transl=tt)
        p64, b64 = pose.double().requires_grad_(True), betas.double().requires_grad_(True)
        t64 = None if t is None else t.double().requires_grad_(True)
        v64, j64 = O.mano_forward(buf, b64, p64[:, :3], p64[:, 3:], transl=t64)
        assert rel(out.vertices, v64.detach()) <= 1e-5 and rel(out.joints, j64.detach()) <= 1e-5
        wv, wj = torch.randn(B, 778, 3, generator=g), torch.randn(B, 21, 3, generator=g)
        ins = (p, b) + (() if tt is None else (tt,))
        ins64 = (p64, b64) + (() if t64 is None else (t64,))
        got = torch.autograd.grad((out.vertices * wv.to(dev)).sum() + (out.joints * wj.to(dev)).sum(), ins)
        ref = torch.autograd.grad((v64 * wv).sum() + (j64 * wj).sum(), ins64)
        for a, r in zip(got, ref):
            assert rel(a, r) <= 1e-4
    assert layer.faces.shape == (1538, 3)
    with torch.no_grad():
        out = layer(betas=betas.to(dev), global_orient=pose[:, :3].to(dev), hand_pose=pose[:, 3:].to(dev))
    assert out.joints.shape == (B, 21, 3)


def test_pre_rot_matches_explicit_fixup(heads, dev):
    from hands_b200.pcl import apply_virtual_rotation

    B = 24
    rotmat, betas, cam, K = synthetic_head_inputs(B, seed=9)
    Rv, _, _, _ = synthetic_head_inputs(B, seed=10)
    Rv = Rv[:, 0].contiguous().to(dev)
    w = torch.randn(B, 21, 3, generator=torch.Generator().manual_seed(1)).to(dev)
    grads = []
    outs = []
    for fused in (True, False):
        r = rotmat.to(dev).requires_grad_(True)
        if fused:
            o = heads[True](r, betas.to(dev), cam.to(dev), K.to(dev), pre_rot=Rv)
        else:
            o = heads[True](apply_virtual_rotation(Rv, r), betas.to(dev), cam.to(dev), K.to(dev))
        outs.append(o["j3d.cam.r"])
        grads.append(torch.autograd.grad((o["j3d.cam.r"] * w).sum(), r)[0])
    assert rel(outs[0], outs[1].cpu()) <= 1e-6
    assert rel(grads[0], grads[1].cpu()) <= 1e-5
    ref = O.pcl_fix_global_orient(Rv.cpu(), rotmat)
    assert rel(apply_virtual_rotation(Rv, rotmat.to(dev)), ref) <= 1e-6


def test_shard_invariance_bit_exact(heads, dev):
    B = 64
    rotmat, betas, cam, K = [t.to(dev) for t in synthetic_head_inputs(B, seed=77)]
    w = torch.randn(B, 778, 3, device=dev)

    def run(sl):
        r, b, c = rotmat[sl].clone().requires_grad_(True), betas[sl].clone().requires_grad_(True), cam[sl].clone().requires_grad_(True)
        o = heads[True](r, b, c, K[sl])
        g, gb, gc = torch.autograd.grad((o["v3d.cam.r"] * w[sl]).sum() + o["j2d.norm.r"].sum(), (r, b, c))
        return o["v3d.cam.r"].detach(), o["j2d.norm.r"].detach(), g, gb, gc

    full = run(slice(0, B))
    again = run(slice(0, B))
    for k in range(5):   # run-to-run: no order-dependent reduction anywhere (g_cam sums 778 vertex gradients per hand)
        assert torch.equal(full[k], again[k]), k
    for n in (2, 4, 8):
        step = B // n
        parts = [run(slice(i * step, (i + 1) * step)) for i in range(n)]
        for k in range(5):
            assert torch.equal(torch.cat([p[k] for p in parts]), full[k]), k


def test_free_functions_against_golden(dev, golden_dir):
    from hands_b200.common import camera, data_utils, rot, transforms

    g = np.load(os.path.join(golden_dir, "logmap.npz"))
    R = torch.from_numpy(g["R"]).to(dev).requires_grad_(True)
    aa = rot.matrix_to_axis_angle(R)
    ref_aa = torch.from_numpy(g["aa"])
    # compare through the rotation both encode (axis-angle near pi is ill-conditioned in the angle itself)
    assert (O.batch_rodrigues(aa.detach().cpu().double()) - O.batch_rodrigues(ref_aa.double())).abs().max() < 2e-6
    ok = ref_aa.norm(dim=1) < 3.0
    assert (aa.detach().cpu()[ok] - ref_aa[ok]).abs().max() < 1e-5
    (gR,) = torch.autograd.grad((aa * torch.from_numpy(g["w"]).to(dev)).sum(), R)
    ref_gR = torch.from_numpy(g["gR"])
    assert rel(gR[ok.to(dev)], ref_gR[ok]) <= 1e-4

    c = np.load(os.path.join(golden_dir, "camera_projection.npz"))
    cam = torch.from_numpy(c["cam"]).to(dev).requires_grad_(True)
    f = torch.from_numpy(c["f"]).to(dev)
    cam_t = camera.weak_perspective_to_perspective_torch(cam, f, 224, 0.1)
    assert torch.equal(cam_t.detach().cpu(), torch.from_numpy(c["cam_t"]))
    (g_cam,) = torch.autograd.grad((cam_t * torch.from_numpy(c["w3"]).to(dev)).sum(), cam)
    assert rel(g_cam, torch.from_numpy(c["g_cam"])) <= 1e-6
    assert torch.equal(camera.perspective_to_weak_perspective_torch(cam_t.detach(), f, 224).cpu(), torch.from_numpy(c["wp"]))
    K = torch.from_numpy(c["K"]).to(dev)
    pts = torch.from_numpy(c["pts"]).to(dev).requires_grad_(True)
    j2d = transforms.project2d_batch(K, pts)
    assert (j2d.detach().cpu() - torch.from_numpy(c["j2d"])).abs().max() < 1e-3
    j2d_n = transforms.project2d_norm_batch(K, pts, 224)
    assert (j2d_n.detach().cpu() - torch.from_numpy(c["j2d_norm"])).abs().max() * 112 < 1e-3
    assert (data_utils.normalize_kp2d(j2d.detach(), 224).cpu() - torch.from_numpy(c["j2d_norm"])).abs().max() * 112 < 1e-3
    (g_pts,) = torch.autograd.grad((j2d_n * torch.from_numpy(c["w2"]).to(dev)).sum(), pts)
    assert rel(g_pts, torch.from_numpy(c["g_pts"])) <= 1e-4
    assert (data_utils.unormalize_kp2d(j2d_n.detach(), 224).cpu() - torch.from_numpy(c["j2d_un"])).abs().max() < 1e-3


@pytest.fixture
def pcl_exact_mode():
    """torch's CPU operation order reproduced exactly (HB_PCL_EXACT=1): the mode the bit-level golden comparison runs in."""
    from hands_b200 import _lib

    prev = _lib.load().hb_pcl_set_exact(1)
    yield
    _lib.load().hb_pcl_set_exact(prev)


def test_pcl_forward_against_golden_default_mode(dev, golden_dir):
    """The reference's own crops (golden) against the DEFAULT forward: 2e-6 of the crop's range."""
    from hands_b200.pcl import perspective_crop

    g = np.load(os.path.join(golden_dir, "pcl.npz"))
    img = torch.from_numpy(g["small_img"]).to(dev)
    bbox = torch.from_numpy(g["small_bbox"].astype(np.int32)).to(dev)
    K = torch.from_numpy(np.repeat(g["small_K"], 2, axis=0)).float().to(dev)
    crop, rot = perspective_crop(img, bbox, K, img_res=64, crops_per_img=2)
    ref = torch.from_numpy(g["small_crop"])
    assert torch.equal(rot.cpu(), torch.from_numpy(g["small_rot"]))
    tol_check("pcl_golden_small_default", float((crop.cpu() - ref).abs().max() / ref.abs().max()), 2e-6)
    img2, bbox2, K2 = synthetic_pcl_inputs(4, seed=int(g["full_seed"]), img_res=224)
    for j in range(4):
        b = (j // 2) * 2
        c2, _ = perspective_crop(img2[b : b + 1].to(dev), bbox2[j : j + 1].to(dev), K2[b : b + 1].to(dev), img_res=224)
        ref2 = torch.from_numpy(g["full_crop_sub4"][j])
        tol_check(f"pcl_golden_full_default[{j}]", float((c2[0, :, ::4, ::4].cpu() - ref2).abs().max() / ref2.abs().max()), 2e-6)


def test_pcl_forward_against_golden(dev, golden_dir, pcl_exact_mode):
    from hands_b200.pcl import perspective_crop

    g = np.load(os.path.join(golden_dir, "pcl.npz"))
    img = torch.from_numpy(g["small_img"]).to(dev)                       # (4,3,64,64), two crops per image
    bbox = torch.from_numpy(g["small_bbox"].astype(np.int32)).to(dev)    # (8,4)
    K = torch.from_numpy(np.repeat(g["small_K"], 2, axis=0)).float().to(dev)
    crop, rot = perspective_crop(img, bbox, K, img_res=64, crops_per_img=2)
    ref = torch.from_numpy(g["small_crop"])
    assert torch.equal(rot.cpu(), torch.from_numpy(g["small_rot"]))
    assert (crop.cpu() - ref).abs().max() <= 1e-6, float((crop.cpu() - ref).abs().max())
    frac_exact = float((crop.cpu() == ref).float().mean())
    assert frac_exact > 0.999, frac_exact
    img2, bbox2, K2 = synthetic_pcl_inputs(4, seed=int(g["full_seed"]), img_res=224)
    for j in range(4):
        b = (j // 2) * 2
        c2, r2 = perspective_crop(img2[b : b + 1].to(dev), bbox2[j : j + 1].to(dev), K2[b : b + 1].to(dev), img_res=224)
        d = (c2[0, :, ::4, ::4].cpu() - torch.from_numpy(g["full_crop_sub4"][j])).abs().max()
        assert d <= 1e-6, float(d)
        assert torch.equal(r2[0].cpu(), torch.from_numpy(g["full_rot"][j]))


@pytest.mark.parametrize("B,cpi,res,smooth", [(6, 1, 224, False), (4, 2, 224, True), (3, 2, 96, False), (2, 5, 100, False), (1, 7, 224, True)])
def test_pcl_forward_backward_against_oracle(dev, B, cpi, res, smooth):
    from hands_b200.pcl import perspective_crop

    n = B * cpi
    img, bbox, K = synthetic_pcl_inputs(n, seed=B, img_res=res, smin=res // 4, smax=3 * res // 4, smooth=smooth)
    img = img[:B].contiguous()
    if B >= 3:
        bbox[0] = torch.tensor([10, 12, 10, 12])            # zero-size box -> s = img_res
        bbox[1] = torch.tensor([0, 0, res - 1, res - 1])    # whole image
        bbox[2] = torch.tensor([res // 2 - 20, res // 2 - 15, res // 2 + 20, res // 2 + 15])  # centred: R = I
    w = torch.randn(n, 3, res, res, generator=torch.Generator().manual_seed(5))
    x = img.to(dev).requires_grad_(True)
    crop, rot = perspective_crop(x, bbox.to(dev), K.to(dev), img_res=res, crops_per_img=cpi)
    (g_img,) = torch.autograd.grad((crop * w.to(dev)).sum(), x)
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        xr = img.clone().requires_grad_(True)
        ref_crop, ref_rot = O.perspective_crop(xr.repeat_interleave(cpi, dim=0), bbox, K, res)
        (ref_g,) = torch.autograd.grad((ref_crop * w).sum(), xr)
    finally:
        torch.set_num_threads(nt)
    # R and P come from a float64 closed-form 3x3 inverse here and from LAPACK in numpy/torch: they can
    # differ in the last fp32 bit, which moves sample positions by ~1e-5 px.  On white-noise images that is
    # up to ~2e-5 in the crop; smooth images stay at 1e-6.
    assert (rot.cpu() - ref_rot).abs().max() <= 1.2e-7
    err = (crop.detach().cpu() - ref_crop.detach()).abs()
    assert err.max() <= (2e-6 if smooth else 5e-5), float(err.max())
    assert float((err <= 1e-6).float().mean()) > 0.99
    assert rel(g_img, ref_g) <= 1e-4


@pytest.mark.parametrize("res,C", [(50, 3), (96, 1), (64, 4)])
def test_pcl_generic_paths(dev, res, C):
    """Resolutions that are not a multiple of 4 (no 16-byte aligned rows -> no bulk copies, generic transposed
    resize) and channel counts other than 3 go through the fallback code paths; same tolerances."""
    from hands_b200.functional import PerspectiveCropFunction

    B = 3
    img, bbox, K = synthetic_pcl_inputs(B, seed=res, img_res=res, smin=res // 4, smax=3 * res // 4)
    g = torch.Generator().manual_seed(res)
    img = torch.randn(B, C, res, res, generator=g)
    w = torch.randn(B, C, res, res, generator=g)
    x = img.to(dev).requires_grad_(True)
    crop, rot = PerspectiveCropFunction.apply(x, bbox.to(dev), K.to(dev), 1)
    (g_img,) = torch.autograd.grad((crop * w.to(dev)).sum(), x)
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        xr = img.clone().requires_grad_(True)
        ref_crop, ref_rot = O.perspective_crop(xr, bbox, K, res)
        (ref_g,) = torch.autograd.grad((ref_crop * w).sum(), xr)
    finally:
        torch.set_num_threads(nt)
    assert (rot.cpu() - ref_rot).abs().max() <= 1.2e-7
    assert (crop.detach().cpu() - ref_crop.detach()).abs().max() <= 5e-5
    assert rel(g_img, ref_g) <= 1e-4


def test_pcl_box_larger_than_image(dev):
    """A box reaching outside the image gives s > img_res (down-sampling): the forward's generic code path."""
    from hands_b200.pcl import perspective_crop

    res = 64
    g = torch.Generator().manual_seed(3)
    img = torch.randn(2, 3, res, res, generator=g)
    bbox = torch.tensor([[-10, -5, 90, 80], [5, -20, 60, 75]], dtype=torch.int32)
    K = torch.tensor([[[80.0, 0, 32], [0, 80.0, 32], [0, 0, 1]], [[120.0, 0, 30], [0, 110.0, 33], [0, 0, 1]]])
    with torch.no_grad():
        crop, rot = perspective_crop(img.to(dev), bbox.to(dev), K.to(dev), img_res=res)
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        ref_crop, ref_rot = O.perspective_crop(img, bbox, K, res)
    finally:
        torch.set_num_threads(nt)
    assert (rot.cpu() - ref_rot).abs().max() <= 1.2e-7
    assert (crop.cpu() - ref_crop).abs().max() <= 5e-5
    # the backward's workspace is sized for s <= img_res (the reference clips boxes to the image): rejected up front
    with pytest.raises(ValueError, match="no larger than the image"):
        perspective_crop(img.to(dev).requires_grad_(True), bbox.to(dev), K.to(dev), img_res=res)


def test_pcl_full_size_properties(dev):
    """BASELINE config C3 size (1024 source images, two crops each = 2048 crops of 3x224x224), checked through properties
    that need no CPU oracle: the backward is the exact adjoint of the forward (<F x, y> == <x, F^T y>), the forward is
    linear in the image, and both are independent of how the batch is sharded (bit-exact)."""
    from hands_b200.pcl import perspective_crop

    B, cpi, res = 1024, 2, 224
    n = B * cpi
    _, bbox, K = synthetic_pcl_inputs(n, seed=3, img_res=res, smin=res // 4, smax=3 * res // 4)
    bbox, K = bbox.to(dev), K.to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(B, 3, res, res, generator=g, device=dev).requires_grad_(True)
    y = torch.randn(n, 3, res, res, generator=g, device=dev)
    crop, _ = perspective_crop(x, bbox, K, img_res=res, crops_per_img=cpi)
    (gx,) = torch.autograd.grad(crop, x, grad_outputs=y)
    lhs = float((crop.detach().double() * y.double()).sum())
    rhs = float((x.detach().double() * gx.double()).sum())
    scale = float(crop.detach().double().norm() * y.double().norm())
    assert abs(lhs - rhs) <= 1e-6 * scale, (lhs, rhs, scale)
    # linearity of the forward
    with torch.no_grad():
        x2 = torch.randn(B, 3, res, res, generator=g, device=dev)
        c2, _ = perspective_crop(x2, bbox, K, img_res=res, crops_per_img=cpi)
        c12, _ = perspective_crop(2.5 * x.detach() + x2, bbox, K, img_res=res, crops_per_img=cpi)
        assert rel(c12, (2.5 * crop.detach() + c2).cpu()) <= 2e-6
        del c2, c12, x2
        # shard invariance, forward and backward, bit-exact (a shard boundary inside the 1024-image backward chunk)
        lo, hi = 300, 812
        cs, _ = perspective_crop(x.detach()[lo:hi].contiguous(), bbox[lo * cpi:hi * cpi], K[lo * cpi:hi * cpi], img_res=res, crops_per_img=cpi)
        assert torch.equal(cs, crop.detach()[lo * cpi:hi * cpi])
    xs = x.detach()[lo:hi].clone().requires_grad_(True)
    cs, _ = perspective_crop(xs, bbox[lo * cpi:hi * cpi], K[lo * cpi:hi * cpi], img_res=res, crops_per_img=cpi)
    (gs,) = torch.autograd.grad(cs, xs, grad_outputs=y[lo * cpi:hi * cpi])
    assert torch.equal(gs, gx[lo:hi])


def test_mano_full_size_properties(heads, dev):
    """BASELINE config C4 per-GPU size (8192 samples -> 8192 hands per side): properties that need no CPU oracle --
    global-rotation equivariance about the root joint, shard invariance (bit-exact), finger tips == gathered vertices,
    and linearity of the backward in the upstream gradients."""
    from hands_b200.synthetic import random_rotmats

    B = 8192
    rotmat, betas, cam, K = [t.to(dev) for t in synthetic_head_inputs(B, seed=11)]
    head = heads[False]
    out = head(rotmat, betas, cam, K)
    v, j = out["vertices.l"], out["joints3d.l"]
    assert torch.equal(j[:, 16:], v[:, list(O.TIP_IDS)])
    Q = random_rotmats(B, torch.Generator().manual_seed(5)).to(dev)
    outq = head(rotmat, betas, cam, K, pre_rot=Q)
    root = j[:, :1]
    assert rel(outq["joints3d.l"][:, 0], j[:, 0].cpu()) <= 1e-5
    want = torch.einsum("bij,bvj->bvi", Q.double(), (v - root).double()) + root.double()
    assert rel(outq["vertices.l"], want.cpu()) <= 2e-5
    sl = slice(5000, 5777)
    part = head(rotmat[sl].contiguous(), betas[sl].contiguous(), cam[sl].contiguous(), K[sl].contiguous())
    for key in ("vertices.l", "j3d.cam.l", "j2d.norm.l", "cam_t.l"):
        assert torch.equal(part[key], out[key][sl]), key
    # backward: linear in the upstream gradients
    g = torch.Generator(device=dev).manual_seed(2)
    w1, w2 = torch.randn(B, 21, 3, generator=g, device=dev), torch.randn(B, 21, 3, generator=g, device=dev)

    def grads(w):
        r, b = rotmat.clone().requires_grad_(True), betas.clone().requires_grad_(True)
        o = head(r, b, cam, K)
        return torch.autograd.grad(o["j3d.cam.l"], (r, b), grad_outputs=w)

    g1, g2, g12 = grads(w1), grads(w2), grads(1.5 * w1 + w2)
    for a, b, c in zip(g1, g2, g12):
        assert rel(c, (1.5 * a + b).cpu()) <= 2e-5


def test_zero_batch_and_error_paths(dev):
    from hands_b200 import _lib
    from hands_b200.common import rot

    lib = _lib.load()
    assert rot.matrix_to_axis_angle(torch.empty(0, 3, 3, device=dev)).shape == (0, 3)
    # workspace too small -> HB_E_WORKSPACE with a message, no launch
    r = torch.eye(3, device=dev).repeat(2, 16, 1, 1).contiguous()
    b = torch.zeros(2, 10, device=dev)
    ws = torch.empty(16, device=dev)
    import ctypes
    P = ctypes.c_void_p
    rc = lib.hb_mano_head_fwd(P(1), P(r.data_ptr()), 1, None, P(b.data_ptr()), None, None, None, 2, 224.0, 0.1,
                              None, None, None, None, None, None, P(ws.data_ptr()), 64, None)
    assert rc == -3 and b"workspace" in lib.hb_last_error_string()


def test_no_cpu_fallback():
    from hands_b200.common import rot

    with pytest.raises(RuntimeError):
        rot.matrix_to_axis_angle(torch.eye(3)[None])


@pytest.mark.parametrize("res,cpi", [(224, 2), (96, 1), (64, 3)])
def test_pcl_fast_forward_matches_exact_forward(dev, res, cpi):
    """The default (fast) forward keeps the reference's sample positions and only evaluates the resize separably: a few ulp
    from the exact-mode forward (which is bit-identical to torch on > 99.9 % of pixels), on white noise."""
    from hands_b200 import _lib
    from hands_b200.pcl import perspective_crop

    B = 5
    n = B * cpi
    img, bbox, K = synthetic_pcl_inputs(n, seed=res, img_res=res, smin=res // 4, smax=3 * res // 4)
    img = img[:B].contiguous().to(dev)
    bbox[0] = torch.tensor([0, 0, 30, 40])                      # touches the top-left image corner: zero-padding border of the tile
    bbox[1] = torch.tensor([res - 41, res - 31, res - 1, res - 1])   # bottom-right corner
    bbox[2] = torch.tensor([7, 9, 7, 9])                         # empty box -> s = img_res
    lib = _lib.load()
    out = {}
    prev = lib.hb_pcl_set_exact(0)
    try:
        for mode in (0, 1):
            lib.hb_pcl_set_exact(mode)
            with torch.no_grad():
                out[mode], _ = perspective_crop(img, bbox.to(dev), K.to(dev), img_res=res, crops_per_img=cpi)
    finally:
        lib.hb_pcl_set_exact(prev)
    tol_check(f"pcl_fast_vs_exact[{res}]", float((out[0] - out[1]).abs().max() / out[1].abs().max()), 2e-6)


@pytest.mark.parametrize("res,cpi", [(224, 2), (96, 1)])
def test_pcl_uint8_source_matches_normalised_fp32_source(dev, res, cpi):
    """hb_pcl_fwd_u8: crops of the 8-bit image with the normalisation fused == crops of the normalised fp32 image
    ((u/255 - mean)/std as torchvision Normalize computes it, hands_light_dataset.py:177-184); and against the oracle."""
    from hands_b200.pcl import perspective_crop

    B = 4
    n = B * cpi
    _, bbox, K = synthetic_pcl_inputs(n, seed=res + 1, img_res=res, smin=res // 4, smax=3 * res // 4)
    bbox[0] = torch.tensor([0, 0, 50, 33])
    g = torch.Generator().manual_seed(4)
    u8 = torch.randint(0, 256, (B, 3, res, res), generator=g, dtype=torch.uint8)
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    x = (u8.float() / 255.0 - torch.tensor(mean).view(1, 3, 1, 1)) / torch.tensor(std).view(1, 3, 1, 1)
    with torch.no_grad():
        c8, r8 = perspective_crop(u8.to(dev), bbox.to(dev), K.to(dev), img_res=res, crops_per_img=cpi, mean=mean, std=std)
        cf, rf = perspective_crop(x.to(dev), bbox.to(dev), K.to(dev), img_res=res, crops_per_img=cpi)
    assert torch.equal(r8, rf)
    tol_check(f"pcl_u8_vs_fp32[{res}]", float((c8 - cf).abs().max() / cf.abs().max()), 1e-6)
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        ref, _ = O.perspective_crop(x.repeat_interleave(cpi, dim=0), bbox, K, res)
    finally:
        torch.set_num_threads(nt)
    tol_check(f"pcl_u8_vs_oracle[{res}]", float((c8.cpu() - ref).abs().max() / ref.abs().max()), 2e-5)
    with pytest.raises(ValueError):
        perspective_crop(u8.to(dev), bbox.to(dev), K.to(dev), img_res=res, crops_per_img=cpi)   # mean/std are required
    with pytest.raises(ValueError, match="inverted"):
        bad = bbox.clone()
        bad[1] = torch.tensor([60, 60, 20, 20])
        perspective_crop(x.to(dev), bad, K.to(dev), img_res=res, crops_per_img=cpi)


def test_compute_loss_light_against_reference_source(dev, golden_dir):
    """f2: every MANO term of the reference's own compute_loss_light (golden from loss_arctic_sf.py:20-158) -- cam_t (+init),
    relative translation, key-points 2D/3D, pose, beta, both hands -- and the gradients of the weighted total w.r.t. every
    prediction, through hands_b200.losses.compute_loss_light (hb_vec_loss_*, hb_kp_loss_*, hb_axis_angle_to_matrix)."""
    from hands_b200.losses import axis_angle_to_matrix, compute_loss_light

    g = {k: v for k, v in np.load(os.path.join(golden_dir, "loss_light.npz")).items()}
    P = {k[5:]: torch.from_numpy(v).to(dev).requires_grad_(True) for k, v in g.items() if k.startswith("pred:")}
    G = {k[3:]: torch.from_numpy(v).to(dev) for k, v in g.items() if k.startswith("gt:")}
    M = {k[5:]: torch.from_numpy(v).to(dev) for k, v in g.items() if k.startswith("meta:")}
    tol_check("aa_to_matrix", float((axis_angle_to_matrix(G["mano.pose.r"].reshape(-1, 3)).cpu() - torch.from_numpy(g["gt_rotmat_r"])).abs().max()), 1e-6)
    out = compute_loss_light(P, G, M)
    keys = [k[5:] for k in g if k.startswith("loss:")]
    assert sorted(out.keys()) == sorted(keys)
    total = 0.0
    for k in keys:
        loss, w = out[k]
        assert loss.shape == (1,) and w == float(g["weight:" + k])
        tol_check(f"loss_light[{k}]", abs(float(loss) - float(g["loss:" + k])) / max(abs(float(g["loss:" + k])), 1e-12), 1e-5)
        total = total + loss * w
    grads = torch.autograd.grad(total, list(P.values()), allow_unused=True)
    for k, gr in zip(P, grads):
        ref = torch.from_numpy(g["grad:" + k])
        if float(ref.abs().max()) == 0.0:
            assert gr is None or float(gr.abs().max()) == 0.0
        else:
            tol_check(f"loss_light.grad[{k}]", rel(gr, ref), 1e-4)
    # run-to-run bit reproducibility of the reductions
    out2 = compute_loss_light(P, G, M)
    assert all(torch.equal(out[k][0], out2[k][0]) for k in keys)


def test_materialise_subset_of_outputs(dev):
    """MANOHead(materialise=...): unread outputs are never written, the rest (and the gradients) are bit-identical."""
    from hands_b200.src.nets.hand_heads.mano_head import MANOHead

    B = 33
    rotmat, betas, cam, K = [t.to(dev) for t in synthetic_head_inputs(B, seed=3)]
    full = MANOHead(True, 1000.0, IMG_RES, synthetic=True).to(dev)
    lean = MANOHead(True, 1000.0, IMG_RES, synthetic=True, materialise=("j3d.cam", "j2d.norm")).to(dev)
    w3, w2 = torch.randn(B, 21, 3, device=dev), torch.randn(B, 21, 2, device=dev)
    res = []
    for head in (full, lean):
        r = rotmat.clone().requires_grad_(True)
        o = head(r, betas, cam, K)
        (gr,) = torch.autograd.grad((o["j3d.cam.r"] * w3).sum() + (o["j2d.norm.r"] * w2).sum(), r)
        res.append((o, gr))
    assert sorted(res[1][0].keys()) == sorted(["cam_t.wp.r", "j3d.cam.r", "j2d.norm.r", "beta.r", "pose.r"])
    for key in ("j3d.cam.r", "j2d.norm.r"):
        assert torch.equal(res[0][0][key], res[1][0][key])
    assert torch.equal(res[0][1], res[1][1])
    with pytest.raises(KeyError):
        res[1][0]["vertices.r"]
    with pytest.raises(ValueError):
        MANOHead(True, 1000.0, IMG_RES, synthetic=True, materialise=("verts",))


def test_mano_decimator_gpu(dev, golden_dir):
    from hands_b200.common.body_models import MANODecimator

    g = np.load(os.path.join(golden_dir, "decimator.npz"))
    dec = MANODecimator(data={"D_right": g["D_right"], "D_left": g["D_left"]})
    out = dec.downsample(torch.from_numpy(g["verts"]).to(dev), True)
    tol_check("decimator", rel(out, torch.from_numpy(g["sub_r"])), 1e-5)   # cuBLAS may use TF32-free fp32 here; 1e-5 relative


def test_pcl_more_than_65535_crops(dev):
    """C4's true shard at 2 GPUs is 32,768 samples = 65,536 crops per launch: crops live on grid.x (no 65,535 limit).
    Small images so the batch stays light; a slice recomputed on its own must match bit for bit, forward and backward."""
    from hands_b200.pcl import perspective_crop

    res, n = 32, 66000
    g = torch.Generator().manual_seed(9)
    img = torch.randn(n, 1, res, res, generator=g).to(dev)
    side = torch.randint(8, 25, (n,), generator=g)
    x0 = torch.randint(0, res - 25, (n,), generator=g)
    y0 = torch.randint(0, res - 25, (n,), generator=g)
    bbox = torch.stack([x0, y0, x0 + side, y0 + side], dim=1).int().to(dev)
    K = torch.tensor([[60.0, 0, 16], [0, 60.0, 16], [0, 0, 1]]).expand(n, 3, 3).contiguous().to(dev)
    w = torch.randn(n, 1, res, res, generator=g).to(dev)
    x = img.clone().requires_grad_(True)
    crop, _ = perspective_crop(x, bbox, K, img_res=res)
    (gx,) = torch.autograd.grad((crop * w).sum(), x)
    sl = slice(65500, 65900)
    xs = img[sl].clone().requires_grad_(True)
    cs, _ = perspective_crop(xs, bbox[sl], K[sl], img_res=res)
    (gs,) = torch.autograd.grad((cs * w[sl]).sum(), xs)
    assert torch.equal(cs, crop[sl]) and torch.equal(gs, gx[sl])
    assert float(crop[-1].abs().max()) > 0


def test_backward_reusing_forward_workspace_is_bit_identical(heads, dev):
    """hb_mano_head_bwd_reuse (the backward picks up the forward's feature rows / transforms / v_posed from the workspace)
    against hb_mano_head_bwd (everything recomputed): the first backward through a node reuses, the second recomputes."""
    B = 40
    rotmat, betas, cam, K = [t.to(dev) for t in synthetic_head_inputs(B, seed=21, small_s_frac=0.2)]
    r, b, c = rotmat.clone().requires_grad_(True), betas.clone().requires_grad_(True), cam.clone().requires_grad_(True)
    o = heads[True](r, b, c, K)
    g = torch.Generator(device=dev).manual_seed(0)
    loss = (o["v3d.cam.r"] * torch.randn(B, 778, 3, generator=g, device=dev)).sum() + (o["j2d.norm.r"] * torch.randn(B, 21, 2, generator=g, device=dev)).sum()
    first = torch.autograd.grad(loss, (r, b, c), retain_graph=True)
    second = torch.autograd.grad(loss, (r, b, c))
    for a, bb in zip(first, second):
        assert torch.equal(a, bb)


def _pcl_grad(dev, img, bbox, K, w, cpi):
    from hands_b200.pcl import perspective_crop

    x = img.to(dev).requires_grad_(True)
    crop, _ = perspective_crop(x, bbox.to(dev), K.to(dev), img_res=224, crops_per_img=cpi)
    (g,) = torch.autograd.grad(crop, x, grad_outputs=w.to(dev))
    return g


@pytest.mark.parametrize("fmin,fmax,cpi", [(300.0, 1500.0, 2), (110.0, 200.0, 2), (60.0, 110.0, 3), (2000.0, 9000.0, 1)])
def test_pcl_backward_gather_form(dev, fmin, fmax, cpi):
    """The gather form of the transposed grid_sample (tile-row CTAs for 3x224x224) against the oracle's autograd, from mild
    to extreme perspective (short focal lengths: rows drift over many pixel rows, samples closer than a pixel, which can
    overflow a cell's list into the region scan), with boxes that leave the image corner regions empty, overlap each other
    and touch the border.  Bit-reproducible run to run."""
    B = 12
    n = B * cpi
    img, bbox, K = synthetic_pcl_inputs(n, seed=int(fmin), img_res=224, smin=40, smax=224)
    img = img[:B].contiguous()
    g = torch.Generator().manual_seed(int(fmax))
    f = fmin + (fmax - fmin) * torch.rand(n, generator=g)
    K[:, 0, 0] = f
    K[:, 1, 1] = f * (0.9 + 0.2 * torch.rand(n, generator=g))
    K[:, 0, 2] += 30 * torch.randn(n, generator=g)
    bbox[0] = torch.tensor([0, 0, 223, 223])
    bbox[1] = torch.tensor([150, 160, 223, 223])
    bbox[2] = torch.tensor([0, 0, 40, 223])
    w = torch.randn(n, 3, 224, 224, generator=g)
    gi = _pcl_grad(dev, img, bbox, K, w, cpi)
    assert torch.equal(gi, _pcl_grad(dev, img, bbox, K, w, cpi))
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        xr = img.clone().requires_grad_(True)
        ref_crop, _ = O.perspective_crop(xr.repeat_interleave(cpi, dim=0), bbox, K, 224)
        (ref_g,) = torch.autograd.grad(ref_crop, xr, grad_outputs=w)
    finally:
        torch.set_num_threads(nt)
    assert rel(gi, ref_g) <= 1e-4
    # per-image check as well (one bad image must not hide behind the batch's largest value)
    for b in range(B):
        assert rel(gi[b], ref_g[b]) <= 1e-4, b
