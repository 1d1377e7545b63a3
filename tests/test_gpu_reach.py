"""GPU paths that the other parity tests do not reach, each against a plain high-precision reference.

- the blendshape kernel's tile-split regimes (more than one column tile per CTA), which only large batches select;
- the gradient of the head's `pre_rot` (the PCL orientation fix-up as a differentiable input), in every pose format;
- the fixed-order loss reductions past one block of 1024 partials, with every optional operand;
- the log map's edge inputs: rotations of exactly pi, argmax ties, near-zero angles.

Tolerances are BASELINE's: values 1e-5 relative, key-points 1e-3 px, gradients 1e-4 relative, counts bit-exact.  Where
fp32 conditioning limits the reference itself (angles near pi) the bound is max(stated, 3 x the fp32 oracle's own error).
"""
import ctypes

import numpy as np
import pytest
import torch

from hands_b200.synthetic import random_rotmats, synthetic_head_inputs, synthetic_mano_buffers
from oracle import geometry_oracle as O
from _tol import tol_check

pytestmark = pytest.mark.gpu

IMG_RES = 224.0
P = ctypes.c_void_p


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


# ---------------------------------------------------------------------------------------------------------------------
# A. blendshape tile-split regimes
# ---------------------------------------------------------------------------------------------------------------------
HEAD_OUT = ("vertices", "v3d.cam", "joints3d", "j3d.cam", "j2d.norm")
HEAD_LOSS = ("v3d.cam", "j3d.cam", "j2d.norm")
TC_M, TC_TILES, NUM_SMS = 128, 10, 148


def blend_nsplit(B):
    """launch_blend_tc (hands_b200/csrc/mano_tc.cu): nsplit = clamp(148 // ceil(B / 128), 1, 10)."""
    return min(max(NUM_SMS // -(-B // TC_M), 1), TC_TILES)


def _head_run(head, pf, rotmat, betas, cam, K, w):
    r, b, c = rotmat.clone().requires_grad_(True), betas.clone().requires_grad_(True), cam.clone().requires_grad_(True)
    o = head(r, b, c, K)
    loss = sum((o[k + pf] * w[k]).sum() for k in HEAD_LOSS)
    g = torch.autograd.grad(loss, (r, b, c))
    return {k: o[k + pf].detach() for k in HEAD_OUT}, dict(zip(("rotmat", "betas", "cam"), g))


@pytest.mark.parametrize("B,nsplit", [(1800, 9), (2200, 8), (2600, 7), (3000, 6), (3300, 5), (4000, 4), (5000, 3), (9601, 1)])
def test_blend_tile_split_regimes(heads, dev, B, nsplit):
    """launch_blend_tc spreads the 10 column tiles of each 128-hand group over
    nsplit = clamp(148 // ceil(B / 128), 1, 10) CTAs; CTA `split` computes tiles split, split + nsplit, ... and cycles its
    two TMEM accumulators, their full/empty phases and the B-stage ring once per tile.  Batches up to 1792 hands
    (14 groups) run nsplit = 10 (one tile per CTA); these batches run every other count:

        B      groups  nsplit  tiles per CTA
        1800   15      9       2,1,...,1
        2200   18      8       2,2,1,...,1
        2600   21      7       2,2,2,1,...,1
        3000   24      6       2,2,2,2,1,1
        3300   26      5       2 each
        4000   32      4       3,3,2,2
        5000   40      3       4,3,3
        9601   76      1       10 (five phases of each accumulator); last group holds one hand

    A hand's result does not depend on the batch around it (DESIGN.md section 3, "Determinism"), so the full batch must
    equal, bit for bit, the same hands run in chunks of <= 1024 (nsplit = 10, the regime the oracle tests pin): outputs
    and the gradients of a weighted sum of v3d.cam, j3d.cam, j2d.norm.  At nsplit 1 and 3 a sample of hands is also
    checked against the fp64 oracle, which catches a regime that would be wrong the same way in both runs."""
    assert blend_nsplit(B) == nsplit and blend_nsplit(1024) == TC_TILES
    is_rhand = B % 2 == 1
    head, pf = heads[is_rhand], (".r" if is_rhand else ".l")
    rotmat, betas, cam, K = synthetic_head_inputs(B, seed=B, small_s_frac=0.05)
    g = torch.Generator().manual_seed(B)
    w = {"v3d.cam": torch.randn(B, 778, 3, generator=g), "j3d.cam": torch.randn(B, 21, 3, generator=g), "j2d.norm": torch.randn(B, 21, 2, generator=g)}
    d = [t.to(dev) for t in (rotmat, betas, cam, K)]
    wd = {k: v.to(dev) for k, v in w.items()}
    out, grads = _head_run(head, pf, *d, wd)
    for lo in range(0, B, 1024):
        sl = slice(lo, min(lo + 1024, B))
        o, gr = _head_run(head, pf, *[t[sl].contiguous() for t in d], {k: v[sl].contiguous() for k, v in wd.items()})
        for k in HEAD_OUT:
            assert torch.equal(o[k], out[k][sl]), (k, lo)
        for k in gr:
            assert torch.equal(gr[k], grads[k][sl]), ("g_" + k, lo)
    if nsplit not in (1, 3):
        return
    # hands from the first and last groups, every lane quarter of a group (TMEM lanes 0-31, ..., 96-127) and the partial
    # last group; every hand's 2334 coordinates span all ten tiles, so each sampled hand reads every split's output
    pick = torch.randperm(B, generator=torch.Generator().manual_seed(7 * B))[:248].tolist()
    idx = torch.tensor(sorted(set(pick) | {0, 31, 32, 95, 127, 128, B - 129, B - 2, B - 1}))
    ref64 = oracle_head(is_rhand, rotmat[idx], betas[idx], cam[idx], K[idx], torch.float64)
    ref32 = oracle_head(is_rhand, rotmat[idx], betas[idx], cam[idx], K[idx], torch.float32)
    ic = idx.to(dev)
    for k in ("vertices", "joints3d", "v3d.cam", "j3d.cam"):
        tol_check(f"blend_split[{B}].{k}", rel(out[k][ic], ref64[k]), 1e-5, rel(ref32[k], ref64[k]))
    px = (out["j2d.norm"][ic].double().cpu() - ref64["j2d.norm"]).abs().max() * IMG_RES / 2
    own_px = (ref32["j2d.norm"].double() - ref64["j2d.norm"]).abs().max() * IMG_RES / 2
    tol_check(f"blend_split[{B}].j2d_px", px, 1e-3, own_px)

    def oracle_grads(dtype):
        r, b, c = rotmat[idx].to(dtype).requires_grad_(True), betas[idx].to(dtype).requires_grad_(True), cam[idx].to(dtype).requires_grad_(True)
        o = oracle_head(is_rhand, r, b, c, K[idx], dtype)
        return torch.autograd.grad(sum((o[k] * w[k][idx].to(dtype)).sum() for k in HEAD_LOSS), (r, b, c))

    g64, g32 = oracle_grads(torch.float64), oracle_grads(torch.float32)
    for name, r64, r32 in zip(("rotmat", "betas", "cam"), g64, g32):
        tol_check(f"blend_split[{B}].g_{name}", rel(grads[name][ic], r64), 1e-4, rel(r32, r64))


# ---------------------------------------------------------------------------------------------------------------------
# B. gradient of pre_rot
# ---------------------------------------------------------------------------------------------------------------------
ROT6D_ORACLE = {"rows": O.rotation_6d_to_matrix, "cols": O.rot6d_to_rotmat_cols, "cols_paired": O.rot6d_to_rotmat_paired}


@pytest.mark.parametrize("fmt", ["rotmat", "rows", "cols", "cols_paired"])
def test_pre_rot_gradient(heads, dev, fmt):
    """A `pre_rot` that requires grad (e.g. a predicted correction of the global orientation) gets the gradient of the
    reference's chain pose[:, 0] <- pre_rot @ pose[:, 0] -> MANOHead, through the geometry outputs (hb_mano_head_bwd*'s
    g_pre_rot) and through the returned `pose`, which the pose loss reads.  fp64 autograd of the oracle on the same inputs
    is the reference.  The first backward through the node reuses the forward's workspace (hb_mano_head_bwd_reuse), the
    second recomputes (hb_mano_head_bwd): both must match the oracle and each other bit for bit."""
    B = 20
    _, betas, cam, K = synthetic_head_inputs(B, seed=31, small_s_frac=0.2)
    g = torch.Generator().manual_seed(32)
    Pm = random_rotmats(B, g)
    pose_in = synthetic_head_inputs(B, seed=33)[0] if fmt == "rotmat" else torch.randn(B, 16, 6, generator=g)
    w = {"v3d.cam": torch.randn(B, 778, 3, generator=g), "j3d.cam": torch.randn(B, 21, 3, generator=g),
         "j2d.norm": torch.randn(B, 21, 2, generator=g), "pose": torch.randn(B, 16, 3, 3, generator=g)}
    keys = ("v3d.cam", "j3d.cam", "j2d.norm", "pose")

    pi, Pi, bi, ci = (t.to(dev).requires_grad_(True) for t in (pose_in, Pm, betas, cam))
    if fmt == "rotmat":
        o = heads[True](pi, bi, ci, K.to(dev), pre_rot=Pi)
    else:
        o = heads[True].forward_rot6d(pi, bi, ci, K.to(dev), layout=fmt, pre_rot=Pi)
    loss = sum((o[k + ".r"] * w[k].to(dev)).sum() for k in keys)
    first = torch.autograd.grad(loss, (Pi, pi, bi, ci), retain_graph=True)
    second = torch.autograd.grad(loss, (Pi, pi, bi, ci))

    def chain(dtype):
        Po, po, bo, co = (t.to(dtype).requires_grad_(True) for t in (Pm, pose_in, betas, cam))
        rotmat = po if fmt == "rotmat" else ROT6D_ORACLE[fmt](po.reshape(-1, 6)).reshape(B, 16, 3, 3)
        ref = oracle_head(True, O.pcl_fix_global_orient(Po, rotmat), bo, co, K, dtype)
        lo = sum((ref[k] * w[k].to(dtype)).sum() for k in keys)
        return ref, torch.autograd.grad(lo, (Po, po, bo, co))

    o64, g64 = chain(torch.float64)
    o32, g32 = chain(torch.float32)
    tol_check(f"pre_rot[{fmt}].pose", rel(o["pose.r"], o64["pose"].detach()), 1e-5, rel(o32["pose"].detach(), o64["pose"].detach()))
    tol_check(f"pre_rot[{fmt}].j3d.cam", rel(o["j3d.cam.r"], o64["j3d.cam"].detach()), 1e-5, rel(o32["j3d.cam"].detach(), o64["j3d.cam"].detach()))
    for name, a, b, r64, r32 in zip(("pre_rot", "pose", "betas", "cam"), first, second, g64, g32):
        assert torch.equal(a, b), name
        tol_check(f"pre_rot[{fmt}].g_{name}", rel(a, r64), 1e-4, rel(r32, r64))


def test_rot_apply_gradients_and_launches(dev):
    """apply_virtual_rotation (out = R @ M on joint 0): g_M = R^T g always, g_R = g M^T only when R requires grad; with the
    crop layer's R_virt2orig (no grad) the backward is the one launch it always was."""
    from hands_b200 import _lib
    from hands_b200.pcl import apply_virtual_rotation

    B = 37
    g = torch.Generator().manual_seed(4)
    R, M = random_rotmats(B, g), random_rotmats(B * 16, g).reshape(B, 16, 3, 3)
    w = torch.randn(B, 16, 3, 3, generator=g)
    for r_grad in (False, True):
        Rd, Md = R.to(dev).requires_grad_(r_grad), M.to(dev).requires_grad_(True)
        out = apply_virtual_rotation(Rd, Md)
        n0 = _lib.launch_count()
        grads = torch.autograd.grad((out * w.to(dev)).sum(), (Rd, Md) if r_grad else (Md,))
        torch.cuda.synchronize()
        assert _lib.launch_count() - n0 == (2 if r_grad else 1)
        R64, M64 = R.double().requires_grad_(r_grad), M.double().requires_grad_(True)
        ref = torch.autograd.grad((O.pcl_fix_global_orient(R64, M64) * w.double()).sum(), (R64, M64) if r_grad else (M64,))
        assert rel(out, O.pcl_fix_global_orient(R64, M64).detach()) <= 1e-6
        for a, r in zip(grads, ref):
            assert rel(a, r) <= 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# C. loss reductions past one block
# ---------------------------------------------------------------------------------------------------------------------
REDUCE_B = [1, 1023, 1024, 1025, 4097]


def _lib_stream():
    from hands_b200 import _lib
    from hands_b200.functional import _stream

    return _lib, _lib.load(), _stream()


def _grid(shape, g):
    """fp32 values on a 2^-10 grid in [-4, 4]: differences of two or four of them are exact in fp32, so the kernels'
    element-wise terms carry only the rounding of the scale factors and squares."""
    return (torch.randint(-4096, 4097, shape, generator=g, dtype=torch.int32).float() / 1024.0)


def _mask(shape, g, p_zero=0.3):
    return (torch.rand(shape, generator=g) >= p_zero).float()


def _ptr(t):
    return None if t is None else P(t.data_ptr())


def _check_sum(name, got, ref):
    assert abs(got - ref) <= 1e-5 * abs(ref), (name, got, ref)


def _check_grad(name, got, ref, scale):
    """element-wise: |got - ref| <= 1e-4 * scale, where scale >= |ref| is the magnitude of the terms the element sums
    (|ref| itself for a single term); a zero reference (masked) must come back as exactly zero"""
    got = got.double().cpu().numpy()
    bad = np.abs(got - ref) > 1e-4 * scale
    assert not bad.any(), (name, int(bad.sum()), got[bad][:4], ref[bad][:4])


@pytest.mark.parametrize("B", REDUCE_B)
def test_kp_loss_reduction(dev, B):
    """hb_kp_loss_fwd/bwd against a float64 numpy restatement of include/hands_b200.h: all eight sums, both gradients
    element by element.  Masks with zero root validity (the root still gets the gradient of every joint taken relative
    to it), invalid hands, zero gates, NULL hand_valid / gates, an all-invalid batch; sums are bit-reproducible."""
    _lib, lib, st = _lib_stream()
    g = torch.Generator().manual_seed(B)
    j3d, gt3, j2d, gt2 = _grid((B, 21, 3), g), _grid((B, 21, 3), g), _grid((B, 21, 2), g), _grid((B, 21, 2), g)
    jv = _mask((B, 21), g)
    jv[::3, 0] = 0.0
    hv, gate3, gate2 = _mask((B,), g), _mask((B,), g), _mask((B,), g)
    gate3[0] = 1.0   # hand 0: root invalid, 3D term on
    variants = {
        "mixed": (jv, hv, gate3, gate2),
        "null": (torch.ones(B, 21), None, None, None),
        "all_invalid": (torch.zeros(B, 21), torch.zeros(B), torch.zeros(B), torch.zeros(B)),
    }
    cd = [t.to(dev) for t in (j3d, j2d, gt3, gt2)]
    g3s, g2s = 0.7, -1.3
    gl3, gl2 = torch.tensor([g3s], device=dev), torch.tensor([g2s], device=dev)
    a3, b3, a2, b2 = (t.double().numpy() for t in (j3d, gt3, j2d, gt2))
    for name, (v, hv, ga3, ga2) in variants.items():
        vd, hvd, ga3d, ga2d = (None if t is None else t.to(dev) for t in (v, hv, ga3, ga2))
        partial = torch.empty(B, 8, device=dev)
        sums = [torch.empty(8, device=dev) for _ in range(2)]
        for s in sums:
            _lib.check(lib.hb_kp_loss_fwd(*map(_ptr, cd + [vd, hvd, ga3d, ga2d]), B, IMG_RES, _ptr(partial), _ptr(s), st), "hb_kp_loss_fwd")
        gj3, gj2 = torch.empty(B, 21, 3, device=dev), torch.empty(B, 21, 2, device=dev)
        _lib.check(lib.hb_kp_loss_bwd(*map(_ptr, cd + [vd, ga3d, ga2d]), B, _ptr(gl3), _ptr(gl2), _ptr(gj3), _ptr(gj2), st), "hb_kp_loss_bwd")
        assert torch.equal(sums[0], sums[1]), name
        got = sums[0].double().cpu().numpy()

        vn = v.double().numpy()
        hvn = np.ones(B) if hv is None else hv.double().numpy()
        g3n = np.ones(B) if ga3 is None else ga3.double().numpy()
        g2n = np.ones(B) if ga2 is None else ga2.double().numpy()
        d3 = (a3 - a3[:, :1]) - (b3 - b3[:, :1])
        d2 = a2 - b2
        sq3, sq2 = (d3 ** 2).sum(-1), (d2 ** 2).sum(-1)
        ref = [(sq3 * vn * g3n[:, None]).sum(), (sq2 * vn * g2n[:, None]).sum(), (hvn * np.sqrt(sq3).mean(1)).sum(), hvn.sum(),
               (np.sqrt(sq2) * 0.5 * IMG_RES * vn * hvn[:, None]).sum(), (vn * hvn[:, None]).sum(), 0.0, 0.0]
        for k in (0, 1, 2, 4):
            _check_sum(f"kp[{B},{name}].sums[{k}]", got[k], ref[k])
        for k in (3, 5, 6, 7):   # counts and the unused slots: exact
            assert got[k] == ref[k], (name, k, got[k], ref[k])
        G3 = 2.0 * g3s / (B * 63) * (vn * g3n[:, None])[..., None] * d3
        S3 = np.abs(G3)
        G3[:, 0] -= G3.sum(1)
        S3[:, 0] += S3.sum(1)
        G2 = 2.0 * g2s / (B * 42) * (vn * g2n[:, None])[..., None] * d2
        _check_grad(f"kp[{B},{name}].g_j3d", gj3, G3, S3)
        _check_grad(f"kp[{B},{name}].g_j2d", gj2, G2, np.abs(G2))
        if name == "mixed":
            root_off = (vn[:, 0] == 0) & (g3n != 0) & (vn[:, 1:].sum(1) > 0)
            assert root_off.any() and (np.abs(G3[root_off, 0]).sum(-1) > 0).all()


@pytest.mark.parametrize("D", [3, 10, 144])
@pytest.mark.parametrize("B", REDUCE_B)
def test_vec_loss_reduction(dev, B, D):
    """hb_vec_loss_fwd/bwd, every operand combination the header allows (pred_minus, gt_minus, pred2, valid, valid2, gate
    each NULL or given; plus an all-invalid batch), against a float64 numpy restatement of the header's formula:
    the sum, and g_pred / g_pred_minus / g_pred2 element by element; the sum is bit-reproducible."""
    import itertools

    _lib, lib, st = _lib_stream()
    g = torch.Generator().manual_seed(B * 1000 + D)
    host = {k: _grid((B, D), g) for k in ("pred", "pred_minus", "gt", "gt_minus", "pred2")}
    host.update({k: _mask((B,), g) for k in ("valid", "valid2", "gate")})
    dv = {k: v.to(dev) for k, v in host.items()}
    npv = {k: v.double().numpy() for k, v in host.items()}
    gs = 0.45
    gl = torch.tensor([gs], device=dev)
    zeros = torch.zeros(B, device=dev)
    opt = ("pred_minus", "gt_minus", "pred2", "valid", "valid2", "gate")
    cases = [dict(zip(opt, c)) for c in itertools.product((False, True), repeat=6)]
    cases.append(dict(zip(opt, (True,) * 6), all_invalid=True))
    partial = torch.empty(B, device=dev)
    out = [torch.empty(1, device=dev) for _ in range(2)]
    gp, gm, g2 = (torch.empty(B, D, device=dev) for _ in range(3))
    for c in cases:
        use = lambda k: dv[k] if c[k] else None  # noqa: E731
        valid = zeros if c.get("all_invalid") else use("valid")
        args = [dv["pred"], use("pred_minus"), dv["gt"], use("gt_minus"), use("pred2"), valid, use("valid2"), use("gate")]
        for o in out:
            _lib.check(lib.hb_vec_loss_fwd(*map(_ptr, args), B, D, _ptr(partial), _ptr(o), st), "hb_vec_loss_fwd")
        _lib.check(lib.hb_vec_loss_bwd(*map(_ptr, args), B, D, _ptr(gl), _ptr(gp), _ptr(gm if c["pred_minus"] else None), _ptr(g2), st),
                   "hb_vec_loss_bwd")
        tag = f"vec[{B},{D},{''.join('1' if c[k] else '0' for k in opt)}{',invalid' if c.get('all_invalid') else ''}]"
        assert torch.equal(out[0], out[1]), tag

        n = lambda k: npv[k] if c[k] else 0.0  # noqa: E731
        m = np.ones(B)
        for k in ("valid", "valid2", "gate"):
            if c[k]:
                m = m * npv[k]
        if c.get("all_invalid"):
            m = m * 0.0
        t = npv["gt"] - n("gt_minus")
        d = (npv["pred"] - n("pred_minus")) - t
        e = (npv["pred2"] - t) if c["pred2"] else np.zeros_like(d)
        ref = (m * ((d ** 2).sum(1) + (e ** 2).sum(1))).sum()
        _check_sum(tag + ".sum", float(out[0]), ref)
        k = 2.0 * gs * m[:, None] / (B * D)
        _check_grad(tag + ".g_pred", gp, k * d, np.abs(k * d))
        _check_grad(tag + ".g_pred2", g2, k * e, np.abs(k * e))
        if c["pred_minus"]:
            _check_grad(tag + ".g_pred_minus", gm, -k * d, np.abs(k * d))


@pytest.mark.parametrize("B", REDUCE_B)
def test_mask_l1_reduction(dev, B):
    """hb_mask_l1_loss_fwd/bwd at n = 224 x 224 against float64: the loss (per-sample |pred - gt| sums in float64, then
    masked and averaged), the gradient sign(pred - gt) * valid * gate / (B n) element by element (zero where pred == gt),
    with valid / gate given (zeros among them), NULL, and an all-invalid batch; the loss is bit-reproducible."""
    _lib, lib, st = _lib_stream()
    n = 224 * 224
    g = torch.Generator(device=dev).manual_seed(B)
    pred = torch.rand(B, n, generator=g, device=dev)
    gt = (torch.rand(B, n, generator=g, device=dev) > 0.5).float()
    tie = torch.rand(B, n, generator=g, device=dev) < 0.01
    pred[tie] = gt[tie]
    gh = torch.Generator().manual_seed(B)
    vm, gm = _mask((B,), gh), _mask((B,), gh)
    row = torch.cat([(pred[i:i + 512].double() - gt[i:i + 512].double()).abs().sum(1) for i in range(0, B, 512)]).cpu().numpy()
    gs = 1.7
    gl = torch.tensor([gs], device=dev)
    partial = torch.empty(B, device=dev)
    g_pred = torch.empty_like(pred)
    for name, valid, gate in (("mixed", vm, gm), ("null", None, None), ("all_invalid", torch.zeros(B), gm)):
        vd, gd = (None if t is None else t.to(dev) for t in (valid, gate))
        loss = [torch.empty(1, device=dev) for _ in range(2)]
        for lo in loss:
            _lib.check(lib.hb_mask_l1_loss_fwd(_ptr(pred), _ptr(gt), _ptr(vd), _ptr(gd), B, n, _ptr(partial), _ptr(lo), st), "hb_mask_l1_loss_fwd")
        _lib.check(lib.hb_mask_l1_loss_bwd(_ptr(pred), _ptr(gt), _ptr(vd), _ptr(gd), _ptr(gl), B, n, _ptr(g_pred), st), "hb_mask_l1_loss_bwd")
        assert torch.equal(loss[0], loss[1]), name
        m = np.ones(B)
        for t in (valid, gate):
            if t is not None:
                m = m * t.double().numpy()
        _check_sum(f"mask[{B},{name}].loss", float(loss[0]), float((m * row).sum() / (B * n)))
        scale = torch.from_numpy(gs * m / (B * n)).to(dev)[:, None]
        for i in range(0, B, 512):
            want = torch.sign(pred[i:i + 512].double() - gt[i:i + 512].double()) * scale[i:i + 512]
            err = (g_pred[i:i + 512].double() - want).abs()
            assert bool((err <= 1e-4 * want.abs()).all()), (name, i, float(err.max()))


# ---------------------------------------------------------------------------------------------------------------------
# D. log-map edges
# ---------------------------------------------------------------------------------------------------------------------
def _axis_angle_rot(axis, ang):
    n = torch.tensor(axis, dtype=torch.float64)
    n = n / n.norm()
    Kx = torch.tensor([[0.0, -n[2], n[1]], [n[2], 0.0, -n[0]], [-n[1], n[0], 0.0]], dtype=torch.float64)
    return torch.eye(3, dtype=torch.float64) + np.sin(ang) * Kx + (1.0 - np.cos(ang)) * Kx @ Kx


def _logmap_edge_cases():
    cases = {}
    for i, name in enumerate("xyz"):   # exact pi about each axis: diag with one +1, w = 0, branches 1-3
        cases[f"pi_{name}"] = torch.diag(torch.tensor([1.0 if k == i else -1.0 for k in range(3)], dtype=torch.float64))
    for axis in ((1, 2, 3), (1, 1, 0), (-1, 0.5, 2), (0.2, -3, 1)):   # oblique pi: 2 n n^T - I
        n = torch.tensor(axis, dtype=torch.float64)
        n = n / n.norm()
        cases[f"pi_{axis}"] = 2.0 * torch.outer(n, n) - torch.eye(3, dtype=torch.float64)
    # near pi the real part w = sin(delta / 2) is the smallest quaternion component, so the argmax lands on the axis'
    # dominant coordinate (branches 1, 2, 3); branch 0 is reached at most up to 120 deg (axis (1,1,1)), taken just below
    for axis, want in (((1, 0.3, -0.2), 1), ((0.1, -1, 0.4), 2), ((-0.3, 0.2, 1), 3)):
        for delta in (1e-3, 1e-5):
            cases[f"near_pi_{want}_{delta}"] = _axis_angle_rot(axis, np.pi - delta)
    cases["idx0_119.9deg"] = _axis_angle_rot((1, 1, 1), 2 * np.pi / 3 - 2e-3)
    cyc = torch.tensor([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]], dtype=torch.float64)
    cases["cyclic_+120"], cases["cyclic_-120"] = cyc, cyc.T.contiguous()   # all four |q| equal: the first maximum wins
    cases["identity"] = torch.eye(3, dtype=torch.float64)
    for axis in ((1, 0, 0), (0.3, -0.5, 0.8), (0, 0, -1)):
        cases[f"tiny_{axis}"] = _axis_angle_rot(axis, 1e-7)
    return {k: v.float() for k, v in cases.items()}


def test_logmap_edges(dev):
    """hb_matrix_to_axis_angle_fwd/bwd (common/rot.py:180-193) on the inputs where its branches and series meet: exact
    pi (w = 0), near pi in each reachable argmax branch, the cyclic permutation matrices (all four |q| tied), identity and
    1e-7 angles (the small-angle series of forward and backward).  Each matrix is checked on its own against fp64
    autograd of the oracle on the same fp32 input: axis-angle 1e-5 absolute, gradient 1e-4 relative, widened to
    3 x the fp32 oracle's own error where fp32 conditioning limits it."""
    from hands_b200.common import rot

    cases = _logmap_edge_cases()
    names = list(cases)
    R = torch.stack([cases[k] for k in names])
    want_idx = {"pi_x": 1, "pi_y": 2, "pi_z": 3, "cyclic_+120": 0, "cyclic_-120": 0, "idx0_119.9deg": 0}
    want_idx.update({k: int(k.split("_")[2]) for k in names if k.startswith("near_pi")})
    for k, i in want_idx.items():   # the inputs land where their names say (fp32 q_abs, first maximum)
        m = cases[k].double()
        t = torch.stack([1 + m[0, 0] + m[1, 1] + m[2, 2], 1 + m[0, 0] - m[1, 1] - m[2, 2], 1 - m[0, 0] + m[1, 1] - m[2, 2], 1 - m[0, 0] - m[1, 1] + m[2, 2]])
        assert int(O.sqrt_positive_part(t).argmax()) == i, k
    w = torch.randn(len(names), 3, generator=torch.Generator().manual_seed(11))
    Rd = R.to(dev).requires_grad_(True)
    aa = rot.matrix_to_axis_angle(Rd)
    (gR,) = torch.autograd.grad((aa * w.to(dev)).sum(), Rd)
    aa, gR = aa.detach().cpu().double(), gR.cpu().double()

    def oracle(dtype):
        x = R.to(dtype).requires_grad_(True)
        a = O.matrix_to_axis_angle(x)
        return a.detach().double(), torch.autograd.grad((a * w.to(dtype)).sum(), x)[0].double()

    a64, g64 = oracle(torch.float64)
    a32, g32 = oracle(torch.float32)
    assert torch.isfinite(aa).all() and torch.isfinite(gR).all()
    for i, k in enumerate(names):
        tol_check(f"logmap[{k}].aa", (aa[i] - a64[i]).abs().max(), 1e-5, (a32[i] - a64[i]).abs().max())
        gs = g64[i].abs().max().clamp_min(1e-30)
        tol_check(f"logmap[{k}].gR", (gR[i] - g64[i]).abs().max() / gs, 1e-4, (g32[i] - g64[i]).abs().max() / gs)
