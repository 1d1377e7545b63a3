"""GPU checks of hb_procrustes_metrics (PA-MPJPE / PA-MPVPE, MPJPE-RA / root-relative MPVPE as device partial sums)
against the fp64 oracle `tests/procrustes_oracle.py::procrustes_errors`, on MANO-head outputs and on edge cases."""
import numpy as np
import pytest
import torch

from hands_b200.synthetic import synthetic_head_inputs, synthetic_mano_buffers
from oracle import geometry_oracle as O
from procrustes_oracle import procrustes_errors
from _tol import tol_check

pytestmark = pytest.mark.gpu

IMG_RES = 224.0


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def hands(dev):
    """gt: the oracle MANO head (camera space) on GT-side parameters; pred: the GPU head on perturbed pose, betas and cam.
    8192 right hands: joints (B,21,3) and vertices (B,778,3) of both, fp32."""
    from hands_b200.src.nets.hand_heads.mano_head import MANOHead

    B = 8192
    rotmat, betas, cam, K = synthetic_head_inputs(B, seed=7)
    g = torch.Generator().manual_seed(8)
    buf = synthetic_mano_buffers(True)
    gt_j, gt_v = [], []
    for lo in range(0, B, 1024):
        o = O.mano_head_forward(buf, rotmat[lo:lo + 1024], betas[lo:lo + 1024], cam[lo:lo + 1024], K[lo:lo + 1024], IMG_RES, 0.1)
        gt_j.append(o["j3d.cam"])
        gt_v.append(o["v3d.cam"])
    dR = O.batch_rodrigues(0.1 * torch.randn(B * 16, 3, generator=g, dtype=torch.float64)).reshape(B, 16, 3, 3)   # ~0.17 rad per joint
    prot = (rotmat.double() @ dR).float()
    pbetas = betas + 0.3 * torch.randn(B, 10, generator=g)
    pcam = cam * (1 + 0.05 * torch.randn(B, 3, generator=g))
    head = MANOHead(True, 1000.0, IMG_RES, synthetic=True).to(dev)
    with torch.no_grad():
        out = head(prot.contiguous().to(dev), pbetas.to(dev), pcam.to(dev), K.to(dev))
    return {"gt_j": torch.cat(gt_j).contiguous().to(dev), "gt_v": torch.cat(gt_v).contiguous().to(dev),
            "pred_j": out["j3d.cam.r"].contiguous(), "pred_v": out["v3d.cam.r"].contiguous()}


def _check_against_oracle(name, pred, gt, per_hand, sums, root_pred=None, root_gt=None, valid=None):
    pa, ra, _ = procrustes_errors(pred.cpu().numpy(), gt.cpu().numpy(),
                                    None if root_pred is None else root_pred.cpu().numpy(), None if root_gt is None else root_gt.cpu().numpy())
    v = np.ones(len(pa), bool) if valid is None else valid.cpu().numpy() != 0
    ph = per_hand.cpu().double().numpy()
    use = v & np.isfinite(pa)
    assert np.isnan(ph[~v]).all() and np.isnan(ph[v & ~np.isfinite(pa), 0]).all()
    err_pa = np.abs(ph[use, 0] - pa[use]) / (2e-7 + 1e-5 * np.abs(pa[use]))
    err_ra = np.abs(ph[v, 1] - ra[v]) / (2e-7 + 1e-5 * np.abs(ra[v]))
    tol_check(f"{name}.pa_per_hand(/(2e-7 m + 1e-5 rel))", err_pa.max(initial=0.0), 1.0)
    tol_check(f"{name}.ra_per_hand(/(2e-7 m + 1e-5 rel))", err_ra.max(initial=0.0), 1.0)
    s = sums.cpu().double().numpy()
    assert s[1] == use.sum() and s[3] == v.sum() and s[4] == (v & ~np.isfinite(pa)).sum() and (s[5:] == 0).all()
    if use.any():
        tol_check(f"{name}.sums0_rel", abs(s[0] - pa[use].sum()) / pa[use].sum(), 1e-5)
    if v.any():
        tol_check(f"{name}.sums2_rel", abs(s[2] - ra[v].sum()) / ra[v].sum(), 1e-5)
    return pa, ra


@pytest.mark.parametrize("kind", ["joints", "vertices", "decimated"])
def test_parity_with_the_fp64_oracle(dev, hands, kind):
    from hands_b200.losses import procrustes_metrics

    if kind == "joints":
        pred, gt, rp, rq = hands["pred_j"], hands["gt_j"], None, None
    elif kind == "vertices":   # root-relative MPVPE: the roots are joint 0 of j3d.cam
        pred, gt, rp, rq = hands["pred_v"], hands["gt_v"], hands["pred_j"][:, 0], hands["gt_j"][:, 0]
    else:                      # a 195-point decimated mesh (row-stochastic 195 x 778 down-sampler), 1000 hands
        g = torch.Generator().manual_seed(9)
        D = torch.rand(195, 778, generator=g) ** 8
        D = (D / D.sum(1, keepdim=True)).to(dev)
        pred, gt = torch.einsum("nv,bvk->bnk", D, hands["pred_v"][:1000]), torch.einsum("nv,bvk->bnk", D, hands["gt_v"][:1000])
        rp = rq = None
    valid = (torch.arange(pred.shape[0], device=dev) % 7 != 3).float()
    sums, per_hand = procrustes_metrics(pred, gt, valid, rp, rq)
    _check_against_oracle(f"procrustes[{kind}]", pred, gt, per_hand, sums, rp, rq, valid)


def test_edge_cases_in_one_batch(dev):
    from hands_b200.losses import procrustes_metrics

    g = torch.Generator().manual_seed(11)
    rng = np.random.default_rng(11)
    B, N = 8, 21
    gt = (torch.randn(B, N, 3, generator=g, dtype=torch.float64) * 0.04 + torch.tensor([0.05, -0.1, 0.8], dtype=torch.float64))
    pred = gt + 0.01 * torch.randn(B, N, 3, generator=g, dtype=torch.float64)
    R = torch.from_numpy(np.linalg.qr(rng.normal(size=(3, 3)))[0])
    R = R * torch.sign(torch.det(R))
    pred[0] = 1.3 * gt[0] @ R.T + torch.tensor([0.2, 0.1, -0.3], dtype=torch.float64)   # exact similarity copy
    pred[1] = gt[1] * torch.tensor([1.0, 1.0, -1.0], dtype=torch.float64) + 0.003 * torch.randn(N, 3, generator=g, dtype=torch.float64)  # mirrored
    gt[2, :, 2] = 0.8                                                                     # planar target
    gt[3] += torch.tensor([5.0, 0.0, 0.0], dtype=torch.float64)                          # 5 m from the origin
    pred[3] += torch.tensor([5.0, 0.0, 0.0], dtype=torch.float64)
    pred[5] = pred[5, 0]                                                                  # degenerate prediction
    pred, gt = pred.float().to(dev), gt.float().to(dev)
    valid = torch.ones(B, device=dev)
    valid[4] = 0.0
    sums, per_hand, aligned = procrustes_metrics(pred, gt, valid, return_aligned=True)
    pa, _ = _check_against_oracle("procrustes[edge]", pred, gt, per_hand, sums, valid=valid)
    ph = per_hand.cpu()
    assert float(ph[0, 0]) <= 2e-7 and torch.isnan(ph[4]).all() and torch.isnan(ph[5, 0]) and torch.isfinite(ph[5, 1])
    assert float(sums[4]) == 1.0 and float(sums[1]) == 6.0 and float(sums[3]) == 7.0
    assert torch.isnan(aligned[5]).all() and torch.isfinite(aligned[[0, 1, 2, 3, 4, 6, 7]]).all()
    # N = 1: every hand is degenerate
    s1, p1 = procrustes_metrics(pred[:, :1], gt[:, :1], valid)
    assert float(s1[1]) == 0.0 and float(s1[4]) == 7.0 and float(s1[3]) == 7.0 and float(s1[2]) == 0.0 and torch.isnan(p1[:, 0]).all()
    # an empty batch still writes the sums
    s0, p0 = procrustes_metrics(pred[:0], gt[:0])
    assert p0.shape == (0, 2) and torch.equal(s0.cpu(), torch.zeros(8))


def test_aligned_points_match_the_oracle_where_the_rotation_is_unique(dev, hands):
    from hands_b200.losses import procrustes_metrics

    for name, pred, gt in (("joints", hands["pred_j"][:2048], hands["gt_j"][:2048]), ("vertices", hands["pred_v"][:512], hands["gt_v"][:512])):
        _, _, aligned = procrustes_metrics(pred, gt, return_aligned=True)
        p, q = pred.cpu().double().numpy(), gt.cpu().double().numpy()
        _, _, ref = procrustes_errors(p, q)
        X, Y = p - p.mean(1, keepdims=True), q - q.mean(1, keepdims=True)
        S = np.linalg.svd(np.einsum("bnk,bnl->bkl", X, Y), compute_uv=False)
        unique = (S[:, 1] - S[:, 2]) >= 1e-2 * S[:, 1]
        extent = np.linalg.norm(Y, axis=2).max(1)
        # plus half an fp32 ulp of the output's magnitude: `aligned` is returned in fp32 camera-space coordinates
        half_ulp = 0.5 * np.spacing(np.abs(ref).max(axis=(1, 2)).astype(np.float32)).astype(np.float64)
        err = np.abs(aligned.cpu().double().numpy() - ref).max(axis=(1, 2)) / (1e-6 * extent + half_ulp)
        assert unique.sum() > 0.9 * len(unique)
        tol_check(f"procrustes_aligned[{name}](/(1e-6 extent + half ulp))", err[unique].max(), 1.0)


def test_bit_reproducible_and_independent_of_the_batch_split(dev, hands):
    from hands_b200.losses import procrustes_metrics

    pred, gt = hands["pred_v"][:1024], hands["gt_v"][:1024]
    rp, rq = hands["pred_j"][:1024, 0], hands["gt_j"][:1024, 0]
    a = procrustes_metrics(pred, gt, None, rp, rq, return_aligned=True)
    b = procrustes_metrics(pred, gt, None, rp, rq, return_aligned=True)
    for x, y in zip(a, b):
        assert torch.equal(x.nan_to_num(7.0), y.nan_to_num(7.0))
    for parts in (2, 4, 8):
        n = 1024 // parts
        ph = torch.cat([procrustes_metrics(pred[i * n:(i + 1) * n], gt[i * n:(i + 1) * n], None, rp[i * n:(i + 1) * n], rq[i * n:(i + 1) * n])[1]
                        for i in range(parts)])
        assert torch.equal(ph, a[1])


def test_ra_on_joints_agrees_with_the_keypoint_metric(dev, hands):
    from hands_b200.losses import keypoint_losses, procrustes_metrics

    pred, gt = hands["pred_j"], hands["gt_j"]
    B = pred.shape[0]
    valid = (torch.arange(B, device=dev) % 5 != 0).float()
    sums, _ = procrustes_metrics(pred, gt, valid)
    z2 = torch.zeros(B, 21, 2, device=dev)
    _, _, kp = keypoint_losses(pred, z2, gt, z2, torch.ones(B, 21, device=dev), valid)
    assert float(sums[3]) == float(kp[3])
    assert abs(float(sums[2] / sums[3]) - float(kp[2] / kp[3])) <= 1e-6 * float(kp[2] / kp[3])


def test_python_wrapper(dev, hands):
    from hands_b200.distributed import PackedMetrics
    from hands_b200.losses import procrustes_metrics

    pred, gt = hands["pred_j"][:64], hands["gt_j"][:64]
    with pytest.raises(RuntimeError, match="no CPU path"):
        procrustes_metrics(pred.cpu(), gt.cpu())
    with pytest.raises(ValueError):
        procrustes_metrics(pred[..., :2], gt[..., :2])
    with pytest.raises(ValueError):
        procrustes_metrics(pred, gt[:, :20])
    with pytest.raises(ValueError):
        procrustes_metrics(pred, gt, torch.ones(63, device=dev))
    with pytest.raises(ValueError):
        procrustes_metrics(pred, gt, None, torch.zeros(64, 2, device=dev))
    x = pred.clone().requires_grad_(True)
    sums, per_hand = procrustes_metrics(x, gt)
    assert not sums.requires_grad and not per_hand.requires_grad
    pm = PackedMetrics(["pa_mpjpe/r", "mpjpe_ra/r"], dev)
    pm.add("pa_mpjpe/r", sums[0], sums[1])
    pm.add("mpjpe_ra/r", sums[2], sums[3])
    out = pm.reduce()
    assert out["pa_mpjpe/r"] == float(sums[0]) / float(sums[1]) and out["mpjpe_ra/r"] == float(sums[2]) / float(sums[3])
