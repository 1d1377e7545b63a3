"""CPU checks of the Procrustes metric's oracle (`tests/procrustes_oracle.py::procrustes_errors`, the similarity fit of the HMR /
ARCTIC `compute_similarity_transform`) and of the argument checks of `hb_procrustes_metrics`, which run without a GPU."""
import numpy as np
import pytest
import torch
from scipy.optimize import minimize
from scipy.spatial.transform import Rotation

from hands_b200 import _lib
from oracle import geometry_oracle as O
from procrustes_oracle import procrustes_errors


def _hands(B, N, seed, noise=0.01):
    rng = np.random.default_rng(seed)
    gt = rng.normal(size=(B, N, 3)) * 0.04 + np.array([0.05, -0.1, 0.8])
    pred = gt + rng.normal(size=(B, N, 3)) * noise
    return pred, gt


def _similarity(rng, x):
    R = Rotation.random(random_state=int(rng.integers(1 << 30))).as_matrix()
    s = rng.uniform(0.5, 2.0)
    t = rng.normal(size=3)
    return s * x @ R.T + t


def _extent(q):
    return np.linalg.norm(q - q.mean(axis=0), axis=1).max()


@pytest.mark.parametrize("N", [3, 21, 778])
def test_exact_similarity_copy_has_zero_pa(N):
    rng = np.random.default_rng(N)
    _, gt = _hands(6, N, N)
    pred = np.stack([_similarity(rng, g) for g in gt])
    pa, _, aligned = procrustes_errors(pred, gt)
    for b in range(6):
        assert pa[b] <= 1e-12 * _extent(gt[b])
        assert np.abs(aligned[b] - gt[b]).max() <= 1e-12 * _extent(gt[b])


def test_closed_form_of_the_squared_objective():
    pred, gt = _hands(8, 21, 1, noise=0.02)
    _, _, aligned = procrustes_errors(pred, gt)
    for b in range(8):
        X, Y = pred[b] - pred[b].mean(0), gt[b] - gt[b].mean(0)
        C = X.T @ Y
        U, S, Vt = np.linalg.svd(C)
        tr = S[0] + S[1] + np.sign(np.linalg.det(U @ Vt)) * S[2]   # trace(R C) at the optimum
        lhs = ((aligned[b] - gt[b]) ** 2).sum()
        rhs = (Y * Y).sum() - tr * tr / (X * X).sum()
        assert abs(lhs - rhs) <= 1e-12 * (Y * Y).sum()


def test_pa_is_invariant_under_similarity_of_pred():
    rng = np.random.default_rng(2)
    pred, gt = _hands(8, 21, 2, noise=0.02)
    pa, _, _ = procrustes_errors(pred, gt)
    moved = np.stack([_similarity(rng, p) for p in pred])
    pa2, _, _ = procrustes_errors(moved, gt)
    np.testing.assert_allclose(pa2, pa, rtol=1e-10, atol=0)


def test_mirrored_prediction_gets_a_proper_rotation_and_the_least_squares_minimum():
    pred, gt = _hands(3, 21, 3, noise=0.005)
    pred = pred * np.array([1.0, 1.0, -1.0])            # mirror: det(U V^T) < 0 without the correction
    _, _, aligned = procrustes_errors(pred, gt)
    for b in range(3):
        X = pred[b] - pred[b].mean(0)
        sRt, *_ = np.linalg.lstsq(X, aligned[b] - aligned[b].mean(0), rcond=None)   # aligned_c = X (sR)^T
        assert np.linalg.det(sRt.T) > 0
        U, S, Vt = np.linalg.svd(X.T @ (gt[b] - gt[b].mean(0)))
        assert np.linalg.det(U @ Vt) < 0                  # the case the determinant correction exists for
        obj = ((aligned[b] - gt[b]) ** 2).sum()

        def f(x):
            R = Rotation.from_rotvec(x[:3]).as_matrix()
            return ((np.exp(x[3]) * pred[b] @ R.T + x[4:] - gt[b]) ** 2).sum()   # s = exp(x3) > 0: a similarity, no reflection

        rng = np.random.default_rng(b)
        best = np.inf
        for _ in range(6):
            x0 = np.concatenate([Rotation.random(random_state=int(rng.integers(1 << 30))).as_rotvec(), [0.0], gt[b].mean(0) - pred[b].mean(0)])
            r = minimize(f, x0, method="BFGS", options={"gtol": 1e-14, "maxiter": 10000})
            best = min(best, r.fun)
        assert abs(obj - best) <= 1e-9 and obj <= best + 1e-12


def test_ra_on_joints_equals_the_keypoint_metric_per_hand():
    pred, gt = _hands(5, 21, 4, noise=0.02)
    _, ra, _ = procrustes_errors(pred, gt)
    p, q = torch.from_numpy(pred), torch.from_numpy(gt)
    j2 = torch.zeros(5, 21, 2, dtype=torch.float64)
    for b in range(5):
        hv = torch.zeros(5, dtype=torch.float64)
        hv[b] = 1.0
        s2, n2, _, _ = O.keypoint_metric_sums(p, j2, q, j2, torch.ones(5, 21, dtype=torch.float64), hv, 224.0)
        assert float(n2) == 1.0 and abs(float(s2) - ra[b]) <= 1e-15


def test_given_roots_and_degenerate_hands():
    pred, gt = _hands(3, 21, 5)
    pred[1] = pred[1, 0]                                  # all predicted points equal: var == 0
    rp, rq = pred[:, 3], gt[:, 7]
    pa, ra, aligned = procrustes_errors(pred, gt, rp, rq)
    assert np.isnan(pa[1]) and np.isnan(aligned[1]).all() and np.isfinite(pa[[0, 2]]).all()
    np.testing.assert_allclose(ra, np.linalg.norm((pred - rp[:, None]) - (gt - rq[:, None]), axis=2).mean(1), rtol=1e-15)
    pa1, _, _ = procrustes_errors(pred[:, :1], gt[:, :1])   # one point: always degenerate
    assert np.isnan(pa1).all()


def test_abi_argument_errors():
    lib = _lib.load()
    rc = lib.hb_procrustes_metrics(None, None, 3, 21, None, None, None, None, None, None, None, None)
    assert rc == -1 and b"hb_procrustes_metrics" in lib.hb_last_error_string()
    dummy = ctypes_ptr()
    rc = lib.hb_procrustes_metrics(dummy, dummy, 2, 0, None, None, None, None, None, dummy, dummy, None)
    assert rc == -1 and b"bad argument" in lib.hb_last_error_string()
    rc = lib.hb_procrustes_metrics(dummy, dummy, 2, 21, None, None, None, None, None, dummy, None, None)
    assert rc == -1 and b"bad argument" in lib.hb_last_error_string()
    assert lib.hb_procrustes_metrics(None, None, -1, 21, None, None, None, None, None, None, dummy, None) == -1


def ctypes_ptr():
    """A non-NULL pointer that the argument checks never dereference (they run before any CUDA call)."""
    import ctypes

    return ctypes.c_void_p(16)


def test_wrapper_rejects_cpu_tensors():
    from hands_b200.losses import procrustes_metrics

    with pytest.raises(RuntimeError, match="no CPU path"):
        procrustes_metrics(torch.zeros(2, 21, 3), torch.zeros(2, 21, 3))
