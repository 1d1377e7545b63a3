"""fp64 reference of the Procrustes point metrics (TEST INFRASTRUCTURE ONLY, never imported by `hands_b200/`).

The HMR / ARCTIC `compute_similarity_transform` as the reference's eval uses it for PA-MPJPE
(src/utils/eval_modules.py:136-219, a numpy SVD per sample).  That file is not in this checkout, so parity with its text
is unpinned (DESIGN.md §4): this module restates the contract of `hb_procrustes_metrics` (include/hands_b200.h)
literally, and tests/test_metrics_oracle.py checks it by known answers."""
import numpy as np


def procrustes_errors(pred, gt, root_pred=None, root_gt=None):
    """Per hand, in float64:
        mu_p, mu_q = means;  X_i = p_i - mu_p;  Y_i = q_i - mu_q;  var = sum |X_i|^2;  C = sum X_i Y_i^T
        U, S, V^T = svd(C);  Z = diag(1, 1, sign(det(U V^T)));  R = V Z U^T;  s = trace(R C) / var;  t = mu_q - s R mu_p
        PA = mean_i |s R p_i + t - q_i|        RA = mean_i |(p_i - r_p) - (q_i - r_q)|
    pred, gt (B,N,3); root_pred, root_gt (B,3) or None (= point 0).  Returns numpy (PA (B,), RA (B,), aligned (B,N,3));
    PA and aligned are NaN where var == 0 (degenerate)."""
    p = np.asarray(pred, dtype=np.float64)
    q = np.asarray(gt, dtype=np.float64)
    rp = p[:, 0] if root_pred is None else np.asarray(root_pred, dtype=np.float64)
    rq = q[:, 0] if root_gt is None else np.asarray(root_gt, dtype=np.float64)
    B, N = p.shape[:2]
    pa = np.full(B, np.nan)
    aligned = np.full((B, N, 3), np.nan)
    for b in range(B):
        mu_p = p[b, 0] + (p[b] - p[b, 0]).mean(axis=0)   # = the mean; exact when all points are equal
        mu_q = q[b, 0] + (q[b] - q[b, 0]).mean(axis=0)
        X, Y = p[b] - mu_p, q[b] - mu_q
        var = float((X * X).sum())
        if var == 0.0:
            continue
        C = X.T @ Y
        U, _, Vt = np.linalg.svd(C)
        V = Vt.T
        Z = np.eye(3)
        Z[2, 2] = np.sign(np.linalg.det(U @ V.T))
        R = V @ Z @ U.T
        s = np.trace(R @ C) / var
        t = mu_q - s * R @ mu_p
        aligned[b] = s * p[b] @ R.T + t
        pa[b] = np.linalg.norm(aligned[b] - q[b], axis=1).mean()
    ra = np.linalg.norm((p - rp[:, None]) - (q - rq[:, None]), axis=2).mean(axis=1)
    return pa, ra, aligned
