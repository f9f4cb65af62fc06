"""ORACLE (test infrastructure) — CPU restatement of the reference's chamfer nearest-neighbour module and of the
points3d energy built on it.  Never imported by the product (humor_b200/): only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline leg may use it.

Follows (paths relative to /root/reference/humor):
  nn_search        utils/chamfer_distance/chamfer_distance.cpp:58-87   (nnsearch, the CPU path of cd.forward)
  chamfer_forward  utils/chamfer_distance/chamfer_distance.cpp:90-111
  chamfer_backward utils/chamfer_distance/chamfer_distance.cpp:114-177
  robust_std / bisquare_robust_weights / apply_robust_weighting   fitting/fitting_utils.py:192-248
  points3d_loss    fitting/fitting_loss.py:378-396

Pinned: bit-exact against what the reference's own C++, compiled from its sources in place (oracle/build_ref.py ->
oracle/_ref/cd_ref.so), wrote: tests/golden/chamfer_*.npz (oracle/make_golden_chamfer.py) and
tests/golden/ref_chamfer_*.npz (oracle/make_golden_ref.py); tests/test_oracle_chamfer.py.  fp32 arithmetic in the reference's order: ((dx*dx)+(dy*dy))+(dz*dz)
with dx = target - query, first strict minimum wins.
"""
import numpy as np


def nn_search(xyz1, xyz2, chunk=256):
    """dist (b,n) fp32, idx (b,n) int32: nearest point of xyz2[i] for every point of xyz1[i]."""
    a = np.ascontiguousarray(xyz1, np.float32)
    b_ = np.ascontiguousarray(xyz2, np.float32)
    b, n, m = a.shape[0], a.shape[1], b_.shape[1]
    dist = np.zeros((b, n), np.float32)
    idx = np.zeros((b, n), np.int32)
    if m == 0:
        return dist, idx                      # best = 0, besti = 0 (chamfer_distance.cpp:69-70)
    for i in range(b):
        for j0 in range(0, n, chunk):
            q = a[i, j0:j0 + chunk]                                   # (c,3)
            d = b_[i][None, :, :] - q[:, None, :]                     # target - query, fp32
            sq = d * d
            dd = (sq[..., 0] + sq[..., 1]) + sq[..., 2]               # separately rounded, reference order
            # `k == 0 || d < best`: first strict minimum; a NaN at k == 0 sticks, later NaNs never win
            first = dd[:, 0]
            nan0 = np.isnan(first)
            safe = np.where(np.isnan(dd), np.float32(np.inf), dd)
            k = np.argmin(safe, axis=1).astype(np.int32)              # argmin returns the first minimum
            best = dd[np.arange(dd.shape[0]), k]
            # all-NaN-or-inf rows: argmin of all-inf is 0, which is what the reference keeps
            k = np.where(nan0, 0, k).astype(np.int32)
            best = np.where(nan0, first, best)
            dist[i, j0:j0 + chunk] = best
            idx[i, j0:j0 + chunk] = k
    return dist, idx


def chamfer_forward(xyz1, xyz2):
    d1, i1 = nn_search(xyz1, xyz2)
    d2, i2 = nn_search(xyz2, xyz1)
    return d1, d2, i1, i2


def chamfer_backward(xyz1, xyz2, graddist1, graddist2, idx1, idx2):
    """Sequential fp32 accumulation in the reference's loop order (the order decides the rounding)."""
    a = np.ascontiguousarray(xyz1, np.float32)
    b_ = np.ascontiguousarray(xyz2, np.float32)
    b, n, m = a.shape[0], a.shape[1], b_.shape[1]
    g1 = np.zeros((b, n, 3), np.float32)
    g2 = np.zeros((b, m, 3), np.float32)
    two = np.float32(2.0)
    for i in range(b):
        if graddist1 is not None and m > 0:
            g = np.asarray(graddist1[i], np.float32) * two
            v = g[:, None] * (a[i] - b_[i][idx1[i]])                  # (n,3), one rounding per op
            g1[i] = g1[i] + v
            for j in range(n):
                g2[i, idx1[i, j]] = g2[i, idx1[i, j]] - v[j]
        if graddist2 is not None and n > 0:
            g = np.asarray(graddist2[i], np.float32) * two
            v = g[:, None] * (b_[i] - a[i][idx2[i]])
            g2[i] = g2[i] + v
            for j in range(m):
                g1[i, idx2[i, j]] = g1[i, idx2[i, j]] - v[j]
    return g1, g2


# ------------------------------------------------------------------------------------------------
# points3d energy (torch, so that autograd supplies the reference gradient)
# ------------------------------------------------------------------------------------------------
def robust_std(res):
    """fitting_utils.py:213-228 — MAD / 0.67449 per row (torch.median = lower median)."""
    import torch
    B = res.size(0)
    med = torch.median(res, dim=-1)[0].reshape((B, 1))
    mad = torch.median(torch.abs(res - med), dim=-1)[0].reshape((B, 1))
    return mad / 0.67449


def bisquare_robust_weights(res, tune_const=4.6851):
    """fitting_utils.py:230-248."""
    norm_res = res / (robust_std(res) * tune_const)
    outlier = norm_res >= 1.0
    w = (1.0 - norm_res ** 2) ** 2
    w[outlier] = 0.0
    return w


def apply_robust_weighting(res, robust_loss_type='bisquare', robust_tuning_const=4.6851):
    """fitting_utils.py:192-211."""
    import torch
    det = res.clone().detach()
    if robust_loss_type == 'none':
        w = torch.ones_like(det)
    elif robust_loss_type == 'bisquare':
        w = bisquare_robust_weights(det, tune_const=robust_tuning_const)
    else:
        raise ValueError(robust_loss_type)
    return w * (res ** 2), w


def points3d_loss(points3d_obs, points3d_pred, robust_loss='bisquare', robust_tuning_const=4.6851):
    """fitting_loss.py:378-396 — one-way chamfer of the observed cloud against the predicted vertices.
    The nearest-neighbour indices come from nn_search; the squared distances are then re-formed in torch from the
    gathered pairs (same fp32 expression) so that autograd yields the reference's gradient
    2*g*(obs - pred[idx]) scattered onto the predicted points (chamfer_distance.cpp:137-156)."""
    import torch
    B, T, N_obs, _ = points3d_obs.shape
    obs = points3d_obs.reshape(B * T, N_obs, 3)
    pred = points3d_pred.reshape(B * T, -1, 3)
    _, idx = nn_search(obs.detach().cpu().numpy(), pred.detach().cpu().numpy())
    idx_t = torch.as_tensor(idx.astype(np.int64), device=pred.device)
    near = torch.gather(pred, 1, idx_t[:, :, None].expand(-1, -1, 3))
    d = near - obs
    sq = d * d
    d1 = (sq[..., 0] + sq[..., 1]) + sq[..., 2]
    d1 = d1.reshape(B, T * N_obs)
    weighted, _ = apply_robust_weighting(d1.sqrt(), robust_loss, robust_tuning_const)
    return 0.5 * torch.sum(weighted)
