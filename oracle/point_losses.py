"""CPU restatement (numpy, fp64) of the reference's DensePose-point losses and the STN key-point loss with their
gradients -- TEST INFRASTRUCTURE ONLY (imported by tests/ alone; the product path never touches it).

dp_uvia_losses follows models/danet/iuv_estimator.py:343-419 (IUV_Estimator.dp_uvia_losses) with the caller-side
has_dp selection of iuv_estimator.py:106-121; stn_kps_losses follows iuv_estimator.py:137-140,159-171 and
utils/keypoints.py:334-394 (softmax_integral_tensor).  Pinned by tests/golden/dp_losses.npz, which
oracle/gen_golden_points.py produces by calling the reference's own code under torch autograd."""
import numpy as np


def _sl1(d):
    a = np.abs(d)
    return np.where(a < 1.0, 0.5 * d * d, a - 0.5)


def grid_corners(X, Y, S, align_corners=False):
    """Bilinear corners of grid_sample (zero padding) at the DensePose points: grid = (X - S/2) * (2/S) in fp32, the
    un-normalisation in fp32 as torch's CPU kernel evaluates it (one fused multiply-add when align_corners=False), so
    that the corner pixels are the ones the reference picks.  Returns [(row, col, weight, inside)] in the order
    nw, ne, sw, se; each array is [B,P], weights in fp64."""
    f = np.float32
    g = [(np.asarray(Z, f) - f(S / 2.0)) * f(2.0 / S) for Z in (X, Y)]
    if align_corners:
        ix, iy = ((c + f(1)) * f((S - 1) / 2.0) for c in g)
    else:
        ix, iy = ((((c + f(1)).astype(np.float64) * (S / 2.0)) - 0.5).astype(f) for c in g)
    x0, y0 = np.floor(ix), np.floor(iy)
    w, n = ix.astype(np.float64) - x0, iy.astype(np.float64) - y0
    e, s = 1.0 - w, 1.0 - n
    out = []
    for dy, dx, wt in ((0, 0, s * e), (0, 1, s * w), (1, 0, n * e), (1, 1, n * w)):
        r, c = y0 + dy, x0 + dx
        inside = (r >= 0) & (r < S) & (c >= 0) & (c < S)
        out.append((np.where(inside, r, 0).astype(np.int64), np.where(inside, c, 0).astype(np.int64), wt, inside))
    return out


def _sample(m, corners):
    """m [B,C,S,S] -> [B,C,P] (fp64)."""
    b = np.arange(m.shape[0])[:, None]
    out = 0.0
    for r, c, w, inside in corners:
        out = out + np.where(inside, w, 0.0)[:, None, :] * m[b, :, r, c].transpose(0, 2, 1).astype(np.float64)
    return out


def _scatter(g, corners, shape):
    """Adjoint of _sample: g [B,C,P] -> [B,C,S,S]."""
    out = np.zeros(shape)
    B, C, P = g.shape
    bi = np.broadcast_to(np.arange(B)[:, None, None], (B, C, P))
    ci = np.broadcast_to(np.arange(C)[None, :, None], (B, C, P))
    for r, c, w, inside in corners:
        np.add.at(out, (bi, ci, np.broadcast_to(r[:, None, :], (B, C, P)), np.broadcast_to(c[:, None, :], (B, C, P))),
                  g * np.where(inside, w, 0.0)[:, None, :])
    return out


def _ce(logits, labels, sel):
    """Mean cross-entropy over the rows of the selected samples.  logits [B,K,M], labels [B,M] (truncated to integers
    like .to(torch.int64)); an out-of-range label makes the loss and its sample's gradient NaN.  Returns (loss,
    d loss / d logits [B,K,M])."""
    x = logits.astype(np.float64)
    K = x.shape[1]
    lab = np.trunc(np.asarray(labels, np.float64))
    ok = (lab >= 0) & (lab < K)
    t = np.where(ok, lab, 0).astype(np.int64)
    m = x.max(axis=1, keepdims=True)
    e = np.exp(x - m)
    s = e.sum(axis=1, keepdims=True)
    lse = (m + np.log(s))[:, 0]
    xt = np.take_along_axis(x, t[:, None], axis=1)[:, 0]
    per = np.where(ok, lse - xt, np.nan)
    cnt = sel.sum() * x.shape[2]
    g = e / s
    np.put_along_axis(g, t[:, None], np.take_along_axis(g, t[:, None], axis=1) - 1.0, axis=1)
    g = np.where(ok[:, None, :], g, np.nan) / cnt
    g[~sel] = 0.0
    return per[sel].sum() / cnt, g


def dp_uvia_losses(U_estimated, V_estimated, Index_UV, Ann_Index, body_uv_X_points, body_uv_Y_points, body_uv_I_points,
                   body_uv_Ind_points, body_uv_U_points, body_uv_V_points, body_uv_point_weights, body_uv_ann_labels,
                   body_uv_ann_weights=None, has_dp=None, align_corners=False, index_weight=2.0, part_weight=0.3,
                   point_weight=0.5):
    """Returns (losses [4] = (loss_Udp, loss_Vdp, loss_IndexUVdp, loss_segAnndp), grads dict of d loss_k / d input
    for u, v, index, ann)."""
    B, C, S = U_estimated.shape[0], U_estimated.shape[1], U_estimated.shape[2]
    P = body_uv_X_points.shape[1]
    Ca = Ann_Index.shape[1]
    sel = np.ones(B, bool) if has_dp is None else np.asarray(has_dp).astype(bool)
    z = {"u": np.zeros(U_estimated.shape), "v": np.zeros(V_estimated.shape), "index": np.zeros(Index_UV.shape),
         "ann": np.zeros(Ann_Index.shape)}
    if not sel.any():                                                     # iuv_estimator.py:116-121
        return np.zeros(4), z
    corners = grid_corners(body_uv_X_points, body_uv_Y_points, S, align_corners)
    on = sel[:, None, None]
    w = np.asarray(body_uv_point_weights, np.float64).reshape(B, C, P)     # view(-1,25,196): channel-major per sample
    L, grads = np.zeros(4), {}
    for k, (pred, tgt) in enumerate(((U_estimated, body_uv_U_points), (V_estimated, body_uv_V_points))):
        d = w * (_sample(pred, corners) - np.asarray(tgt, np.float64).reshape(B, C, P))       # utils/net.py:18-35
        L[k] = point_weight * (w * _sl1(d) * on).sum()
        grads["uv"[k]] = _scatter(point_weight * w * w * np.clip(d, -1.0, 1.0) * on, corners, pred.shape)
    li, gi = _ce(_sample(Index_UV, corners), np.asarray(body_uv_I_points).reshape(B, P), sel)
    L[2] = part_weight * li
    grads["index"] = _scatter(part_weight * gi, corners, Index_UV.shape)
    la, ga = _ce(Ann_Index.reshape(B, Ca, S * S), np.asarray(body_uv_ann_labels).reshape(B, S * S), sel)
    L[3] = index_weight * la
    grads["ann"] = (index_weight * ga).reshape(Ann_Index.shape)
    return L, grads


def stn_kps_losses(skps_hm_pred, smpl_kps_gt, weight=1.0):
    """Returns (loss_roi, stn_centers [B,J,2], d loss_roi / d skps_hm_pred)."""
    B, J, H, W = skps_hm_pred.shape
    x = 10.0 * skps_hm_pred.astype(np.float64).reshape(B, J, H * W)
    e = np.exp(x - x.max(axis=2, keepdims=True))
    sm = e / e.sum(axis=2, keepdims=True)
    col = np.tile(np.arange(W, dtype=np.float64), H)
    row = np.repeat(np.arange(H, dtype=np.float64), W)
    xh, yh = (sm * col).sum(axis=2), (sm * row).sum(axis=2)
    half = 0.5 * W
    c = np.stack([xh / half - 1.0, yh / half - 1.0], axis=2)
    gt = smpl_kps_gt.astype(np.float64)
    wk = gt[:, :, 2]
    d = c - gt[:, :, :2]
    loss = weight * (wk[:, :, None] * _sl1(d)).sum() / B
    gc = weight * wk[:, :, None] * np.clip(d, -1.0, 1.0) / B
    g = (10.0 / half) * sm * (gc[:, :, 0:1] * (col - xh[:, :, None]) + gc[:, :, 1:2] * (row - yh[:, :, None]))
    return loss, c, g.reshape(B, J, H, W)
