"""IUV-branch losses of the training step (SURVEY section 8f-2) with the reference's call surface:

    loss_U, loss_V, loss_IndexUV, loss_segAnn = body_uv_losses(u_pred, v_pred, index_pred, ann_pred, uvia_list, has_iuv)
    loss_pU, loss_pV, loss_pIndexUV           = part_iuv_losses(part_iuv_pred, part_iuv_gt, has_iuv)
    loss_Udp, loss_Vdp, loss_IndexUVdp, loss_segAnndp = dp_uvia_losses(u_pred, v_pred, index_pred, ann_pred,
                                                                       **uvia_dp_gt, has_dp=has_dp)
    loss_roi, stn_centers                     = stn_kps_losses(skps_hm_pred, smpl_kps_gt)

`body_uv_losses` is models/danet/iuv_estimator.py:304-341; `part_iuv_losses` is the loop over the 24 part crops of
iuv_estimator.py:232-255 as one launch.  Forward and backward are ONE fused CUDA pass (csrc/losses.cu,
danet_body_uv_losses): the gradients w.r.t. the predictions are produced with the losses and handed to autograd by a
torch.autograd.Function.  No CPU path.

`dp_uvia_losses` is iuv_estimator.py:343-419 with the has_dp selection of :106-121 (csrc/point_losses.cu,
danet_dp_uvia_losses); `stn_kps_losses` is the soft-argmax of :137-140 with loss_roi of :159-171 (danet_stn_kps_losses).

Deviations from the reference, stated:
- when no image has IUV / DensePose ground truth the reference returns `torch.zeros(1)` per loss after a host
  synchronisation (`torch.sum(has_iuv) > 0`); here the losses are 0-dim zeros and nothing synchronises (the count stays
  on the device);
- a DensePose part or annotation label outside its class range makes the reference raise (inside cross_entropy); here
  the affected loss is NaN, because raising would need a host synchronisation."""
import torch
from torch.autograd.function import once_differentiable

from . import _lib

POINT_REGRESSION_WEIGHTS = 0.5                  # configs/danet_default.yaml:23 (cfg.DANET.POINT_REGRESSION_WEIGHTS)
INDEX_WEIGHTS = 2.0                             # configs/danet_default.yaml:19 (cfg.DANET.INDEX_WEIGHTS)
PART_WEIGHTS = 0.3                              # configs/danet_default.yaml:21 (cfg.DANET.PART_WEIGHTS)
STN_KPS_WEIGHTS = 1.0                           # configs/danet_default.yaml:35 (cfg.DANET.STN_KPS_WEIGHTS)


def _launch(N, C, Cann, HW, pred_stride, map_stride, u, v, idx, ann, U, V, I, A, has, batch_size, point_weight, dev,
            gu, gv, gi, ga):
    """Pointers are integer device addresses (or None); returns losses [4] on `dev`."""
    lib = _lib.load()
    p = lambda x: _lib.c_p(x if x else 0)
    with torch.cuda.device(dev):
        ws = torch.empty(int(lib.danet_body_uv_losses_workspace_bytes(N, HW)), dtype=torch.uint8, device=dev)
        losses = torch.empty(4, device=dev)
        _lib.check(lib.danet_body_uv_losses(N, C, Cann, HW, pred_stride, map_stride, p(u), p(v), p(idx), p(ann), p(U), p(V),
                                            p(I), p(A), p(has), float(batch_size), float(point_weight), _lib.ptr(losses),
                                            p(gu), p(gv), p(gi), p(ga), _lib.ptr(ws), _lib.stream_ptr(dev)),
                   "body_uv_losses")
    return losses


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _has_u8(has_iuv, dev, repeat=1):
    if has_iuv is None:
        return None
    h = (has_iuv.to(dev) != 0).to(torch.uint8)
    if repeat > 1:
        h = h.repeat_interleave(repeat)
    return h.contiguous()


class _BodyUvLosses(torch.autograd.Function):
    """losses [4] = (loss_U, loss_V, loss_IndexUV, loss_segAnn); the backward multiplies the gradients the fused pass
    already wrote by the incoming d/d losses[k]."""

    @staticmethod
    def forward(ctx, u, v, idx, ann, U, V, I, A, has, point_weight):
        dev = u.device
        B, C = u.shape[0], u.shape[1]
        HW = u.shape[2] * u.shape[3]
        u_, v_, i_ = _f32(u, dev), _f32(v, dev), _f32(idx, dev)
        U_, V_, I_ = _f32(U, dev), _f32(V, dev), _f32(I, dev)
        a_ = _f32(ann, dev) if ann is not None else None
        A_ = _f32(A, dev) if ann is not None else None
        need = [ctx.needs_input_grad[k] for k in range(4)]
        gu = torch.empty_like(u_) if need[0] else None
        gv = torch.empty_like(v_) if need[1] else None
        gi = torch.empty_like(i_) if need[2] else None
        ga = torch.empty_like(a_) if (ann is not None and need[3]) else None
        d = lambda t: t.data_ptr() if t is not None else 0
        losses = _launch(B, C, a_.shape[1] if a_ is not None else 0, HW, 0, 0, d(u_), d(v_), d(i_), d(a_), d(U_), d(V_),
                         d(I_), d(A_), d(has), float(B), point_weight, dev, d(gu), d(gv), d(gi), d(ga))
        ctx.grads = (gu, gv, gi, ga)
        ctx.dtypes = (u.dtype, v.dtype, idx.dtype, ann.dtype if ann is not None else None)
        return losses

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        out = []
        for k, t in enumerate(ctx.grads):
            out.append(None if t is None else (t * g[k]).to(ctx.dtypes[k]))
        return (*out, None, None, None, None, None, None)


def body_uv_losses(u_pred, v_pred, index_pred, ann_pred, uvia_list, has_iuv=None,
                   point_weight=POINT_REGRESSION_WEIGHTS):
    """models/danet/iuv_estimator.py:304-341.  u/v/index_pred [B,C,S,S]; ann_pred [B,Cann,S,S] or None;
    uvia_list = (Umap, Vmap, Imap, Annmap) as utils/iuvmap.py iuv_img2map returns them; has_iuv [B] or None.
    Returns (loss_U, loss_V, loss_IndexUV, loss_segAnn | None), differentiable w.r.t. the predictions."""
    _lib.require_cuda(u_pred, "u_pred")
    Umap, Vmap, Imap, Annmap = uvia_list
    if u_pred.dim() != 4 or u_pred.shape != v_pred.shape or u_pred.shape != index_pred.shape or u_pred.shape != Imap.shape:
        raise ValueError("body_uv_losses: u/v/index predictions and the target maps must share one [B,C,S,S] shape")
    if ann_pred is not None and (Annmap is None or ann_pred.shape != Annmap.shape):
        raise ValueError("body_uv_losses: ann_pred needs an Annmap of the same shape")
    if has_iuv is not None and has_iuv.shape[0] != u_pred.shape[0]:
        raise ValueError("body_uv_losses: has_iuv must have one entry per image")
    if u_pred.shape[0] == 0 or u_pred.shape[2] * u_pred.shape[3] == 0:      # nothing to sum: zeros that still carry a graph
        z = u_pred.sum() * 0 + v_pred.sum() * 0 + index_pred.sum() * 0
        return z, z, z, (ann_pred.sum() * 0 if ann_pred is not None else None)
    has = _has_u8(has_iuv, u_pred.device)
    L = _BodyUvLosses.apply(u_pred, v_pred, index_pred, ann_pred, Umap, Vmap, Imap, Annmap if ann_pred is not None else None,
                            has, point_weight)
    return L[0], L[1], L[2], (L[3] if ann_pred is not None else None)


class _PartIuvLosses(torch.autograd.Function):
    """The 24 body_uv_losses calls of iuv_estimator.py:232-255 (+ the /24 means) over part_iuv_pred [B,24,3,7,S,S]
    in place: image = (batch, part) row, u / v / index = the three 7-channel groups of a row."""

    @staticmethod
    def forward(ctx, pred, gt, has, point_weight):
        dev = pred.device
        B, P, three, C = pred.shape[:4]
        HW = pred.shape[4] * pred.shape[5]
        p_, g_ = _f32(pred, dev), _f32(gt, dev)
        grad = torch.empty_like(p_) if ctx.needs_input_grad[0] else None
        step = C * HW * 4                                         # bytes between the u, v and index groups of a row
        pb, gb, qb = p_.data_ptr(), g_.data_ptr(), (grad.data_ptr() if grad is not None else 0)
        q = lambda k: qb + k * step if qb else 0
        losses = _launch(B * P, C, 0, HW, three * C * HW, three * C * HW, pb, pb + step, pb + 2 * step, 0,
                         gb, gb + step, gb + 2 * step, 0, has.data_ptr() if has is not None else 0, float(B * P),
                         point_weight, dev, q(0), q(1), q(2), 0)
        ctx.grad = grad
        ctx.dtype = pred.dtype
        return losses[:3]

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        if ctx.grad is None:
            return None, None, None, None
        return (ctx.grad * g.reshape(1, 1, 3, 1, 1, 1)).to(ctx.dtype), None, None, None


def part_iuv_losses(part_iuv_pred, part_iuv_gt, has_iuv=None, point_weight=POINT_REGRESSION_WEIGHTS):
    """iuv_estimator.py:232-255: part_iuv_pred / part_iuv_gt [B,24,3,7,S,S] (u, v, index groups of the part crops).
    Returns (loss_pU, loss_pV, loss_pIndexUV) = the means over the 24 parts of body_uv_losses per part."""
    _lib.require_cuda(part_iuv_pred, "part_iuv_pred")
    if part_iuv_pred.dim() != 6 or part_iuv_pred.shape[2] != 3 or part_iuv_pred.shape != part_iuv_gt.shape:
        raise ValueError("part_iuv_losses: expected part_iuv_pred and part_iuv_gt of one shape [B,P,3,C,S,S]")
    if has_iuv is not None and has_iuv.shape[0] != part_iuv_pred.shape[0]:
        raise ValueError("part_iuv_losses: has_iuv must have one entry per image")
    if part_iuv_pred.numel() == 0:
        z = part_iuv_pred.sum() * 0
        return z, z, z
    has = _has_u8(has_iuv, part_iuv_pred.device, repeat=part_iuv_pred.shape[1])
    L = _PartIuvLosses.apply(part_iuv_pred, part_iuv_gt, has, point_weight)
    return L[0], L[1], L[2]


class _DpUviaLosses(torch.autograd.Function):
    """losses [4] = (loss_Udp, loss_Vdp, loss_IndexUVdp, loss_segAnndp) of the DensePose points; the backward multiplies
    the gradients the fused pass already wrote by the incoming d/d losses[k]."""

    @staticmethod
    def forward(ctx, u, v, idx, ann, X, Y, I, Up, Vp, Wp, alab, has, align, weights):
        dev = u.device
        B, C, S = u.shape[0], u.shape[1], u.shape[2]
        P = X.shape[1]
        preds = [_f32(t, dev) for t in (u, v, idx, ann)]
        pts = [_f32(t, dev) for t in (X, Y, I, Up, Vp, Wp, alab)]
        grads = [torch.empty_like(t) if ctx.needs_input_grad[k] else None for k, t in enumerate(preds)]
        lib = _lib.load()
        with torch.cuda.device(dev):
            ws = torch.empty(int(lib.danet_dp_uvia_losses_workspace_bytes(B, C, S, P)), dtype=torch.uint8, device=dev)
            losses = torch.empty(4, device=dev)
            _lib.check(lib.danet_dp_uvia_losses(B, C, ann.shape[1], S, P, *[_lib.ptr(t) for t in preds + pts], _lib.ptr(has),
                                                int(align), *[float(w) for w in weights], _lib.ptr(losses),
                                                *[_lib.ptr(g) for g in grads], _lib.ptr(ws), _lib.stream_ptr(dev)),
                       "dp_uvia_losses")
        ctx.grads = grads
        ctx.dtypes = [t.dtype for t in (u, v, idx, ann)]
        return losses

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        out = [None if t is None else (t * g[k]).to(ctx.dtypes[k]) for k, t in enumerate(ctx.grads)]
        return (*out,) + (None,) * 10


def dp_uvia_losses(U_estimated, V_estimated, Index_UV, Ann_Index, body_uv_X_points, body_uv_Y_points, body_uv_I_points,
                   body_uv_Ind_points, body_uv_U_points, body_uv_V_points, body_uv_point_weights, body_uv_ann_labels,
                   body_uv_ann_weights=None, has_dp=None, align_corners=False, index_weight=INDEX_WEIGHTS,
                   part_weight=PART_WEIGHTS, point_weight=POINT_REGRESSION_WEIGHTS):
    """models/danet/iuv_estimator.py:343-419 with the has_dp selection of :106-121 done on the device.
    U_estimated / V_estimated / Index_UV [B,C,S,S], Ann_Index [B,Cann,S,S]; the DensePose targets with the reference's
    keyword names: X / Y / I / Ind points [B,P], U / V points and point weights [B,C*P], ann labels [B,S*S];
    has_dp [B] or None (every sample).  body_uv_Ind_points and body_uv_ann_weights are accepted and not used, as in the
    reference.  align_corners=True samples like torch 1.1's grid_sample.  Returns (loss_Udp, loss_Vdp, loss_IndexUVdp,
    loss_segAnndp), 0-dim, differentiable w.r.t. the four predictions."""
    _lib.require_cuda(U_estimated, "U_estimated")
    u = U_estimated
    if u.dim() != 4 or u.shape[2] != u.shape[3] or V_estimated.shape != u.shape or Index_UV.shape != u.shape:
        raise ValueError("dp_uvia_losses: U/V/Index predictions must share one [B,C,S,S] shape")
    B, C, S = u.shape[0], u.shape[1], u.shape[2]
    if Ann_Index.dim() != 4 or Ann_Index.shape[0] != B or Ann_Index.shape[2:] != u.shape[2:] or Ann_Index.shape[1] < 1:
        raise ValueError("dp_uvia_losses: Ann_Index must be [B,Cann,S,S] like the predictions")
    if body_uv_X_points.dim() != 2 or body_uv_X_points.shape[0] != B or body_uv_X_points.shape[1] < 1:
        raise ValueError("dp_uvia_losses: body_uv_X_points must be [B,P] with P >= 1")
    P = body_uv_X_points.shape[1]
    for name, t in (("body_uv_Y_points", body_uv_Y_points), ("body_uv_I_points", body_uv_I_points),
                    ("body_uv_Ind_points", body_uv_Ind_points)):
        if tuple(t.shape) != (B, P):
            raise ValueError("dp_uvia_losses: %s must be [B,P] = [%d,%d]" % (name, B, P))
    for name, t in (("body_uv_U_points", body_uv_U_points), ("body_uv_V_points", body_uv_V_points),
                    ("body_uv_point_weights", body_uv_point_weights)):
        if t.shape[0] != B or t.numel() != B * C * P:
            raise ValueError("dp_uvia_losses: %s must be [B,C*P] = [%d,%d]" % (name, B, C * P))
    if body_uv_ann_labels.shape[0] != B or body_uv_ann_labels.numel() != B * S * S:
        raise ValueError("dp_uvia_losses: body_uv_ann_labels must be [B,S*S] = [%d,%d]" % (B, S * S))
    if has_dp is not None and tuple(has_dp.shape) != (B,):
        raise ValueError("dp_uvia_losses: has_dp must have one entry per sample")
    if B == 0 or C == 0 or S == 0:                                 # nothing to sum: zeros that still carry a graph
        z = U_estimated.sum() * 0 + V_estimated.sum() * 0 + Index_UV.sum() * 0 + Ann_Index.sum() * 0
        return z, z, z, z
    flat = lambda t, n: t.reshape(B, n)
    L = _DpUviaLosses.apply(U_estimated, V_estimated, Index_UV, Ann_Index, body_uv_X_points, body_uv_Y_points,
                            body_uv_I_points, flat(body_uv_U_points, C * P), flat(body_uv_V_points, C * P),
                            flat(body_uv_point_weights, C * P), flat(body_uv_ann_labels, S * S),
                            _has_u8(has_dp, u.device), bool(align_corners), (index_weight, part_weight, point_weight))
    return L[0], L[1], L[2], L[3]


class _StnKpsLosses(torch.autograd.Function):
    """(loss_roi [1], stn_centers [B,J,2]); the centres are not differentiable (every later use of them in the reference
    is detached or thresholded)."""

    @staticmethod
    def forward(ctx, hm, kps, weight):
        dev = hm.device
        B, J, S = hm.shape[0], hm.shape[1], hm.shape[2]
        h_, k_ = _f32(hm, dev), _f32(kps, dev)
        grad = torch.empty_like(h_) if ctx.needs_input_grad[0] else None
        lib = _lib.load()
        with torch.cuda.device(dev):
            ws = torch.empty(int(lib.danet_stn_kps_losses_workspace_bytes(B, J)), dtype=torch.uint8, device=dev)
            loss = torch.empty(1, device=dev)
            centers = torch.empty(B, J, 2, device=dev)
            _lib.check(lib.danet_stn_kps_losses(B, J, S, _lib.ptr(h_), _lib.ptr(k_), float(weight), _lib.ptr(loss),
                                                _lib.ptr(centers), _lib.ptr(grad), _lib.ptr(ws), _lib.stream_ptr(dev)),
                       "stn_kps_losses")
        ctx.grad = grad
        ctx.dtype = hm.dtype
        ctx.mark_non_differentiable(centers)
        return loss, centers

    @staticmethod
    @once_differentiable
    def backward(ctx, g, _g_centers):
        if ctx.grad is None:
            return None, None, None
        return (ctx.grad * g[0]).to(ctx.dtype), None, None


def stn_kps_losses(skps_hm_pred, smpl_kps_gt, weight=STN_KPS_WEIGHTS):
    """iuv_estimator.py:137-140 and 159-171.  skps_hm_pred [B,J,S,S] (the key-point heat maps), smpl_kps_gt [B,J,3]
    (x, y in [-1, 1], weight).  Returns (loss_roi 0-dim, differentiable w.r.t. skps_hm_pred; stn_centers [B,J,2] fp32,
    x from columns and y from rows, not differentiable)."""
    _lib.require_cuda(skps_hm_pred, "skps_hm_pred")
    hm = skps_hm_pred
    if hm.dim() != 4 or hm.shape[2] != hm.shape[3] or hm.shape[1] < 1:
        raise ValueError("stn_kps_losses: skps_hm_pred must be [B,J,S,S]")
    if tuple(smpl_kps_gt.shape) != (hm.shape[0], hm.shape[1], 3):
        raise ValueError("stn_kps_losses: smpl_kps_gt must be [B,J,3] = [%d,%d,3]" % (hm.shape[0], hm.shape[1]))
    if hm.shape[0] == 0 or hm.shape[2] == 0:
        return hm.sum() * 0, torch.zeros(hm.shape[0], hm.shape[1], 2, device=hm.device)
    loss, centers = _StnKpsLosses.apply(hm, smpl_kps_gt, weight)
    return loss[0], centers
