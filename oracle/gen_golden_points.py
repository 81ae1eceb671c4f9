"""Generates tests/golden/dp_losses.npz by running the REFERENCE'S OWN code (imported with the shims in
oracle/ref_import.py) under torch autograd.  Run in this container only:

    python -m oracle.gen_golden_points

- IUV_Estimator.dp_uvia_losses (models/danet/iuv_estimator.py:343-419) behind the has_dp selection of
  iuv_estimator.py:106-121, for torch's grid_sample with align_corners=False and =True (the torch 1.1 behaviour);
- loss_roi: softmax_integral_tensor (utils/keypoints.py:334-394) with iuv_estimator.py:137-140,159-171 verbatim.

The reference sizes its maps by cfg.DANET.HEATMAP_SIZE; it is set to 14 while generating (so that the file stays
small) and restored afterwards.  The 196 points per sample are fixed by the reference."""
import functools
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _dp_inputs(torch, g, B, C, CA, S, P):
    """Points at random sub-pixel positions, at exact integers on and beyond the border, several sharing one pixel,
    and padded slots (X = Y = I = 0, weight 0) at the end of every sample."""
    X = torch.rand(B, P, generator=g) * (S + 3) - 1.5
    Y = torch.rand(B, P, generator=g) * (S + 3) - 1.5
    ints = torch.tensor([-1.0, 0.0, 1.0, S / 2.0, S - 1.0, float(S), S + 1.0, 3.0])
    X[:, :40] = ints[torch.randint(0, len(ints), (B, 40), generator=g)]
    Y[:, :40] = ints[torch.randint(0, len(ints), (B, 40), generator=g)]
    X[:, 40:60] = X[:, 60:61] + 0.25                                     # twenty points on one pixel's corners
    Y[:, 40:60] = Y[:, 60:61] - 0.5
    I = torch.randint(0, C, (B, P), generator=g).float()
    W = torch.zeros(B, C, P)
    W.scatter_(1, I.long().unsqueeze(1), 1.0)                            # weight 1 on the point's part channel ...
    W[:, :, 100:110] *= 2.0                                              # ... 2 on a few, so w_in * d leaves the knee
    U = torch.rand(B, C, P, generator=g) * (W > 0)
    V = torch.rand(B, C, P, generator=g) * (W > 0)
    npad = 16
    X[:, -npad:] = 0.0
    Y[:, -npad:] = 0.0
    I[:, -npad:] = 0.0
    W[:, :, -npad:] = 0.0
    U[:, :, -npad:] = 0.0
    V[:, :, -npad:] = 0.0
    Ind = torch.arange(B).float()[:, None].expand(B, P).contiguous()
    lab = torch.randint(0, CA, (B, S * S), generator=g).float()
    return dict(body_uv_X_points=X, body_uv_Y_points=Y, body_uv_I_points=I, body_uv_Ind_points=Ind,
                body_uv_U_points=U.reshape(B, C * P), body_uv_V_points=V.reshape(B, C * P),
                body_uv_point_weights=W.reshape(B, C * P), body_uv_ann_labels=lab, body_uv_ann_weights=torch.ones(B, S * S))


def gen_dp_losses(ns):
    torch = ns.torch
    F = torch.nn.functional
    cfg = ns.cfg
    g = torch.Generator().manual_seed(3141)
    B, C, CA, S, P = 3, 25, 15, 14, 196
    fn = ns.IUV_Estimator.dp_uvia_losses                         # `self` is unused apart from the module-level cfg
    gt = _dp_inputs(torch, g, B, C, CA, S, P)
    u, v, i = (torch.randn(B, C, S, S, generator=g).mul_(1.5).requires_grad_() for _ in range(3))
    a = torch.randn(B, CA, S, S, generator=g).mul_(2.0).requires_grad_()
    wts = torch.tensor([1.0, 2.0, 3.0, 4.0])
    out = {}
    saved_size, saved_gs = cfg.DANET.HEATMAP_SIZE, F.grid_sample
    cfg.DANET.HEATMAP_SIZE = S
    try:
        for ac in (0, 1):
            F.grid_sample = functools.partial(saved_gs, align_corners=bool(ac))
            for tag, has in (("all", torch.ones(B, dtype=torch.bool)), ("some", torch.tensor([True, False, True]))):
                for t in (u, v, i, a):
                    t.grad = None
                dp_on = (has == 1)                                       # iuv_estimator.py:106-109
                gt_ = {k: x[dp_on] if isinstance(x, torch.Tensor) else x for k, x in gt.items()}
                L = fn(None, u[dp_on], v[dp_on], i[dp_on], a[dp_on], **gt_)
                sum(w * l for w, l in zip(wts, L)).backward()
                out["L_%s_ac%d" % (tag, ac)] = torch.stack([l.detach().reshape(()) for l in L]).numpy()
                for k, t in (("u", u), ("v", v), ("i", i), ("a", a)):   # gradient of sum_k (k+1) loss_k
                    out["g%s_%s_ac%d" % (k, tag, ac)] = t.grad.numpy().copy()
    finally:
        F.grid_sample = saved_gs
        cfg.DANET.HEATMAP_SIZE = saved_size
    out.update(u=u.detach().numpy(), v=v.detach().numpy(), i=i.detach().numpy(), a=a.detach().numpy(),
               has_some=np.array([1, 0, 1], np.uint8), grad_weights=wts.numpy(),
               **{k: x.numpy() for k, x in gt.items()})
    out.update(gen_stn_kps(ns, g))
    np.savez_compressed(os.path.join(GOLD, "dp_losses.npz"), **out)
    print("dp_losses.npz written")


def gen_stn_kps(ns, g):
    """loss_roi through the soft-argmax: iuv_estimator.py:137-140 and 159-171 verbatim (STN_KPS_WEIGHTS = 1.0)."""
    torch = ns.torch
    F = torch.nn.functional
    from utils.keypoints import softmax_integral_tensor
    B, J, S = 3, 24, 14
    skps_hm_pred = (torch.randn(B, J, S, S, generator=g) * 0.3).requires_grad_()
    smpl_kps_gt = torch.cat([torch.rand(B, J, 2, generator=g) * 2.4 - 1.2,
                             torch.tensor([0.0, 0.5, 1.0, 2.0])[torch.randint(0, 4, (B, J, 1), generator=g)]], dim=2)
    smpl_kps_hm_size = skps_hm_pred.size(-1)
    stn_centers = softmax_integral_tensor(10 * skps_hm_pred, skps_hm_pred.size(1), skps_hm_pred.size(-2),
                                          skps_hm_pred.size(-1))
    stn_centers /= 0.5 * smpl_kps_hm_size
    stn_centers -= 1
    loss_roi = 0
    for w in torch.unique(smpl_kps_gt[:, :, 2]):
        if w == 0:
            continue
        kps_w_idx = smpl_kps_gt[:, :, 2] == w
        loss_roi += F.smooth_l1_loss(stn_centers[kps_w_idx], smpl_kps_gt[:, :, :2][kps_w_idx], size_average=False) * w
    loss_roi /= smpl_kps_gt.size(0)
    loss_roi *= ns.cfg.DANET.STN_KPS_WEIGHTS
    loss_roi.backward()
    return {"hm": skps_hm_pred.detach().numpy(), "kps": smpl_kps_gt.numpy(), "roi_loss": loss_roi.detach().numpy(),
            "roi_centers": stn_centers.detach().numpy(), "roi_grad": skps_hm_pred.grad.numpy()}


def main():
    sys.path.insert(0, ROOT)
    from oracle import ref_import
    ns = ref_import.load(48)
    os.makedirs(GOLD, exist_ok=True)
    gen_dp_losses(ns)


if __name__ == "__main__":
    main()
