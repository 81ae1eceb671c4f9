"""GPU tests of the DensePose-point losses and the STN key-point loss (csrc/point_losses.cu through the C ABI) --
SURVEY section 8f-2.  Oracles: tests/golden/dp_losses.npz (the reference's own dp_uvia_losses and soft-argmax code under
torch autograd, oracle/gen_golden_points.py) and, at the training configuration's sizes, the reference's expressions
restated with torch ops on the device.

Tolerances: golden point losses 5e-6 relative, gradients 5e-7 absolute, as the dense-loss tests.  STN golden: centres
1e-6 and gradients 3e-6 absolute -- the gradient reaches 2.4 there and the golden's own fp32 rounding is 1.1e-6 (the fp64
oracle against it, tests/test_point_losses_cpu.py).  Training size (torch's fp32 sums and atomic scatter on the other
side): losses 2e-5 relative, gradients 2e-4 relative with 1e-6 of the largest gradient as the absolute floor (pixels
where the contributions of several points cancel)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

PTS = ["body_uv_X_points", "body_uv_Y_points", "body_uv_I_points", "body_uv_Ind_points", "body_uv_U_points",
       "body_uv_V_points", "body_uv_point_weights", "body_uv_ann_labels", "body_uv_ann_weights"]


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "dp_losses.npz"))


def _dev(x, grad=False, dev="cuda:0"):
    t = torch.tensor(np.asarray(x), dtype=torch.float32, device=dev)
    return t.requires_grad_() if grad else t


@pytest.mark.parametrize("ac", [0, 1])
def test_dp_uvia_losses_match_reference_golden(gold, ac):
    from danet_b200 import losses
    g = gold
    w = _dev(g["grad_weights"])
    gt = {k: _dev(g[k]) for k in PTS}
    for tag, has in (("all", None), ("some", torch.tensor(g["has_some"]).cuda()), ("none", torch.zeros(3).cuda())):
        preds = [_dev(g[k], True) for k in ("u", "v", "i", "a")]
        L = losses.dp_uvia_losses(*preds, **gt, has_dp=has, align_corners=bool(ac))
        assert all(l.dim() == 0 for l in L)
        ref = g["L_%s_ac%d" % (tag, ac)] if tag != "none" else np.zeros(4)
        np.testing.assert_allclose(torch.stack(L).detach().cpu().numpy(), ref, rtol=5e-6)
        sum(wk * l for wk, l in zip(w, L)).backward()
        for t, n in zip(preds, "uvia"):
            ref = g["g%s_%s_ac%d" % (n, tag, ac)] if tag != "none" else 0.0
            np.testing.assert_allclose(t.grad.cpu().numpy(), ref, atol=5e-7)


def test_stn_kps_losses_match_reference_golden(gold):
    from danet_b200 import losses
    g = gold
    hm = _dev(g["hm"], True)
    loss, centers = losses.stn_kps_losses(hm, _dev(g["kps"]))
    assert loss.dim() == 0 and not centers.requires_grad
    np.testing.assert_allclose(loss.item(), g["roi_loss"], rtol=5e-6)
    np.testing.assert_allclose(centers.cpu().numpy(), g["roi_centers"], atol=1e-6)
    loss.backward()
    np.testing.assert_allclose(hm.grad.cpu().numpy(), g["roi_grad"], atol=3e-6)


def _torch_dp(u, v, idx, ann, X, Y, I, Up, Vp, Wp, lab, has, ac, iw=2.0, pw=0.3, ptw=0.5):
    """iuv_estimator.py:106-121,343-419 restated with current torch spellings."""
    if has is not None:
        u, v, idx, ann, X, Y, I, Up, Vp, Wp, lab = (t[has] for t in (u, v, idx, ann, X, Y, I, Up, Vp, Wp, lab))
    B, C, S = u.shape[0], u.shape[1], u.shape[2]
    P, Ca = X.shape[1], ann.shape[1]
    grid = torch.stack([(X - S / 2.) * (2. / S), (Y - S / 2.) * (2. / S)], dim=2).unsqueeze(1)
    samp = lambda m: F.grid_sample(m, grid, align_corners=ac)[:, :, 0]                        # [B,C,P]
    W = Wp.view(B, C, P)
    out = []
    for m, T in ((u, Up), (v, Vp)):
        d = W * (samp(m) - T.view(B, C, P))
        a = d.abs()
        out.append(ptw * (W * torch.where(a < 1, 0.5 * d * d, a - 0.5)).sum())
    out.append(pw * F.cross_entropy(samp(idx).transpose(1, 2).reshape(-1, C), I.long().view(-1)))
    out.append(iw * F.cross_entropy(ann.reshape(B, Ca, S * S).transpose(1, 2).reshape(-1, Ca), lab.long().view(-1)))
    return out


def _torch_stn(hm, kps, weight=1.0):
    """iuv_estimator.py:137-140,159-171 with utils/keypoints.py:334-394."""
    B, J, S = hm.shape[0], hm.shape[1], hm.shape[2]
    sm = F.softmax((10 * hm).reshape(B, J, -1), 2).reshape(B, J, S, S)
    ar = torch.arange(S, dtype=torch.float32, device=hm.device)
    c = torch.stack([(sm.sum(2) * ar).sum(2), (sm.sum(3) * ar).sum(2)], dim=2) / (0.5 * S) - 1
    loss = 0
    for w in torch.unique(kps[:, :, 2]):
        if w == 0:
            continue
        idx = kps[:, :, 2] == w
        loss = loss + F.smooth_l1_loss(c[idx], kps[:, :, :2][idx], reduction="sum") * w
    return loss / B * weight, c


def _training_batch(gen, B=16, C=25, Ca=15, S=56, P=196, dev="cuda:0"):
    rnd = lambda *s: torch.randn(*s, generator=gen, device=dev)
    X = torch.rand(B, P, generator=gen, device=dev) * (S + 2) - 1
    Y = torch.rand(B, P, generator=gen, device=dev) * (S + 2) - 1
    X[:, :30], Y[:, :30] = X[:, :30].round(), Y[:, :30].round()          # exact integer positions
    X[1], Y[1] = 20.5, 31.25                                             # sample 1: all points on one pixel
    I = torch.randint(0, C, (B, P), generator=gen, device=dev).float()
    W = torch.zeros(B, C, P, device=dev).scatter_(1, I.long().unsqueeze(1), 1.0)
    X[:, -20:], Y[:, -20:], I[:, -20:], W[:, :, -20:] = 0, 0, 0, 0       # padded slots
    U = torch.rand(B, C, P, generator=gen, device=dev) * W
    V = torch.rand(B, C, P, generator=gen, device=dev) * W
    lab = torch.randint(0, Ca, (B, S * S), generator=gen, device=dev).float()
    gt = dict(body_uv_X_points=X, body_uv_Y_points=Y, body_uv_I_points=I, body_uv_Ind_points=torch.zeros(B, P, device=dev),
              body_uv_U_points=U.view(B, -1), body_uv_V_points=V.view(B, -1), body_uv_point_weights=W.view(B, -1),
              body_uv_ann_labels=lab, body_uv_ann_weights=torch.ones(B, S * S, device=dev))
    preds = [rnd(B, C, S, S) * 2, rnd(B, C, S, S) * 2, rnd(B, C, S, S) * 3, rnd(B, Ca, S, S) * 3]
    return preds, gt


def _close(got, ref):
    torch.testing.assert_close(got, ref, rtol=2e-4, atol=1e-6 * ref.abs().max().item())


@pytest.mark.parametrize("ac", [False, True])
def test_losses_at_training_size_match_torch(ac):
    """Per-GPU training batch: 16 samples, 56 x 56 maps, 196 points, 24 joints."""
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(8)
    preds, gt = _training_batch(gen)
    has = torch.rand(16, generator=gen, device="cuda:0") > 0.3
    has[:2] = True
    ours = [p.clone().requires_grad_() for p in preds]
    ref = [p.clone().requires_grad_() for p in preds]
    L = losses.dp_uvia_losses(*ours, **gt, has_dp=has, align_corners=ac)
    R = _torch_dp(*ref, *[gt[k] for k in PTS if k not in ("body_uv_Ind_points", "body_uv_ann_weights")], has, ac)
    for l, r in zip(L, R):
        assert abs(l.item() - r.item()) <= 2e-5 * abs(r.item())
    sum((k + 1.0) * l for k, l in enumerate(L)).backward()
    sum((k + 1.0) * r for k, r in enumerate(R)).backward()
    for o, r in zip(ours, ref):
        assert r.grad.abs().max().item() > 0
        _close(o.grad, r.grad)
    hm = torch.randn(16, 24, 56, 56, generator=gen, device="cuda:0") * 0.2
    kps = torch.cat([torch.rand(16, 24, 2, generator=gen, device="cuda:0") * 2.2 - 1.1,
                     torch.tensor([0.0, 0.5, 1.0, 2.0], device="cuda:0")[torch.randint(0, 4, (16, 24, 1), generator=gen,
                                                                                      device="cuda:0")]], dim=2)
    a, b = hm.clone().requires_grad_(), hm.clone().requires_grad_()
    loss, c = losses.stn_kps_losses(a, kps)
    rl, rc = _torch_stn(b, kps)
    assert abs(loss.item() - rl.item()) <= 2e-5 * abs(rl.item())
    torch.testing.assert_close(c, rc.detach(), rtol=0, atol=2e-6)
    loss.backward()
    rl.backward()
    _close(a.grad, b.grad)


def test_repeatable_bit_for_bit():
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(9)
    preds, gt = _training_batch(gen)
    runs = []
    for _ in range(2):
        p = [x.clone().requires_grad_() for x in preds]
        L = losses.dp_uvia_losses(*p, **gt)
        sum(L).backward()
        runs.append([l.detach() for l in L] + [x.grad for x in p])
    assert all(torch.equal(x, y) for x, y in zip(*runs))
    hm = torch.randn(16, 24, 56, 56, generator=gen, device="cuda:0")
    kps = torch.rand(16, 24, 3, generator=gen, device="cuda:0")
    runs = []
    for _ in range(2):
        h = hm.clone().requires_grad_()
        loss, c = losses.stn_kps_losses(h, kps)
        loss.backward()
        runs.append([loss.detach(), c, h.grad])
    assert all(torch.equal(x, y) for x, y in zip(*runs))


def test_gradients_only_where_requested():
    from danet_b200 import losses, _lib
    gen = torch.Generator(device="cuda:0").manual_seed(10)
    preds, gt = _training_batch(gen, B=3)
    full = [p.clone().requires_grad_() for p in preds]
    L = losses.dp_uvia_losses(*full, **gt)
    sum(L).backward()
    part = [p.clone().requires_grad_(k == 2) for k, p in enumerate(preds)]
    L2 = losses.dp_uvia_losses(*part, **gt)
    assert all(torch.equal(a.detach(), b.detach()) for a, b in zip(L, L2))
    L2[2].backward()
    assert part[0].grad is None and part[1].grad is None and part[3].grad is None
    assert torch.equal(part[2].grad, full[2].grad)
    # at the C ABI: NULL gradient pointers, losses alone
    lib = _lib.load()
    B, C, S, P = 3, 25, 56, 196
    pts = [gt[k].contiguous() for k in PTS if k not in ("body_uv_Ind_points", "body_uv_ann_weights")]
    ws = torch.empty(int(lib.danet_dp_uvia_losses_workspace_bytes(B, C, S, P)), dtype=torch.uint8, device="cuda:0")
    out = torch.empty(4, device="cuda:0")
    _lib.check(lib.danet_dp_uvia_losses(B, C, 15, S, P, *[_lib.ptr(t) for t in preds + pts], None, 0, 2.0, 0.3, 0.5,
                                        _lib.ptr(out), None, None, None, None, _lib.ptr(ws), _lib.stream_ptr()))
    assert torch.equal(out, torch.stack([l.detach() for l in L]))
    hm = torch.randn(2, 24, 8, 8, device="cuda:0")
    loss, c = losses.stn_kps_losses(hm, torch.rand(2, 24, 3, device="cuda:0"))
    assert not loss.requires_grad and c.shape == (2, 24, 2)


def test_non_contiguous_fp16_and_empty_inputs():
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(11)
    preds, gt = _training_batch(gen, B=4, S=20, P=50)
    ref = losses.dp_uvia_losses(*preds, **gt)
    wide = [torch.stack([p, p], dim=2)[:, :, 0] for p in preds]                         # stride 2 in the channel dim
    gtn = {k: torch.stack([t, t], dim=1)[:, 0] if t.dim() == 2 else t for k, t in gt.items()}
    assert not wide[0].is_contiguous() and not gtn["body_uv_X_points"].is_contiguous()
    got = losses.dp_uvia_losses(*wide, **gtn)
    assert all(torch.equal(a, b) for a, b in zip(got, ref))
    half = [p.half().requires_grad_() for p in preds]
    L = losses.dp_uvia_losses(*half, **gt)
    Lf = losses.dp_uvia_losses(*[p.detach().float() for p in half], **gt)
    assert all(torch.equal(a.detach(), b) for a, b in zip(L, Lf))
    sum(L).backward()
    assert all(p.grad.dtype == torch.float16 and torch.isfinite(p.grad).all() for p in half)
    e = [p[:0].clone().requires_grad_() for p in preds]
    L = losses.dp_uvia_losses(*e, **{k: t[:0] for k, t in gt.items()})
    assert [float(l) for l in L] == [0.0] * 4
    sum(L).backward()
    assert all(p.grad is not None and p.grad.numel() == 0 for p in e)
    hm = torch.randn(3, 24, 14, 14, device="cuda:0")
    kps = torch.rand(3, 24, 3, device="cuda:0")
    l0, c0 = losses.stn_kps_losses(hm, kps)
    l1, c1 = losses.stn_kps_losses(hm.transpose(2, 3).contiguous().transpose(2, 3), kps.transpose(0, 1).contiguous().transpose(0, 1))
    assert torch.equal(l0, l1) and torch.equal(c0, c1)
    l2, _ = losses.stn_kps_losses(hm.half(), kps)
    l3, _ = losses.stn_kps_losses(hm.half().float(), kps)
    assert torch.equal(l2, l3)
    le, ce = losses.stn_kps_losses(torch.zeros(0, 24, 14, 14, device="cuda:0", requires_grad=True), torch.zeros(0, 24, 3, device="cuda:0"))
    assert float(le) == 0.0 and ce.shape == (0, 24, 2)


def test_nothing_selected_gives_zeros_that_backpropagate():
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(12)
    preds, gt = _training_batch(gen, B=3, S=14)
    p = [x.clone().requires_grad_() for x in preds]
    L = losses.dp_uvia_losses(*p, **gt, has_dp=torch.zeros(3, dtype=torch.bool, device="cuda:0"))
    assert all(l.dim() == 0 and float(l) == 0.0 and l.requires_grad for l in L)
    sum(L).backward()
    assert all(x.grad is not None and float(x.grad.abs().max()) == 0.0 for x in p)


def test_out_of_range_label_gives_nan():
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(13)
    preds, gt = _training_batch(gen, B=3, S=14)
    bad = dict(gt)
    bad["body_uv_I_points"] = gt["body_uv_I_points"].clone()
    bad["body_uv_I_points"][1, 3] = 25
    L = losses.dp_uvia_losses(*preds, **bad)
    assert torch.isnan(L[2]) and all(torch.isfinite(L[k]) for k in (0, 1, 3))
    bad = dict(gt)
    bad["body_uv_ann_labels"] = gt["body_uv_ann_labels"].clone()
    bad["body_uv_ann_labels"][0, 7] = -1
    L = losses.dp_uvia_losses(*preds, **bad)
    assert torch.isnan(L[3]) and all(torch.isfinite(L[k]) for k in (0, 1, 2))


def test_bad_shapes_raise_value_error():
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(14)
    preds, gt = _training_batch(gen, B=2, S=14, P=10)
    u, v, i, a = preds
    with pytest.raises(ValueError):
        losses.dp_uvia_losses(u, v[:, :24], i, a, **gt)
    with pytest.raises(ValueError):
        losses.dp_uvia_losses(u, v, i, a[:, :, :13], **gt)
    for k, t in (("body_uv_X_points", gt["body_uv_X_points"][:, :9]), ("body_uv_U_points", gt["body_uv_U_points"][:, 1:]),
                 ("body_uv_ann_labels", gt["body_uv_ann_labels"][:, 1:]), ("body_uv_I_points", gt["body_uv_I_points"][:1])):
        with pytest.raises(ValueError):
            losses.dp_uvia_losses(*preds, **dict(gt, **{k: t}))
    with pytest.raises(ValueError):
        losses.dp_uvia_losses(*preds, **gt, has_dp=torch.ones(3, device="cuda:0"))
    with pytest.raises(ValueError):
        losses.stn_kps_losses(torch.zeros(2, 24, 8, 7, device="cuda:0"), torch.zeros(2, 24, 3, device="cuda:0"))
    with pytest.raises(ValueError):
        losses.stn_kps_losses(torch.zeros(2, 24, 8, 8, device="cuda:0"), torch.zeros(2, 24, 2, device="cuda:0"))


def test_second_device_while_current_is_zero():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from danet_b200 import losses
    gen = torch.Generator(device="cuda:0").manual_seed(15)
    preds, gt = _training_batch(gen, B=3, S=14)
    assert torch.cuda.current_device() == 0
    p0 = [x.clone().requires_grad_() for x in preds]
    p1 = [x.to("cuda:1").requires_grad_() for x in preds]
    L0 = losses.dp_uvia_losses(*p0, **gt)
    L1 = losses.dp_uvia_losses(*p1, **{k: t.to("cuda:1") for k, t in gt.items()})
    assert all(l.device == torch.device("cuda:1") for l in L1)
    sum(L0).backward()
    sum(L1).backward()
    assert all(torch.equal(a.detach(), b.detach().cpu().to("cuda:0")) for a, b in zip(L0, L1))
    assert all(torch.equal(a.grad, b.grad.to("cuda:0")) for a, b in zip(p0, p1))
    hm = torch.randn(2, 24, 14, 14, device="cuda:0")
    kps = torch.rand(2, 24, 3, device="cuda:0")
    l0, c0 = losses.stn_kps_losses(hm, kps)
    l1, c1 = losses.stn_kps_losses(hm.to("cuda:1"), kps.to("cuda:1"))
    assert l1.device == torch.device("cuda:1") and torch.equal(l0, l1.to("cuda:0")) and torch.equal(c0, c1.to("cuda:0"))
