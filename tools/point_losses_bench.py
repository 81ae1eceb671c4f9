"""Times the fused DensePose-point loss pass and the STN key-point loss pass (csrc/point_losses.cu), forward + backward,
at the training configuration's per-GPU batch (16 samples, 56 x 56 maps, 196 points, 24 joints) with CUDA events, and
rates them against the HBM roofline: algorithmic bytes = the inputs each pass must read + every gradient written once.
Also times the same losses + backward through torch ops and autograd (the reference's expressions,
iuv_estimator.py:343-419 and :137-140,159-171) on the same device.  Inputs stay L2-resident between iterations (the
working set is ~25 MB): the numbers are the warm-cache steady state of a training step.  Dev tool; prints one JSON
object, `--out FILE` also writes it to FILE."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
from danet_b200 import losses

ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
ap.add_argument("--out", help="also write the JSON result to this file")
args = ap.parse_args()
dev = torch.device("cuda:0")
gen = torch.Generator(device=dev).manual_seed(0)
B, C, CA, S, P, J = 16, 25, 15, 56, 196, 24
HW = S * S
peak = 6581.2                                                    # GB/s, measured HBM copy rate of the B200 (DESIGN §6)


def timed(f, n):
    for _ in range(3):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


X = torch.rand(B, P, generator=gen, device=dev) * S
Y = torch.rand(B, P, generator=gen, device=dev) * S
I = torch.randint(0, C, (B, P), generator=gen, device=dev).float()
W = torch.zeros(B, C, P, device=dev).scatter_(1, I.long().unsqueeze(1), 1.0)
U, V = torch.rand(B, C, P, generator=gen, device=dev) * W, torch.rand(B, C, P, generator=gen, device=dev) * W
lab = torch.randint(0, CA, (B, HW), generator=gen, device=dev).float()
gt = dict(body_uv_X_points=X, body_uv_Y_points=Y, body_uv_I_points=I, body_uv_Ind_points=torch.zeros(B, P, device=dev),
          body_uv_U_points=U.view(B, -1), body_uv_V_points=V.view(B, -1), body_uv_point_weights=W.view(B, -1),
          body_uv_ann_labels=lab, body_uv_ann_weights=torch.ones(B, HW, device=dev))
preds = [torch.randn(B, c, S, S, generator=gen, device=dev).requires_grad_() for c in (C, C, C, CA)]


def fused_dp():
    sum(losses.dp_uvia_losses(*preds, **gt)).backward()


def torch_dp():
    u, v, idx, ann = preds
    grid = torch.stack([(X - S / 2.) * (2. / S), (Y - S / 2.) * (2. / S)], dim=2).unsqueeze(1)
    samp = lambda m: F.grid_sample(m, grid, align_corners=False)[:, :, 0]
    tot = 0
    for m, T in ((u, U), (v, V)):
        d = W * (samp(m) - T)
        a = d.abs()
        tot = tot + 0.5 * (W * torch.where(a < 1, 0.5 * d * d, a - 0.5)).sum()
    tot = tot + 0.3 * F.cross_entropy(samp(idx).transpose(1, 2).reshape(-1, C), I.long().view(-1))
    tot = tot + 2.0 * F.cross_entropy(ann.reshape(B, CA, HW).transpose(1, 2).reshape(-1, CA), lab.long().view(-1))
    tot.backward()


hm = (torch.randn(B, J, S, S, generator=gen, device=dev) * 0.2).requires_grad_()
kps = torch.cat([torch.rand(B, J, 2, generator=gen, device=dev) * 2 - 1, torch.ones(B, J, 1, device=dev)], dim=2)


def fused_stn():
    losses.stn_kps_losses(hm, kps)[0].backward()


def torch_stn():
    sm = F.softmax((10 * hm).reshape(B, J, -1), 2).reshape(B, J, S, S)
    ar = torch.arange(S, dtype=torch.float32, device=dev)
    c = torch.stack([(sm.sum(2) * ar).sum(2), (sm.sum(3) * ar).sum(2)], dim=2) / (0.5 * S) - 1
    F.smooth_l1_loss(c, kps[:, :, :2], reduction="sum").div(B).backward()


res = {}
n = 200
# dp: the four gradient planes written (3 x 25 + 15 channels), Ann_Index read; the point inputs and the 4 x 3 x 25
# gathered values per point are < 0.5 MB
dp_bytes = B * HW * 4 * (3 * C + CA) + B * HW * 4 * CA
stn_bytes = B * J * HW * 4 * 2                                    # the heat maps read once, their gradient written once
for name, f, by in (("dp_uvia_fused", fused_dp, dp_bytes), ("stn_kps_fused", fused_stn, stn_bytes)):
    ms = timed(f, n)
    res[name] = {"ms_fwd_bwd": ms, "bytes": by, "GB/s": by / ms / 1e6, "frac_of_hbm_peak": by / ms / 1e6 / peak,
                 "note": "includes the wrapper's fp32-contiguous pass-through, gradient and workspace allocation, "
                         "and the autograd backward that scales the gradients"}
res["dp_uvia_torch_ops"] = {"ms_fwd_bwd": timed(torch_dp, n)}
res["stn_kps_torch_ops"] = {"ms_fwd_bwd": timed(torch_stn, n)}
res["dp_uvia_speedup"] = res["dp_uvia_torch_ops"]["ms_fwd_bwd"] / res["dp_uvia_fused"]["ms_fwd_bwd"]
res["stn_kps_speedup"] = res["stn_kps_torch_ops"]["ms_fwd_bwd"] / res["stn_kps_fused"]["ms_fwd_bwd"]
res["hbm_peak_gbs"] = peak
res["shape"] = {"B": B, "S": S, "P": P, "C": C, "Cann": CA, "J": J}
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
except Exception:
    q = "unknown"
res["gpu"] = q
res["torch"] = torch.__version__
print(json.dumps(res, indent=1))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
