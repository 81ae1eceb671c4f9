"""Golden vectors of the network half, produced by the REFERENCE'S OWN modules
(models/danet/iuv_estimator.py IUV_Estimator, models/danet/smpl_regressor.py DecomposedPredictor,
utils/iuvmap.py iuvmap_clean, glue of models/danet/danet.py:78-98,118) imported on CPU with the
SURVEY Appendix-C shims, with deterministic keyed weights (danet_b200.synthetic.keyed_state_dict:
a pure function of the state_dict key) so the GPU box can rebuild the same parameters without a
checkpoint.  Called from oracle/gen_golden.py (this container only)."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def make_image(torch, B, seed):
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(seed)
    low = torch.randn(B, 3, 7, 7, generator=g)
    return F.interpolate(low, size=224, mode="bilinear", align_corners=False) * 2 + 0.3 * torch.randn(B, 3, 224, 224, generator=g)


def build_reference(ns, width, seed):
    import torch
    from danet_b200 import synthetic
    from oracle import ref_import
    ref_import._set_width(ns.cfg, width)
    est = ns.IUV_Estimator(pretrained=False).eval()
    mp = synthetic.make_mean_params(seed)
    pred = ns.DecomposedPredictor(None, (torch.tensor(mp["cam"]).reshape(1, 3), torch.tensor(mp["shape"]).reshape(1, 10),
                                         torch.tensor(mp["pose"]).reshape(1, 144)), pretrained=False).eval()
    rsd = {}
    for k, v in est.state_dict().items():
        rsd["img2iuv." + k] = v
    for k, v in pred.state_dict().items():
        rsd["iuv2smpl.smpl_para_Outs." + k] = v
    ksd = synthetic.keyed_state_dict(rsd, seed)
    est.load_state_dict({k[len("img2iuv."):]: v for k, v in ksd.items() if k.startswith("img2iuv.")}, strict=True)
    pred.load_state_dict({k[len("iuv2smpl.smpl_para_Outs."):]: v for k, v in ksd.items() if k.startswith("iuv2smpl.")}, strict=True)
    return est, pred, rsd


def top2_margin(x, dim=1):
    v = x.topk(2, dim=dim)[0]
    return (v.select(dim, 0) - v.select(dim, 1))


def gen(ns, width, B, seed, detail=None, chunk=8):
    """detail = number of leading images whose per-part maps / sums are stored (all when None); the batch runs
    through the reference in chunks of `chunk` images (eval-mode network: images are independent)."""
    import torch
    from oracle import ref_import
    est, pred, rsd = build_reference(ns, width, seed)
    img = make_image(torch, B, 100 + seed)
    nd = B if detail is None else detail
    acc = {}
    for s0 in range(0, B, chunk):
        r = ref_import.infer_para(ns, est, pred, img[s0:s0 + chunk])
        ret = r["ret"]
        u, v, i, a = r["uvia_clean"]
        I_raw, A_raw = ret["uvia_pred"][2], ret["uvia_pred"][3]
        pp = ret["part_iuv_pred"]                                    # [b,24,3,7,56,56]
        part = dict(
            para=r["para"].numpy(), stn_kps=ret["stn_kps_pred"].numpy(),
            index_argmax=I_raw.argmax(1).numpy().astype(np.uint8), index_margin=top2_margin(I_raw).numpy().astype(np.float16),
            ann_argmax=A_raw.argmax(1).numpy().astype(np.uint8), ann_margin=top2_margin(A_raw).numpy().astype(np.float16))
        pm = top2_margin(pp[:, :, 2], dim=2)
        if detail is not None:
            # every image: the per-part argmax maps and, bit-packed, where the reference's own top-2 margin is below 1e-3
            # (near-ties: any implementation may pick the other index there, and the regressor's output then moves)
            part.update(part_argmax_all=pp[:, :, 2].argmax(2).numpy().astype(np.uint8),
                        part_tie_bits=np.packbits((pm < 1e-3).numpy().reshape(pm.shape[0], -1), axis=1))
        if s0 < nd:
            part.update(
                part_argmax=pp[:, :, 2].argmax(2).numpy().astype(np.uint8),
                part_margin=pm.numpy().astype(np.float16),
                u_sum=u.sum(1).numpy().astype(np.float32), v_sum=v.sum(1).numpy().astype(np.float32))
            if detail is None:
                part.update(
                    hm=ret["skps_hm_pred"].numpy().astype(np.float16),
                    part_u_sum=r["part_iuv_map"][:, :, 0].sum(2).numpy().astype(np.float16),
                    heads_sub=torch.cat(ret["uvia_pred"], 1)[:, :, ::4, ::4].numpy().astype(np.float32),
                    parts_sub=pp[:, ::5, :, :, ::8, ::8].numpy().astype(np.float32))
        for k, val in part.items():
            acc.setdefault(k, []).append(val)
    out = {k: np.concatenate(v, 0) for k, v in acc.items()}
    out.update(width=np.int32(width), B=np.int32(B), seed=np.int32(seed), detail=np.int32(nd))
    path = os.path.join(GOLD, "net_w%d.npz" % width if detail is None else "net_w%d_b%d.npz" % (width, B))
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path) // 1024, "KiB; para[0,:6] =", out["para"][0, :6])
    return rsd


def main(ns, big=True):
    rsd = gen(ns, 32, 2, 0)
    rsd48 = gen(ns, 48, 2, 0)
    if big:
        # BASELINE config 3: the benched configuration; only what check_batch_against_golden reads (per-part
        # margins of even a few images would take the file above 1 MB)
        gen(ns, 48, 64, 0, detail=0)
    # the reference's state_dict keys + shapes: the drop-in surface (SURVEY section 8b)
    with open(os.path.join(GOLD, "state_dict_keys_w48.txt"), "w") as f:
        for k, v in rsd48.items():
            f.write("%s %s\n" % (k, "x".join(str(d) for d in v.shape) or "scalar"))
    print("state_dict_keys_w48.txt:", len(rsd48), "keys")
