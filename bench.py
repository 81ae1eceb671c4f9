"""Benchmark of the DaNet inference hot path (BASELINE.json metric: images/sec, DaNet forward
bs=64 224x224, HRNet-W48 + SMPL + IUV_Renderer; plus SMPL LBS vertices/sec and roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); batches are sharded image-parallel (weak
scaling: 64 images per GPU) and the only collective is one all_gather of the outputs per step.
Prints ONE JSON line on rank 0 (contract in the task statement)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_IMG = {48: 46.5e9, 32: 29.5e9}            # SURVEY section 8d: 2 x conv/linear MACs of a2+a3+a6
LBS_BYTES_PER_BODY = 84460.0                        # SURVEY section 8d compulsory HBM bytes / body
LBS_FLOP_PER_BODY = 15.8e6


def metric_name(batch, width):
    """ONE metric string for both arms (the driver computes the ratio only when they agree)."""
    return "images/sec DaNet fwd bs=%d 224x224 (HRNet-W%d + part regressors + SMPL LBS + IUV render)" % (batch, width)


def host_threads():
    """Threads for the CPU arms: the cores this process may run on, capped at 32 (oneDNN on small
    batches degrades badly when a 128-core box is oversubscribed)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, int(os.environ.get("DANET_CPU_THREADS", "32"))))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = []
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                out["sm_max_mhz"] = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active") and name not in out["reasons"]:
                        out["reasons"].append(name)
            except Exception:
                continue
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
            out["samples"] = len(sm)
        return out


# ---------------------------------------------------------------------------------------------
# CPU arms (reference's own modules when /root/reference exists, else the oracle port)
# ---------------------------------------------------------------------------------------------
def cpu_step_factory(width, B, seed=0):
    """Returns (step_fn, kind, description).  One step = B images through the CPU implementation of
    the same path: network half + SMPL LBS + IUV rasteriser."""
    import numpy as np
    import torch
    from danet_b200 import synthetic
    from oracle import lbs as olbs, raster as oraster, ref_import
    torch.set_num_threads(host_threads())
    model, mesh = synthetic.make_smpl_model(seed), synthetic.make_dp_mesh(seed)
    tex = synthetic.dp_textures(mesh)
    g = torch.Generator().manual_seed(0)
    img = torch.randn(B, 3, 224, 224, generator=g)
    if ref_import.available():
        import contextlib
        from oracle import gen_golden_net
        with contextlib.redirect_stdout(sys.stderr):          # the reference prints banners on import
            ns = ref_import.load(width)
            est, pred, _ = gen_golden_net.build_reference(ns, width, seed)
        kind = "reference"
        desc = ("the reference's own modules (IUV_Estimator + iuvmap_clean + DecomposedPredictor) imported from %s" %
                ("/root/reference" if ref_import.REF.startswith("/root/reference") else "oracle/_ref (oracle/make_ref.py)"))

        def net(x):
            return ref_import.infer_para(ns, est, pred, x)["para"]
    else:
        import danet_b200
        from oracle.net_ops import TorchEmulOps
        m = danet_b200.DaNet(None, synthetic.make_mean_params(seed), pretrained=False, width=width,
                             smpl_model=model, dp_mesh=mesh)
        m.load_state_dict(synthetic.keyed_state_dict(m.state_dict(), seed))
        m.eval()
        emul = TorchEmulOps()
        kind = "port"
        desc = "oracle port: the same graph through torch CPU ops (oracle/net_ops.py)"

        def net(x):
            plan = m.plan_for(x.shape[0], "cpu", ops=emul)
            plan.run(x)
            return m.outputs_of(plan, x.shape[0])["para"]

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=min(B, host_threads()))
    oraster.build()

    def step():
        para = net(img).numpy()
        R = para[:, 13:].reshape(B, 24, 3, 3)
        out = olbs.smpl_forward(model, para[:, 3:13], R[:, 1:], R[:, :1], pose2rot=False, dtype=np.float32)
        verts, cam = out["vertices"].astype(np.float32), para[:, :3].copy()
        # the C rasteriser is single-threaded per call; ctypes drops the GIL, so images run in parallel
        list(pool.map(lambda b: oraster.verts2uvimg(verts[b:b + 1], cam[b:b + 1], mesh, tex), range(B)))
        return B

    return step, kind, desc + " + oracle/lbs.py (numpy fp32) + oracle/raster.c"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.cpu_batch
    step, kind, desc = cpu_step_factory(args.width, B)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        n += step()
    dt = time.perf_counter() - t0
    val = n / dt
    cores = host_threads()
    sample = "%d steps x %d images, W%d, %s" % (args.steps, B, args.width, desc)
    line = {"impl": "reference", "metric": metric_name(args.batch, args.width),
            "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[2]: DaNet forward batch=64 synthetic 224x224, HRNet-W%d + IUV_Renderer" % args.width,
                       "cpu_step_batch": B},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    import danet_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # libraries (NCCL's version banner) write to fd 1; keep stdout clean for the single JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if args.gpus > 1 and world == 1:
        raise SystemExit("bench.py --gpus %d must be launched with torchrun (one rank per GPU)" % args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, W = args.batch, args.width
    net = danet_b200.build_synthetic_danet(width=W, seed=0, device=dev, conv_algo=args.conv, precision=args.precision,
                                           use_cuda_graph=not args.no_graph, group_convs=not args.no_group)
    smpl, rend = net.iuv2smpl.smpl, net.iuv_renderer
    nrot = 4                                          # 4 x 38.5 MB input batches > 126 MB L2
    g = torch.Generator().manual_seed(1234 + rank)
    host_in = [torch.randn(B, 3, 224, 224, generator=g).pin_memory() for _ in range(nrot)]
    dev_in = [t.to(dev) for t in host_in]
    gathered = torch.empty(world * B, 229, device=dev) if world > 1 else None

    def hot_path(x):
        para = net.infer_net(x)["para"]
        R = para[:, 13:].reshape(B, 24, 3, 3)
        out = smpl(betas=para[:, 3:13].contiguous(), body_pose=R[:, 1:], global_orient=R[:, :1], pose2rot=False)
        img = rend.verts2uvimg(out.vertices, para[:, :3].contiguous())
        if world > 1:
            dist.all_gather_into_tensor(gathered, para)      # the single NCCL gather of outputs
        return para, out.vertices, img

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        hot_path(dev_in[i % nrot])
    sync()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for i in range(args.steps):
        last = hot_path(dev_in[i % nrot])
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("para", "vertices", "iuv_image"), last)))
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B * args.steps / (ms * 1e-3)

    # ---- end-to-end through the public API with host buffers (H2D + D2H inside the timed region) ----
    host_para = torch.empty(B, 229).pin_memory()
    host_img = torch.empty(B, 3, 56, 56).pin_memory()

    # the user-facing loop a server would run: the H2D copy of step i+1 is issued on a copy stream while step i
    # computes (two device input buffers), results are read back on the compute stream; every step's H2D and
    # D2H lie inside the timed region
    copy_s = torch.cuda.Stream(device=dev)
    cur_s = torch.cuda.current_stream(dev)
    in_buf = [torch.empty_like(dev_in[0]) for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]

    def issue_h2d(i):
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(ev_free[i % 2])                 # the step that last read this buffer is done
            in_buf[i % 2].copy_(host_in[i % nrot], non_blocking=True)
            ev_in[i % 2].record(copy_s)

    def e2e_run(n):
        issue_h2d(0)
        for i in range(n):
            if i + 1 < n:
                issue_h2d(i + 1)
            cur_s.wait_event(ev_in[i % 2])
            para, _, img = hot_path(in_buf[i % 2])
            ev_free[i % 2].record(cur_s)
            host_para.copy_(para, non_blocking=True)
            host_img.copy_(img, non_blocking=True)

    e2e_run(3)
    sync()
    e0.record()
    e2e_run(args.steps)
    e1.record()
    sync()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t.item()) * 1e-3)

    plan = net.plan_for(B, dev)
    launches_per_step = plan.n_launch + 3 + 4 + (1 if world > 1 else 0)
    line = None
    if rank == 0:
        pk = peaks()
        # ---- per-kernel-class timing of one profiled step (CUDA events on the launch stream) ----
        prof = profile_step(net, plan, dev_in[0], dev)
        # the convolutions' time inside the measured (CUDA-graph) step = step time x their share of an eager pass in
        # which every launch is timed with CUDA events (eager launches do not overlap, the graph's do: the share, not
        # the absolute eager sum, carries over)
        eager_total = prof["conv_ms"] + sum(prof["other_ms"].values())
        conv_share = prof["conv_ms"] / max(1e-9, eager_total)
        conv_ms = conv_share * (ms / args.steps)
        flops = FLOP_PER_IMG.get(W, 0.0) * B
        conv_tflops = flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        tc_peak = pk["bf16_tflops_sustained"]
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            if tj.get("width") == W and tj.get("batch") == B:
                traffic, traffic_src = tj.get("dram_bytes_per_step"), tj.get("source")
        roof = {"bound": "tensor", "kernel": prof["conv_kernel"], "achieved": conv_tflops, "peak": tc_peak,
                "unit": "TFLOP/s", "frac": conv_tflops / tc_peak if tc_peak else None, "traffic": traffic,
                "traffic_note": traffic_src,
                "peak_note": "16-bit dense tensor peak = the %s sustained cuBLAS bf16 figure (%.0f TFLOP/s; kernel timed "
                             "inside a long step); achieved = algorithmic conv FLOPs of one step / summed duration of "
                             "its conv launches (CUDA events per launch); the few fp32-FMA launches are rated against "
                             "the same denominator" % (pk["source"], pk["bf16_tflops_sustained"]),
                "algorithmic_flop_per_launch_group": flops, "conv_ms_per_step": conv_ms,
                # share within the same eager, individually timed pass (under the CUDA graph + programmatic
                # dependent launch the step is shorter than the sum of its separately timed launches)
                "conv_share_of_step": conv_share, "conv_ms_eager_sum": prof["conv_ms"],
                "eager_sum_vs_graph_step": eager_total / (ms / args.steps),
                "precision": plan.precision, "mma_per_k_step": 3 if (plan.n_tc and plan.precision == "exact") else 1,
                "n_conv_tc": plan.n_tc,
                "n_conv_total": prof["n_conv"], "other_ms": prof["other_ms"]}
        lbs = lbs_bench(smpl, dev, pk)
        parity = parity_block(net, dev, W, B) if world == 1 else None
        extras = {}
        if world == 1 and not args.no_extras:
            # BASELINE config 2: single 224x224 image, HRNet-W32, batch 1 (latency)
            n32 = danet_b200.build_synthetic_danet(width=32, seed=0, device=dev, conv_algo=args.conv, precision=args.precision,
                                                   use_cuda_graph=not args.no_graph)
            ms1 = time_net(n32, n32.iuv2smpl.smpl, n32.iuv_renderer, torch.randn(1, 3, 224, 224, device=dev), 30)
            extras["latency_b1_w32"] = {"workload": "configs[1]: DaNet forward single 224x224 image, batch=1, HRNet-W32", "ms": ms1,
                                        "images_per_s": 1e3 / ms1}
            del n32
            # the other precision of the tensor-core path, same workload (device-resident), with its own parity block
            other = "fast" if plan.precision == "exact" else "exact"
            n2 = danet_b200.build_synthetic_danet(width=W, seed=0, device=dev, conv_algo=args.conv, precision=other,
                                                  use_cuda_graph=not args.no_graph)
            ms2 = time_net(n2, n2.iuv2smpl.smpl, n2.iuv_renderer, dev_in[0], max(5, args.steps))
            extras["precision_" + other] = {"value": B / (ms2 * 1e-3), "unit": "images/s", "ms_per_step": ms2,
                                            "tensor_frac_of_sustained_peak": (FLOP_PER_IMG.get(W, 0.0) * B / (ms2 * 1e-3) / 1e12) / tc_peak,
                                            "parity": parity_block(n2, dev, W, B)}
            del n2
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_baseline(W, args.cpu_batch)
        line = {"metric": metric_name(B, W),
                "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": ("split-f16 operands (hi+lo, 22 bits; 3 MMAs per K step), f32 accumulate" if plan.precision == "exact"
                          else "f16 operands, f32 accumulate") if plan.n_tc else "f32", "data": "synthetic",
                "config": {"workload": "configs[2]: DaNet forward batch=64 synthetic 224x224, HRNet-W%d + IUV_Renderer" % W,
                           "per_gpu_batch": B, "global_batch": B * world, "parallelism": "image-sharded x%d, one all_gather of para" % world,
                           "conv_path": "tcgen05 kind::f16, precision=%s: %d convolutions in %d launches" % (plan.precision, plan.n_tc, prof["n_conv"]),
                           "cuda_graph": not args.no_graph,
                           "l2": "inputs rotate over %d batches (%.0f MB > 126 MB L2); activations (%.1f GB/step) exceed L2"
                                 % (nrot, nrot * B * 3 * 224 * 224 * 4 / 1e6, plan.bytes_alloc / 1e9),
                           "weights": "deterministic keyed random init of the reference architecture (synthetic.keyed_state_dict)"},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * 3 * 224 * 224 * 4,
                        "d2h_bytes_per_step": B * 229 * 4 + B * 3 * 56 * 56 * 4},
                "gpu_launches": launches_per_step * args.steps,
                "roofline": roof, "lbs": lbs, "parity": parity, "cpu_baseline": cpu}
        line.update(extras)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


DUMP_LIMIT_BYTES = 60 * 10 ** 6                     # array data: the files with their .npy headers stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each [B, ...] array as out_dir/<name>.npy in float32, so that two builds run with the same arguments
    (same seeded inputs and weights) can be compared output for output.  Above DUMP_LIMIT_BYTES in all, only the
    first images of the batch are written (the same images for every array)."""
    import numpy as np
    per_image = sum(t[0].numel() * 4 for t in arrays.values())
    n = max(1, min(next(iter(arrays.values())).shape[0], DUMP_LIMIT_BYTES // per_image))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[:n].detach().float().cpu().numpy())


def parity_block(net, dev, width, B):
    """The benched configuration against the reference's own outputs for the same images
    (tests/golden/net_w48_b64.npz, produced by the reference's modules -- oracle/gen_golden_net.py): para / STN
    centre error, integer-map agreement, and the para error carried through the SMPL layer in millimetres."""
    import numpy as np
    import torch
    import torch.nn.functional as F
    gp = os.path.join(ROOT, "tests", "golden", "net_w%d_b%d.npz" % (width, B))
    if not os.path.exists(gp):
        return None
    g = np.load(gp)
    gen = torch.Generator().manual_seed(100 + int(g["seed"]))
    low = torch.randn(B, 3, 7, 7, generator=gen)
    img = F.interpolate(low, size=224, mode="bilinear", align_corners=False) * 2 + 0.3 * torch.randn(B, 3, 224, 224, generator=gen)
    out = net.infer_net(img.to(dev))
    para = out["para"]
    ref = torch.from_numpy(g["para"]).to(dev)
    smpl = net.iuv2smpl.smpl

    def verts(p):
        R = p[:, 13:].reshape(-1, 24, 3, 3)
        return smpl(betas=p[:, 3:13].contiguous(), body_pose=R[:, 1:], global_orient=R[:, :1], pose2rot=False).vertices
    dv = (verts(para) - verts(ref)).norm(dim=-1)
    # eval.py:196-212 on both: MPJPE against synthetic ground-truth joints, from our para and from the reference's
    from danet_b200.smpl import mpjpe_h36m
    gt = (torch.randn(B, 14, 3, generator=torch.Generator().manual_seed(5)) * 0.2).to(dev)
    mp = []
    for p in (para, ref):
        verts(p)
        j17 = smpl.joints_h36m()
        mp.append(mpjpe_h36m(j17, gt).cpu().numpy() * 1e3 if j17 is not None else None)
    u, v, i, a = out["visualization"]["iuv_pred"]
    idx = i.argmax(1).cpu().numpy()
    ann = a.argmax(1).cpu().numpy()
    parts = out["visualization"]["part_iuv_pred"][:, :, 2].argmax(2).cpu().numpy()
    tie = np.unpackbits(g["part_tie_bits"], axis=1)[:, :parts[0].size].reshape(parts.shape).astype(bool)
    flip_i, flip_a, flip_p = idx != g["index_argmax"], ann != g["ann_argmax"], parts != g["part_argmax_all"]
    bad = int((flip_i & (g["index_margin"].astype(np.float32) > 1e-3)).sum() + (flip_a & (g["ann_margin"].astype(np.float32) > 1e-3)).sum()
              + (flip_p & ~tie).sum())
    dirty = flip_i.reshape(B, -1).any(1) | flip_p.reshape(B, -1).any(1)
    err = (para - ref).abs().max(1)[0].cpu().numpy()
    dvn = dv.max(1)[0].cpu().numpy() * 1e3
    return {"golden": os.path.relpath(gp, ROOT), "images": B, "para_tolerance": 1e-4,
            "note": "integer decisions (iuvmap_clean argmax) may flip only where the REFERENCE's own top-2 margin is < 1e-3 "
                    "(near-ties); images whose integer maps equal the reference's are held to the 1e-4 tolerance",
            "images_with_identical_integer_maps": int((~dirty).sum()),
            "para_max_abs_err_identical_maps": float(err[~dirty].max()) if (~dirty).any() else None,
            "verts_max_err_mm_identical_maps": float(dvn[~dirty].max()) if (~dirty).any() else None,
            "images_with_near_tie_flips": int(dirty.sum()), "flipped_pixels_total": int(flip_i.sum() + flip_p.sum()),
            "flips_outside_reference_near_ties": bad,
            "para_max_abs_err_flipped_images": float(err[dirty].max()) if dirty.any() else 0.0,
            "verts_max_err_mm_flipped_images": float(dvn[dirty].max()) if dirty.any() else 0.0,
            "stn_kps_max_abs_err": float((out["stn_kps_pred"].cpu() - torch.from_numpy(g["stn_kps"])).abs().max()),
            "verts_mean_err_mm": float(dv.mean()) * 1e3,
            "mpjpe_mm": None if mp[0] is None else {
                "note": "eval.py:196-212 on synthetic ground truth, from this path's para vs from the reference's para",
                "mean_this": float(mp[0].mean()), "mean_reference": float(mp[1].mean()),
                "mean_abs_diff": float(abs(mp[0].mean() - mp[1].mean())),
                "per_image_max_abs_diff": float(np.abs(mp[0] - mp[1]).max()),
                "per_image_median_abs_diff": float(np.median(np.abs(mp[0] - mp[1])))}}


def time_net(net, smpl, rend, x, iters):
    """ms per call of infer_net + SMPL + render on a resident batch (CUDA events, graph replay)."""
    import torch

    def f():
        para = net.infer_net(x)["para"]
        R = para[:, 13:].reshape(-1, 24, 3, 3)
        out = smpl(betas=para[:, 3:13].contiguous(), body_pose=R[:, 1:], global_orient=R[:, :1], pose2rot=False)
        return rend.verts2uvimg(out.vertices, para[:, :3].contiguous())
    for _ in range(3):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def profile_step(net, plan, x, dev):
    """One eager (non-graph) step with CUDA events around every launch; groups by kernel class."""
    import torch
    saved = plan.use_cuda_graph
    plan.use_cuda_graph = False
    ops = plan.ops
    events = []

    class Timed(object):
        def __getattr__(self, name):
            fn = getattr(ops, name)
            if name.startswith("conv_tc") or not callable(fn):
                return fn

            def wrapped(*a, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = fn(*a, **k)
                e1.record()
                tag = {"conv2d": "conv_simt", "conv_group": "conv_tc"}.get(name, name)
                events.append((tag, e0, e1))
                return r
            return wrapped
    plan.ops = Timed()
    plan.run(x)
    torch.cuda.synchronize()
    plan.ops = ops
    plan.use_cuda_graph = saved
    agg = {}
    for tag, e0, e1 in events:
        agg[tag] = agg.get(tag, 0.0) + e0.elapsed_time(e1)
    conv_ms = agg.get("conv_tc", 0.0) + agg.get("conv_simt", 0.0)
    n_conv = sum(1 for t, _, _ in events if t.startswith("conv"))
    kern = "k_conv_tc (tcgen05 kind::f16, TMA tensor-map operands, fp32 TMEM accumulators)" if agg.get("conv_tc") else "k_conv_simt (fp32 FMA implicit GEMM)"
    return {"conv_ms": conv_ms, "n_conv": n_conv, "conv_kernel": kern,
            "other_ms": {k: v for k, v in agg.items() if not k.startswith("conv")},
            "conv_tc_ms": agg.get("conv_tc", 0.0), "conv_simt_ms": agg.get("conv_simt", 0.0)}


def lbs_bench(smpl, dev, pk, B=8192):
    """SMPL LBS vertices/sec on a batch whose output (B*82.7 KB = 677 MB) exceeds L2."""
    import torch
    betas = torch.randn(B, 10, device=dev)
    x6 = torch.randn(B, 24, 6, device=dev)
    for _ in range(3):
        smpl(betas=betas, pose6d=x6)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 10
    e0.record()
    for _ in range(n):
        smpl(betas=betas, pose6d=x6)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    bodies = B / (ms * 1e-3)
    gbs = bodies * LBS_BYTES_PER_BODY / 1e9
    return {"metric": "SMPL LBS vertices/sec (forward incl. 49 joints)", "value": bodies * 6890, "unit": "vertices/s",
            "batch": B, "ms": ms, "bodies_per_s": bodies,
            "roofline_hbm": {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                             "algorithmic_bytes_per_body": LBS_BYTES_PER_BODY},
            "roofline_fma": {"achieved_tflops": bodies * LBS_FLOP_PER_BODY / 1e12, "nominal_fp32_tflops": 80.0,
                             "note": "dense pose-corrective contraction (4.28 MMAC/body) makes the fused kernel FMA-bound (SURVEY 8d)"}}


def cpu_baseline(width, B):
    step, kind, desc = cpu_step_factory(width, B)
    t0 = time.perf_counter()
    step()                                            # warm-up (also bounds the sample: see below)
    warm = time.perf_counter() - t0
    t0 = time.perf_counter()
    n, it = 0, 0
    while it < 1 or (time.perf_counter() - t0 + warm < 20.0 and it < 20):
        n += step()
        it += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "images/s", "cores": host_threads(), "kind": kind,
            "sample": "%d steps x %d images (%.1f s), W%d; %s" % (it, B, dt, width, desc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--width", type=int, default=48)
    ap.add_argument("--conv", default="auto", choices=["auto", "tc", "simt"])
    ap.add_argument("--cpu-batch", type=int, default=4)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--precision", default="exact", choices=["exact", "fast"],
                    help="tensor-core path: exact = split-fp16 operands, 3 MMAs per K step (fp32-grade, default); fast = one fp16 pass")
    ap.add_argument("--no-group", action="store_true", help="one convolution per launch (no multi-problem launches)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the B=1 W32 latency line and the other-precision run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0: para, SMPL vertices, IUV image) to DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
