"""CPU tests of the DensePose-point losses and the STN key-point loss (SURVEY section 8f-2,
models/danet/iuv_estimator.py:343-419,106-121,137-140,159-171): the numpy oracle against the golden the reference's own
code produced under torch autograd (oracle/gen_golden_points.py), and the kernels' per-point / per-pixel / per-joint
arithmetic (csrc/point_losses.cu compiled with DANET_POINT_LOSSES_HOST_CHECK: the same __host__ __device__ functions
walked on the host) against the same golden -- no GPU involved.

Tolerances: the point losses as the dense-loss tests (losses 2e-6 / 3e-6 relative, gradients 3e-7 absolute).  The STN
gradient reaches 2.4 on these maps and is (10 / (S/2)) * softmax * (col - x^) summed by the reference in fp32, so the
golden itself carries ~1e-6 of rounding there (the fp64 oracle differs from it by 1.1e-6): 3e-6 absolute."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import point_losses as opl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PTS = ["body_uv_X_points", "body_uv_Y_points", "body_uv_I_points", "body_uv_Ind_points", "body_uv_U_points",
       "body_uv_V_points", "body_uv_point_weights", "body_uv_ann_labels", "body_uv_ann_weights"]
CASES = [(ac, tag) for ac in (0, 1) for tag in ("all", "some")]


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "dp_losses.npz"))


def _has(g, tag):
    return None if tag == "all" else g["has_some"]


@pytest.mark.parametrize("ac,tag", CASES)
def test_oracle_dp_uvia_losses_match_reference_golden(gold, ac, tag):
    g = gold
    L, gr = opl.dp_uvia_losses(g["u"], g["v"], g["i"], g["a"], *[g[k] for k in PTS], has_dp=_has(g, tag),
                               align_corners=bool(ac))
    np.testing.assert_allclose(L, g["L_%s_ac%d" % (tag, ac)], rtol=2e-6)
    for k, (name, n) in enumerate((("u", "u"), ("v", "v"), ("index", "i"), ("ann", "a"))):
        np.testing.assert_allclose(gr[name] * g["grad_weights"][k], g["g%s_%s_ac%d" % (n, tag, ac)], atol=5e-7)


def test_oracle_dp_uvia_losses_none_selected_and_bad_label(gold):
    g = gold
    L, gr = opl.dp_uvia_losses(g["u"], g["v"], g["i"], g["a"], *[g[k] for k in PTS], has_dp=np.zeros(3))
    assert np.all(L == 0) and all(np.abs(x).max() == 0 for x in gr.values())
    pts = {k: g[k].copy() for k in PTS}
    pts["body_uv_I_points"][0, 5] = 25
    L, _ = opl.dp_uvia_losses(g["u"], g["v"], g["i"], g["a"], **pts)
    assert np.isnan(L[2]) and np.isfinite(L[[0, 1, 3]]).all()


def test_oracle_stn_kps_losses_match_reference_golden(gold):
    g = gold
    loss, c, gr = opl.stn_kps_losses(g["hm"], g["kps"])
    np.testing.assert_allclose(loss, g["roi_loss"], rtol=2e-6)
    np.testing.assert_allclose(c, g["roi_centers"], atol=1e-6)
    np.testing.assert_allclose(gr, g["roi_grad"], atol=3e-6)
    assert set(np.unique(g["kps"][:, :, 2])) == {0.0, 0.5, 1.0, 2.0}


@pytest.fixture(scope="module")
def hostlib(tmp_path_factory):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = shutil.which("nvcc")
    if not nvcc:
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("point_losses_host") / "libpoint_losses_host.so")
    csrc = os.path.join(ROOT, "danet-densepose2smpl_b200", "csrc")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "-Xcompiler", "-fPIC",
                           "-DDANET_POINT_LOSSES_HOST_CHECK", "-shared", os.path.join(csrc, "point_losses.cu"),
                           os.path.join(csrc, "api.cu"), "-o", out])
    lib = ctypes.CDLL(out)
    p, i32, f = ctypes.c_void_p, ctypes.c_int32, ctypes.c_float
    lib.danet_test_dp_uvia_losses_host.argtypes = [i32] * 5 + [p] * 12 + [i32, f, f, f] + [p] * 5
    lib.danet_test_dp_uvia_losses_host.restype = ctypes.c_int
    lib.danet_test_stn_kps_losses_host.argtypes = [i32, i32, i32, p, p, f, p, p, p]
    lib.danet_test_stn_kps_losses_host.restype = ctypes.c_int
    return lib


def _c(x):
    return np.ascontiguousarray(x, np.float32)


def _P(x):
    return None if x is None else x.ctypes.data_as(ctypes.c_void_p)


def _host_dp(lib, preds, pts, has, ac, grads, weights=(2.0, 0.3, 0.5)):
    """preds = (u, v, index, ann); pts = (X, Y, I, U, V, W, ann_labels); grads: 4 arrays or None."""
    B, C, S = preds[0].shape[:3]
    L = np.zeros(4, np.float32)
    assert lib.danet_test_dp_uvia_losses_host(B, C, preds[3].shape[1], S, pts[0].shape[1], *[_P(x) for x in preds + pts],
                                              _P(has), ac, *weights, _P(L), *[_P(x) for x in grads]) == 0
    return L


@pytest.mark.parametrize("ac,tag", CASES + [(0, "none")])
def test_kernel_arithmetic_on_host_matches_reference_golden(gold, hostlib, ac, tag):
    g = gold
    preds = [_c(g[k]) for k in ("u", "v", "i", "a")]
    pts = [_c(g[k]) for k in PTS if k not in ("body_uv_Ind_points", "body_uv_ann_weights")]
    has = {"all": None, "some": np.ascontiguousarray(g["has_some"], np.uint8), "none": np.zeros(3, np.uint8)}[tag]
    grads = [np.full_like(x, 7) for x in preds]
    L = _host_dp(hostlib, preds, pts, has, ac, grads)
    if tag == "none":
        assert np.all(L == 0) and all(np.abs(x).max() == 0 for x in grads)
        return
    np.testing.assert_allclose(L, g["L_%s_ac%d" % (tag, ac)], rtol=3e-6)
    for k, n in enumerate("uvia"):
        np.testing.assert_allclose(grads[k] * g["grad_weights"][k], g["g%s_%s_ac%d" % (n, tag, ac)], atol=3e-7)


def test_stn_kernel_arithmetic_on_host_matches_reference_golden(gold, hostlib):
    g = gold
    hm, kps = _c(g["hm"]), _c(g["kps"])
    B, J, S = hm.shape[:3]
    L, cen, gh = np.zeros(1, np.float32), np.zeros((B, J, 2), np.float32), np.full_like(hm, 7)
    assert hostlib.danet_test_stn_kps_losses_host(B, J, S, _P(hm), _P(kps), 1.0, _P(L), _P(cen), _P(gh)) == 0
    np.testing.assert_allclose(L[0], g["roi_loss"], rtol=3e-6)
    np.testing.assert_allclose(cen, g["roi_centers"], atol=1e-6)
    np.testing.assert_allclose(gh, g["roi_grad"], atol=3e-6)


def test_kernel_arithmetic_on_host_matches_oracle_on_other_shapes(hostlib):
    """Shapes and inputs the golden does not cover: few channels, odd map sizes, more points than pixels, all points of
    a sample on one pixel, an out-of-range part label (NaN loss), other loss weights, non-square STN key-point sets."""
    rng = np.random.default_rng(7)
    for (B, C, Ca, S, P, ac) in ((1, 1, 1, 1, 3, 0), (2, 3, 2, 5, 40, 1), (3, 25, 15, 9, 196, 0), (2, 4, 3, 7, 11, 1)):
        preds = [_c(rng.normal(0, 1.5, (B, c, S, S))) for c in (C, C, C, Ca)]
        X, Y = (_c(rng.uniform(-2, S + 1, (B, P))) for _ in range(2))
        X[0], Y[0] = 1.5, 2.0                                          # sample 0: every point on one pixel pair
        I = _c(rng.integers(0, C, (B, P)))
        W = _c(rng.choice([0.0, 0.5, 1.0, 2.0], (B, C * P)))
        U, V = _c(rng.random((B, C * P))), _c(rng.random((B, C * P)))
        lab = _c(rng.integers(0, Ca, (B, S * S)))
        has = np.ones(B, np.uint8)
        has[-1] = B == 1
        weights = (1.5, 0.7, 0.25)
        Lr, gr = opl.dp_uvia_losses(*preds, X, Y, I, None, U, V, W, lab, has_dp=has, align_corners=bool(ac),
                                    index_weight=weights[0], part_weight=weights[1], point_weight=weights[2])
        grads = [np.full_like(x, 7) for x in preds]
        L = _host_dp(hostlib, preds, [X, Y, I, U, V, W, lab], has, ac, grads, weights)
        np.testing.assert_allclose(L, Lr, rtol=5e-6, atol=1e-7)
        for got, name in zip(grads, ("u", "v", "index", "ann")):                # the one-pixel sample adds 4P fp32
            np.testing.assert_allclose(got, gr[name], atol=1e-6 * max(1.0, np.abs(gr[name]).max()))   # terms
        I[0, 1] = C                                                    # out-of-range part label: NaN part loss
        L = _host_dp(hostlib, preds, [X, Y, I, U, V, W, lab], has, ac, [None] * 4, weights)
        assert np.isnan(L[2]) and np.isfinite(L[[0, 1, 3]]).all()
    for (B, J, S) in ((1, 1, 1), (2, 5, 7), (4, 24, 56)):
        hm = _c(rng.normal(0, 0.3, (B, J, S, S)))
        kps = _c(np.concatenate([rng.uniform(-1.2, 1.2, (B, J, 2)), rng.choice([0, 0.5, 1, 2], (B, J, 1))], axis=2))
        lr, cr, gr = opl.stn_kps_losses(hm, kps, weight=0.8)
        L, cen, gh = np.zeros(1, np.float32), np.zeros((B, J, 2), np.float32), np.full_like(hm, 7)
        assert hostlib.danet_test_stn_kps_losses_host(B, J, S, _P(hm), _P(kps), 0.8, _P(L), _P(cen), _P(gh)) == 0
        np.testing.assert_allclose(L[0], lr, rtol=5e-6, atol=1e-7)
        np.testing.assert_allclose(cen, cr, atol=2e-6)
        np.testing.assert_allclose(gh, gr, atol=3e-6 * max(1.0, np.abs(gr).max()))


def test_point_losses_refuse_cpu_tensors():
    import torch
    from danet_b200 import losses
    z = torch.zeros
    with pytest.raises(RuntimeError):
        losses.dp_uvia_losses(z(1, 25, 4, 4), z(1, 25, 4, 4), z(1, 25, 4, 4), z(1, 15, 4, 4), z(1, 2), z(1, 2), z(1, 2),
                              z(1, 2), z(1, 50), z(1, 50), z(1, 50), z(1, 16), z(1, 16))
    with pytest.raises(RuntimeError):
        losses.stn_kps_losses(z(1, 24, 4, 4), z(1, 24, 3))
