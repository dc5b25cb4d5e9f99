"""GPU checks of the pointnet2_cls_bga training engine: the feature-propagation kernels (psa_fp_conv1_prebn / psa_fp_conv1_bwd),
the joint loss (psa_cls_seg_xent) and PointNet2BgaTrainer against the float64 restatement oracle/train_bga_oracle.py, the autograd
assembly pointnet2_cls_bga._get_model_training, and over two NCCL ranks."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import train_bga_oracle as BO
from oracle import train_model_oracle as M
from scanobjectnn_b200 import _lib
from scanobjectnn_b200 import pointnet2_cls_bga as bga
from scanobjectnn_b200._lib import PsaGradIn
from scanobjectnn_b200.synthetic import make_clouds
from scanobjectnn_b200.training import BGA_FP, LevelSpec, PointNet2BgaTrainer, _plain_grad

from . import gpu_util as G

pytestmark = pytest.mark.gpu
GTOL = 1e-4


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _vp(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _rel(got, want):
    return float(np.abs(np.asarray(got, np.float64) - want).max() / max(1e-30, np.abs(want).max()))


def _ws(nbytes):
    return torch.empty(nbytes // 4 + 64, device="cuda")


# (b, n unknown, m known, C1, interpolated channels, skip channels): m = 1, m < 3, m above the 2048-point tile, n not a multiple of
# the CTA, no skip, and the three FP fronts of pointnet2_cls_bga at B=32, N=2048
FP_SHAPES = [(2, 300, 1, 256, 256, 256), (3, 200, 2, 128, 64, 0), (1, 130, 2500, 128, 32, 16), (2, 77, 5, 128, 16, 8),
             (32, 128, 1, 256, 256, 256), (32, 512, 128, 256, 256, 128), (32, 2048, 512, 128, 128, 0)]


@pytest.mark.parametrize("b,n,m,c1,c_a,c_s", FP_SHAPES)
def test_fp_conv1_prebn_matches_float64_interpolate_concat_conv(b, n, m, c1, c_a, c_s):
    lib = _lib.load()
    rng = np.random.default_rng(n + m)
    xyz1 = rng.random((b, n, 3)).astype(np.float32)
    xyz2 = np.zeros((b, 1, 3), np.float32) if m == 1 else rng.random((b, m, 3)).astype(np.float32)
    P2 = rng.standard_normal((b, m, c_a)).astype(np.float32)
    skip = rng.standard_normal((b, n, c_s)).astype(np.float32)
    W = (rng.standard_normal((c_a + c_s, c1)) / np.sqrt(c_a + c_s)).astype(np.float32)
    bias = (rng.standard_normal(c1) * 0.1).astype(np.float32)
    W64 = W.astype(np.float64)
    U = G.cu((P2.astype(np.float64) @ W64[:c_a]).astype(np.float32).reshape(b * m, c1))
    x1, x2, bd = G.cu(xyz1), G.cu(xyz2), G.cu(bias)
    idx = torch.empty((b, n, 3), dtype=torch.int32, device="cuda")
    w = torch.empty((b, n, 3), device="cuda")
    stats = torch.empty((2, c1), device="cuda")
    need = lib.psa_fp_conv1_prebn_workspace_bytes(b, n, c1)
    ws = _ws(need)
    pre0 = (skip.astype(np.float64) @ W64[c_a:] + bias).astype(np.float32).reshape(b * n, c1) if c_s else None

    def run():
        pre = G.cu(pre0) if c_s else torch.empty((b * n, c1), device="cuda")
        assert lib.psa_fp_conv1_prebn(b, n, m, c1, _vp(x1), _vp(x2), _vp(U), _vp(bd), 1 if c_s else 0, _vp(pre), _vp(idx), _vp(w),
                                      _vp(stats), _vp(ws), C.c_size_t(need), _st()) == 0
        return pre, stats.clone()

    pre, st = run()
    # idx / weight bit-identical to the inference interpolation
    P2d = G.cu(P2)
    out_r = torch.empty((b, n, c_a), device="cuda")
    idx_r = torch.empty_like(idx)
    w_r = torch.empty_like(w)
    assert lib.psa_three_nn_interpolate(b, n, m, c_a, _vp(x1), _vp(x2), _vp(P2d), _vp(out_r), None, _vp(idx_r), _vp(w_r), _st()) == 0
    assert torch.equal(idx, idx_r) and torch.equal(w, w_r)
    # float64 [interp, skip] . W + b with the same idx / weight
    ii, ww = G.npy(idx).astype(np.int64), G.npy(w).astype(np.float64)
    interp = BO.interpolate_fwd(P2.astype(np.float64), ii, ww)
    x = np.concatenate([interp, skip.astype(np.float64)], axis=-1) if c_s else interp
    want = (x @ W64 + bias).reshape(b * n, c1)
    G.contract_close(G.npy(pre), want, f"fp_conv1_prebn b={b} n={n} m={m}")
    y = G.npy(pre).astype(np.float64)
    assert _rel(G.npy(st)[0], y.sum(0)) < 2e-5 and _rel(G.npy(st)[1], (y * y).sum(0)) < 2e-5
    pre2, st2 = run()
    assert torch.equal(pre, pre2) and torch.equal(st, st2), "fp_conv1_prebn must be bit-reproducible"


@pytest.mark.parametrize("b,n,m,c1", [(2, 300, 1, 256), (3, 200, 2, 128), (2, 513, 129, 256), (4, 2048, 512, 128)])
def test_fp_conv1_bwd_is_ordered_three_interpolate_grad(b, n, m, c1):
    lib = _lib.load()
    rng = np.random.default_rng(m)
    xyz1 = G.cu(rng.random((b, n, 3)).astype(np.float32))
    xyz2 = G.cu(rng.random((b, m, 3)).astype(np.float32))
    idx = torch.empty((b, n, 3), dtype=torch.int32, device="cuda")
    w = torch.empty((b, n, 3), device="cuda")
    dist = torch.empty_like(w)
    assert lib.psa_three_nn_interpolate(b, n, m, 0, _vp(xyz1), _vp(xyz2), None, None, _vp(dist), _vp(idx), _vp(w), _st()) == 0
    dh = G.cu(rng.standard_normal((b * n, c1)).astype(np.float32))
    need = max(lib.psa_fp_conv1_bwd_workspace_bytes(b, n, m), lib.psa_scatter_workspace_bytes(b, m, 3 * n))
    ws = _ws(need)
    dU = torch.empty((b * m, c1), device="cuda")
    g = _plain_grad(dh)
    assert lib.psa_fp_conv1_bwd(b, n, m, c1, _vp(idx), _vp(w), C.byref(g), _vp(dU), _vp(ws), C.c_size_t(need), _st()) == 0
    ref = torch.empty_like(dU)
    assert lib.psa_three_interpolate_grad(b, n, c1, m, _vp(dh), _vp(idx), _vp(w), _vp(ref), _vp(ws), C.c_size_t(need), _st()) == 0
    assert torch.equal(dU, ref), "plain-gradient fp_conv1_bwd must be bit-identical to psa_three_interpolate_grad"
    # with batch-norm backward coefficients evaluated on load
    y = rng.standard_normal((b * n, c1)).astype(np.float32)
    s, t = rng.uniform(0.5, 1.5, c1).astype(np.float32), (rng.standard_normal(c1) * 0.3).astype(np.float32)
    ca, cb, cc = rng.uniform(0.5, 1.5, c1).astype(np.float32), (rng.standard_normal(c1) * 0.01).astype(np.float32), (rng.standard_normal(c1) * 0.01).astype(np.float32)
    yd, sd, td, cad, cbd, ccd = map(G.cu, (y, s, t, ca, cb, cc))
    gb = PsaGradIn()
    gb.y = yd.data_ptr(); gb.ld = c1; gb.s = sd.data_ptr(); gb.t = td.data_ptr(); gb.relu = 1
    gb.ca = cad.data_ptr(); gb.cb = cbd.data_ptr(); gb.cc = ccd.data_ptr(); gb.dh = dh.data_ptr(); gb.ld_dh = c1; gb.mask = None
    gb.dp = None; gb.pv = None; gb.argk = None; gb.pool_k = 1; gb.C = c1; gb.mode = 0
    assert lib.psa_fp_conv1_bwd(b, n, m, c1, _vp(idx), _vp(w), C.byref(gb), _vp(dU), _vp(ws), C.c_size_t(need), _st()) == 0
    y64 = y.astype(np.float64)
    dz = G.npy(dh).astype(np.float64) * ((y64 * s + t) > 0)
    dy0 = ca * dz + cb * y64 + cc
    want = BO.interpolate_bwd(dy0.reshape(b, n, c1), G.npy(idx).astype(np.int64), G.npy(w).astype(np.float64), m).reshape(b * m, c1)
    assert _rel(G.npy(dU), want) < GTOL


@pytest.mark.parametrize("b,n,w", [(4, 1024, 0.5), (32, 2048, 0.3), (3, 17, 1.0)])
def test_cls_seg_xent_matches_float64_and_get_loss(b, n, w):
    lib = _lib.load()
    rng = np.random.default_rng(n)
    cls = (rng.standard_normal((b, 15)) * 3).astype(np.float32)
    seg = (rng.standard_normal((b, n, 2)) * 2).astype(np.float32)
    labels = rng.integers(0, 15, b).astype(np.int32)
    mask = (rng.random((b, n)) > 0.4).astype(np.int32)
    cd, sd, ld, md = G.cu(cls), G.cu(seg), G.cu(labels), G.cu(mask)
    loss = torch.empty(3, device="cuda")
    dcls, dseg = torch.empty_like(cd), torch.empty_like(sd)
    need = lib.psa_cls_seg_xent_workspace_bytes(b, n)
    ws = _ws(need)
    assert lib.psa_cls_seg_xent(b, 15, n, _vp(cd), _vp(ld), _vp(sd), _vp(md), C.c_float(w), _vp(loss), _vp(dcls), _vp(dseg), _vp(ws),
                                C.c_size_t(need), _st()) == 0
    lc, gc = BO._xent(cls.astype(np.float64), labels)
    ls, gs = BO._xent(seg.astype(np.float64).reshape(-1, 2), mask.reshape(-1))
    want = np.array([(1 - w) * lc + w * ls, lc, ls])
    assert np.abs(G.npy(loss) - want).max() < 1e-6 * max(1.0, np.abs(want).max())
    assert _rel(G.npy(dcls), (1 - w) * gc) < 1e-6 if w < 1 else np.abs(G.npy(dcls)).max() == 0.0
    assert _rel(G.npy(dseg).reshape(-1, 2), w * gs) < 1e-6
    tl = bga.get_loss(cd.double(), sd.double(), ld, md, seg_weight=w)
    assert np.abs(G.npy(loss) - np.array([float(v) for v in tl])).max() < 1e-6 * max(1.0, np.abs(want).max())
    loss2 = torch.empty(3, device="cuda")
    assert lib.psa_cls_seg_xent(b, 15, n, _vp(cd), _vp(ld), _vp(sd), _vp(md), C.c_float(w), _vp(loss2), _vp(dcls), _vp(dseg), _vp(ws),
                                C.c_size_t(need), _st()) == 0
    assert torch.equal(loss, loss2)


SMALL_LEVELS = [LevelSpec("layer1", 64, 0.3, 16, [64, 64, 128]), LevelSpec("layer2", 16, 0.6, 16, [128, 128, 256]),
                LevelSpec("layer3", None, None, None, [256, 512, 1024], group_all=True)]


def _np_params(p):
    return {k: v.detach().cpu().numpy().astype(np.float64) for k, v in p.items()}


def _mask_by_plane(xyz):
    return (xyz[..., 2] > 0).astype(np.int32)


def _bga_layers(tr):
    """scope -> _Layer of every layer of a PointNet2BgaTrainer, in BACKWARD order (the order the gradients are computed in)"""
    order = list(reversed(tr.seg))
    for f in reversed(tr.fps):
        order += list(reversed(f.layers))
    order += list(reversed(tr.head))
    for lv in reversed(tr.levels):
        order += list(reversed(lv.layers))
    return {ly.scope: ly for ly in order}


def _relu_decisions(ly):
    """the relu decisions the kernels take on load, fmaf(y, scale, shift) > 0 (its sign is that of the exact value, as here)"""
    return (ly.y.double() * ly.scale.double() + ly.shift.double() > 0).cpu().numpy()


def test_bga_training_step_matches_float64_restatement():
    """whole BGA step at a small shape with the dp1 / dp2 / seg_dp1 masks drawn: both logit tensors, the three losses, every gradient,
    moving averages, one Adam step against oracle/train_bga_oracle.py.  The oracle takes the kernels' relu decisions for the layers it
    evaluates itself (group-all level, FC head, FP modules, seg head): a z within rounding of 0 may come out positive in fp32 and not in
    fp64, which would route that row's gradient differently; the test checks every overridden decision is such a rounding-level z."""
    B, N = 8, 256
    p = bga.init_params(seed=3, randomize_bn=True)
    tr = PointNet2BgaTrainer(p, B, N, 15, levels=SMALL_LEVELS)
    xyz = make_clouds("ball", B, N, seed=11)
    labels = np.random.default_rng(0).integers(0, 15, B).astype(np.int32)
    mask = _mask_by_plane(xyz)
    before = _np_params(p)
    tr.draw_dropout()
    masks = {ly.scope: G.npy(ly.mask).astype(np.float64) for ly, _ in tr._masked()}
    assert sorted(masks) == ["fc1", "fc2", "seg_fc1"] and all(0.3 < (m > 0).mean() < 0.7 for m in masks.values())
    masks["seg_fc1"] = masks["seg_fc1"].reshape(B, N, -1)
    cls, seg = tr.forward(G.cu(xyz), bn_decay=0.7)
    loss, dcls, dseg = tr.loss_and_grad(cls, seg, G.cu(labels), G.cu(mask), seg_weight=0.5)
    tr.backward(dcls, dseg)
    torch.cuda.synchronize()
    levels = [(s.scope, s.npoint, s.radius, s.nsample, s.mlp, s.group_all) for s in SMALL_LEVELS]
    relu = {sc: _relu_decisions(ly) for sc, ly in _bga_layers(tr).items() if ly.bn and not sc.startswith(("layer1/", "layer2/"))}
    want = BO.bga_train_step(xyz, labels, mask, before, levels, [f.mlp for f in BGA_FP], masks, 15, seg_weight=0.5, relu=relu)
    print("relu decisions taken from the kernels (count, max |z|):", {k: v for k, v in want["relu_forced"].items() if v[0]})
    assert all(zmax < 1e-4 for _, zmax in want["relu_forced"].values()), want["relu_forced"]
    for lv, oidx in zip(tr.levels[:2], want["idx"]):
        assert np.array_equal(G.npy(lv.idx), oidx)
    for f, (oidx, ow) in zip(tr.fps, want["fp_idx"]):
        assert np.array_equal(G.npy(f.idx), oidx) and np.array_equal(G.npy(f.weight).astype(np.float64), ow)
    assert np.abs(G.npy(cls) - want["class_logits"]).max() < 1e-4 * max(1.0, np.abs(want["class_logits"]).max())
    assert np.abs(G.npy(seg) - want["seg_logits"]).max() < 1e-4 * max(1.0, np.abs(want["seg_logits"]).max())
    assert np.abs(G.npy(loss) - np.array(want["loss"])).max() < 1e-5 * max(1.0, abs(want["loss"][0]))
    worst = {}
    for name, gw in want["grads"].items():
        got = G.npy(tr.fp.grad_of(name)).reshape(gw.shape).astype(np.float64)
        if name.endswith("/biases") and f"{name[:-7]}/bn/gamma" in before:
            assert np.abs(got).max() == 0.0 and np.abs(gw).max() < 1e-9, name
            continue
        if np.abs(gw).max() < 1e-9:
            assert np.abs(got).max() < 1e-5, (name, np.abs(got).max())
            continue
        worst[name] = _rel(got, gw)
    assert len(worst) >= 60
    bad = {k: v for k, v in worst.items() if v > GTOL}
    print("max relative gradient error:", max(worst.values()), "over", len(worst), "tensors")
    assert not bad, bad
    for scope, (mean, var) in want["batch_stats"].items():
        np.testing.assert_allclose(G.npy(p[f"{scope}/bn/moving_mean"]), 0.7 * before[f"{scope}/bn/moving_mean"] + 0.3 * mean, rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(G.npy(p[f"{scope}/bn/moving_variance"]), 0.7 * before[f"{scope}/bn/moving_variance"] + 0.3 * var, rtol=2e-4,
                                   atol=1e-6)
    g_before = {k: G.npy(tr.fp.grad_of(k)).astype(np.float64) for k in want["grads"]}
    tr.adam(1e-3)
    for name in ("layer1/conv1/weights", "fa_layer1/conv_0/weights", "fa_layer3/conv_2/bn/gamma", "seg_fc2/biases", "fc3/weights"):
        pw, _, _ = M.adam_update(before[name], g_before[name].reshape(before[name].shape), 0.0, 0.0, 1, 1e-3)
        np.testing.assert_allclose(G.npy(p[name]).astype(np.float64), pw, rtol=1e-6, atol=1e-7)


def test_bga_dropout_masks_in_the_seg_head_backward():
    """seg_dp1 (and the dp1 / dp2 masks) drawn: the seg head's backward against float64 recomputed from the trainer's own stored
    activations -- the input gradient of seg_fc2, the batch-norm sums and the weight / input gradients of seg_fc1."""
    B, N = 8, 256
    p = bga.init_params(seed=3, randomize_bn=True)
    tr = PointNet2BgaTrainer(p, B, N, 15, levels=SMALL_LEVELS)
    xyz = make_clouds("ball", B, N, seed=11)
    tr.draw_dropout()
    assert all(0.3 < float((ly.mask > 0).float().mean()) < 0.7 for ly, _ in tr._masked())
    cls, seg = tr.forward(G.cu(xyz), 0.7)
    _, dcls, dseg = tr.loss_and_grad(cls, seg, G.cu(np.arange(B, dtype=np.int32)), G.cu(_mask_by_plane(xyz)))
    tr.backward(dcls, dseg)
    torch.cuda.synchronize()
    s1, s2 = tr.seg
    d = lambda t: t.double()  # noqa: E731
    seg_dh = d(dseg.reshape(-1, 2)) @ d(s2.W).T
    assert _rel(G.npy(tr.seg_dh), G.npy(seg_dh)) < 1e-6
    y = d(s1.y)
    mean, var = y.mean(0), y.var(0, unbiased=False)
    inv = 1 / torch.sqrt(var + 1e-3)
    xhat = (y - mean) * inv
    dz = seg_dh * d(s1.mask) * ((xhat * d(s1.gamma) + d(s1.beta)) > 0).double()
    assert _rel(G.npy(s1.dbeta), G.npy(dz.sum(0))) < 1e-5 and _rel(G.npy(s1.dgamma), G.npy((dz * xhat).sum(0))) < 1e-5
    R = y.shape[0]
    dy = d(s1.gamma) * inv / R * (R * dz - dz.sum(0) - xhat * (dz * xhat).sum(0))
    f3 = tr.fps[2].layers[-1]
    h = torch.relu(d(f3.y) * d(f3.scale) + d(f3.shift))
    assert _rel(G.npy(s1.dW), G.npy(h.T @ dy)) < 1e-5 and _rel(G.npy(tr.fp_dout), G.npy(dy @ d(s1.W).T)) < 1e-5


def test_bga_training_step_is_bit_reproducible_and_learns():
    B, N = 8, 256
    xyz_np = np.concatenate([make_clouds("ball", B // 2, N, seed=2), make_clouds("shell", B // 2, N, seed=3)])
    xyz = G.cu(xyz_np)
    labels = G.cu((np.arange(B) >= B // 2).astype(np.int32))
    mask = G.cu(_mask_by_plane(xyz_np))
    grads = []
    for _ in range(2):
        p = bga.init_params(seed=5)
        tr = PointNet2BgaTrainer(p, B, N, 15, levels=SMALL_LEVELS)
        tr._gen.manual_seed(7)
        tr.draw_dropout()
        cls, seg = tr.forward(xyz, 0.5)
        _, dcls, dseg = tr.loss_and_grad(cls, seg, labels, mask)
        tr.backward(dcls, dseg)
        grads.append(tr.fp.grad.clone())
    assert torch.equal(grads[0], grads[1]), "two runs of the same step must give bit-identical gradients"
    losses = [float(tr.train_step(xyz, labels, mask, lr=2e-3, bn_decay=0.5)[0].item()) for _ in range(30)]
    print("loss", losses[0], "->", losses[-1])
    assert losses[-1] < 0.5 * losses[0]


def test_bga_trainer_matches_autograd_path_at_real_hyper_parameters():
    """PointNet2BgaTrainer against pointnet2_cls_bga._get_model_training + get_loss + backward (dropout off), same seed, B=4, N=1024"""
    B, N = 4, 1024
    xyz = G.cu(make_clouds("ball", B, N, seed=8))
    labels = G.cu(np.array([1, 4, 7, 11], dtype=np.int32))
    mask = G.cu((np.random.default_rng(0).random((B, N)) > 0.5).astype(np.int32))
    pa = bga.init_params(seed=3)
    cp, sp = bga._get_model_training(xyz, 0.5, 15, pa, False, dropout=False)
    la = bga.get_loss(cp, sp, labels, mask)
    la[0].backward()
    ga = pa._flat
    pt = bga.init_params(seed=3)
    tr = PointNet2BgaTrainer(pt, B, N, 15)
    for ly, _ in tr._masked():
        ly.mask.fill_(1.0)
    cls, seg = tr.forward(xyz, 0.5)
    loss, dcls, dseg = tr.loss_and_grad(cls, seg, labels, mask)
    tr.backward(dcls, dseg)
    torch.cuda.synchronize()
    assert _rel(G.npy(cls), G.npy(cp).astype(np.float64)) < 1e-4 and _rel(G.npy(seg), G.npy(sp).astype(np.float64)) < 1e-4
    assert np.abs(G.npy(loss) - np.array([float(v) for v in la])).max() < 1e-5
    # the two paths round the FP modules' first conv differently (interpolate + concat + GEMM vs U = P2 . W1[:C_a] interpolated), so a
    # relu decision at |z| ~ 1e-7 can differ between them and reroute one row of a ~4096-row sum.  Such a flip changes the gradients
    # computed from that layer on (backward order); the ones computed before it, and fc3's (its input and dlogits come from the forward
    # alone), keep the 1e-4 bound.
    mine = _bga_layers(tr)
    theirs = {}
    for mt in pa.__dict__["_trainers"].values():
        for ly in getattr(mt, "layers", []):
            theirs[ly.scope] = ly
        for lv in getattr(mt, "levels", []):
            for ly in lv.layers:
                theirs[ly.scope] = ly
    order = list(mine)
    flips = {sc: int((_relu_decisions(mine[sc]) != _relu_decisions(theirs[sc])).sum()) for sc in order if mine[sc].bn}
    print("relu decisions that differ between the two paths:", {k: v for k, v in flips.items() if v})
    first = min((order.index(sc) for sc, v in flips.items() if v), default=len(order))
    loose = {sc for sc in order[first:] if sc != "fc3"}
    worst, checked = 0.0, 0
    for name in tr.fp.names:
        want = G.npy(ga.flat.grad[(ga.views[name].data_ptr() - ga.flat.data_ptr()) // 4:][:ga.views[name].numel()]).astype(np.float64)
        got = G.npy(tr.fp.grad_of(name)).reshape(-1).astype(np.float64)
        if name.endswith("/biases") and f"{name[:-7]}/bn/gamma" in tr.fp.views:
            assert np.abs(got).max() == 0.0 and np.abs(want).max() < 1e-5, name
            continue
        if np.abs(want).max() < 1e-7:
            assert np.abs(got).max() < 1e-5, name
            continue
        r = _rel(got, want)
        assert r < (2e-2 if name.rsplit("/", 2 if "/bn/" in name else 1)[0] in loose else GTOL), (name, r, flips)
        worst, checked = max(worst, r), checked + 1
    print("trainer vs autograd: max relative gradient difference", worst, "over", checked, "tensors")


def test_bga_full_size_step_is_finite():
    B, N = 32, 2048
    torch.cuda.reset_peak_memory_stats()
    p = bga.init_params(seed=1)
    tr = PointNet2BgaTrainer(p, B, N, 15)
    xyz_np = make_clouds("ball", B, N, seed=9)
    loss = tr.train_step(G.cu(xyz_np), G.cu((np.arange(B) % 15).astype(np.int32)), G.cu(_mask_by_plane(xyz_np)), lr=1e-3)
    torch.cuda.synchronize()
    assert torch.isfinite(loss).all() and torch.isfinite(tr.fp.grad).all() and torch.isfinite(tr.fp.flat).all()
    print(f"B={B} N={N}: loss {G.npy(loss)}, peak memory {torch.cuda.max_memory_allocated() / 2**20:.0f} MiB")


# ---- two ranks over NCCL ----
B_LOCAL, N_MP, STEPS = 4, 512, 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _data(rank):
    xyz = make_clouds("ball", B_LOCAL, N_MP, seed=500 + rank)
    return xyz, ((np.arange(B_LOCAL) * 3 + rank) % 15).astype(np.int32), _mask_by_plane(xyz)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    tr = PointNet2BgaTrainer(bga.init_params(seed=11, device=dev), B_LOCAL, N_MP, device=dev)
    assert tr.world == world
    xyz, labels, mask = (torch.from_numpy(a).to(dev) for a in _data(rank))
    out = []
    for _ in range(STEPS):
        cls, seg = tr.forward(xyz, 0.5)
        loss, dcls, dseg = tr.loss_and_grad(cls, seg, labels, mask)
        tr.backward(dcls, dseg)
        local = tr.fp.grad.clone()
        tr.allreduce_grads()
        reduced = tr.fp.grad.clone()
        tr.adam(1e-3)
        out.append((local.cpu().numpy(), reduced.cpu().numpy(), tr.fp.flat.detach().cpu().numpy().copy(), G.npy(loss)))
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, out))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_bga_two_rank_gradient_allreduce_and_identical_parameters():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    res = dict(q.get(timeout=600) for _ in range(world))
    for pr in procs:
        pr.join(timeout=120)
        assert pr.exitcode == 0
    for s in range(STEPS):
        l0, r0, p0, loss0 = res[0][s]
        l1, r1, p1, loss1 = res[1][s]
        assert np.array_equal(r0, r1), "ranks disagree on the reduced gradient"
        assert np.array_equal(r0, l0 + l1), "all-reduce is not the plain sum of the two local buckets"
        assert np.array_equal(p0, p1), "parameters diverged between the ranks"
        assert np.isfinite(loss0).all() and np.isfinite(loss1).all()
