"""The float64 restatement of one pointnet2_cls_bga training step (oracle/train_bga_oracle.py) against central finite differences,
and the argument checks of the FP-module / joint-loss entry points (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

from oracle import train_bga_oracle as BO
from scanobjectnn_b200.synthetic import make_clouds

# small BGA-shaped model: SA2 keeps 2 points, so fa_layer1 has m = 1 (group-all centroid), fa_layer2 m = 2, fa_layer3 m = 8 (>= 3)
LEVELS = [("layer1", 8, 0.5, 6, [6, 8], False), ("layer2", 2, 0.9, 4, [8, 10], False), ("layer3", None, None, None, [12], True)]
FP_MLPS = [[8, 7], [6, 5], [5, 4]]
B, N, NC = 3, 32, 4


def _params(seed=0):
    rng = np.random.default_rng(seed)
    p = {}

    def add(scope, cin, cout, bn=True):
        p[f"{scope}/weights"] = rng.standard_normal((cin, cout)) * (1.0 / np.sqrt(cin))
        p[f"{scope}/biases"] = rng.standard_normal(cout) * 0.1
        if bn:
            p[f"{scope}/bn/gamma"] = rng.uniform(0.5, 1.5, cout)
            p[f"{scope}/bn/beta"] = rng.standard_normal(cout) * 0.1

    c = 0
    for scope, _, _, _, mlp, _ in LEVELS:
        cin = 3 + c
        for i, w in enumerate(mlp):
            add(f"{scope}/conv{i}", cin, w)
            cin = w
        c = mlp[-1]
    add("fc1", c, 9)
    add("fc2", 9, 6)
    add("fc3", 6, NC, bn=False)
    c_a = 6
    for scope, mlp, c_s in zip(BO.FP_MODULES, FP_MLPS, (LEVELS[1][4][-1], LEVELS[0][4][-1], 0)):
        cin = c_a + c_s
        for i, w in enumerate(mlp):
            add(f"{scope}/conv_{i}", cin, w)
            cin = w
        c_a = mlp[-1]
    add("seg_fc1", c_a, 5)
    add("seg_fc2", 5, 2, bn=False)
    return p


def _inputs():
    xyz = make_clouds("ball", B, N, seed=21)
    rng = np.random.default_rng(3)
    labels = rng.integers(0, NC, B)
    mask = (rng.random((B, N)) > 0.5).astype(np.int64)
    masks = {s: (rng.random(shape) < 0.5) * 2.0 for s, shape in (("fc1", (B, 9)), ("fc2", (B, 6)), ("seg_fc1", (B, N, 5)))}
    return xyz, labels, mask, masks


def test_bga_oracle_gradients_match_finite_differences():
    p = _params()
    xyz, labels, mask, masks = _inputs()
    out = BO.bga_train_step(xyz, labels, mask, p, LEVELS, FP_MLPS, masks, NC, seg_weight=0.3)
    # FP modules with m = 1, 2 and >= 3 known points
    assert [w.shape[1] for _, w in out["fp_idx"]] == [2, 8, N]
    idx1, w1 = out["fp_idx"][0]
    assert np.all(idx1 == 0) and np.all(w1[..., 0] == 1.0) and np.all(w1[..., 1:] == 0.0)
    idx2, w2 = out["fp_idx"][1]
    assert np.all(w2[..., 2] == 0.0) and np.allclose(w2.sum(-1), 1.0)
    total, cls, seg = out["loss"]
    assert abs(total - (0.7 * cls + 0.3 * seg)) < 1e-12

    def loss_of(q):
        return BO.bga_train_step(xyz, labels, mask, q, LEVELS, FP_MLPS, masks, NC, seg_weight=0.3)["loss"][0]

    rng = np.random.default_rng(7)
    eps = 1e-6
    checked = 0
    for name, g in out["grads"].items():
        for _ in range(2):
            pick = tuple(int(rng.integers(0, s)) for s in g.shape)
            q = {k: v.copy() for k, v in p.items()}
            q[name][pick] += eps
            lp = loss_of(q)
            q[name][pick] -= 2 * eps
            lm = loss_of(q)
            fd = (lp - lm) / (2 * eps)
            assert abs(fd - g[pick]) < 1e-6 + 1e-4 * abs(g[pick]), (name, pick, fd, g[pick])
            checked += 1
    assert checked == 2 * len(p)
    # every FP layer, the seg head and both skip fan-ins received gradient
    for name in ("fa_layer1/conv_0/weights", "fa_layer2/conv_0/weights", "fa_layer3/conv_0/weights", "seg_fc2/weights", "fc3/weights"):
        assert np.abs(out["grads"][name]).max() > 0, name
    # biases under batch norm: zero up to rounding
    for name, g in out["grads"].items():
        if name.endswith("/biases") and f"{name[:-7]}/bn/gamma" in p:
            assert np.abs(g).max() < 1e-9, name


def test_bga_oracle_joint_loss_gradient_is_the_mixture():
    """seg_weight 0 and 1 pick one loss each: the classification head gets no gradient from the seg loss and vice versa"""
    p = _params(1)
    xyz, labels, mask, masks = _inputs()
    only_cls = BO.bga_train_step(xyz, labels, mask, p, LEVELS, FP_MLPS, masks, NC, seg_weight=0.0)
    only_seg = BO.bga_train_step(xyz, labels, mask, p, LEVELS, FP_MLPS, masks, NC, seg_weight=1.0)
    assert np.abs(only_cls["grads"]["seg_fc2/weights"]).max() == 0.0
    assert np.abs(only_seg["grads"]["fc3/weights"]).max() == 0.0
    assert only_cls["loss"][0] == only_cls["loss"][1] and only_seg["loss"][0] == only_seg["loss"][2]


def test_fp_and_loss_entries_reject_bad_arguments_without_a_gpu():
    from scanobjectnn_b200 import _lib
    lib = _lib.load()
    null = C.c_void_p(0)
    sz0 = C.c_size_t(0)
    for name in ("psa_fp_conv1_prebn", "psa_fp_conv1_bwd", "psa_cls_seg_xent"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)
    # C1 not a multiple of 4 / too wide, negative dims, no known points, null buffers
    assert lib.psa_fp_conv1_prebn(2, 16, 4, 130, null, null, null, null, 0, null, null, null, null, null, sz0, null) == -1
    assert lib.psa_fp_conv1_prebn(2, 16, 4, 1024, null, null, null, null, 0, null, null, null, null, null, sz0, null) == -1
    assert lib.psa_fp_conv1_prebn(-1, 16, 4, 128, null, null, null, null, 0, null, null, null, null, null, sz0, null) == -1
    assert lib.psa_fp_conv1_prebn(2, 16, 0, 128, null, null, null, null, 0, null, null, null, null, null, sz0, null) == -1
    assert b"known point" in lib.psa_last_error()
    assert lib.psa_fp_conv1_prebn(2, 16, 4, 128, null, null, null, null, 0, null, null, null, null, null, sz0, null) == -1
    assert lib.psa_fp_conv1_prebn(0, 16, 4, 128, null, null, null, null, 0, null, null, null, null, null, sz0, null) == 0   # b = 0: no-op
    assert lib.psa_fp_conv1_bwd(2, 16, 4, 126, null, null, None, null, null, sz0, null) == -1
    assert lib.psa_fp_conv1_bwd(2, 16, 4, 128, null, null, None, null, null, sz0, null) == -1
    # a misaligned gradient buffer is an argument error, caught before any launch (fake device addresses: nothing is dereferenced)
    from scanobjectnn_b200.training import _plain_grad

    class _Fake:
        def __init__(self, addr):
            self.addr, self.shape = addr, (16, 128)

        def data_ptr(self):
            return self.addr

    fake = C.c_void_p(0x10000)
    g = _plain_grad(_Fake(0x20004))
    assert lib.psa_fp_conv1_bwd(2, 16, 4, 128, fake, fake, C.byref(g), fake, fake, C.c_size_t(1 << 20), null) == -1
    assert b"16-byte aligned" in lib.psa_last_error()
    g = _plain_grad(_Fake(0x20000))
    g.ca = 0x30000                                 # coefficients without y / cb / cc
    assert lib.psa_fp_conv1_bwd(2, 16, 4, 128, fake, fake, C.byref(g), fake, fake, C.c_size_t(1 << 20), null) == -1
    assert lib.psa_cls_seg_xent(0, 15, 16, null, null, null, null, C.c_float(0.5), null, null, null, null, sz0, null) == -1
    assert lib.psa_cls_seg_xent(2, 15, 16, null, null, null, null, C.c_float(0.5), null, null, null, null, sz0, null) == -1
    assert lib.psa_fp_conv1_prebn_workspace_bytes(32, 2048, 128) >= 32 * 16 * 2 * 128 * 4
    assert lib.psa_fp_conv1_bwd_workspace_bytes(32, 2048, 512) >= (32 * 513 + 32 * 3 * 2048) * 4
    assert lib.psa_cls_seg_xent_workspace_bytes(32, 2048) >= 8


def test_bga_trainer_hyper_parameters():
    from scanobjectnn_b200.training import BGA_FP, BGA_LEVELS, BGA_SEG_HEAD
    assert [(s.npoint, s.radius, s.nsample, s.mlp, s.group_all) for s in BGA_LEVELS] == [
        (512, 0.2, 64, [64, 64, 128], False), (128, 0.4, 64, [128, 128, 256], False), (None, None, None, [256, 512, 1024], True)]
    assert [(f.scope, f.mlp) for f in BGA_FP] == [("fa_layer1", [256, 256]), ("fa_layer2", [256, 128]), ("fa_layer3", [128, 128, 128])]
    assert BGA_SEG_HEAD == [("seg_fc1", 128, True, 0.5), ("seg_fc2", 2, False, None)]


@pytest.mark.parametrize("m", [1, 2, 5])
def test_interpolation_restatement_is_linear_with_scatter_adjoint(m):
    """<interpolate(P), D> == <P, interpolate_bwd(D)>: the backward is the exact adjoint of the forward for any m"""
    rng = np.random.default_rng(m)
    xyz1 = rng.standard_normal((2, 11, 3)).astype(np.float32)
    xyz2 = rng.standard_normal((2, m, 3)).astype(np.float32)
    idx, w = BO.fp_weights(xyz1, xyz2)
    P = rng.standard_normal((2, m, 4))
    D = rng.standard_normal((2, 11, 4))
    lhs = (BO.interpolate_fwd(P, idx, w) * D).sum()
    rhs = (P * BO.interpolate_bwd(D, idx, w, m)).sum()
    assert abs(lhs - rhs) < 1e-12 * max(1.0, abs(lhs))


def test_bga_oracle_relu_override_follows_the_given_decisions():
    """relu={scope: decisions}: an empty override changes nothing; overridden decisions are applied and reported with their largest |z|"""
    p = _params(2)
    xyz, labels, mask, masks = _inputs()
    base = BO.bga_train_step(xyz, labels, mask, p, LEVELS, FP_MLPS, masks, NC)
    assert base["relu_forced"] == {}
    own = BO.bga_train_step(xyz, labels, mask, p, LEVELS, FP_MLPS, masks, NC, relu={})
    assert own["relu_forced"] == {} and all(np.array_equal(own["grads"][k], g) for k, g in base["grads"].items())
    h2_scope = "fa_layer1/conv_1"
    probe = BO.bga_train_step(xyz, labels, mask, p, LEVELS, FP_MLPS, masks, NC, relu={h2_scope: np.ones((B, 2, FP_MLPS[0][1]), bool)})
    cnt, zmax = probe["relu_forced"][h2_scope]
    assert cnt > 0 and zmax > 0
    assert not np.array_equal(probe["grads"][f"{h2_scope}/bn/gamma"], base["grads"][f"{h2_scope}/bn/gamma"])
