"""Training step of pointnet2_cls_bga restated in float64 numpy (TEST INFRASTRUCTURE ONLY -- nothing in the product imports it).
Composes oracle/train_oracle.py's layer and set-abstraction level restatements and train_model_oracle.py's parameter reader / Adam
with the feature-propagation modules, the segmentation head and the joint loss.

PARITY UNPINNED like the rest of the floating-point half.  Restated call sites:
  pointnet2/models/pointnet2_cls_bga.py:21-75   levels (SA1 nsample 64), fc1/dp1/fc2, class_vector = fc2's output BEFORE dp2,
                                                dp2/fc3, fa_layer1..3, seg_fc1/seg_dp1/seg_fc2
  pointnet2/models/pointnet2_cls_bga.py:78-93   loss = (1-w) * mean CE(class) + w * mean over instances of mean per-point CE
  pointnet2/utils/pointnet_util.py:199-229      pointnet_fp_module: three_nn, dist = max(dist, 1e-10), inverse-distance weights,
                                                three_interpolate, concat [interpolated, points1], 1x1 convs + BN + relu
  3d_interpolation/tf_interpolate.cpp:60-153    three_nn / three_interpolate / ThreeInterpolateGrad (scatter-add of w * grad)
idx / weights come from oracle.three_nn + oracle.three_weights (bit-exact to the reference's CPU op); they carry no gradient.
Gradients are checked against central finite differences in tests/test_train_bga_oracle.py."""
from __future__ import annotations

import numpy as np

from . import oracle as orc
from . import train_oracle as T
from .train_model_oracle import _layer_params

FP_MODULES = ("fa_layer1", "fa_layer2", "fa_layer3")


def _xent(logits, labels):
    """mean softmax cross-entropy over the rows and d(mean)/d(logits)"""
    mx = logits.max(axis=1, keepdims=True)
    e = np.exp(logits - mx)
    rows = logits.shape[0]
    lab = np.asarray(labels).astype(np.int64)
    loss = float(np.mean(np.log(e.sum(axis=1)) + mx[:, 0] - logits[np.arange(rows), lab]))
    d = e / e.sum(axis=1, keepdims=True)
    d[np.arange(rows), lab] -= 1.0
    return loss, d / rows


def _mlp_fwd(h, layers, stats, scopes, relu=None, forced=None):
    """1x1 conv + batch-statistics BN + relu chain; -> output, caches.  relu {scope: bool array}: take these relu decisions instead of
    z > 0 (a float32 run's own decisions, so that a z within rounding of 0 cannot route its row differently); forced[scope] records
    (how many decisions were overridden, the largest |z| among them)."""
    caches = []
    for scope, (w, b, gamma, beta) in zip(scopes, layers):
        y, c_conv = T.conv1x1_fwd(h, w, b)
        z, c_bn, mean, var = T.bn_train_fwd(y, gamma, beta)
        h, mask = T.relu_fwd(z)
        if relu is not None and scope in relu:
            want = np.asarray(relu[scope], dtype=bool).reshape(z.shape)
            diff = want != mask
            forced[scope] = (int(diff.sum()), float(np.abs(z[diff]).max()) if diff.any() else 0.0)
            mask = want
            h = z * mask
        caches.append((c_conv, c_bn, mask))
        stats[scope] = (mean, var)
    return h, caches


def _mlp_bwd(dh, caches, scopes, grads):
    for scope, (c_conv, c_bn, mask) in zip(reversed(scopes), reversed(caches)):
        dy, dgamma, dbeta = T.bn_train_bwd(dh * mask, c_bn)
        dh, dw, db = T.conv1x1_bwd(dy, c_conv)
        grads[f"{scope}/weights"], grads[f"{scope}/biases"] = dw, db
        grads[f"{scope}/bn/gamma"], grads[f"{scope}/bn/beta"] = dgamma, dbeta
    return dh


def fp_weights(xyz1, xyz2):
    """three_nn + inverse-distance weights of pointnet_fp_module (float32 coordinates) -> idx (B,n,3) int64, weight (B,n,3) float64"""
    dist, idx = orc.three_nn(np.asarray(xyz1, np.float32), np.asarray(xyz2, np.float32))
    return idx.astype(np.int64), orc.three_weights(dist).astype(np.float64)


def interpolate_fwd(points2, idx, weight):
    """three_interpolate: points2 (B,m,C), idx / weight (B,n,3) -> (B,n,C)"""
    b = np.arange(points2.shape[0])[:, None, None]
    return (points2[b, idx] * weight[..., None]).sum(axis=2)


def interpolate_bwd(dout, idx, weight, m):
    """ThreeInterpolateGrad: scatter-add of w * dout into the known points (tf_interpolate.cpp:131-153)"""
    bsz, n, c = dout.shape
    d = np.zeros((bsz, m, c))
    for b in range(bsz):
        np.add.at(d[b], idx[b].reshape(-1), (dout[b][:, None, :] * weight[b][..., None]).reshape(-1, c))
    return d


def fp_module_fwd(idx, weight, points1, points2, layers, stats, scopes, relu=None, forced=None):
    """pointnet_fp_module(is_training=True) on fixed idx / weight -> (B,n,C_L), cache"""
    interp = interpolate_fwd(points2, idx, weight)
    h = interp if points1 is None else np.concatenate([interp, points1], axis=-1)
    out, caches = _mlp_fwd(h, layers, stats, scopes, relu, forced)
    return out, (caches, scopes, idx, weight, points2.shape, points2.shape[-1])


def fp_module_bwd(dout, cache, grads):
    """-> d points1 (or None), d points2"""
    caches, scopes, idx, weight, p2_shape, c_a = cache
    dh = _mlp_bwd(dout, caches, scopes, grads)
    dp1 = dh[..., c_a:] if dh.shape[-1] > c_a else None
    return dp1, interpolate_bwd(dh[..., :c_a], idx, weight, p2_shape[1])


def bga_train_step(xyz, labels, mask, params, levels, fp_mlps, masks, num_class, seg_weight=0.5, relu=None):
    """xyz (B,N,3) float32, labels (B,) int, mask (B,N) int in {0,1}, params {tf name: array}, levels = [(scope, npoint, radius,
    nsample, mlp, group_all)] x 3 (the last group_all), fp_mlps = [mlp of fa_layer1, fa_layer2, fa_layer3], masks = {"fc1", "fc2",
    "seg_fc1": dropout mask of 0 / 1/keep, or absent for none}, relu = {scope: relu decisions} for the layers outside the ball-query
    levels (group-all level, FC head, FP modules, seg head), or None.
    -> dict(class_logits, seg_logits, loss (total, classify, seg), grads {name: array}, batch_stats {scope: (mean, var)},
            idx [ball-query idx of SA1, SA2], fp_idx [(idx, weight) of fa_layer1..3], relu_forced {scope: (count, max |z|)})"""
    xyz32 = np.asarray(xyz, dtype=np.float32)
    B, N = xyz32.shape[:2]
    stats, grads, forced = {}, {}, {}
    # ---- set-abstraction levels ----
    cur_xyz32, cur_pts = xyz32, None
    sa, lxyz, lpts, idxs = [], [xyz32], [None], []
    for (scope, npoint, radius, nsample, mlp, group_all) in levels:
        layers = [_layer_params(params, f"{scope}/conv{i}") for i in range(len(mlp))]
        scopes = [f"{scope}/conv{i}" for i in range(len(mlp))]
        if group_all:
            # sample_and_group_all: one group of every point, rows [xyz, points] (new_xyz = 0, no centring)
            x = cur_xyz32.astype(np.float64)
            h = (x if cur_pts is None else np.concatenate([x, cur_pts], axis=-1))[:, None, :, :]
            h, lc = _mlp_fwd(h, layers, stats, scopes, relu, forced)
            pooled, c_pool = T.maxpool_fwd(h, axis=2)
            sa.append(("all", lc, c_pool, scopes, None if cur_pts is None else cur_pts.shape[-1]))
            new_xyz32 = np.zeros((B, 1, 3), dtype=np.float32)
        else:
            fps_idx = orc.fps(cur_xyz32, npoint)
            new_xyz32 = orc.gather_point(cur_xyz32, fps_idx)
            idx, _ = orc.query_ball_point(radius, nsample, cur_xyz32, new_xyz32, contract=True)
            pooled, cache, st = T.sa_level_train_fwd(cur_xyz32, cur_pts, fps_idx.astype(np.int64), idx.astype(np.int64), layers)
            for s, v in zip(scopes, st):
                stats[s] = v
            sa.append(("sa", cache, scopes))
            idxs.append(idx)
        cur_xyz32, cur_pts = new_xyz32, pooled
        lxyz.append(new_xyz32)
        lpts.append(pooled)
    # ---- classification head: fc1 -> dp1 -> fc2 (-> class_vector) -> dp2 -> fc3 ----
    feat = cur_pts.reshape(B, -1)
    fc = [_layer_params(params, s) for s in ("fc1", "fc2", "fc3")]
    ones = lambda s: masks.get(s, 1.0)  # noqa: E731
    h1, c1 = _mlp_fwd(feat, [fc[0]], stats, ["fc1"], relu, forced)
    h1d = h1 * ones("fc1")
    h2, c2 = _mlp_fwd(h1d, [fc[1]], stats, ["fc2"], relu, forced)
    h2d = h2 * ones("fc2")
    class_logits, c3 = T.conv1x1_fwd(h2d, fc[2][0], fc[2][1])
    # ---- feature propagation: (unknown xyz, known xyz, skip, source) ----
    fp_caches, fp_idx = [], []
    src = h2[:, None, :]                                           # class_vector (B,1,256), before dp2
    for k, scope in enumerate(FP_MODULES):
        xyz1, xyz2, skip = lxyz[2 - k], lxyz[3 - k], lpts[2 - k]
        scopes = [f"{scope}/conv_{i}" for i in range(len(fp_mlps[k]))]
        layers = [_layer_params(params, s) for s in scopes]
        idx, w = fp_weights(xyz1, xyz2)
        fp_idx.append((idx, w))
        src, cache = fp_module_fwd(idx, w, skip, src, layers, stats, scopes, relu, forced)
        fp_caches.append(cache)
    # ---- segmentation head: seg_fc1 -> seg_dp1 -> seg_fc2 ----
    f1, cs1 = _mlp_fwd(src, [_layer_params(params, "seg_fc1")], stats, ["seg_fc1"], relu, forced)
    f1d = f1 * ones("seg_fc1")
    w2, b2, _, _ = _layer_params(params, "seg_fc2")
    seg_logits, cs2 = T.conv1x1_fwd(f1d, w2, b2)
    # ---- joint loss ----
    cls_loss, dcls = _xent(class_logits, labels)
    seg_loss, dseg = _xent(seg_logits.reshape(-1, 2), np.asarray(mask).reshape(-1))
    w = seg_weight
    loss = ((1 - w) * cls_loss + w * seg_loss, cls_loss, seg_loss)
    dcls, dseg = (1 - w) * dcls, (w * dseg).reshape(seg_logits.shape)
    # ---- backward: segmentation head ----
    d, grads["seg_fc2/weights"], grads["seg_fc2/biases"] = T.conv1x1_bwd(dseg, cs2)
    d = _mlp_bwd(d * ones("seg_fc1"), cs1, ["seg_fc1"], grads)
    # ---- FP modules, last to first; skip gradients collected for the fan-ins ----
    dskip = {}
    for k in (2, 1, 0):
        dp1, d = fp_module_bwd(d, fp_caches[k], grads)
        dskip[2 - k] = dp1
    dclass_vector = d[:, 0, :]
    # ---- classification head; h2 feeds fc3 through dp2 and fa_layer1 directly ----
    dh2d, grads["fc3/weights"], grads["fc3/biases"] = T.conv1x1_bwd(dcls, c3)
    dh2 = dh2d * ones("fc2") + dclass_vector
    dh1 = _mlp_bwd(dh2, c2, ["fc2"], grads) * ones("fc1")
    dfeat = _mlp_bwd(dh1, c1, ["fc1"], grads)
    # ---- levels, last to first; l2_points / l1_points also fed fa_layer1 / fa_layer2 as skip features ----
    dpooled = dfeat.reshape(B, 1, -1)
    for li in (2, 1, 0):
        entry = sa[li]
        if entry[0] == "all":
            _, lc, c_pool, scopes, cfeat = entry
            dd = _mlp_bwd(T.maxpool_bwd(dpooled, c_pool), lc, scopes, grads)
            dpts = None if cfeat is None else dd[:, 0, :, 3:]
        else:
            _, cache, scopes = entry
            _, dpts, lg = T.sa_level_train_bwd(dpooled, cache)
            for s, (dw, db, dgamma, dbeta) in zip(scopes, lg):
                grads[f"{s}/weights"], grads[f"{s}/biases"] = dw, db
                grads[f"{s}/bn/gamma"], grads[f"{s}/bn/beta"] = dgamma, dbeta
        if li > 0 and dskip.get(li) is not None:
            dpts = dpts + dskip[li]
        dpooled = dpts
    return dict(class_logits=class_logits, seg_logits=seg_logits, loss=loss, grads=grads, batch_stats=stats, idx=idxs, fp_idx=fp_idx,
                relu_forced=forced)
