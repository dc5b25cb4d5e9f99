"""Pin the CPU restatement (oracle/psa_oracle.c) against the reference's OWN CPU code (the digests of its outputs on these
inputs, tests/golden/ref_cpu_pins.json, written by tests/golden/make_golden_ref.py) and against the reference's only
deterministic known-answer test (grouping/test/selection_sort.cpp:68-78)."""
import numpy as np
import pytest

from oracle import oracle as orc
from scanobjectnn_b200.synthetic import make_clouds

from . import golden_util as golden

D = golden.digest


def _ref(key):
    return golden.load("ref_cpu_pins.json")[key]


def test_selection_sort_kat():
    # selection_sort.cpp:68-78: b=2,n=4,m=2,k=3, dist[i]=10-i -> each row's first 3 slots are 3,2,1
    b, n, m, k = 2, 4, 2, 3
    dist = (10.0 - np.arange(b * m * n, dtype=np.float32)).reshape(b, m, n)
    outi, out = orc.selection_sort(k, dist)
    assert (outi[..., :k] == np.array([3, 2, 1])).all()
    assert (np.diff(out[..., :k], axis=-1) > 0).all()
    # the full permutation the harness prints: 3 2 1 0 for every row
    assert (outi == np.array([3, 2, 1, 0])).all()


def test_selection_sort_matches_reference_cpu():
    rng = np.random.default_rng(5)
    dist = rng.random((3, 7, 50), dtype=np.float32)
    dist[0, 0, 10:20] = dist[0, 0, 3]          # ties: resolved by current array position
    dist[1, 2, :] = 0.5
    for k in (1, 5, 50):
        oi, ov = orc.selection_sort(k, dist)
        assert [D(oi), D(ov)] == _ref(f"selection_sort/{k}"), k


@pytest.mark.parametrize("kind", ["ball", "shell", "dup"])
def test_ball_query_matches_reference_cpu(kind):
    xyz = make_clouds(kind, 4, 512, seed=11)
    q = xyz[:, ::4, :].copy()
    for r, k in ((0.1, 64), (0.2, 32), (0.4, 16)):
        oi, cnt = orc.query_ball_point(r, k, xyz, q, contract=False, fill=-7)
        assert D(oi) == _ref(f"ball_query/{kind}/{r}/{k}"), (r, k)
        assert cnt.min() >= 1          # queries are dataset points: self-distance 1e-20 < r


def test_ball_query_empty_ball_leaves_row_untouched():
    xyz = make_clouds("ball", 2, 64, seed=3)
    q = np.full((2, 5, 3), 9.0, np.float32)
    oi, cnt = orc.query_ball_point(0.2, 8, xyz, q, contract=False, fill=-7)
    assert (oi == -7).all() and (cnt == 0).all()
    assert D(oi) == _ref("ball_query_empty")                # the reference leaves the row untouched too


def test_group_point_and_grad_match_reference_cpu():
    rng = np.random.default_rng(9)
    pts = rng.standard_normal((3, 40, 7)).astype(np.float32)
    idx = rng.integers(0, 40, size=(3, 11, 5), dtype=np.int32)
    go = rng.standard_normal((3, 11, 5, 7)).astype(np.float32)
    assert [D(orc.group_point(pts, idx)), D(orc.group_point_grad(pts.shape, idx, go))] == _ref("group_point")


@pytest.mark.parametrize("n,m", [(128, 1), (128, 2), (512, 128), (300, 77)])
def test_three_nn_matches_reference_cpu(n, m):
    xyz1 = make_clouds("shell", 3, n, seed=21)
    xyz2 = make_clouds("dup", 3, max(m, 4), seed=22)[:, :m, :].copy()
    od, oi = orc.three_nn(xyz1, xyz2)
    assert [D(od), D(oi)] == _ref(f"three_nn/{n}/{m}")     # inf == inf for the m<3 slots
    if m < 3:
        assert np.isinf(od[..., m:]).all() and (oi[..., m:] == 0).all()


def test_three_interpolate_and_grad_match_reference_cpu():
    rng = np.random.default_rng(2)
    pts = rng.standard_normal((2, 30, 9)).astype(np.float32)
    idx = rng.integers(0, 30, size=(2, 50, 3), dtype=np.int32)
    w = rng.random((2, 50, 3), dtype=np.float32)
    go = rng.standard_normal((2, 50, 9)).astype(np.float32)
    assert [D(orc.three_interpolate(pts, idx, w)), D(orc.three_interpolate_grad(pts.shape, idx, w, go))] == _ref("three_interpolate")


def test_fps_basic_properties():
    xyz = make_clouds("ball", 2, 700, seed=1)
    idx = orc.fps(xyz, 64)
    assert (idx[:, 0] == 0).all()
    for b in range(2):
        assert len(set(idx[b].tolist())) == 64          # distinct while distinct points remain
    # second pick is the farthest from point 0 (no ties in random data)
    d = ((xyz - xyz[:, :1]) ** 2).sum(-1)
    assert (idx[:, 1] == d.argmax(1)).all()


def test_fps_tie_key_is_kmod512_then_k():
    # 1100 points: point 0 at origin, every other point at one of two antipodal spots at equal
    # distance -> all maxima tie; the reference's winner is min over (k mod 512, k).
    n = 1100
    xyz = np.zeros((1, n, 3), np.float32)
    xyz[0, 1:, 0] = 1.0
    xyz[0, 600:, 0] = -1.0
    idx = orc.fps(xyz, 3)
    # round 1: all k>=1 tie at d=1; slots t=k mod 512: slot 0 holds k=512,1024 -> wins -> 512
    assert idx[0, 1] == 512
    # round 2: points at -1 (k>=600) have d=4 from x=+1; candidates k in [600,1100): slot (k mod 512):
    # k=1024 -> slot 0 -> wins
    assert idx[0, 2] == 1024


def test_dgcnn_knn_self_first_and_sorted():
    x = make_clouds("ball", 2, 100, seed=4)
    idx, adj = orc.dgcnn_knn(x, 5, want_adj=True)
    rows = np.take_along_axis(adj, idx, axis=-1)
    assert (np.diff(rows, axis=-1) >= 0).all()
    assert (idx == orc.topk_smallest(adj, 5)).all()


def test_dgcnn_knn_agrees_with_torch_topk_at_the_reference_call_site():
    """dgcnn/utils/tf_util.py:638-671 evaluated by an independent library (torch CPU, float64): adj = |x|^2 - 2 x x^T + |x|^2^T,
    top_k(-adj, k).  On tie-free data the oracle's float32 canonical-order evaluation must select the same neighbours."""
    import torch
    for c, n, k in [(3, 300, 20), (64, 200, 20)]:
        x = np.random.default_rng(c).standard_normal((2, n, c)).astype(np.float32)
        idx = orc.dgcnn_knn(x, k)
        t = torch.from_numpy(x).double()
        inner = -2 * torch.matmul(t, t.transpose(2, 1))
        sq = (t * t).sum(-1, keepdim=True)
        adj = sq + inner + sq.transpose(2, 1)
        ref = torch.topk(-adj, k).indices.numpy()
        # float32 rounding can swap two neighbours whose float64 distances differ by less than a few ulp: compare as sets per row,
        # and require exact order wherever the float64 gaps are clear
        gaps = np.diff(np.sort(adj.numpy(), axis=-1)[..., : k + 1], axis=-1).min(-1)
        scale = float((sq.max() * 4).item())                      # magnitude of the terms that cancel in adj
        clear = gaps > 64 * np.finfo(np.float32).eps * scale         # well above the float32 evaluation error
        assert clear.mean() > 0.5, clear.mean()
        assert np.array_equal(idx[clear], ref[clear])
