"""GPU parity: this repo's sm_100a kernels (through the C ABI via scanobjectnn_b200.ops) against
(1) the CPU oracle and (2) the REFERENCE's own CUDA kernels compiled for sm_100a, through the digests of their outputs on
the same inputs (tests/golden/ref_gpu_ops.json, written by tests/golden/make_golden_ref.py on a B200).
Index outputs must be bit-exact."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from scanobjectnn_b200 import ops
from scanobjectnn_b200.synthetic import make_clouds

from . import golden_util as golden
from . import gpu_util as G

pytestmark = pytest.mark.gpu
D = golden.digest


def _ref(key):
    """digests of the reference kernel's outputs for this test case"""
    return golden.load("ref_gpu_ops.json")[key]


# ----------------------------------------------------------------------------------------------- FPS
@pytest.mark.parametrize("kind", ["ball", "shell", "dup"])
@pytest.mark.parametrize("n,m", [(1, 1), (7, 3), (100, 40), (512, 128), (513, 64), (1000, 250), (2048, 512),
                                 (3000, 100), (4096, 64), (8192, 32)])
def test_fps_matches_oracle(kind, n, m):
    xyz = make_clouds(kind, 3, n, seed=100 + n)
    got = G.npy(ops.farthest_point_sample(m, G.cu(xyz)))
    assert (got == orc.fps(xyz, m)).all()


@pytest.mark.parametrize("kind,b,n,m", [("ball", 32, 2048, 512), ("dup", 32, 2048, 512), ("shell", 40, 512, 128),
                                        ("dup", 5, 4096, 256), ("ball", 2, 8192, 128), ("dup", 3, 700, 700)])
def test_fps_matches_reference_kernel(kind, b, n, m):
    xyz = G.cu(make_clouds(kind, b, n, seed=7 + n))
    idx, new_xyz = ops.farthest_point_sample_and_gather(m, xyz)
    assert [D(idx), D(new_xyz)] == _ref(f"fps/{kind}/{b}/{n}/{m}")


def test_fps_tie_break_and_oversampling():
    n = 1100
    xyz = np.zeros((2, n, 3), np.float32)
    xyz[:, 1:, 0] = 1.0
    xyz[:, 600:, 0] = -1.0
    xyz[1, :, 1] = 0.25            # second cloud: same ties, shifted
    t = G.cu(xyz)
    got = ops.farthest_point_sample(5, t)
    assert D(got) == _ref("fps_ties")
    assert G.npy(got)[0, :3].tolist() == [0, 512, 1024]
    # m > n: once every point is taken the reference keeps returning the (k mod 512, k)-minimal index
    small = G.cu(make_clouds("ball", 2, 5, seed=1))
    assert D(ops.farthest_point_sample(9, small)) == _ref("fps_oversampled")


def test_fps_nan_and_inf_inputs_match_oracle():
    xyz = make_clouds("ball", 2, 300, seed=5)
    xyz[0, 17] = np.nan
    xyz[1, 3, 0] = np.inf
    xyz[1, 200] = 1e30
    got = G.npy(ops.farthest_point_sample(20, G.cu(xyz)))
    assert (got == orc.fps(xyz, 20)).all()


def test_fps_argument_errors():
    with pytest.raises(ValueError):
        ops.farthest_point_sample(4, torch.zeros((2, 10, 4), device="cuda"))
    with pytest.raises(ValueError):
        ops.farthest_point_sample(4, torch.zeros((2, 0, 3), device="cuda"))
    with pytest.raises(RuntimeError):
        ops.farthest_point_sample(4, torch.zeros((2, 10, 3)))
    assert ops.farthest_point_sample(0, torch.zeros((2, 10, 3), device="cuda")).shape == (2, 0)


def test_gather_point_and_grad():
    rng = np.random.default_rng(0)
    inp = rng.standard_normal((3, 50, 3)).astype(np.float32)
    idx = rng.integers(0, 50, size=(3, 20), dtype=np.int32)
    t = G.cu(inp).requires_grad_(True)
    out = ops.gather_point(t, G.cu(idx))
    assert np.array_equal(G.npy(out), orc.gather_point(inp, idx))
    go = rng.standard_normal((3, 20, 3)).astype(np.float32)
    out.backward(G.cu(go))
    # ordered scatter-add: the sum order of the reference's sequential CPU loop -> bit-identical, not just close
    assert np.array_equal(G.npy(t.grad), orc.gather_point_grad(inp.shape, idx, go))


# ----------------------------------------------------------------------------------------------- ball query
@pytest.mark.parametrize("kind", ["ball", "shell", "dup"])
@pytest.mark.parametrize("n,m,r,k", [(2048, 512, 0.2, 32), (512, 128, 0.4, 64), (512, 128, 0.1, 64), (100, 33, 0.3, 5),
                                     (1, 1, 0.2, 4), (77, 77, 2.5, 100)])
def test_ball_query_matches_oracle(kind, n, m, r, k):
    xyz = make_clouds(kind, 3, n, seed=n + k)
    q = xyz[:, :: max(1, n // m), :][:, :m].copy()
    idx, cnt = ops.query_ball_point(r, k, G.cu(xyz), G.cu(q))
    oi, oc = orc.query_ball_point(r, k, xyz, q, contract=True, fill=0)
    assert (G.npy(idx) == oi).all() and (G.npy(cnt) == oc).all()


@pytest.mark.parametrize("kind,b,n,m,r,k", [("ball", 32, 2048, 512, 0.2, 32), ("shell", 32, 2048, 512, 0.2, 64),
                                            ("dup", 32, 512, 128, 0.4, 64), ("ball", 4, 4096, 1024, 0.1, 16)])
def test_ball_query_matches_reference_kernel(kind, b, n, m, r, k):
    xyz = G.cu(make_clouds(kind, b, n, seed=n + k + 1))
    q = ops.gather_point(xyz, ops.farthest_point_sample(m, xyz))
    idx, cnt = ops.query_ball_point(r, k, xyz, q)
    assert [D(idx), D(cnt)] == _ref(f"ball_query/{kind}/{b}/{n}/{m}/{r}/{k}")


def test_ball_query_radius_boundary_and_specials():
    # distances that land exactly on / next to the radius: lattice points at multiples of 0.05 from the query
    g = np.arange(-8, 9, dtype=np.float32) * np.float32(0.05)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(1, -1, 3).astype(np.float32)
    q = np.zeros((1, 3, 3), np.float32)
    q[0, 1] = [0.05, 0.1, -0.15]
    q[0, 2] = [1e-3, -2e-3, 3e-3]
    xt, qt = G.cu(xyz), G.cu(q)
    for r in (0.05, 0.1, 0.15, 0.2, 0.25, 0.3, 0.0707, 0.0866, np.nextafter(np.float32(0.2), np.float32(1))):
        idx, cnt = ops.query_ball_point(float(r), 64, xt, qt)
        assert [D(idx), D(cnt)] == _ref(f"ball_query_radius/{float(r)!r}"), r
    # NaN / inf coordinates in the dataset: CUDA's max(NaN,1e-20f) makes a NaN distance count as inside
    x2 = make_clouds("ball", 2, 200, seed=3)
    x2[0, 5] = np.nan
    x2[1, 9, 2] = np.inf
    xt2 = G.cu(x2)
    qt2 = G.cu(x2[:, 20:40].copy())
    idx, cnt = ops.query_ball_point(0.3, 16, xt2, qt2)
    assert [D(idx), D(cnt)] == _ref("ball_query_nonfinite")


def test_ball_query_empty_ball_and_errors():
    xyz = G.cu(make_clouds("ball", 2, 64, seed=3))
    q = torch.full((2, 5, 3), 9.0, device="cuda")
    idx, cnt = ops.query_ball_point(0.2, 8, xyz, q)
    assert (idx == 0).all() and (cnt == 0).all()
    with pytest.raises(ValueError):
        ops.query_ball_point(-1.0, 8, xyz, q)
    with pytest.raises(ValueError):
        ops.query_ball_point(0.2, 0, xyz, q)
    with pytest.raises(ValueError):
        ops.query_ball_point(0.2, 8, xyz, q[:1])


# ----------------------------------------------------------------------------------------------- group
@pytest.mark.parametrize("c", [3, 7, 64, 128])
def test_group_point_and_grad(c):
    rng = np.random.default_rng(c)
    pts = rng.standard_normal((3, 90, c)).astype(np.float32)
    idx = rng.integers(0, 90, size=(3, 17, 9), dtype=np.int32)
    t = G.cu(pts).requires_grad_(True)
    out = ops.group_point(t, G.cu(idx))
    assert np.array_equal(G.npy(out), orc.group_point(pts, idx))
    assert D(out) == _ref(f"group_point/{c}")
    go = rng.standard_normal(out.shape).astype(np.float32)
    out.backward(G.cu(go))
    assert np.array_equal(G.npy(t.grad), orc.group_point_grad(pts.shape, idx, go))


# ----------------------------------------------------------------------------------------------- selection sort / knn_point
def test_selection_sort_kat_and_oracle():
    dist = (10.0 - np.arange(16, dtype=np.float32)).reshape(2, 2, 4)
    outi, out = ops.select_top_k(3, G.cu(dist))
    assert (G.npy(outi) == np.array([3, 2, 1, 0])).all()          # selection_sort.cpp:68-92
    rng = np.random.default_rng(1)
    d = rng.random((3, 9, 300), dtype=np.float32)
    d[0, 0, 10:40] = d[0, 0, 3]
    d[1, 1, :] = 0.25
    d[2, 2, ::7] = np.nan
    for k in (1, 8, 32, 300):
        oi, ov = orc.selection_sort(k, d)
        gi, gv = ops.select_top_k(k, G.cu(d))
        assert np.array_equal(G.npy(gi), oi) and np.array_equal(G.npy(gv), ov, equal_nan=True)
        assert [D(gi), D(gv)] == _ref(f"selection_sort/{k}"), k


@pytest.mark.parametrize("kind", ["ball", "dup"])
def test_knn_point_matches_oracle(kind):
    xyz = make_clouds(kind, 2, 400, seed=2)
    q = xyz[:, ::5].copy()
    val, idx = ops.knn_point(16, G.cu(xyz), G.cu(q))
    ov, oi = orc.knn_point(16, xyz, q)
    assert np.array_equal(G.npy(idx), oi) and np.array_equal(G.npy(val), ov)


# ----------------------------------------------------------------------------------------------- three_nn / interpolate
@pytest.mark.parametrize("n,m", [(128, 1), (128, 2), (512, 128), (2048, 512), (300, 77), (5000, 2500)])
def test_three_nn_matches_oracle(n, m):
    xyz1 = make_clouds("shell", 2, n, seed=21)
    xyz2 = make_clouds("dup", 2, max(m, 4), seed=22)[:, :m].copy()
    dist, idx = ops.three_nn(G.cu(xyz1), G.cu(xyz2))
    od, oi = orc.three_nn(xyz1, xyz2)
    assert np.array_equal(G.npy(idx), oi) and np.array_equal(G.npy(dist), od)


@pytest.mark.parametrize("c", [1, 6, 128, 256])
def test_three_interpolate_and_grad(c):
    rng = np.random.default_rng(c)
    pts = rng.standard_normal((2, 30, c)).astype(np.float32)
    idx = rng.integers(0, 30, size=(2, 70, 3), dtype=np.int32)
    w = rng.random((2, 70, 3), dtype=np.float32)
    t = G.cu(pts).requires_grad_(True)
    out = ops.three_interpolate(t, G.cu(idx), G.cu(w))
    assert np.array_equal(G.npy(out), orc.three_interpolate(pts, idx, w))
    go = rng.standard_normal(out.shape).astype(np.float32)
    out.backward(G.cu(go))
    assert np.array_equal(G.npy(t.grad), orc.three_interpolate_grad(pts.shape, idx, w, go))


def test_scatter_gradients_are_ordered_at_model_shapes():
    """SA-1 shapes (B=8, N=2048 -> 512 x 32 rows, hot destinations hit hundreds of times): the three gradients equal the
    reference's sequential CPU sums bit for bit, twice in a row, and unreferenced destinations are exact zeros."""
    rng = np.random.default_rng(77)
    b, n, m, k, c = 8, 2048, 512, 32, 64
    idx = (rng.integers(0, n // 4, size=(b, m, k)) * rng.integers(1, 5, size=(b, m, 1))).astype(np.int32) % n
    idx[:, :, :4] = 5                                                     # one very hot destination
    go = rng.standard_normal((b, m, k, c)).astype(np.float32)
    pts = torch.zeros((b, n, c), device="cuda", requires_grad=True)
    want = orc.group_point_grad((b, n, c), idx, go)
    for _ in range(2):
        pts.grad = None
        ops.group_point(pts, G.cu(idx)).backward(G.cu(go))
        assert np.array_equal(G.npy(pts.grad), want)
    untouched = np.ones((b, n), bool)
    for i in range(b):
        untouched[i, np.unique(idx[i])] = False
    assert untouched.any() and not G.npy(pts.grad)[untouched].any()
    # FP-module shapes: 2048 unknown points interpolate from 128 known ones
    idx3 = rng.integers(0, 128, size=(b, n, 3), dtype=np.int32)
    w3 = rng.random((b, n, 3), dtype=np.float32)
    g3 = rng.standard_normal((b, n, 256)).astype(np.float32)
    known = torch.zeros((b, 128, 256), device="cuda", requires_grad=True)
    ops.three_interpolate(known, G.cu(idx3), G.cu(w3)).backward(G.cu(g3))
    assert np.array_equal(G.npy(known.grad), orc.three_interpolate_grad((b, 128, 256), idx3, w3, g3))
    # FPS gather: every centre index once, most inputs untouched
    fidx = np.stack([rng.permutation(n)[:m] for _ in range(b)]).astype(np.int32)
    gg = rng.standard_normal((b, m, 3)).astype(np.float32)
    xyz = torch.zeros((b, n, 3), device="cuda", requires_grad=True)
    ops.gather_point(xyz, G.cu(fidx)).backward(G.cu(gg))
    assert np.array_equal(G.npy(xyz.grad), orc.gather_point_grad((b, n, 3), fidx, gg))


def test_scatter_gradient_workspace_is_checked():
    import ctypes as C

    from scanobjectnn_b200 import _lib
    lib = _lib.load()
    need = lib.psa_scatter_workspace_bytes(2, 16, 8)
    assert need >= (2 * 17 + 2 * 8) * 4
    g = torch.zeros((2, 16, 3), device="cuda")
    og = torch.zeros((2, 8, 3), device="cuda")
    ix = torch.zeros((2, 8), dtype=torch.int32, device="cuda")
    small = torch.empty((16,), dtype=torch.uint8, device="cuda")
    rc = lib.psa_gather_point_grad(2, 16, 8, C.c_void_p(og.data_ptr()), C.c_void_p(ix.data_ptr()), C.c_void_p(g.data_ptr()),
                                   C.c_void_p(small.data_ptr()), C.c_size_t(16), None)
    assert rc == -1 and b"workspace" in lib.psa_last_error()


@pytest.mark.parametrize("n,m,c", [(128, 1, 16), (512, 128, 256), (2048, 512, 128), (333, 50, 7)])
def test_three_nn_interpolate_fused(n, m, c):
    rng = np.random.default_rng(n)
    xyz1 = make_clouds("ball", 2, n, seed=31)
    xyz2 = make_clouds("ball", 2, max(m, 4), seed=32)[:, :m].copy()
    p2 = rng.standard_normal((2, m, c)).astype(np.float32)
    out, dist, idx, w = ops.three_nn_interpolate(G.cu(xyz1), G.cu(xyz2), G.cu(p2), return_aux=True)
    od, oi = orc.three_nn(xyz1, xyz2)
    ow = orc.three_weights(od)
    assert np.array_equal(G.npy(idx), oi) and np.array_equal(G.npy(dist), od)
    assert np.array_equal(G.npy(w), ow)
    assert np.array_equal(G.npy(out), orc.three_interpolate(p2, oi, ow))


# ----------------------------------------------------------------------------------------------- dgcnn graph
@pytest.mark.parametrize("n,c,k", [(100, 3, 5), (257, 64, 20), (1024, 3, 20), (300, 128, 20)])
def test_dgcnn_graph_matches_oracle(n, c, k):
    rng = np.random.default_rng(n + c)
    x = rng.standard_normal((2, n, c)).astype(np.float32) if c != 3 else make_clouds("dup", 2, n, seed=n)
    oi, oadj = orc.dgcnn_knn(x, k, want_adj=True)
    xt = G.cu(x)
    adj = ops.pairwise_distance(xt)
    assert np.array_equal(G.npy(adj), oadj)
    assert np.array_equal(G.npy(ops.knn(adj, k)), oi)
    assert np.array_equal(G.npy(ops.knn_graph(xt, k)), oi)
    edge = ops.get_edge_feature(xt.unsqueeze(2), G.cu(oi), k)
    nb = x[np.arange(2)[:, None, None], oi]
    ctr = np.broadcast_to(x[:, :, None, :], nb.shape)
    assert np.array_equal(G.npy(edge), np.concatenate([ctr, nb - ctr], -1))


@pytest.mark.parametrize("kind,n,c,k", [("gauss", 2048, 64, 20), ("ball", 2048, 3, 20), ("dup", 1024, 3, 20), ("gauss", 300, 16, 8),
                                        ("gauss", 256, 64, 32), ("scaled", 1024, 64, 20), ("nan", 512, 8, 10),
                                        ("lattice", 1024, 3, 20), ("jitter", 1024, 64, 20), ("offset", 2048, 64, 20), ("relu", 2048, 64, 20),
                                        ("jitter", 640, 12, 16)])
def test_knn_graph_tensor_core_path_is_index_exact(kind, n, c, k):
    """csrc/knn_tc.cu: bf16 / bf16x3 tensor-core distances only PRUNE; the neighbours come from the canonical fp32 distances of the
    survivors, so the result equals the oracle (and the fp32 kernel) bit for bit -- incl. the BASELINE configs[2] size n = 2048,
    clouds with many exactly equidistant points (list overflow -> exhaustive rows) and a cloud holding a NaN."""
    rng = np.random.default_rng(n + c + k)
    if kind in ("ball", "dup"):
        x = make_clouds(kind, 2, n, seed=n + 1)
    else:
        x = rng.standard_normal((2, n, c)).astype(np.float32)
        if kind == "lattice":                 # integer grid: most distances tie exactly -> everything is decided canonically / by index
            x = rng.integers(0, 7, size=(2, n, c)).astype(np.float32)
        if kind == "jitter":                  # a few hundred distinct sites + noise from 1e-7 to 1e-2: near-ties on every scale around
            sites = rng.standard_normal((2, 40, c)).astype(np.float32)          # the fine/canonical decision boundary
            pick = rng.integers(0, 40, size=(2, n))
            amp = (10.0 ** rng.uniform(-7, -2, size=(2, n, 1))).astype(np.float32)
            x = np.take_along_axis(sites, pick[:, :, None].repeat(c, 2), 1) + amp * rng.standard_normal((2, n, c)).astype(np.float32)
        if kind == "offset":                  # large common offset: |x|^2 terms dwarf the distances (cancellation in adj)
            x = (x * 0.05 + 3.0).astype(np.float32)
        if kind == "relu":
            x = np.maximum(x, 0)
        if kind == "scaled":
            x[1] *= 37.5                      # per-cloud scale: the error bounds are relative to the cloud's norms
            x[0, : n // 2] *= 1e-3            # a dense cluster far below the cloud's largest distances
    if kind == "nan":
        x[1, 7, 2] = np.nan
    xt = G.cu(x)
    assert _lib_ws(2, n, c, k) > 0
    got = G.npy(ops.knn_graph(xt, k))
    if kind == "nan":
        want0 = orc.dgcnn_knn(x[:1], k)
        assert np.array_equal(got[0], want0[0])            # the finite cloud is exact; the NaN cloud only has to complete
        assert got[1].min() >= 0 and got[1].max() < n
        return
    assert np.array_equal(got, orc.dgcnn_knn(x, k))
    ops._KNN_FP32_ONLY = True
    try:
        assert np.array_equal(got, G.npy(ops.knn_graph(xt, k)))
    finally:
        ops._KNN_FP32_ONLY = False


def _lib_ws(b, n, c, k):
    from scanobjectnn_b200 import _lib
    return _lib.load().psa_knn_graph_workspace_bytes(b, n, c, k)
