"""Property-based pin of the CPU restatement (oracle/psa_oracle.c) against the reference's OWN CPU code (grouping/test/
query_ball_point.cpp, selection_sort.cpp, tf_interpolate.cpp:57-153): random shapes down to the degenerate ones (n = 1, m = 1,
nsample > n, k = n) and adversarial values -- points on a lattice so that many distances sit exactly on the radius, duplicated
points (ties), tiny and large magnitudes.  Bit-exact, CPU only.

The cases are 200 derandomised hypothesis examples per property, drawn by tests/golden/make_golden_ref.py, which stored each
case's parameters (ARGS) with the digests of the reference's outputs in tests/golden/ref_cpu_fuzz.json.  INPUTS rebuilds a
case's input from its parameters."""
import numpy as np

from oracle import oracle as orc

from . import golden_util as golden

ARGS = {
    "ball_query": ["seed", "b", "n", "m", "nsample", "flavour", "radius"],
    "selection_sort": ["seed", "b", "m", "n", "ties", "kfrac"],
    "three_nn": ["seed", "b", "n", "m", "flavour"],
    "three_interpolate": ["seed", "b", "m", "n", "c", "dup"],
    "group_point": ["seed", "b", "n", "c", "m", "k"],
}


def _cloud(rng, b, n, flavour):
    if flavour == 0:                                   # lattice: distances repeat and land exactly on round radii
        x = rng.integers(-4, 5, size=(b, n, 3)).astype(np.float32) * np.float32(0.125)
    elif flavour == 1:                                 # duplicates of a few points
        base = rng.standard_normal((b, max(n // 4, 1), 3)).astype(np.float32)
        x = base[:, rng.integers(0, base.shape[1], size=n), :]
    elif flavour == 2:                                 # tiny magnitudes (denormal squares)
        x = (rng.standard_normal((b, n, 3)) * 1e-20).astype(np.float32)
    elif flavour == 3:                                 # large offset: catastrophic cancellation in the differences
        x = (rng.standard_normal((b, n, 3)) * 0.1 + 1000.0).astype(np.float32)
    else:
        x = rng.standard_normal((b, n, 3)).astype(np.float32)
    return np.ascontiguousarray(x)


def _ball_query(seed, b, n, m, nsample, flavour, radius):
    rng = np.random.default_rng(seed)
    xyz = _cloud(rng, b, n, flavour)
    q = _cloud(rng, b, m, flavour) if seed % 2 else np.ascontiguousarray(xyz[:, rng.integers(0, n, size=m), :])
    return dict(xyz=xyz, q=q, radius=radius, nsample=nsample)


def _selection_sort(seed, b, m, n, ties, kfrac):
    rng = np.random.default_rng(seed)
    dist = rng.random((b, m, n), dtype=np.float32)
    if ties:
        dist = np.round(dist * 4).astype(np.float32) / 4           # five distinct values: position-dependent tie resolution
    return dict(dist=dist, k=max(1, min(n, int(round(kfrac * n)))))


def _three_nn(seed, b, n, m, flavour):
    rng = np.random.default_rng(seed)
    xyz1 = _cloud(rng, b, n, flavour)
    return dict(xyz1=xyz1, xyz2=_cloud(rng, b, m, flavour))


def _three_interpolate(seed, b, m, n, c, dup):
    rng = np.random.default_rng(seed)
    pts = rng.standard_normal((b, m, c)).astype(np.float32)
    idx = rng.integers(0, m, size=(b, n, 3), dtype=np.int32)
    if dup:
        idx[..., 1] = idx[..., 0]                                  # the same source twice in a row: order of the scatter adds matters
    w = rng.random((b, n, 3), dtype=np.float32)
    return dict(pts=pts, idx=idx, w=w, go=rng.standard_normal((b, n, c)).astype(np.float32))


def _group_point(seed, b, n, c, m, k):
    rng = np.random.default_rng(seed)
    pts = rng.standard_normal((b, n, c)).astype(np.float32)
    idx = rng.integers(0, n, size=(b, m, k), dtype=np.int32)
    return dict(pts=pts, idx=idx, go=rng.standard_normal((b, m, k, c)).astype(np.float32))


INPUTS = {"ball_query": _ball_query, "selection_sort": _selection_sort, "three_nn": _three_nn,
          "three_interpolate": _three_interpolate, "group_point": _group_point}


def _cases(name):
    """(parameters, input, reference output digests) of every stored case of one property"""
    rows = golden.load("ref_cpu_fuzz.json")[name]
    assert len(rows) >= 150, len(rows)
    for row in rows:
        args = row[:len(ARGS[name])]
        yield args, INPUTS[name](*args), row[len(ARGS[name]):]


def test_ball_query_fuzz():
    for args, a, want in _cases("ball_query"):
        oi, cnt = orc.query_ball_point(a["radius"], a["nsample"], a["xyz"], a["q"], contract=False, fill=-7)   # the CPU harness's arithmetic
        assert [golden.digest(oi)] == want, args
        assert ((cnt == 0) == (oi[..., 0] == -7)).all() and cnt.max() <= a["nsample"]


def test_selection_sort_fuzz():
    for args, a, want in _cases("selection_sort"):
        oi, ov = orc.selection_sort(a["k"], a["dist"])
        assert [golden.digest(oi), golden.digest(ov)] == want, args


def test_three_nn_fuzz():
    for args, a, want in _cases("three_nn"):
        od, oi = orc.three_nn(a["xyz1"], a["xyz2"])
        assert [golden.digest(od), golden.digest(oi)] == want, args


def test_three_interpolate_and_grad_fuzz():
    for args, a, want in _cases("three_interpolate"):
        out = orc.three_interpolate(a["pts"], a["idx"], a["w"])
        grad = orc.three_interpolate_grad(a["pts"].shape, a["idx"], a["w"], a["go"])
        assert [golden.digest(out), golden.digest(grad)] == want, args


def test_group_point_and_grad_fuzz():
    for args, a, want in _cases("group_point"):
        out = orc.group_point(a["pts"], a["idx"])
        grad = orc.group_point_grad(a["pts"].shape, a["idx"], a["go"])
        assert [golden.digest(out), golden.digest(grad)] == want, args
