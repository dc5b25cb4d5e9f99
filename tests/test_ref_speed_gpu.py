"""GPU-vs-GPU: the libpsa kernels against the reference's own CUDA kernels (compiled unmodified for sm_100a) at the SSG shapes
(SURVEY 8d "timing the ref beside it").  tests/golden/make_golden_ref.py ran the reference's kernels on the same seeded inputs on a
B200 and stored their output digests and CUDA-event medians in tests/golden/ref_gpu_ops.json, with the GPU's name and power limit.
Here the outputs must be identical (index-exact) and every kernel faster than the reference's stored time."""
import json

import numpy as np
import pytest
import torch

from scanobjectnn_b200 import ops
from scanobjectnn_b200.synthetic import make_clouds
from tests import golden_util as golden
from tests import gpu_util as G

pytestmark = pytest.mark.gpu
B = 32


def time_us(fn, reps=7, warm=2):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def ssg_inputs():
    """seeded: B=32 clouds of 2048 points, SA2 features (B,512,128), a (B,128,512) distance matrix for SelectionSort"""
    rng = np.random.default_rng(1001)
    return (G.cu(make_clouds("ball", B, 2048, seed=1001)), G.cu(rng.standard_normal((B, 512, 128), dtype=np.float32)),
            G.cu(rng.random((B, 128, 512), dtype=np.float32)))


def test_libpsa_kernels_beat_the_reference_kernels():
    gold = golden.load("ref_gpu_ops.json")
    xyz, feats, dist = ssg_inputs()
    out = {}
    rows = {}

    def case(name, ours, outs):
        t_ours, t_ref = time_us(ours), gold["reference_kernel_us"][name]
        assert [golden.digest(o) for o in outs()] == gold[f"ssg/{name}"], f"{name}: output differs from the reference kernel's"
        rows[name] = {"libpsa_us": round(t_ours, 1), "reference_kernel_us": t_ref, "speedup": round(t_ref / t_ours, 2)}

    def fps1():
        out["i1"], out["x1"] = ops.farthest_point_sample_and_gather(512, xyz)
    case("fps+gather 2048->512", fps1, lambda: [out["i1"], out["x1"]])
    l1 = out["x1"].contiguous()

    def fps2():
        out["i2"], out["x2"] = ops.farthest_point_sample_and_gather(128, l1)
    case("fps+gather 512->128", fps2, lambda: [out["i2"], out["x2"]])
    l2 = out["x2"].contiguous()

    for name, (r, k, a, q) in {"query_ball_point r=0.2 k=32 (2048, 512)": (0.2, 32, xyz, l1),
                               "query_ball_point r=0.4 k=64 (512, 128)": (0.4, 64, l1, l2)}.items():
        def ours(r=r, k=k, a=a, q=q, key=name):
            out[key] = ops.query_ball_point(r, k, a, q)
        case(name, ours, lambda key=name: list(out[key]))
    idx2 = out["query_ball_point r=0.4 k=64 (512, 128)"][0]

    # group_point at the SA2 size (the tensor the fused path never writes): (B,512,128) by (B,128,64)
    def group():
        out["g"] = ops.group_point(feats, idx2)
    case("group_point C=128 (128 MiB out)", group, lambda: [out["g"]])

    # SelectionSort (knn_point's op) at b*m = 4096 rows of 512
    def sel():
        out["s"] = ops.select_top_k(32, dist)
    case("selection_sort k=32 (4096 rows x 512)", sel, lambda: [out["s"][0][..., :32]])

    print(json.dumps({"reference_measured_on": gold["measured_on"], **rows}, indent=1))
    slow = {k: v for k, v in rows.items() if v["speedup"] < 1.0}
    assert not slow, f"slower than the reference kernel: {slow}"
