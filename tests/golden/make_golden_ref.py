"""Generate the digest files of tests/golden_util.py from the REFERENCE's own code.

    python tests/golden/make_golden_ref.py cpu OUTDIR    # oracle/_ref/libref_cpu.so   -> ref_cpu_pins.json, ref_cpu_fuzz.json
    python tests/golden/make_golden_ref.py gpu OUTDIR    # oracle/_ref/libref_tfops.so -> ref_gpu_ops.json (needs a B200)

oracle/_ref/ is built by `make -C oracle ref` from a checkout of the reference.  Inputs are NOT stored: every case below
builds its input exactly as the test that reads its digests does (tests/test_oracle_pins.py, test_oracle_fuzz.py,
test_ops_gpu.py, test_ref_speed_gpu.py), from seeds.  The fuzz cases are the 200 derandomised hypothesis examples per
property; their parameters are stored with the digests.  The gpu mode also times the reference's kernels at the SSG shapes
(CUDA-event medians) and records the GPU's name and power limit beside the times.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np

from oracle import oracle as orc
from scanobjectnn_b200.synthetic import make_clouds
from tests.golden_util import digest as D


def _dump(path, obj):
    """one case per line: reviewable diffs, small files"""
    with open(path, "w") as f:
        f.write("{\n")
        items = list(obj.items())
        for i, (k, v) in enumerate(items):
            if isinstance(v, list) and v and isinstance(v[0], list):
                f.write(f"{json.dumps(k)}: [\n" + ",\n".join("  " + json.dumps(r) for r in v) + "\n]")
            else:
                f.write(f"{json.dumps(k)}: {json.dumps(v)}")
            f.write(",\n" if i + 1 < len(items) else "\n")
        f.write("}\n")


def cpu(outdir):
    assert orc.refcpu_available(), "oracle/_ref/libref_cpu.so not built (make -C oracle ref)"
    # ---- tests/test_oracle_pins.py
    pins = {}
    rng = np.random.default_rng(5)
    dist = rng.random((3, 7, 50), dtype=np.float32)
    dist[0, 0, 10:20] = dist[0, 0, 3]
    dist[1, 2, :] = 0.5
    for k in (1, 5, 50):
        ri, rv = orc.refcpu_selection_sort(k, dist)
        pins[f"selection_sort/{k}"] = [D(ri), D(rv)]
    for kind in ("ball", "shell", "dup"):
        xyz = make_clouds(kind, 4, 512, seed=11)
        q = xyz[:, ::4, :].copy()
        for r, k in ((0.1, 64), (0.2, 32), (0.4, 16)):
            pins[f"ball_query/{kind}/{r}/{k}"] = D(orc.refcpu_query_ball_point(r, k, xyz, q, fill=-7))
    xyz = make_clouds("ball", 2, 64, seed=3)
    q = np.full((2, 5, 3), 9.0, np.float32)
    pins["ball_query_empty"] = D(orc.refcpu_query_ball_point(0.2, 8, xyz, q, fill=-7))
    rng = np.random.default_rng(9)
    pts = rng.standard_normal((3, 40, 7)).astype(np.float32)
    idx = rng.integers(0, 40, size=(3, 11, 5), dtype=np.int32)
    go = rng.standard_normal((3, 11, 5, 7)).astype(np.float32)
    pins["group_point"] = [D(orc.refcpu_group_point(pts, idx)), D(orc.refcpu_group_point_grad(pts.shape, idx, go))]
    for n, m in [(128, 1), (128, 2), (512, 128), (300, 77)]:
        xyz1 = make_clouds("shell", 3, n, seed=21)
        xyz2 = make_clouds("dup", 3, max(m, 4), seed=22)[:, :m, :].copy()
        pins[f"three_nn/{n}/{m}"] = [D(a) for a in orc.refcpu_three_nn(xyz1, xyz2)]
    rng = np.random.default_rng(2)
    pts = rng.standard_normal((2, 30, 9)).astype(np.float32)
    idx = rng.integers(0, 30, size=(2, 50, 3), dtype=np.int32)
    w = rng.random((2, 50, 3), dtype=np.float32)
    go = rng.standard_normal((2, 50, 9)).astype(np.float32)
    pins["three_interpolate"] = [D(orc.refcpu_three_interpolate(pts, idx, w)), D(orc.refcpu_three_interpolate_grad(pts.shape, idx, w, go))]
    _dump(os.path.join(outdir, "ref_cpu_pins.json"), pins)

    # ---- tests/test_oracle_fuzz.py: the parameters hypothesis draws, then the reference's outputs for each
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as st

    from tests import test_oracle_fuzz as F
    fuzz = settings(max_examples=200, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    seed = st.integers(0, 2 ** 31 - 1)
    drawn = {k: [] for k in F.ARGS}

    @fuzz
    @given(seed=seed, b=st.integers(1, 3), n=st.integers(1, 70), m=st.integers(1, 20), nsample=st.integers(1, 80),
           flavour=st.integers(0, 4), radius=st.sampled_from([0.125, 0.25, 0.5, 0.2, 1e-3, 3.0, 1e-19]))
    def ball_query(**a):
        drawn["ball_query"].append(a)

    @fuzz
    @given(seed=seed, b=st.integers(1, 3), m=st.integers(1, 6), n=st.integers(1, 40), ties=st.booleans(), kfrac=st.floats(0.0, 1.0))
    def selection_sort(**a):
        drawn["selection_sort"].append(a)

    @fuzz
    @given(seed=seed, b=st.integers(1, 3), n=st.integers(1, 50), m=st.integers(1, 30), flavour=st.integers(0, 4))
    def three_nn(**a):
        drawn["three_nn"].append(a)

    @fuzz
    @given(seed=seed, b=st.integers(1, 3), m=st.integers(1, 20), n=st.integers(1, 30), c=st.integers(1, 9), dup=st.booleans())
    def three_interpolate(**a):
        drawn["three_interpolate"].append(a)

    @fuzz
    @given(seed=seed, b=st.integers(1, 3), n=st.integers(1, 30), c=st.integers(1, 9), m=st.integers(1, 12), k=st.integers(1, 9))
    def group_point(**a):
        drawn["group_point"].append(a)

    for f in (ball_query, selection_sort, three_nn, three_interpolate, group_point):
        f()
    ref = {
        "ball_query": lambda xyz, q, radius, nsample: [orc.refcpu_query_ball_point(radius, nsample, xyz, q, fill=-7)],
        "selection_sort": lambda dist, k: orc.refcpu_selection_sort(k, dist),
        "three_nn": lambda xyz1, xyz2: orc.refcpu_three_nn(xyz1, xyz2),
        "three_interpolate": lambda pts, idx, w, go: [orc.refcpu_three_interpolate(pts, idx, w),
                                                      orc.refcpu_three_interpolate_grad(pts.shape, idx, w, go)],
        "group_point": lambda pts, idx, go: [orc.refcpu_group_point(pts, idx), orc.refcpu_group_point_grad(pts.shape, idx, go)],
    }
    out = {}
    for name, cases in drawn.items():
        rows, seen = [], set()
        for a in cases:
            args = [a[k] for k in F.ARGS[name]]
            if json.dumps(args) in seen:
                continue
            seen.add(json.dumps(args))
            rows.append(args + [D(x) for x in ref[name](**F.INPUTS[name](*args))])
        out[name] = rows
    _dump(os.path.join(outdir, "ref_cpu_fuzz.json"), out)


def gpu(outdir):
    import torch

    from tests import gpu_util as G
    from tests.test_ref_speed_gpu import ssg_inputs, time_us
    assert orc.refgpu_available(), "oracle/_ref/libref_tfops.so not built (make -C oracle ref)"
    cases = {}
    # ---- tests/test_ops_gpu.py
    for kind, b, n, m in [("ball", 32, 2048, 512), ("dup", 32, 2048, 512), ("shell", 40, 512, 128),
                          ("dup", 5, 4096, 256), ("ball", 2, 8192, 128), ("dup", 3, 700, 700)]:
        xyz = G.cu(make_clouds(kind, b, n, seed=7 + n))
        ref = G.ref_fps(xyz, m)
        cases[f"fps/{kind}/{b}/{n}/{m}"] = [D(ref), D(G.ref_gather_point(xyz, ref))]
    n = 1100
    xyz = np.zeros((2, n, 3), np.float32)
    xyz[:, 1:, 0] = 1.0
    xyz[:, 600:, 0] = -1.0
    xyz[1, :, 1] = 0.25
    cases["fps_ties"] = D(G.ref_fps(G.cu(xyz), 5))
    cases["fps_oversampled"] = D(G.ref_fps(G.cu(make_clouds("ball", 2, 5, seed=1)), 9))
    for kind, b, n, m, r, k in [("ball", 32, 2048, 512, 0.2, 32), ("shell", 32, 2048, 512, 0.2, 64),
                                ("dup", 32, 512, 128, 0.4, 64), ("ball", 4, 4096, 1024, 0.1, 16)]:
        xyz = G.cu(make_clouds(kind, b, n, seed=n + k + 1))
        q = G.ref_gather_point(xyz, G.ref_fps(xyz, m))            # FPS + gather are bit-exact to the reference's (fps/...)
        cases[f"ball_query/{kind}/{b}/{n}/{m}/{r}/{k}"] = [D(a) for a in G.ref_query_ball_point(r, k, xyz, q)]
    g = np.arange(-8, 9, dtype=np.float32) * np.float32(0.05)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(1, -1, 3).astype(np.float32)
    q = np.zeros((1, 3, 3), np.float32)
    q[0, 1] = [0.05, 0.1, -0.15]
    q[0, 2] = [1e-3, -2e-3, 3e-3]
    for r in (0.05, 0.1, 0.15, 0.2, 0.25, 0.3, 0.0707, 0.0866, np.nextafter(np.float32(0.2), np.float32(1))):
        cases[f"ball_query_radius/{float(r)!r}"] = [D(a) for a in G.ref_query_ball_point(float(r), 64, G.cu(xyz), G.cu(q))]
    x2 = make_clouds("ball", 2, 200, seed=3)
    x2[0, 5] = np.nan
    x2[1, 9, 2] = np.inf
    cases["ball_query_nonfinite"] = [D(a) for a in G.ref_query_ball_point(0.3, 16, G.cu(x2), G.cu(x2[:, 20:40].copy()))]
    for c in (3, 7, 64, 128):
        rng = np.random.default_rng(c)
        pts = rng.standard_normal((3, 90, c)).astype(np.float32)
        idx = rng.integers(0, 90, size=(3, 17, 9), dtype=np.int32)
        cases[f"group_point/{c}"] = D(G.ref_group_point(G.cu(pts), G.cu(idx)))
    rng = np.random.default_rng(1)
    d = rng.random((3, 9, 300), dtype=np.float32)
    d[0, 0, 10:40] = d[0, 0, 3]
    d[1, 1, :] = 0.25
    d[2, 2, ::7] = np.nan
    for k in (1, 8, 32, 300):
        cases[f"selection_sort/{k}"] = [D(a) for a in G.ref_selection_sort(k, G.cu(d))]

    # ---- tests/test_ref_speed_gpu.py: outputs and CUDA-event times of the reference's kernels at the SSG shapes, each level
    # fed by the reference's own previous level
    import ctypes as C
    ref = orc.refgpu()
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    B = 32
    xyz, feats, dist = ssg_inputs()
    temp = torch.empty((32, 2048), dtype=torch.float32, device="cuda")
    i1, x1 = torch.zeros((B, 512), dtype=torch.int32, device="cuda"), torch.zeros((B, 512, 3), device="cuda")
    i2, x2 = torch.zeros((B, 128), dtype=torch.int32, device="cuda"), torch.zeros((B, 128, 3), device="cuda")
    q1, c1 = torch.zeros((B, 512, 32), dtype=torch.int32, device="cuda"), torch.zeros((B, 512), dtype=torch.int32, device="cuda")
    q2, c2 = torch.zeros((B, 128, 64), dtype=torch.int32, device="cuda"), torch.zeros((B, 128), dtype=torch.int32, device="cuda")
    grouped = torch.empty((B, 128, 64, 128), device="cuda")
    so, sv = torch.empty((B, 128, 512), dtype=torch.int32, device="cuda"), torch.empty((B, 128, 512), device="cuda")

    def fps1():
        ref.ref_fps(B, 2048, 512, p(xyz), p(temp), p(i1), 0)
        ref.ref_gather_point(B, 2048, 512, p(xyz), p(i1), p(x1), 0)

    def fps2():
        ref.ref_fps(B, 512, 128, p(x1), p(temp), p(i2), 0)
        ref.ref_gather_point(B, 512, 128, p(x1), p(i2), p(x2), 0)

    launches = [
        ("fps+gather 2048->512", fps1, lambda: [i1, x1]),
        ("fps+gather 512->128", fps2, lambda: [i2, x2]),
        ("query_ball_point r=0.2 k=32 (2048, 512)",
         lambda: ref.ref_query_ball_point(B, 2048, 512, C.c_float(0.2), 32, p(xyz), p(x1), p(q1), p(c1), 0), lambda: [q1, c1]),
        ("query_ball_point r=0.4 k=64 (512, 128)",
         lambda: ref.ref_query_ball_point(B, 512, 128, C.c_float(0.4), 64, p(x1), p(x2), p(q2), p(c2), 0), lambda: [q2, c2]),
        ("group_point C=128 (128 MiB out)", lambda: ref.ref_group_point(B, 512, 128, 128, 64, p(feats), p(q2), p(grouped), 0),
         lambda: [grouped]),
        ("selection_sort k=32 (4096 rows x 512)", lambda: ref.ref_selection_sort(B, 512, 128, 32, p(dist), p(so), p(sv), 0),
         lambda: [so[..., :32]]),
    ]
    ref_us = {}
    for name, launch, outs in launches:
        ref_us[name] = round(time_us(launch), 1)
        cases[f"ssg/{name}"] = [D(o) for o in outs()]
    smi = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    _dump(os.path.join(outdir, "ref_gpu_ops.json"),
          {"measured_on": smi or torch.cuda.get_device_name(), "reference_kernel_us": ref_us, **cases})


if __name__ == "__main__":
    mode, outdir = sys.argv[1], sys.argv[2]
    os.makedirs(outdir, exist_ok=True)
    {"cpu": cpu, "gpu": gpu}[mode](outdir)
    print("golden written to", outdir, sorted(os.listdir(outdir)))
