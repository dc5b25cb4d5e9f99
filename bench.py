#!/usr/bin/env python
"""bench.py -- clouds/s of the PointNet++ (SSG) point-set-abstraction forward on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one inference forward of pointnet2_cls_ssg (FPS -> fused ball-query/group/MLP/max-pool x2 ->
group-all MLP -> FC head, BN in moving-average mode) over one batch of B=32 synthetic clouds of N=2048 points
(BASELINE.json configs[1]).  Prints ONE JSON line (contract in the task statement):
  value     clouds/s with the batch already resident in HBM (inputs rotate through a pool > L2);
  e2e       same metric through the public API with HOST (pinned) buffers: H2D of the batch + forward + D2H logits;
  roofline  the dominant kernel of the step, timed live with CUDA events on the launching stream;
  cpu_baseline  the oracle port of the same forward on the host cores, on a bounded sample.
`--dump-outputs DIR` writes the logits of the last timed step (rank 0) as DIR/logits.npy, float32 (B, 15).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.
`--impl reference` times only the CPU arm (there is no runnable TensorFlow here; see DESIGN.md).
"""
from __future__ import annotations

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

if "reference" in sys.argv and os.environ.get("RANK", "0") == "0" and "TORCHELASTIC_RUN_ID" in os.environ:
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0 alone and is meant to use every host core
    # (set before numpy / the OpenMP runtime load)
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = str(os.cpu_count() or 1)

B, N, NUM_CLASS = 32, 2048, 15
WORKLOAD = "pointnet2_cls_ssg inference forward, B=32 N=2048 K=32/64, 15 classes (BASELINE.json configs[1])"
METRIC = "point-clouds/sec (B=32, N=2048, 15-class)"

# algorithmic work per step (SURVEY.md 8d / DESIGN.md): fp32 flops of the grouped MLPs per 32-cloud batch
SA_FLOPS = {"sa1": 2 * 524288 * (3 * 64 + 64 * 64 + 64 * 128), "sa2": 2 * 262144 * (131 * 128 + 128 * 128 + 128 * 256),
            "sa3": 2 * 4096 * (259 * 256 + 256 * 512 + 512 * 1024)}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


class CpuForward:
    """Oracle port of the SSG forward on the host cores: C restatement (OpenMP over the batch) for FPS / ball query / group,
    fp32 GEMMs on every core for conv+BN+ReLU+max (oracle.mlp_oracle.pointnet2_cls_ssg_fast: one GEMM per layer over all
    grouped rows through torch-CPU, batch norm folded, in-place ReLU).  Weights and clouds are made once, outside any timer."""

    def __init__(self):
        from oracle import mlp_oracle as mo
        from scanobjectnn_b200 import pointnet2_cls_ssg
        from scanobjectnn_b200.synthetic import make_clouds

        self.mo = mo
        try:
            self.cores = len(os.sched_getaffinity(0)) or 1           # the cores this process may run on
        except AttributeError:
            self.cores = os.cpu_count() or 1
        self.params = pointnet2_cls_ssg.init_params(seed=1, device="cpu", randomize_bn=True)
        self.xyz = make_clouds("ball", B, N, seed=1001)
        self.run(1)                                                   # warm-up (page in the GEMM library, thread pools)

    def run(self, n_clouds: int) -> float:
        """one forward over the first n_clouds clouds of the batch; returns seconds"""
        t0 = time.perf_counter()
        self.mo.pointnet2_cls_ssg_fast(self.xyz[:n_clouds], self.params, threads=self.cores)
        return time.perf_counter() - t0


def run_reference(args):
    """The reference arm: the CPU implementation of the same forward on the box's host cores (the reference's TF1 path
    is not installable here -- DESIGN.md section 4 -- so this is the oracle port: C/OpenMP restatement of the reference
    kernels for FPS / ball query / group, one fp32 GEMM per layer on all cores (torch-CPU) for conv+BN+ReLU+max).  Each step is a
    bounded sample of the 32-cloud batch, sized so that the whole run stays within ~90 s of CPU work."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cpu = CpuForward()
    cores = cpu.cores
    probe = 8 / min(cpu.run(8), cpu.run(8))                # clouds/s, also the warm-up at batch scale
    budget_s = 90.0
    sample = int(max(1, min(B, budget_s * probe / max(args.steps, 1))))
    for _ in range(max(args.warmup, 1)):
        cpu.run(sample)
    t0 = time.perf_counter()
    done = 0
    for _ in range(args.steps):
        cpu.run(sample)
        done += sample
    dt = time.perf_counter() - t0
    value = done / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "clouds/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": f"{sample} of the 32 clouds per step"},
        "cpu_baseline": {"value": value, "unit": "clouds/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} clouds x {args.steps} steps ({dt:.1f} s), oracle port (C/OpenMP index ops + fp32 GEMMs on all cores, torch-CPU); "
                                   "the reference's TF1 path is not installable here"},
        "e2e": {"value": value, "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _ev_time(fn, reps, flush=None, sink=None, spin=400_000):
    """median CUDA-event time (us) of fn(); with `flush`, L2 is flushed by READING it (clean lines) before every launch and
    a ~0.2 ms spin kernel sits in front so the host has enqueued e0 / fn / e1 before the GPU gets there"""
    import torch
    ts = []
    for _ in range(reps):
        if flush is not None:
            sink.copy_(flush.sum())
            torch.cuda._sleep(spin)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def run_training_bench(args, dev, rank, world, local_rank):
    """Second workload of the line: one TRAINING step of pointnet2_cls_ssg per B=32 batch and GPU (pointnet2/train.py:246-252:
    forward with batch-statistics BN, loss, backward, one flat-bucket NCCL all-reduce of the gradients, Adam).  Returns the
    `train` object (rank 0) or None."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from scanobjectnn_b200 import pointnet2_cls_ssg
    from scanobjectnn_b200.shard import max_over_ranks, rank_seed
    from scanobjectnn_b200.synthetic import make_clouds
    from scanobjectnn_b200.training import PointNet2ClsTrainer

    if args.no_train:
        return None
    params = pointnet2_cls_ssg.init_params(seed=1, device=dev)          # identical initial weights on every rank
    tr = PointNet2ClsTrainer(params, B, N, NUM_CLASS, device=dev)
    NPOOL = 8
    pool = [torch.from_numpy(make_clouds("ball", B, N, seed=rank_seed(2001 + i, rank))).to(dev) for i in range(NPOOL)]
    labels = torch.from_numpy(np.random.default_rng(rank).integers(0, NUM_CLASS, B).astype(np.int32)).to(dev)
    steps = max(4, min(args.steps, args.train_steps))
    warm = 3

    def step(i):
        return tr.train_step(pool[i % NPOOL], labels, lr=1e-3, bn_decay=0.5)

    for i in range(warm):
        step(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loss = step(warm + i)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), device=dev)
    # the all-reduce alone (the only data-path collective of the whole framework): flat fp32 bucket, NCCL over NVLink
    ar_us = None
    if world > 1:
        for _ in range(3):
            dist.all_reduce(tr.fp.grad)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        a0.record()
        for _ in range(20):
            dist.all_reduce(tr.fp.grad)
        a1.record()
        torch.cuda.synchronize()
        ar_us = max_over_ranks(a0.elapsed_time(a1) * 1e3 / 20, device=dev)
    # phases of one step on rank 0 (device time, eager launches)
    phases = {}
    if rank == 0 and world == 1:
        x = pool[0]
        tr.draw_dropout()
        torch.cuda.synchronize()
        out = {}
        phases["forward_us"] = _ev_time(lambda: out.__setitem__("l", tr.forward(x, 0.5)), 5)
        dl = tr.loss_and_grad(out["l"], labels)[1]
        phases["backward_us"] = _ev_time(lambda: tr.backward(dl), 5)
        phases["adam_us"] = _ev_time(lambda: tr.adam(1e-3), 5)
    if rank != 0:
        return None
    flops_fwd = sum(SA_FLOPS.values()) + 2 * B * (1024 * 512 + 512 * 256 + 256 * NUM_CLASS)
    return {"workload": "pointnet2_cls_ssg TRAINING step (fwd with batch-stat BN + loss + bwd + grad all-reduce + Adam), B=32 N=2048 per GPU",
            "clouds_per_s": B * world * steps / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps, "n_gpus": world,
            "allreduce_us": ar_us, "allreduce_bytes": int(tr.fp.total * 4), "params": int(tr.fp.total),
            "loss_last": float(loss.item()), "dtype": "f32 (fp32 FMA GEMMs, fixed-order reductions: bit-reproducible gradients)",
            "approx_tflops_fp32": 3 * flops_fwd / (ms / steps * 1e-3) / 1e12, **phases}


def run_sweep(dev, peaks):
    """BASELINE.json configs[4]: FPS + ball-query sweep N x B on one GPU -- us, algorithmic GB/s vs the measured HBM peak,
    ns per FPS round.  m = N/4, r = 0.2, K = 32, uniform-ball clouds (SURVEY 8d)."""
    import torch

    from scanobjectnn_b200 import ops
    from scanobjectnn_b200.synthetic import make_clouds
    rows = []
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    sink = torch.zeros((), dtype=torch.float32, device=dev)
    for n in (1024, 2048, 4096, 8192):
        base = torch.from_numpy(make_clouds("ball", 4, n, seed=1004 + n)).to(dev)
        for b in (1, 4, 16, 64, 256):
            x = base.repeat((b + 3) // 4, 1, 1)[:b].contiguous()
            m = n // 4
            _, q = ops.farthest_point_sample_and_gather(m, x)
            ops.query_ball_point(0.2, 32, x, q)
            t_fps = _ev_time(lambda: ops.farthest_point_sample_and_gather(m, x), 3, flush, sink)
            t_bq = _ev_time(lambda: ops.query_ball_point(0.2, 32, x, q), 3, flush, sink)
            by_fps = b * (12 * n + 4 * m + 12 * m)
            by_bq = b * (12 * n + 12 * m + 4 * m * 32 + 4 * m)
            rows.append({"N": n, "B": b, "fps_us": round(t_fps, 1), "fps_ns_per_round": round(t_fps * 1e3 / max(m - 1, 1), 1),
                         "fps_gbs": round(by_fps / t_fps / 1e3, 2), "ballq_us": round(t_bq, 1), "ballq_gbs": round(by_bq / t_bq / 1e3, 1),
                         "ballq_hbm_frac": round(by_bq / t_bq / 1e3 / peaks["hbm"], 4)})
    del flush
    return {"config": "FPS (m=N/4) + ball query (r=0.2, K=32), uniform-ball clouds, L2 read-flushed before every launch, median of 3",
            "note": "FPS is bound by its m-1 dependent arg-max rounds (ns_per_round), the ball query by issue/latency: both far below "
                    "the HBM roofline by construction -- their algorithmic bytes are a few MB", "rows": rows}


def run_ref_gpu(dev, x, l1_xyz, l2_xyz, l1_pts_shape_c=128):
    """R-GPU contender (SURVEY 8d): the reference's own CUDA kernels, compiled unmodified for sm_100a by oracle/Makefile into
    oracle/_ref/libref_tfops.so, timed on the same tensors in the same run.  Reported baseline only (like cpu_baseline)."""
    import ctypes as C

    import torch
    path = os.path.join(ROOT, "oracle", "_ref", "libref_tfops.so")
    if not os.path.exists(path):
        return None
    ref = C.CDLL(path)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    out = {}
    temp = torch.empty((32, N), dtype=torch.float32, device=dev)
    i1 = torch.zeros((B, 512), dtype=torch.int32, device=dev)
    g1 = torch.zeros((B, 512, 3), dtype=torch.float32, device=dev)

    def fps1():
        ref.ref_fps(B, N, 512, p(x), p(temp), p(i1), 0)
        ref.ref_gather_point(B, N, 512, p(x), p(i1), p(g1), 0)
    out["fps1"] = _ev_time(fps1, 5)
    i2 = torch.zeros((B, 128), dtype=torch.int32, device=dev)
    g2 = torch.zeros((B, 128, 3), dtype=torch.float32, device=dev)

    def fps2():
        ref.ref_fps(B, 512, 128, p(l1_xyz), p(temp), p(i2), 0)
        ref.ref_gather_point(B, 512, 128, p(l1_xyz), p(i2), p(g2), 0)
    out["fps2"] = _ev_time(fps2, 5)
    q1 = torch.zeros((B, 512, 32), dtype=torch.int32, device=dev)
    c1 = torch.zeros((B, 512), dtype=torch.int32, device=dev)
    out["ballq1"] = _ev_time(lambda: ref.ref_query_ball_point(B, N, 512, C.c_float(0.2), 32, p(x), p(l1_xyz), p(q1), p(c1), 0), 5)
    q2 = torch.zeros((B, 128, 64), dtype=torch.int32, device=dev)
    c2 = torch.zeros((B, 128), dtype=torch.int32, device=dev)
    out["ballq2"] = _ev_time(lambda: ref.ref_query_ball_point(B, 512, 128, C.c_float(0.4), 64, p(l1_xyz), p(l2_xyz), p(q2), p(c2), 0), 5)
    # the grouping the reference needs in front of its convolutions (group_point of xyz at SA1, of xyz + features at SA2)
    gx = torch.empty((B, 512, 32, 3), dtype=torch.float32, device=dev)
    out["group_sa1"] = _ev_time(lambda: ref.ref_group_point(B, N, 3, 512, 32, p(x), p(q1), p(gx), 0), 5)
    feats = torch.randn((B, 512, l1_pts_shape_c), device=dev)
    gf = torch.empty((B, 128, 64, l1_pts_shape_c), dtype=torch.float32, device=dev)
    out["group_sa2"] = _ev_time(lambda: ref.ref_group_point(B, 512, l1_pts_shape_c, 128, 64, p(feats), p(q2), p(gf), 0), 5)
    return {k: round(v, 1) for k, v in out.items()}


def _traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu summary (profiles/traffic.json), else None"""
    pth = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(pth):
        return None, None
    with open(pth) as f:
        d = json.load(f)
    e = d.get(kernel_key)
    return (e["bytes"], e["source"]) if e else (None, None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=6, help="batches kept in flight (1 = strictly one step at a time; measured 4: 93.9 k, 6: 95.8 k, 8: 95.4 k clouds/s)")
    ap.add_argument("--no-extra", action="store_true", help="skip the BGA / DGCNN / single-op / sweep measurements")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step measurement")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's logits (rank 0) as DIR/logits.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from scanobjectnn_b200 import _lib, ops, pointnet2_cls_ssg
    from scanobjectnn_b200.shard import max_over_ranks, rank_seed
    from scanobjectnn_b200.synthetic import make_clouds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)      # communicator bound to this rank's GPU up front
    _lib.load()       # fail loudly if the CUDA library is missing
    solo = world == 1  # the side measurements (per-kernel times, other models, sweep, CPU arm) run on the single-GPU line only

    params = pointnet2_cls_ssg.init_params(seed=1, device=dev, randomize_bn=True)
    # input pool larger than L2 (126 MB): 192 distinct batches x 786 KB = 151 MB, rotated every step
    POOL = 192
    base = make_clouds("ball", B, N, seed=rank_seed(1001, rank))
    rng = np.random.default_rng(rank)
    pool_host = torch.empty((POOL, B, N, 3), dtype=torch.float32).pin_memory()
    for i in range(POOL):
        perm = rng.permutation(N)
        pool_host[i] = torch.from_numpy(base[:, perm, :])          # same geometry, different point order
    pool_dev = pool_host.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    # ---- the public inference API: CUDA graph of one forward per slot, `slots` independent batches in flight ----
    # (step i -> slot i % slots; the next step's FPS -- one CTA per cloud, latency-bound -- overlaps the current step's
    #  tensor-core kernels, which hand their tiles out dynamically)
    from scanobjectnn_b200.engine import pointnet2_cls_ssg_engine
    NSTREAMS = max(1, args.streams)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(engine, host, steps, warmup):
        def step_fn(i):
            if host:
                return engine.submit(pool_host[i % POOL], to_host=True)    # pinned host batch in, logits back to pinned host memory
            return engine.submit(pool_dev[i % POOL])                       # device-resident batch (rotating pool > L2)
        for i in range(warmup):
            step_fn(i)
        barrier()
        main = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        engine.fence_begin(e0)
        for i in range(steps):
            last = step_fn(warmup + i)
        engine.fence_end(main)
        e1.record(main)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), device=dev), last       # ms, slot holding the last step's logits

    engine = pointnet2_cls_ssg_engine(params, batch=B, npoints=N, num_class=NUM_CLASS, slots=NSTREAMS, device=dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_res, last_slot = timed(engine, False, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:           # read now: the host-buffer run below reuses the slots
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "logits.npy"), engine.result(last_slot).cpu().numpy().astype(np.float32))
    ms_e2e, _ = timed(engine, True, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    ms_res_1 = None
    if solo and NSTREAMS > 1:
        engine1 = pointnet2_cls_ssg_engine(params, batch=B, npoints=N, num_class=NUM_CLASS, slots=1, device=dev)
        n1 = max(args.steps // 4, 8)
        ms_res_1 = timed(engine1, False, n1, args.warmup)[0] / n1
        del engine1

    train = run_training_bench(args, dev, rank, world, local_rank)

    # ---- per-stage device times (eager launches, CUDA events on the launching stream) ----
    stages, ref_gpu, f1 = {}, None, {}
    if rank == 0 and solo:
        import ctypes as C
        x = pool_dev[1].contiguous()
        p = params
        mlp1 = p.mlp([f"layer1/conv{i}" for i in range(3)])
        mlp2 = p.mlp([f"layer2/conv{i}" for i in range(3)])
        mlp3 = p.mlp([f"layer3/conv{i}" for i in range(3)])
        head = p.mlp(["fc1", "fc2", "fc3"], [True, True, False])
        _, l1_xyz = ops.farthest_point_sample_and_gather(512, x)
        l1_pts, idx1, _ = ops.sa_module_infer(x, l1_xyz, None, 0.2, 32, mlp1, return_idx=True)
        _, l2_xyz = ops.farthest_point_sample_and_gather(128, l1_xyz)
        l2_pts, idx2, _ = ops.sa_module_infer(l1_xyz, l2_xyz, l1_pts, 0.4, 64, mlp2, return_idx=True)
        l3 = ops.sa_group_all_infer(l2_xyz, l2_pts, mlp3)
        cases = {
            "fps1": lambda: ops.farthest_point_sample_and_gather(512, x),
            "ballq1": lambda: ops.query_ball_point(0.2, 32, x, l1_xyz),
            "sa1_mlp": lambda: ops.sa_module_infer(x, l1_xyz, None, 0.2, 32, mlp1, idx=idx1),
            "fps2": lambda: ops.farthest_point_sample_and_gather(128, l1_xyz),
            "ballq2": lambda: ops.query_ball_point(0.4, 64, l1_xyz, l2_xyz),
            "sa2_mlp": lambda: ops.sa_module_infer(l1_xyz, l2_xyz, l1_pts, 0.4, 64, mlp2, idx=idx2),
            "sa3_mlp": lambda: ops.sa_group_all_infer(l2_xyz, l2_pts, mlp3),
            "head": lambda: ops.shared_mlp(l3, head),
        }
        flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)   # 256 MB > L2
        flush_sink = torch.zeros((), dtype=torch.float32, device=dev)
        for name, fn in cases.items():
            for _ in range(3):
                fn()
            stages[name] = _ev_time(fn, 10, flush, flush_sink)
        # variant F1 (training-mode front of SA1): ball query + group + centre + conv1 -> pre-BN (B,m,K,64) + idx + BN stats.
        # Timed through the C ABI with preallocated buffers (one ctypes call per launch): (a) isolated, L2 read-flushed in
        # front; (b) steady state, 50 launches back to back into the same buffers (every byte has to reach HBM).
        lib = _lib.load()
        w1 = p["layer1/conv0/weights"].reshape(3, 64).contiguous()
        b1 = p["layer1/conv0/biases"]
        pre = torch.empty((B, 512, 32, 64), device=dev)
        fidx = torch.empty((B, 512, 32), dtype=torch.int32, device=dev)
        fcnt = torch.empty((B, 512), dtype=torch.int32, device=dev)
        fstats = torch.empty((2, 64), device=dev)
        need = lib.psa_sa_conv1_prebn_workspace_bytes(B, N, 512, 0, 64, 1)
        fws = torch.empty(need // 4 + 1, device=dev)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        vp = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

        def f1_launch():
            rc = lib.psa_sa_conv1_prebn(B, N, 512, 0, C.c_float(0.2), 32, vp(x), vp(l1_xyz), C.c_void_p(0), vp(w1), vp(b1), 64, vp(pre), vp(fidx),
                                        vp(fcnt), vp(fstats), vp(fws), C.c_size_t(need), st)
            assert rc == 0, rc
        for _ in range(3):
            f1_launch()
        f1["isolated_us"] = _ev_time(f1_launch, 15, flush, flush_sink)
        torch.cuda._sleep(2_000_000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            f1_launch()
        e1.record()
        torch.cuda.synchronize()
        f1["steady_us"] = e0.elapsed_time(e1) * 1e3 / 50
        assert torch.equal(fidx, idx1), "F1 neighbourhoods differ from the ball query's"
        del flush
        ref_gpu = run_ref_gpu(dev, x, l1_xyz, l2_xyz)

    extra = {}
    if rank == 0 and solo and not args.no_extra:
        from scanobjectnn_b200 import dgcnn, pointnet2_cls_bga, pointnet_cls
        from scanobjectnn_b200.engine import InferenceEngine

        pool_dev_full = pool_dev

        def time_graph(fn, out_shape, reps=12, bs=B, n=N):
            """The same engine as the main workload (CUDA graph per slot, NSTREAMS batches in flight): ms per forward."""
            eng = InferenceEngine(fn, (bs, n, 3), out_shape, slots=NSTREAMS, device=dev)
            pool_dev = [t[:bs, :n].contiguous() for t in pool_dev_full] if (bs, n) != (B, N) else pool_dev_full
            for i in range(NSTREAMS):
                eng.submit(pool_dev[(3 + i) % POOL])
            torch.cuda.synchronize()
            main = torch.cuda.current_stream()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(main)
            eng.fence_begin(e0)
            for i in range(reps):
                eng.submit(pool_dev[(7 + i) % POOL])
            eng.fence_end(main)
            e1.record(main)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        p_bga = pointnet2_cls_bga.init_params(seed=2, device=dev, randomize_bn=True)
        ms = time_graph(lambda t: pointnet2_cls_bga.get_model(t, False, params=p_bga)[0], (B, NUM_CLASS))
        extra["pointnet2_cls_bga"] = {"workload": "inference forward B=32 N=2048 (BASELINE.json configs[3] per-GPU shape)", "ms_per_step": ms,
                                      "clouds_per_s": B / (ms * 1e-3)}
        p_dg = dgcnn.init_params(seed=3, device=dev, randomize_bn=True)
        ms = time_graph(lambda t: dgcnn.get_model(t, False, params=p_dg)[0], (B, NUM_CLASS), reps=8)
        extra["dgcnn"] = {"workload": "inference forward k=20 B=32 N=2048 (BASELINE.json configs[2])", "ms_per_step": ms,
                          "clouds_per_s": B / (ms * 1e-3)}
        p_pn = pointnet_cls.init_params(seed=4, device=dev, randomize_bn=True)
        ms = time_graph(lambda t: pointnet_cls.get_model(t, False, params=p_pn)[0], (8, NUM_CLASS), reps=24, bs=8, n=1024)
        extra["pointnet_cls_vanilla"] = {"workload": "inference forward B=8 N=1024 (BASELINE.json configs[0])", "ms_per_step": ms,
                                         "clouds_per_s": 8 / (ms * 1e-3)}
        # single ops of the remaining scope rows, event-timed with an L2 flush + spin in front
        xq = pool_dev[5].contiguous()
        feats64 = torch.randn((B, N, 64), device=dev)
        nn20 = ops.knn_graph(feats64, 20)
        _, l1x = ops.farthest_point_sample_and_gather(512, xq)
        f128 = torch.randn((B, 512, 128), device=dev)
        mlp_e = ops.MlpParams([(torch.randn((128, 64), device=dev) * 0.1, torch.ones(64, device=dev), torch.zeros(64, device=dev), True)])
        bidx, _ = ops.query_ball_point(0.2, 32, xq, l1x)
        fidx2 = ops.farthest_point_sample(512, xq)
        nn3_d, nn3_i = ops.three_nn(xq, l1x)
        w3 = torch.full((B, N, 3), 1.0 / 3, device=dev)
        adj = ops.pairwise_distance(xq)
        aug = ops.draw_augmentation(B, N, N, dev)
        opcases = {
            "augment_batch_subset_rotate_jitter": (lambda: ops.augment_batch(xq, N, **aug), None, B * (12 * N + 12 * N + 12 * N) + 4 * N),
            "gather_point_512": (lambda: ops.gather_point(xq, fidx2), None, B * (12 * N + 4 * 512 + 12 * 512)),
            "group_point_c64_k32": (lambda: ops.group_point(feats64, bidx), None, B * (4 * N * 64 + 4 * 512 * 32 + 4 * 512 * 32 * 64)),
            "knn_point_k32": (lambda: ops.knn_point(32, xq, l1x), None, B * (12 * N + 12 * 512 + 8 * 512 * 32)),
            "three_nn_2048from512": (lambda: ops.three_nn(xq, l1x), None, B * (12 * N + 12 * 512 + 24 * N)),
            "three_interpolate_c128": (lambda: ops.three_interpolate(f128, nn3_i, w3), None, B * (4 * 512 * 128 + 24 * N + 4 * N * 128)),
            "pairwise_distance_c3": (lambda: ops.pairwise_distance(xq), 2.0 * B * N * N * 3, B * (12 * N + 4 * N * N)),
            "knn_top20_of_adj": (lambda: ops.knn(adj, 20), None, B * (4 * N * N + 4 * N * 20)),
            "get_edge_feature_c64_k20": (lambda: ops.get_edge_feature(feats64, nn20, 20), None, B * (4 * N * 64 + 4 * N * 20 + 4 * N * 20 * 128)),
            "knn_graph_c3": (lambda: ops.knn_graph(xq, 20), 2.0 * B * N * N * 3, B * (4 * N * 3 + 4 * N * 20)),
            "knn_graph_c64": (lambda: ops.knn_graph(feats64, 20), 2.0 * B * N * N * 64, B * (4 * N * 64 + 4 * N * 20)),
            "edgeconv_128to64": (lambda: ops.edgeconv_infer(feats64, nn20, mlp_e), 2.0 * B * N * 64 * 128, B * (4 * N * 64 + 4 * N * 20 + 4 * N * 64)),
            "three_nn_interp_2048from512_c128": (lambda: ops.three_nn_interpolate(xq, l1x, f128), None, B * (12 * N + 12 * 512 + 4 * 512 * 128 + 4 * N * 128)),
        }
        flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
        flush_sink = torch.zeros((), dtype=torch.float32, device=dev)
        extra["ops"] = {}
        for name, (fn, flops, nbytes) in opcases.items():
            for _ in range(2):
                fn()
            us = _ev_time(fn, 5, flush, flush_sink)
            extra["ops"][name] = {"us": us, "alg_bytes": nbytes, "gbs": nbytes / (us * 1e-6) / 1e9,
                                  **({"tflops_fp32": flops / (us * 1e-6) / 1e12} if flops else {})}
        del flush
        extra["fps_ballq_sweep"] = run_sweep(dev, _peaks())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = _peaks()
    clouds = B * world * args.steps
    value = clouds / (ms_res * 1e-3)
    e2e_v = clouds / (ms_e2e * 1e-3)
    roofline = roofline_f1 = None
    kern = {}
    if stages:
        # dominant kernel of the step
        dom = max(stages, key=stages.get)
        flops = {"sa1_mlp": SA_FLOPS["sa1"], "sa2_mlp": SA_FLOPS["sa2"], "sa3_mlp": SA_FLOPS["sa3"]}.get(dom)
        if flops:
            ach = flops / (stages[dom] * 1e-6) / 1e12
            # share of the level's flops that runs on the tensor cores (layers after the first); each fp32 product is three f16 MMAs
            tc_flops = {"sa1_mlp": 2 * 524288 * (64 * 64 + 64 * 128), "sa2_mlp": 2 * 262144 * (128 * 128 + 128 * 256) + 2 * 16384 * 128 * 128,
                        "sa3_mlp": 2 * 4096 * (256 * 256 + 256 * 512 + 512 * 1024)}[dom]
            traffic, tsrc = _traffic(dom)
            roofline = {"kernel": dom + " (tc_sa_dual_kernel + its per-source-point first-layer GEMM)" if dom != "sa3_mlp" else dom + " (3 x tc_dense3_kernel)",
                        "bound": "tensor", "achieved": ach, "peak": peaks["tf"], "unit": "TFLOP/s",
                        "frac": ach / peaks["tf"], "traffic": traffic, "traffic_source": tsrc, "peak_source": peaks["src"] + " bf16 burst",
                        "algorithmic_flops": flops,
                        "note": "achieved = SURVEY 8d fp32 MLP flops of the level / measured stage time. fp32 parity (1e-5) is kept by splitting "
                                "both operands into two fp16 pieces: three f16 MMAs per product (fp32 accumulate), so the tensor pipe executes "
                                "3x the tensor-core share of these flops (tensor_pipe_frac; the bf16x3 mode of round 1 executed 6x).",
                        "tensor_pipe_frac": 3.0 * tc_flops / (stages[dom] * 1e-6) / 1e12 / peaks["tf"]}
        else:
            fps_bytes = B * (12 * N + 4 * 512)
            ach = fps_bytes / (stages[dom] * 1e-6) / 1e9
            roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                        "traffic": None, "peak_source": peaks["src"], "note": "latency-bound dependent arg-max rounds"}
        # HBM-class kernels of the metric's second half ("FPS+ballq HBM GB/s")
        kern = {
            "fps1": {"us": stages["fps1"], "alg_bytes": B * (12 * N + 4 * 512 + 12 * 512), "ns_per_round": stages["fps1"] * 1e3 / 511},
            "ballq1": {"us": stages["ballq1"], "alg_bytes": B * (12 * N + 12 * 512 + 4 * 512 * 32 + 4 * 512)},
            "fps2": {"us": stages["fps2"], "alg_bytes": B * (12 * 512 + 4 * 128 + 12 * 128), "ns_per_round": stages["fps2"] * 1e3 / 127},
            "ballq2": {"us": stages["ballq2"], "alg_bytes": B * (12 * 512 + 12 * 128 + 4 * 128 * 64 + 4 * 128)},
        }
        for k, v in kern.items():
            v["gbs"] = v["alg_bytes"] / (v["us"] * 1e-6) / 1e9
            v["hbm_frac"] = v["gbs"] / peaks["hbm"]
            if ref_gpu and k in ref_gpu:
                v["ref_gpu_us"] = ref_gpu[k]          # the reference's own kernel (sm_100a build) on the same tensors
        for k in ("sa1_mlp", "sa2_mlp", "sa3_mlp"):
            kern[k] = {"us": stages[k], "tflops_fp32": SA_FLOPS[k[:3]] / (stages[k] * 1e-6) / 1e12}
        if ref_gpu:
            kern["sa1_mlp"]["ref_gpu_us_group_point_only"] = ref_gpu["group_sa1"]    # the reference's convs are cuDNN (TF absent):
            kern["sa2_mlp"]["ref_gpu_us_group_point_only"] = ref_gpu["group_sa2"]    # its grouping alone is a lower bound
        kern["head"] = {"us": stages["head"]}
        # F1: B*(12n + 12m) in, 4*B*m*K*C1 (pre-BN) + 4*B*m*K (idx) + 4*B*m (pts_cnt) out  (SURVEY 8d: 137.3 MB)
        f1_bytes = B * (12 * N + 12 * 512) + 4 * B * 512 * 32 * 64 + 4 * B * 512 * 32 + 4 * B * 512
        gbs_iso = f1_bytes / (f1["isolated_us"] * 1e-6) / 1e9
        gbs_std = f1_bytes / (f1["steady_us"] * 1e-6) / 1e9
        kern["sa1_f1"] = {"us": f1["isolated_us"], "steady_us": f1["steady_us"], "alg_bytes": f1_bytes, "gbs": gbs_iso, "hbm_frac": gbs_iso / peaks["hbm"],
                          "steady_gbs": gbs_std, "steady_hbm_frac": gbs_std / peaks["hbm"]}
        traffic, tsrc = _traffic("sa1_f1")
        roofline_f1 = {"kernel": "sa_conv1_stream_kernel (variant F1: fused ball-query + group + conv1, pre-BN output + BN statistics, SA1 B=32 N=2048 K=32)",
                       "bound": "hbm", "achieved": gbs_iso, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs_iso / peaks["hbm"],
                       "steady_state": {"achieved": gbs_std, "frac": gbs_std / peaks["hbm"],
                                        "note": "50 launches back to back into the same 137 MB of outputs: every byte reaches HBM inside the window"},
                       "timing": "CUDA events around one C-ABI call (memset node + kernel), L2 read-flushed (clean lines) and a spin kernel in front; median of 15",
                       "traffic": traffic, "traffic_source": tsrc, "peak_source": peaks["src"],
                       "in_timed_step": "training step only (train object); the inference step never writes the (B,m,K,C) tensor"}

    cpu = None
    if solo and not args.no_cpu_baseline:
        cf = CpuForward()
        times = []
        while len(times) < 5 or (sum(times) < 10.0 and len(times) < 60):       # ~10 s of CPU work, best forward reported
            times.append(cf.run(B))
        secs = min(times)
        cpu = {"value": B / secs, "unit": "clouds/s", "cores": cf.cores, "kind": "port",
               "sample": f"the full 32-cloud batch, best of {len(times)} forwards ({secs:.2f} s; {sum(times):.1f} s of CPU work in all): oracle port = "
                         "C/OpenMP FPS+ball-query+group, one fp32 GEMM per layer on all host cores (torch-CPU), folded BN, ReLU, max"}

    line = {
        "metric": METRIC, "value": value, "unit": "clouds/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": B * world, "per_gpu_batch": B, "points": N,
                   "l2_policy": "inputs larger than L2: 192 distinct 786 KB batches (151 MB) rotated every step",
                   "mode": "inference (BN moving averages folded); CUDA graph replay of one forward per step",
                   "streams": NSTREAMS, "in_flight": f"{NSTREAMS} independent B=32 steps in flight on {NSTREAMS} streams (step i on stream i % {NSTREAMS})",
                   "parallelism": f"dp{world} (independent batches, no data-path collective; training adds one gradient all-reduce)"},
        "one_step_at_a_time": None if ms_res_1 is None else {"ms_per_step": ms_res_1, "clouds_per_s": B / (ms_res_1 * 1e-3),
                                                             "note": "same engine with ONE slot: a step starts when the previous one has finished"},
        "e2e": {"value": e2e_v, "unit": "clouds/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": B * N * 3 * 4,
                "d2h_bytes_per_step": B * NUM_CLASS * 4},
        # kernels of libpsa.so per step: 2 FPS (+ fused gather), 2 ball queries, SA1 level + its guarded rerun, SA2 per-point GEMM + level +
        # their reruns, SA3 3 x (layer + rerun), head 3 x (K-split partial + reduce); reruns are no-ops unless a value left the fp16 range
        "gpu_launches": 22 * args.steps,
        "roofline": roofline,
        "roofline_f1": roofline_f1,
        "kernels": kern,
        "train": train,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "other_workloads": extra,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
