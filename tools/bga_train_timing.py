"""Step time of one pointnet2_cls_bga training step at B=32, N=2048 (pointnet2/train_seg.py's sess.run(train_op)) on the B200:
  - PointNet2BgaTrainer.train_step (hand-written kernels: FP modules without the interpolated / concatenated tensors, fused loss);
  - the autograd assembly on the same inputs: pointnet2_cls_bga.get_model(is_training=True) + get_loss().backward() + torch Adam;
  - the trainer's per-stage split: dropout masks, SA levels, FC head, FP modules, seg head, loss, backward, Adam.
CUDA events after warm-up; the L2 (126 MB) is flushed before every timed step by overwriting a 256 MB buffer, outside the timed window.
The GPU name and power limit are read in the same run.  Writes profiles/<name>.json (default bga_train_timing) and prints it."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from scanobjectnn_b200 import pointnet2_cls_bga as bga
from scanobjectnn_b200.synthetic import make_clouds
from scanobjectnn_b200.training import PointNet2BgaTrainer

B, N, WARMUP, STEPS = 32, 2048, 5, 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout.strip() else (torch.cuda.get_device_name(), "not read")
    return name, power


def main(out_name="bga_train_timing"):
    assert torch.cuda.is_available(), "bga_train_timing needs a GPU"
    torch.cuda.set_device(0)
    flush = torch.empty(64 * 2**20, device="cuda")
    xyz_np = make_clouds("ball", B, N, seed=1001)
    xyz = torch.from_numpy(xyz_np).cuda()
    labels = torch.from_numpy((np.arange(B) % 15).astype(np.int32)).cuda()
    mask = torch.from_numpy((xyz_np[..., 2] > 0).astype(np.int32)).cuda()

    def timed(fn):
        for _ in range(WARMUP):
            fn(None)
        torch.cuda.synchronize()
        tot, parts = [], {}
        for _ in range(STEPS):
            flush.fill_(1.0)
            ev = {}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(ev)
            e1.record()
            torch.cuda.synchronize()
            tot.append(e0.elapsed_time(e1))
            names = list(ev)
            prev = e0
            for k in names:
                parts.setdefault(k, []).append(prev.elapsed_time(ev[k]))
                prev = ev[k]
        return float(np.median(tot)), {k: float(np.median(v)) for k, v in parts.items()}

    # ---- trainer ----
    tr = PointNet2BgaTrainer(bga.init_params(seed=1), B, N, 15)

    def mark(ev, key):
        if ev is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            ev[key] = e

    def trainer_step(ev):
        tr.train_step(xyz, labels, mask, lr=1e-3)

    def trainer_stages(ev):
        if ev is None:
            return trainer_step(ev)
        # the calls train_step makes, with an event after each stage
        tr.draw_dropout()
        mark(ev, "dropout_masks")
        feat = tr._levels_forward(xyz, None, 0.5)
        mark(ev, "sa_levels_forward")
        cls = tr._head_forward(feat, 0.5)
        mark(ev, "fc_head_forward")
        tr._fps_forward(0.5)
        mark(ev, "fp_modules_forward")
        tr._seg_forward(0.5)
        mark(ev, "seg_head_forward")
        seg = tr.seg[-1].y.view(B, N, -1)
        loss, dcls, dseg = tr.loss_and_grad(cls, seg, labels, mask)
        mark(ev, "loss")
        tr.backward(dcls, dseg)
        mark(ev, "backward")
        tr.allreduce_grads()
        tr.adam(1e-3)
        mark(ev, "adam")

    step_ms, _ = timed(trainer_step)
    stages_ms, split = timed(trainer_stages)
    peak_trainer = torch.cuda.max_memory_allocated() / 2**20
    # ---- autograd assembly ----
    pa = bga.init_params(seed=1)
    bga.get_model(xyz, True, bn_decay=0.5, params=pa)
    flat = pa._flat.flat
    opt = torch.optim.Adam([flat], lr=1e-3)

    def autograd_step(ev):
        flat.grad = None
        cp, sp = bga.get_model(xyz, True, bn_decay=0.5, params=pa)
        loss = bga.get_loss(cp, sp, labels, mask)[0]
        loss.backward()
        with torch.no_grad():
            opt.step()
        pa.invalidate()

    auto_ms, _ = timed(autograd_step)
    name, power = gpu_info()
    res = dict(workload=f"pointnet2_cls_bga training step, B={B}, N={N}", gpu=name, power_limit=power, warmup=WARMUP, steps=STEPS,
               l2="flushed before every timed step (256 MB overwrite outside the timed window)",
               trainer_train_step_ms=step_ms, autograd_step_ms=auto_ms, speedup=auto_ms / step_ms,
               trainer_stage_ms=split, trainer_staged_step_ms=stages_ms,
               stage_note="a separate timed pass of the same step with an event between consecutive stages (the calls train_step makes); "
                          "median over the steps of each stage's time since the previous event",
               peak_memory_mib_after_trainer=peak_trainer)
    out_dir = os.environ.get("BGA_TIMING_OUT", os.path.join(ROOT, "profiles"))
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f"{out_name}.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main(*sys.argv[1:2])
