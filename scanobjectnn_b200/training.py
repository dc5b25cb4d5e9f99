"""Training mode of the PointNet++ classifier (pointnet2_cls_ssg) on the B200 kernels: forward with batch-statistics
batch norm through every layer, backward of the fused set-abstraction levels and the FC head, Adam, and the
data-parallel gradient all-reduce.

Reference: pointnet2/train.py:139-171 (graph: get_model(is_training) -> get_loss -> AdamOptimizer.minimize), :246-252
(the per-batch feed: rotate + jitter, one sess.run of train_op), pointnet2/utils/tf_util.py:155-185,512-531 (conv2d /
batch norm in training mode), pointnet_util.py:87-154 (set-abstraction level), tf_grouping.py:43-47 (GroupPointGrad).

How a level is stored: ONE tensor per layer, the PRE-batch-norm activations y_l (B*m*K, C_l).  relu(BN(y_l)) is recomputed
inside the next layer's GEMM operand load, the batch-norm backward inside the backward GEMMs' operand loads
(csrc/train_gemm.cuh), the max-pool keeps the winning row per (group, channel).  The first layer of a level is the fused
ball-query + group + conv1 kernel (psa_sa_conv1_prebn); its backward is a coordinate reduction plus, for levels with
features, an ORDERED gather that replaces the reference's atomicAdd GroupPointGrad, and two dense products on the source
points instead of the grouped rows.

Everything numeric runs in libpsa.so; torch provides memory, streams and torch.distributed (one flat gradient bucket,
one NCCL all-reduce per step -- SURVEY 8e).  All buffers are allocated once, so a step can be captured in a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import torch

from . import _lib, ops
from ._lib import PsaActIn, PsaGradIn, check
from .tf_util import VariableStore

_p = lambda t: C.c_void_p(0 if t is None else t.data_ptr())  # noqa: E731


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@dataclass
class LevelSpec:
    """One pointnet_sa_module call (pointnet2_cls_ssg.py:35-37)."""
    scope: str
    npoint: int | None
    radius: float | None
    nsample: int | None
    mlp: list
    group_all: bool = False


SSG_LEVELS = [LevelSpec("layer1", 512, 0.2, 32, [64, 64, 128]), LevelSpec("layer2", 128, 0.4, 64, [128, 128, 256]),
              LevelSpec("layer3", None, None, None, [256, 512, 1024], group_all=True)]
SSG_HEAD = [("fc1", 512, True, 0.5), ("fc2", 256, True, 0.5), ("fc3", None, False, None)]   # (scope, width, bn, keep_prob)


class FlatParams:
    """The trainable variables of a VariableStore re-homed as views of ONE flat fp32 tensor (same TF names), with a
    matching flat gradient tensor and Adam moments.  One bucket = one all-reduce, one Adam launch."""

    def __init__(self, params: VariableStore):
        self.params = params
        names = [k for k in params.keys() if not k.endswith(("/moving_mean", "/moving_variance"))]
        self.names = names
        dev = params[names[0]].device
        sizes = [params[k].numel() for k in names]
        pad = lambda n: (n + 63) // 64 * 64          # 256-byte aligned segments: float4 loads of the views stay legal  # noqa: E731
        offs, o = [], 0
        for n in sizes:
            offs.append(o)
            o += pad(n)
        self.total = o
        self.flat = torch.zeros(o, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(o, dtype=torch.float32, device=dev)
        self.adam_m = torch.zeros(o, dtype=torch.float32, device=dev)
        self.adam_v = torch.zeros(o, dtype=torch.float32, device=dev)
        self.views, self.gviews = {}, {}
        for k, off, n in zip(names, offs, sizes):
            shape = params[k].shape
            v = self.flat[off:off + n].view(shape)
            v.copy_(params[k])
            dict.__setitem__(params, k, v)            # the store now aliases the flat buffer
            self.views[k] = v
            self.gviews[k] = self.grad[off:off + n].view(shape)
        params.invalidate()
        self.step_count = 0

    def grad_of(self, name):
        return self.gviews[name]

    def live(self, name) -> torch.Tensor:
        """a view of the flat parameter vector taken NOW (autograd-tracked when flat.requires_grad): for variables used directly in
        torch ops (e.g. the T-net's transform_XYZ matrix) rather than through the hand-written layers"""
        v = self.views[name]
        off = (v.data_ptr() - self.flat.data_ptr()) // 4
        return self.flat[off:off + v.numel()].view(v.shape)


class _Layer:
    """conv1x1 / fully_connected (+ batch norm + relu): parameter views, gradient views and per-step buffers."""

    def __init__(self, fp: FlatParams, scope: str, rows: int, bn: bool, dev):
        p = fp.params
        w = fp.views[f"{scope}/weights"]
        self.scope = scope
        self.W = w.view(-1, w.shape[-1])
        self.K, self.N = self.W.shape
        self.b = fp.views[f"{scope}/biases"]
        self.dW = fp.gviews[f"{scope}/weights"].view(self.K, self.N)
        self.db = fp.gviews[f"{scope}/biases"]
        self.bn = bn
        self.rows = rows
        f32 = dict(dtype=torch.float32, device=dev)
        self.y = torch.empty((rows, self.N), **f32)
        if bn:
            self.gamma, self.beta = fp.views[f"{scope}/bn/gamma"], fp.views[f"{scope}/bn/beta"]
            self.dgamma, self.dbeta = fp.gviews[f"{scope}/bn/gamma"], fp.gviews[f"{scope}/bn/beta"]
            self.mov_mean, self.mov_var = p[f"{scope}/bn/moving_mean"], p[f"{scope}/bn/moving_variance"]
            self.stats = torch.empty((2, self.N), **f32)
            self.scale = torch.empty(self.N, **f32)
            self.shift = torch.empty(self.N, **f32)
            self.mean_inv = torch.empty((2, self.N), **f32)
            self.ca = torch.empty(self.N, **f32)
            self.cb = torch.empty(self.N, **f32)
            self.cc = torch.empty(self.N, **f32)
        self.mask = None      # dropout mask applied to this layer's OUTPUT (rows, N), or None

    def act_in(self) -> PsaActIn:
        """this layer's output as the next layer's input"""
        a = PsaActIn()
        a.x = self.y.data_ptr(); a.ld = self.N
        if self.bn:
            a.scale = self.scale.data_ptr(); a.shift = self.shift.data_ptr(); a.relu = 1
        else:
            a.scale = None; a.shift = None; a.relu = 0
        a.mask = self.mask.data_ptr() if self.mask is not None else None
        return a


def _raw_in(x: torch.Tensor) -> PsaActIn:
    a = PsaActIn()
    a.x = x.data_ptr(); a.ld = x.shape[-1]; a.scale = None; a.shift = None; a.mask = None; a.relu = 0
    return a


def _grad_dense(layer: _Layer, dh: torch.Tensor, with_coeffs: bool) -> PsaGradIn:
    g = PsaGradIn()
    g.y = layer.y.data_ptr(); g.ld = layer.N
    if layer.bn:
        g.s = layer.scale.data_ptr(); g.t = layer.shift.data_ptr(); g.relu = 1
    else:
        g.s = None; g.t = None; g.relu = 0
    if layer.bn and with_coeffs:
        g.ca = layer.ca.data_ptr(); g.cb = layer.cb.data_ptr(); g.cc = layer.cc.data_ptr()
    else:
        g.ca = None; g.cb = None; g.cc = None
    g.dh = dh.data_ptr(); g.ld_dh = dh.shape[-1]
    g.mask = layer.mask.data_ptr() if layer.mask is not None else None
    g.dp = None; g.pv = None; g.argk = None; g.pool_k = 1; g.C = layer.N; g.mode = 0
    return g


def _grad_pooled(layer: _Layer, dp: torch.Tensor, pv: torch.Tensor, argk: torch.Tensor, pool_k: int, with_coeffs: bool) -> PsaGradIn:
    g = _grad_dense(layer, dp, with_coeffs)
    g.dh = None; g.ld_dh = 0; g.mask = None
    g.dp = dp.data_ptr(); g.pv = pv.data_ptr(); g.argk = argk.data_ptr(); g.pool_k = pool_k; g.C = layer.N; g.mode = 1
    return g


def _plain_grad(dh: torch.Tensor) -> PsaGradIn:
    g = PsaGradIn()
    g.y = None; g.ld = 0; g.s = None; g.t = None; g.relu = 0; g.ca = None; g.cb = None; g.cc = None
    g.dh = dh.data_ptr(); g.ld_dh = dh.shape[-1]; g.mask = None
    g.dp = None; g.pv = None; g.argk = None; g.pool_k = 1; g.C = dh.shape[-1]; g.mode = 0
    return g


@dataclass
class _Level:
    spec: LevelSpec
    n: int
    m: int
    k: int
    c_in: int
    layers: list = field(default_factory=list)
    new_xyz: torch.Tensor = None
    idx: torch.Tensor = None
    cnt: torch.Tensor = None
    pooled: torch.Tensor = None
    argk: torch.Tensor = None
    dh: list = field(default_factory=list)      # dh[l] = gradient w.r.t. layer l's post-relu output (dense), l < L-1
    dU: torch.Tensor = None
    x_cat: torch.Tensor = None                  # group_all: [xyz, points] rows
    d_in: torch.Tensor = None                   # gradient w.r.t. the level's input features (B*n, c_in)


class _TrainOps:
    """Per-layer training operations shared by the trainers below (they provide self.lib, self.ws, self.ws_bytes)."""

    def _c(self, rc, what):
        check(rc, what)

    def _bn_finalize(self, ly: _Layer, count: int, decay: float):
        self._c(self.lib.psa_bn_finalize(ly.N, count, _p(ly.stats), _p(ly.gamma), _p(ly.beta), C.c_float(decay), _p(ly.mov_mean),
                                         _p(ly.mov_var), _p(ly.scale), _p(ly.shift), _p(ly.mean_inv), _stream()), "bn_finalize")

    def _dense_fwd(self, ly: _Layer, a: PsaActIn):
        self._c(self.lib.psa_train_dense_fwd(ly.rows, ly.K, ly.N, C.byref(a), _p(ly.W), _p(ly.b), _p(ly.y),
                                             _p(ly.stats) if ly.bn else None, _p(self.ws), C.c_size_t(self.ws_bytes), _stream()), "train_dense_fwd")

    def _layer_bwd(self, ly: _Layer, g_nocoef: PsaGradIn, g: PsaGradIn, a_in: PsaActIn, dx: torch.Tensor | None, col_skip: int = 0):
        """gradients of one conv/fc(+BN+relu) layer: BN sums/coefficients, dW, (db), dx."""
        lib = self.lib
        if ly.bn:
            self._c(lib.psa_bn_bwd_coeffs(ly.rows, ly.N, C.byref(g_nocoef), _p(ly.gamma), _p(ly.mean_inv), _p(ly.dgamma), _p(ly.dbeta),
                                          _p(ly.ca), _p(ly.cb), _p(ly.cc), _p(self.ws), C.c_size_t(self.ws_bytes), _stream()), "bn_bwd_coeffs")
            ly.db.zero_()          # sum_r dy = 0 under batch norm
        else:
            self._c(lib.psa_train_bias_grad(ly.rows, ly.N, C.byref(g), _p(ly.db), _stream()), "train_bias_grad")
        if a_in is not None:
            self._c(lib.psa_train_dense_bwd_weight(ly.rows, ly.K, ly.N, C.byref(a_in), C.byref(g), _p(ly.dW), _p(self.ws), C.c_size_t(self.ws_bytes),
                                                   _stream()), "train_dense_bwd_weight")
        if dx is not None:
            self._c(lib.psa_train_dense_bwd_input(ly.rows, ly.K, ly.N, C.byref(g), _p(ly.W), _p(dx), dx.shape[-1], col_skip, _p(self.ws),
                                                  C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_input")


def _flat_grad_of_layers(fp: FlatParams, layers) -> torch.Tensor:
    """a gradient bucket that holds the given layers' gradients and zeros elsewhere (several autograd nodes share one bucket)"""
    g = torch.zeros_like(fp.grad)
    base = fp.grad.data_ptr()
    for ly in layers:
        for t in ([ly.dW, ly.db] + ([ly.dgamma, ly.dbeta] if ly.bn else [])):
            off = (t.data_ptr() - base) // 4
            g[off:off + t.numel()].copy_(t.reshape(-1))
    return g


class MlpTrainer(_TrainOps):
    """Training-mode shared MLP on dense rows -- tf_util.conv1d / conv2d(1x1) / fully_connected chains with batch-statistics batch
    norm + ReLU (tf_util.py:120-185,512-531): the FP modules' MLPs, FC heads, per-point heads.  layers = [(scope, bn), ...];
    a layer with bn=False has no activation (the reference's logits layers)."""

    def __init__(self, params: VariableStore, rows: int, in_channels: int, layers, device=None):
        self.lib = _lib.load()
        self.params = params
        self.dev = torch.device(device) if device is not None else params.device
        self.fp = params._flat if getattr(params, "_flat", None) is not None else FlatParams(params)
        params._flat = self.fp
        self.rows, self.in_channels = rows, in_channels
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.layers: list[_Layer] = []
        cin, ws_bytes = in_channels, 0
        for scope, bn in layers:
            ly = _Layer(self.fp, scope, rows, bn, self.dev)
            assert ly.K == cin, (scope, ly.W.shape, cin)
            ws_bytes = max(ws_bytes, self.lib.psa_train_dense_workspace_bytes(rows, ly.K, ly.N), self.lib.psa_bn_bwd_workspace_bytes(ly.N))
            self.layers.append(ly)
            cin = ly.N
        self.dh = [torch.empty((rows, ly.N), **f32) for ly in self.layers[:-1]]
        self.d_in = torch.empty((rows, in_channels), **f32)
        last = self.layers[-1]
        if last.bn:
            assert last.N % 4 == 0, "an activated last layer needs a width that is a multiple of 4"
            self.out = torch.empty((rows, last.N), **f32)
            self.argk = torch.empty((rows, last.N), dtype=torch.int32, device=self.dev)
        self.ws = torch.empty(ws_bytes // 4 + 64, **f32)
        self.ws_bytes = ws_bytes

    def forward(self, x: torch.Tensor, bn_decay: float = 0.5) -> torch.Tensor:
        assert x.shape == (self.rows, self.in_channels) and x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        self.x = x
        a = _raw_in(x)
        for ly in self.layers:
            self._dense_fwd(ly, a)
            if ly.bn:
                self._bn_finalize(ly, ly.rows, bn_decay)
            a = ly.act_in()
        last = self.layers[-1]
        if not last.bn:
            return last.y
        # the stack's output is the activated tensor: relu(BN(y)) through the pooling kernel with runs of one row
        self._c(self.lib.psa_train_pool_fwd(self.rows, 1, last.N, _p(last.y), _p(last.scale), _p(last.shift), _p(self.out), _p(self.argk),
                                            _stream()), "train_pool_fwd")
        return self.out

    def backward(self, dout: torch.Tensor) -> torch.Tensor:
        """dout = gradient w.r.t. forward()'s return value -> gradient w.r.t. x; the layers' gradients go to the flat bucket"""
        dh = dout.contiguous()
        for i in range(len(self.layers) - 1, -1, -1):
            ly = self.layers[i]
            a_in = self.layers[i - 1].act_in() if i > 0 else _raw_in(self.x)
            dx = self.dh[i - 1] if i > 0 else self.d_in
            self._layer_bwd(ly, _grad_dense(ly, dh, False), _grad_dense(ly, dh, True), a_in, dx)
            dh = dx
        return self.d_in


class _MlpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, flat, x, trainer, bn_decay):
        ctx.trainer = trainer
        return trainer.forward(x, bn_decay).clone()

    @staticmethod
    def backward(ctx, dout):
        tr = ctx.trainer
        dx = tr.backward(dout)
        return _flat_grad_of_layers(tr.fp, tr.layers), dx.clone(), None, None


def mlp_training(x: torch.Tensor, layers, bn_decay, params: VariableStore) -> torch.Tensor:
    """Training-mode shared MLP with autograd: x (..., C_in) -> (..., C_out); layers = [(scope, bn), ...].  Buffers are cached on
    `params` per (scopes, shape)."""
    shape = x.shape
    rows = x.numel() // shape[-1]
    key = ("mlp", tuple(layers), rows, shape[-1])
    cache = params.__dict__.setdefault("_trainers", {})
    if key not in cache:
        cache[key] = MlpTrainer(params, rows, shape[-1], list(layers), device=x.device)
    tr = cache[key]
    tr.fp.flat.requires_grad_(True)
    out = _MlpFn.apply(tr.fp.flat, x.reshape(rows, shape[-1]).contiguous(), tr, 0.5 if bn_decay is None else float(bn_decay))
    return out.view(*shape[:-1], out.shape[-1])


class PointNet2ClsTrainer(_TrainOps):
    """Training engine of pointnet2_cls_ssg (or any stack of LevelSpec + FC head with the same structure)."""

    def __init__(self, params: VariableStore, batch: int, npoints: int, num_class: int = 15, levels=None, head=None,
                 device=None, process_group=None, in_channels: int = 0):
        self.lib = _lib.load()
        self.params = params
        self.dev = torch.device(device) if device is not None else params.device
        self.B, self.N0, self.num_class = batch, npoints, num_class
        self.fp = params._flat if getattr(params, "_flat", None) is not None else FlatParams(params)
        params._flat = self.fp
        self.pg = process_group
        self.world = torch.distributed.get_world_size(process_group) if (process_group is not None or
                                                                          (torch.distributed.is_available() and torch.distributed.is_initialized())) else 1
        dev = self.dev
        f32 = dict(dtype=torch.float32, device=dev)
        specs = levels if levels is not None else SSG_LEVELS
        self.levels: list[_Level] = []
        n, c = npoints, in_channels          # in_channels > 0: the first level takes per-point features (a level used on its own)
        self.in_channels = in_channels
        ws_bytes = 0
        lib = self.lib
        for sp in specs:
            if sp.group_all:
                m, k = 1, n
            else:
                m, k = sp.npoint, sp.nsample
            lv = _Level(sp, n, m, k, c)
            rows = batch * m * k
            cin = 3 + c
            for i, cout in enumerate(sp.mlp):
                lv.layers.append(_Layer(self.fp, f"{sp.scope}/conv{i}", rows, True, dev))
                assert lv.layers[-1].K == cin and lv.layers[-1].N == cout, (sp.scope, i, lv.layers[-1].W.shape, cin, cout)
                ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(rows, cin, cout), lib.psa_bn_bwd_workspace_bytes(cout))
                cin = cout
            L = len(sp.mlp)
            lv.pooled = torch.empty((batch * m, sp.mlp[-1]), **f32)
            lv.argk = torch.empty((batch * m, sp.mlp[-1]), dtype=torch.int32, device=dev)
            lv.dh = [torch.empty((rows, sp.mlp[i]), **f32) for i in range(L - 1)]
            if sp.group_all:
                lv.x_cat = torch.empty((batch * n, 3 + c), **f32)
                if c:
                    lv.d_in = torch.empty((batch * n, c), **f32)
            else:
                lv.idx = torch.empty((batch, m, k), dtype=torch.int32, device=dev)
                lv.cnt = torch.empty((batch, m), dtype=torch.int32, device=dev)
                c1 = sp.mlp[0]
                ws_bytes = max(ws_bytes, lib.psa_sa_conv1_prebn_workspace_bytes(batch, n, m, c, c1, 1), lib.psa_sa_conv1_bwd_workspace_bytes(batch, n, m, k, c1, 1 if c else 0))
                if c:
                    lv.dU = torch.empty((batch * n, c1), **f32)
                    lv.d_in = torch.empty((batch * n, c), **f32)
                    ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(batch * n, c, c1))
            self.levels.append(lv)
            n, c = m, sp.mlp[-1]
        # FC head on the (B, C) global feature
        self.head: list[_Layer] = []
        self.keep: list = []
        cin = c
        for scope, width, bn, keep in (head if head is not None else SSG_HEAD):
            width = width if width is not None else num_class
            ly = _Layer(self.fp, scope, batch, bn, dev)
            assert ly.K == cin and ly.N == width, (scope, ly.W.shape)
            if keep is not None:
                ly.mask = torch.ones((batch, width), **f32)
            self.head.append(ly)
            self.keep.append(keep)
            ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(batch, cin, width), lib.psa_bn_bwd_workspace_bytes(width))
            cin = width
        self.head_dh = [torch.empty((batch, ly.N), **f32) for ly in self.head[:-1]]
        self.d_feat = torch.empty_like(self.levels[-1].pooled)          # (B, C) under a head; (B*m, C) for a bare level stack
        self.dlogits = torch.empty((batch, num_class), **f32)
        self.loss = torch.zeros(1, **f32)
        self.ws = torch.empty(ws_bytes // 4 + 64, **f32)
        self.ws_bytes = ws_bytes
        self._gen = torch.Generator(device=dev)
        self._gen.manual_seed(1234)

    # ------------------------------------------------------------------------------------------------
    def draw_dropout(self):
        """tf.nn.dropout masks of the head (0 or 1/keep_prob), drawn on the device before the step."""
        for ly, keep in zip(self.head, self.keep):
            if keep is not None:
                r = torch.rand(ly.mask.shape, generator=self._gen, device=self.dev)
                ly.mask.copy_((r < keep).to(torch.float32) / keep)

    # ------------------------------------------------------------------------------------------------
    def _level_forward(self, lv: _Level, cur_xyz: torch.Tensor, cur_pts: torch.Tensor | None, bn_decay: float):
        """one set-abstraction level in training mode: lv.new_xyz, the layers' pre-BN activations, lv.pooled"""
        lib = self.lib
        B = self.B
        sp = lv.spec
        L0 = lv.layers[0]
        if sp.group_all:
            # sample_and_group_all (pointnet_util.py:59-84): rows = [xyz, points], one group per cloud
            lv.x_cat[:, :3].copy_(cur_xyz.reshape(-1, 3))
            if cur_pts is not None:
                lv.x_cat[:, 3:].copy_(cur_pts.reshape(B * lv.n, -1))
            self._dense_fwd(L0, _raw_in(lv.x_cat))
            lv.new_xyz = torch.zeros((B, 1, 3), dtype=torch.float32, device=self.dev)
        else:
            _, lv.new_xyz = ops.farthest_point_sample_and_gather(lv.m, cur_xyz)
            self._c(lib.psa_sa_conv1_prebn(B, lv.n, lv.m, lv.c_in, C.c_float(sp.radius), lv.k, _p(cur_xyz), _p(lv.new_xyz), _p(cur_pts),
                                           _p(L0.W), _p(L0.b), L0.N, _p(L0.y), _p(lv.idx), _p(lv.cnt), _p(L0.stats), _p(self.ws),
                                           C.c_size_t(self.ws_bytes), _stream()), "sa_conv1_prebn")
        self._bn_finalize(L0, L0.rows, bn_decay)
        prev = L0
        for ly in lv.layers[1:]:
            self._dense_fwd(ly, prev.act_in())
            self._bn_finalize(ly, ly.rows, bn_decay)
            prev = ly
        self._c(lib.psa_train_pool_fwd(B * lv.m, lv.k, prev.N, _p(prev.y), _p(prev.scale), _p(prev.shift), _p(lv.pooled), _p(lv.argk),
                                       _stream()), "train_pool_fwd")

    def forward(self, xyz: torch.Tensor, bn_decay: float = 0.5, points: torch.Tensor | None = None) -> torch.Tensor:
        """Training-mode forward (batch statistics, moving averages updated with `bn_decay`) -> logits (B, num_class); without a head
        -> the last level's pooled features (B*m, C).  `points` (B, N, in_channels): input features of the first level."""
        feat = self._levels_forward(xyz, points, bn_decay)
        if not self.head:
            return feat
        return self._head_forward(feat, bn_decay)

    def _levels_forward(self, xyz: torch.Tensor, points: torch.Tensor | None, bn_decay: float) -> torch.Tensor:
        """the set-abstraction levels -> the last level's pooled features"""
        B = self.B
        assert xyz.shape == (B, self.N0, 3) and xyz.is_cuda and xyz.dtype == torch.float32
        assert (points is None) == (self.in_channels == 0), "points must be given exactly when the trainer was built with in_channels > 0"
        cur_xyz, cur_pts = xyz.contiguous(), None
        if points is not None:
            assert points.shape == (B, self.N0, self.in_channels) and points.dtype == torch.float32
            cur_pts = points.contiguous()
        self.in_xyz = []
        for lv in self.levels:
            self.in_xyz.append((cur_xyz, cur_pts))
            self._level_forward(lv, cur_xyz, cur_pts, bn_decay)
            cur_xyz, cur_pts = lv.new_xyz, lv.pooled.view(B, lv.m, -1)
        return self.levels[-1].pooled

    def _head_forward(self, feat: torch.Tensor, bn_decay: float) -> torch.Tensor:
        """the FC head on the global feature (B, C) -> logits"""
        a = _raw_in(feat)
        for ly in self.head:
            self._dense_fwd(ly, a)
            if ly.bn:
                self._bn_finalize(ly, ly.rows, bn_decay)
            a = ly.act_in()
        return self.head[-1].y

    # ------------------------------------------------------------------------------------------------
    def _level_backward(self, li: int, dpool: torch.Tensor):
        """gradients of level li's variables for d(loss)/d(pooled) = dpool; the gradient of its input features goes to lv.d_in"""
        lib = self.lib
        B = self.B
        lv = self.levels[li]
        sp = lv.spec
        L = len(lv.layers)
        cur_xyz, cur_pts = self.in_xyz[li]
        for l in range(L - 1, 0, -1):
            ly = lv.layers[l]
            if l == L - 1:
                g0 = _grad_pooled(ly, dpool, lv.pooled, lv.argk, lv.k, False)
                g1 = _grad_pooled(ly, dpool, lv.pooled, lv.argk, lv.k, True)
            else:
                g0 = _grad_dense(ly, lv.dh[l], False)
                g1 = _grad_dense(ly, lv.dh[l], True)
            self._layer_bwd(ly, g0, g1, lv.layers[l - 1].act_in(), lv.dh[l - 1])
        L0 = lv.layers[0]
        if L == 1:
            g0 = _grad_pooled(L0, dpool, lv.pooled, lv.argk, lv.k, False)
            g1 = _grad_pooled(L0, dpool, lv.pooled, lv.argk, lv.k, True)
        else:
            g0 = _grad_dense(L0, lv.dh[0], False)
            g1 = _grad_dense(L0, lv.dh[0], True)
        if sp.group_all:
            self._layer_bwd(L0, g0, g1, _raw_in(lv.x_cat), lv.d_in, col_skip=3)
        else:
            self._c(lib.psa_bn_bwd_coeffs(L0.rows, L0.N, C.byref(g0), _p(L0.gamma), _p(L0.mean_inv), _p(L0.dgamma), _p(L0.dbeta),
                                          _p(L0.ca), _p(L0.cb), _p(L0.cc), _p(self.ws), C.c_size_t(self.ws_bytes), _stream()), "bn_bwd_coeffs")
            L0.db.zero_()
            self._c(lib.psa_sa_conv1_bwd(B, lv.n, lv.m, lv.k, L0.N, _p(cur_xyz), _p(lv.new_xyz), _p(lv.idx), C.byref(g1), _p(L0.dW[:3]),
                                         _p(lv.dU), _p(self.ws), C.c_size_t(self.ws_bytes), _stream()), "sa_conv1_bwd")
            if lv.c_in:
                pts = cur_pts.reshape(B * lv.n, lv.c_in)
                gU = _plain_grad(lv.dU)
                wf = L0.W[3:]
                self._c(lib.psa_train_dense_bwd_weight(B * lv.n, lv.c_in, L0.N, C.byref(_raw_in(pts)), C.byref(gU), _p(L0.dW[3:]), _p(self.ws),
                                                       C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_weight")
                self._c(lib.psa_train_dense_bwd_input(B * lv.n, lv.c_in, L0.N, C.byref(gU), _p(wf), _p(lv.d_in), lv.c_in, 0, _p(self.ws),
                                                      C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_input")

    def backward(self, dlogits: torch.Tensor):
        """Gradients of every trainable variable for d(loss)/d(logits) = dlogits, into the flat gradient bucket."""
        # ---- head ----  (a bare level stack: dlogits is the gradient of the last level's pooled features)
        dh = dlogits.contiguous()
        if not self.head:
            self.d_feat.copy_(dh.reshape(self.d_feat.shape))
        feat = self.levels[-1].pooled
        for i in range(len(self.head) - 1, -1, -1):
            ly = self.head[i]
            a_in = self.head[i - 1].act_in() if i > 0 else _raw_in(feat)
            dx = self.head_dh[i - 1] if i > 0 else self.d_feat
            self._layer_bwd(ly, _grad_dense(ly, dh, False), _grad_dense(ly, dh, True), a_in, dx)
            dh = dx
        # ---- set-abstraction levels, last to first ----
        dpool = self.d_feat
        for li in range(len(self.levels) - 1, -1, -1):
            self._level_backward(li, dpool)
            dpool = self.levels[li].d_in

    # ------------------------------------------------------------------------------------------------
    def loss_and_grad(self, logits: torch.Tensor, labels: torch.Tensor):
        """mean sparse softmax cross-entropy (pointnet2_cls_ssg.py:50-57) -> loss (1,) and d loss / d logits."""
        self._c(self.lib.psa_softmax_xent(self.B, self.num_class, _p(logits), _p(labels), _p(self.loss), _p(self.dlogits), _stream()), "softmax_xent")
        return self.loss, self.dlogits

    def allreduce_grads(self):
        """data parallelism: ONE all-reduce (sum) of the flat gradient bucket; averaged inside the Adam kernel"""
        if self.world > 1:
            torch.distributed.all_reduce(self.fp.grad, group=self.pg)

    def adam(self, lr: float, beta1=0.9, beta2=0.999, eps=1e-8):
        fp = self.fp
        fp.step_count += 1
        self._c(self.lib.psa_adam_step(fp.total, _p(fp.flat), _p(fp.grad), _p(fp.adam_m), _p(fp.adam_v), C.c_float(lr), C.c_float(beta1),
                                       C.c_float(beta2), C.c_float(eps), fp.step_count, C.c_float(1.0 / self.world), _stream()), "adam_step")
        self.params.invalidate()

    def train_step(self, xyz: torch.Tensor, labels: torch.Tensor, lr: float = 1e-3, bn_decay: float = 0.5, dropout: bool = True):
        """one sess.run(train_op) of pointnet2/train.py:246-252: forward, loss, backward, (all-reduce), Adam.  -> loss (1,)"""
        if dropout:
            self.draw_dropout()
        logits = self.forward(xyz, bn_decay)
        loss, dl = self.loss_and_grad(logits, labels)
        self.backward(dl)
        self.allreduce_grads()
        self.adam(lr)
        return loss


@dataclass
class FpSpec:
    """One pointnet_fp_module call (pointnet2_cls_bga.py:51-53)."""
    scope: str
    mlp: list


# pointnet2_cls_bga.py:30-67 (SA1 takes nsample 64 here, 32 in pointnet2_cls_ssg)
BGA_LEVELS = [LevelSpec("layer1", 512, 0.2, 64, [64, 64, 128]), LevelSpec("layer2", 128, 0.4, 64, [128, 128, 256]),
              LevelSpec("layer3", None, None, None, [256, 512, 1024], group_all=True)]
BGA_FP = [FpSpec("fa_layer1", [256, 256]), FpSpec("fa_layer2", [256, 128]), FpSpec("fa_layer3", [128, 128, 128])]
BGA_SEG_HEAD = [("seg_fc1", 128, True, 0.5), ("seg_fc2", 2, False, None)]      # (scope, width, bn, keep_prob)


@dataclass
class _Fp:
    """buffers of one feature-propagation module: n unknown / m known points per cloud, c_a interpolated and c_s skip channels"""
    spec: FpSpec
    n: int
    m: int
    c_a: int
    c_s: int
    layers: list = field(default_factory=list)
    U: torch.Tensor = None                      # (B*m, C1) = P2 . W1[:c_a]
    idx: torch.Tensor = None                    # (B, n, 3)
    weight: torch.Tensor = None                 # (B, n, 3)
    dh: list = field(default_factory=list)      # dh[l] = gradient w.r.t. layer l's post-relu output, l < L-1
    dU: torch.Tensor = None                     # (B*m, C1)
    dP2: torch.Tensor = None                    # (B*m, c_a): gradient w.r.t. the interpolated features' source
    dskip: torch.Tensor = None                  # (B*n, c_s)
    p2_in: PsaActIn = None                      # the forward's P2 operand (kept for the weight gradient)
    skip: torch.Tensor = None


class PointNet2BgaTrainer(PointNet2ClsTrainer):
    """Training engine of pointnet2_cls_bga (classification + background-mask segmentation): one sess.run(train_op) of
    pointnet2/train_seg.py on the hand-written kernels.  The set-abstraction levels and the FC head are PointNet2ClsTrainer's; the
    feature-propagation modules never build the interpolated or concatenated inputs (psa_fp_conv1_prebn / psa_fp_conv1_bwd), the
    joint loss is psa_cls_seg_xent.  Three tensors feed two consumers each, and their gradients are summed before their producer's
    backward: l2_points (SA3 and fa_layer1's skip), l1_points (SA2 and fa_layer2's skip), fc2's activated output (fc3 through the dp2
    mask, fa_layer1 without it: class_vector is tapped before dp2, pointnet2_cls_bga.py:45-48)."""

    def __init__(self, params: VariableStore, batch: int, npoints: int, num_class: int = 15, device=None, process_group=None,
                 levels=None):
        super().__init__(params, batch, npoints, num_class, levels=levels if levels is not None else BGA_LEVELS, head=SSG_HEAD,
                         device=device, process_group=process_group)
        assert len(self.levels) == 3 and self.levels[2].spec.group_all and len(self.head) == 3
        lib = self.lib
        dev = self.dev
        f32 = dict(dtype=torch.float32, device=dev)
        B = batch
        lv1, lv2, _ = self.levels
        fc2 = self.head[1]
        ws_bytes = self.ws_bytes
        # pointnet2_cls_bga.py:51-53: (unknown points, known points, skip channels); interpolated channels = the producer's width
        wiring = [(lv2.m, 1, lv2.spec.mlp[-1]), (lv1.m, lv2.m, lv1.spec.mlp[-1]), (npoints, lv1.m, 0)]
        self.fps: list[_Fp] = []
        c_a = fc2.N
        for sp, (n, m, c_s) in zip(BGA_FP, wiring):
            f = _Fp(sp, n, m, c_a, c_s)
            cin = c_a + c_s
            for i, cout in enumerate(sp.mlp):
                ly = _Layer(self.fp, f"{sp.scope}/conv_{i}", B * n, True, dev)
                assert ly.K == cin and ly.N == cout, (sp.scope, i, ly.W.shape, cin, cout)
                ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(B * n, cin, cout), lib.psa_bn_bwd_workspace_bytes(cout))
                f.layers.append(ly)
                cin = cout
            c1 = sp.mlp[0]
            ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(B * m, c_a, c1), lib.psa_fp_conv1_prebn_workspace_bytes(B, n, c1),
                           lib.psa_fp_conv1_bwd_workspace_bytes(B, n, m))
            if c_s:
                ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(B * n, c_s, c1))
                f.dskip = torch.empty((B * n, c_s), **f32)
            f.U = torch.empty((B * m, c1), **f32)
            f.dU = torch.empty((B * m, c1), **f32)
            f.dP2 = torch.empty((B * m, c_a), **f32)
            f.idx = torch.empty((B, n, 3), dtype=torch.int32, device=dev)
            f.weight = torch.empty((B, n, 3), **f32)
            f.dh = [torch.empty((B * n, w), **f32) for w in sp.mlp[:-1]]
            self.fps.append(f)
            c_a = sp.mlp[-1]
        # per-point segmentation head on the B*N rows of fa_layer3's output
        self.seg: list[_Layer] = []
        self.seg_keep: list = []
        rows = B * npoints
        cin = c_a
        for scope, width, bn, keep in BGA_SEG_HEAD:
            ly = _Layer(self.fp, scope, rows, bn, dev)
            assert ly.K == cin and ly.N == width, (scope, ly.W.shape)
            if keep is not None:
                ly.mask = torch.ones((rows, width), **f32)
            ws_bytes = max(ws_bytes, lib.psa_train_dense_workspace_bytes(rows, cin, width), lib.psa_bn_bwd_workspace_bytes(width))
            self.seg.append(ly)
            self.seg_keep.append(keep)
            cin = width
        self.seg_dh = torch.empty((rows, self.seg[0].N), **f32)        # gradient w.r.t. seg_fc1's (masked) output
        self.fp_dout = torch.empty((rows, c_a), **f32)                 # gradient w.r.t. fa_layer3's output
        self.d_h2 = torch.empty((B, fc2.N), **f32)                      # gradient w.r.t. fc2's activated output (both consumers)
        self.dseg = torch.empty((rows, 2), **f32)
        self.loss = torch.zeros(3, **f32)
        ws_bytes = max(ws_bytes, lib.psa_cls_seg_xent_workspace_bytes(B, npoints))
        if ws_bytes > self.ws_bytes:
            self.ws = torch.empty(ws_bytes // 4 + 64, **f32)
            self.ws_bytes = ws_bytes

    # ------------------------------------------------------------------------------------------------
    def _masked(self):
        return [(ly, keep) for ly, keep in zip(self.head + self.seg, self.keep + self.seg_keep) if keep is not None]

    def draw_dropout(self):
        """tf.nn.dropout masks of dp1, dp2 and seg_dp1 (0 or 1/keep_prob), drawn on the device before the step."""
        for ly, keep in self._masked():
            r = torch.rand(ly.mask.shape, generator=self._gen, device=self.dev)
            ly.mask.copy_((r < keep).to(torch.float32) / keep)

    def _fp_forward(self, f: _Fp, xyz1: torch.Tensor, xyz2: torch.Tensor, p2_in: PsaActIn, skip: torch.Tensor | None, bn_decay: float):
        lib = self.lib
        B = self.B
        L0 = f.layers[0]
        f.p2_in, f.skip = p2_in, skip
        self._c(lib.psa_train_dense_fwd(B * f.m, f.c_a, L0.N, C.byref(p2_in), _p(L0.W[:f.c_a]), None, _p(f.U), None, _p(self.ws),
                                        C.c_size_t(self.ws_bytes), _stream()), "train_dense_fwd")
        if skip is not None:
            self._c(lib.psa_train_dense_fwd(B * f.n, f.c_s, L0.N, C.byref(_raw_in(skip)), _p(L0.W[f.c_a:]), _p(L0.b), _p(L0.y), None,
                                            _p(self.ws), C.c_size_t(self.ws_bytes), _stream()), "train_dense_fwd")
        self._c(lib.psa_fp_conv1_prebn(B, f.n, f.m, L0.N, _p(xyz1), _p(xyz2), _p(f.U), _p(L0.b), 1 if skip is not None else 0, _p(L0.y),
                                       _p(f.idx), _p(f.weight), _p(L0.stats), _p(self.ws), C.c_size_t(self.ws_bytes), _stream()),
                "fp_conv1_prebn")
        self._bn_finalize(L0, L0.rows, bn_decay)
        prev = L0
        for ly in f.layers[1:]:
            self._dense_fwd(ly, prev.act_in())
            self._bn_finalize(ly, ly.rows, bn_decay)
            prev = ly

    def _fps_forward(self, bn_decay: float):
        """fa_layer1..3 (pointnet2_cls_bga.py:51-53) after the levels and the FC head have run"""
        lv1, lv2, lv3 = self.levels
        p2 = self.head[1].act_in()
        p2.mask = None                                   # class_vector: fc2's output before dp2
        self._fp_forward(self.fps[0], lv2.new_xyz, lv3.new_xyz, p2, lv2.pooled, bn_decay)
        self._fp_forward(self.fps[1], lv1.new_xyz, lv2.new_xyz, self.fps[0].layers[-1].act_in(), lv1.pooled, bn_decay)
        self._fp_forward(self.fps[2], self.in_xyz[0][0], lv1.new_xyz, self.fps[1].layers[-1].act_in(), None, bn_decay)

    def _seg_forward(self, bn_decay: float):
        """seg_fc1 -> seg_dp1 -> seg_fc2 on fa_layer3's output"""
        a = self.fps[2].layers[-1].act_in()
        for ly in self.seg:
            self._dense_fwd(ly, a)
            if ly.bn:
                self._bn_finalize(ly, ly.rows, bn_decay)
            a = ly.act_in()

    def forward(self, xyz: torch.Tensor, bn_decay: float = 0.5):
        """Training-mode forward (batch statistics, moving averages updated with `bn_decay`) -> (class logits (B, num_class),
        seg logits (B, N, 2))."""
        B = self.B
        class_logits = super().forward(xyz, bn_decay)
        self._fps_forward(bn_decay)
        self._seg_forward(bn_decay)
        return class_logits, self.seg[-1].y.view(B, self.N0, -1)

    # ------------------------------------------------------------------------------------------------
    def loss_and_grad(self, class_logits: torch.Tensor, seg_logits: torch.Tensor, labels: torch.Tensor, mask: torch.Tensor,
                      seg_weight: float = 0.5):
        """pointnet2_cls_bga.get_loss (pointnet2_cls_bga.py:78-93) -> loss (3,) = [total, classify, seg], d loss / d class_logits,
        d loss / d seg_logits.  labels (B,) and mask (B, N) int32."""
        assert labels.dtype == torch.int32 and mask.dtype == torch.int32 and mask.shape == (self.B, self.N0)
        self._c(self.lib.psa_cls_seg_xent(self.B, self.num_class, self.N0, _p(class_logits), _p(labels), _p(seg_logits), _p(mask),
                                          C.c_float(seg_weight), _p(self.loss), _p(self.dlogits), _p(self.dseg), _p(self.ws),
                                          C.c_size_t(self.ws_bytes), _stream()), "cls_seg_xent")
        return self.loss, self.dlogits, self.dseg.view(self.B, self.N0, 2)

    def _fp_backward(self, f: _Fp, dout: torch.Tensor):
        """gradients of one FP module's variables for d(loss)/d(output) = dout -> f.dP2 (and f.dskip)"""
        lib = self.lib
        B = self.B
        L = len(f.layers)
        for l in range(L - 1, 0, -1):
            ly = f.layers[l]
            dh = dout if l == L - 1 else f.dh[l]
            self._layer_bwd(ly, _grad_dense(ly, dh, False), _grad_dense(ly, dh, True), f.layers[l - 1].act_in(), f.dh[l - 1])
        L0 = f.layers[0]
        dh = dout if L == 1 else f.dh[0]
        g1 = _grad_dense(L0, dh, True)
        self._layer_bwd(L0, _grad_dense(L0, dh, False), g1, None, None)          # batch-norm sums and coefficients
        self._c(lib.psa_fp_conv1_bwd(B, f.n, f.m, L0.N, _p(f.idx), _p(f.weight), C.byref(g1), _p(f.dU), _p(self.ws),
                                     C.c_size_t(self.ws_bytes), _stream()), "fp_conv1_bwd")
        gU = _plain_grad(f.dU)
        self._c(lib.psa_train_dense_bwd_weight(B * f.m, f.c_a, L0.N, C.byref(f.p2_in), C.byref(gU), _p(L0.dW[:f.c_a]), _p(self.ws),
                                               C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_weight")
        self._c(lib.psa_train_dense_bwd_input(B * f.m, f.c_a, L0.N, C.byref(gU), _p(L0.W[:f.c_a]), _p(f.dP2), f.c_a, 0, _p(self.ws),
                                              C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_input")
        if f.c_s:
            self._c(lib.psa_train_dense_bwd_weight(B * f.n, f.c_s, L0.N, C.byref(_raw_in(f.skip)), C.byref(g1), _p(L0.dW[f.c_a:]),
                                                   _p(self.ws), C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_weight")
            self._c(lib.psa_train_dense_bwd_input(B * f.n, L0.K, L0.N, C.byref(g1), _p(L0.W), _p(f.dskip), f.c_s, f.c_a, _p(self.ws),
                                                  C.c_size_t(self.ws_bytes), _stream()), "train_dense_bwd_input")

    def backward(self, dcls: torch.Tensor, dseg: torch.Tensor):
        """Gradients of every trainable variable for d(loss)/d(class logits) = dcls and d(loss)/d(seg logits) = dseg, into the flat
        gradient bucket."""
        dseg = dseg.reshape(-1, 2).contiguous()
        s1, s2 = self.seg
        fa3_out = self.fps[2].layers[-1].act_in()
        self._layer_bwd(s2, _grad_dense(s2, dseg, False), _grad_dense(s2, dseg, True), s1.act_in(), self.seg_dh)
        self._layer_bwd(s1, _grad_dense(s1, self.seg_dh, False), _grad_dense(s1, self.seg_dh, True), fa3_out, self.fp_dout)
        dout = self.fp_dout
        for f in reversed(self.fps):
            self._fp_backward(f, dout)
            dout = f.dP2
        fc1, fc2, fc3 = self.head
        self._layer_bwd(fc3, _grad_dense(fc3, dcls, False), _grad_dense(fc3, dcls, True), fc2.act_in(), self.head_dh[1])
        # fc2's activated output h2 feeds fc3 through the dp2 mask and fa_layer1 directly: d h2 = mask * dx_fc3 + dP2
        torch.addcmul(self.fps[0].dP2, fc2.mask, self.head_dh[1], out=self.d_h2)
        g0, g1 = _grad_dense(fc2, self.d_h2, False), _grad_dense(fc2, self.d_h2, True)
        g0.mask = None
        g1.mask = None
        self._layer_bwd(fc2, g0, g1, fc1.act_in(), self.head_dh[0])
        self._layer_bwd(fc1, _grad_dense(fc1, self.head_dh[0], False), _grad_dense(fc1, self.head_dh[0], True),
                        _raw_in(self.levels[-1].pooled), self.d_feat)
        # set-abstraction levels; l2_points / l1_points also fed fa_layer1 / fa_layer2 as skip features
        _, lv2, lv3 = self.levels
        self._level_backward(2, self.d_feat)
        lv3.d_in.add_(self.fps[0].dskip)
        self._level_backward(1, lv3.d_in)
        lv2.d_in.add_(self.fps[1].dskip)
        self._level_backward(0, lv2.d_in)

    def train_step(self, xyz: torch.Tensor, labels: torch.Tensor, mask: torch.Tensor, lr: float = 1e-3, bn_decay: float = 0.5,
                   seg_weight: float = 0.5, dropout: bool = True):
        """one sess.run(train_op) of pointnet2/train_seg.py: forward, joint loss, backward, (all-reduce), Adam.  dropout=False runs
        with every keep mask at 1.  -> loss (3,) = [total, classify, seg]"""
        if dropout:
            self.draw_dropout()
        else:
            for ly, _ in self._masked():
                ly.mask.fill_(1.0)
        class_logits, seg_logits = self.forward(xyz, bn_decay)
        loss, dcls, dseg = self.loss_and_grad(class_logits, seg_logits, labels, mask, seg_weight)
        self.backward(dcls, dseg)
        self.allreduce_grads()
        self.adam(lr)
        return loss


class _TrainFn(torch.autograd.Function):
    """get_model(is_training=True) for autograd users: logits whose backward fills the flat gradient bucket."""

    @staticmethod
    def forward(ctx, flat, trainer, xyz, bn_decay):
        ctx.trainer = trainer
        return trainer.forward(xyz, bn_decay).clone()

    @staticmethod
    def backward(ctx, dlogits):
        tr = ctx.trainer
        tr.backward(dlogits.contiguous())
        return tr.fp.grad.clone(), None, None, None


class _LevelFn(torch.autograd.Function):
    """One pointnet_sa_module(is_training=True): pooled features whose backward returns the gradient of the input features and
    of this level's variables (a flat bucket that is zero outside the level -- several levels may share one store)."""

    @staticmethod
    def forward(ctx, flat, points, trainer, xyz, bn_decay):
        ctx.trainer = trainer
        ctx.has_points = points is not None
        out = trainer.forward(xyz, bn_decay, points)
        lv = trainer.levels[-1]
        return out.clone().view(trainer.B, lv.m, -1)

    @staticmethod
    def backward(ctx, dout):
        tr = ctx.trainer
        tr.backward(dout.contiguous())
        g = _flat_grad_of_layers(tr.fp, [ly for lv in tr.levels for ly in lv.layers])
        dp = tr.levels[0].d_in.view(tr.B, tr.N0, tr.in_channels).clone() if ctx.has_points else None
        return g, dp, None, None, None


def sa_module_training(xyz, points, spec: LevelSpec, bn_decay, params: VariableStore):
    """Training-mode pointnet_sa_module (max pooling, use_xyz): -> (new_xyz, new_points (B,m,C) with a grad_fn, idx).  The level's
    buffers are cached on `params` per (scope, shape); gradients of its variables arrive in `params._flat.grad_of(name)` /
    through autograd on `params._flat.flat`, the gradient of `points` through autograd."""
    b, n, _ = xyz.shape
    c = 0 if points is None else points.shape[-1]
    key = ("level", spec.scope, b, n, c, spec.npoint, spec.radius, spec.nsample, tuple(spec.mlp), spec.group_all)
    cache = params.__dict__.setdefault("_trainers", {})
    if key not in cache:
        cache[key] = PointNet2ClsTrainer(params, b, n, levels=[spec], head=[], device=xyz.device, in_channels=c)
    tr = cache[key]
    tr.fp.flat.requires_grad_(True)
    out = _LevelFn.apply(tr.fp.flat, points, tr, xyz, 0.5 if bn_decay is None else float(bn_decay))
    lv = tr.levels[0]
    idx = lv.idx
    if spec.group_all:            # sample_and_group_all: one group holding every point in order (pointnet_util.py:75-77)
        idx = torch.arange(n, dtype=torch.int32, device=xyz.device).view(1, 1, n).repeat(b, 1, 1)
    return lv.new_xyz, out, idx


def get_model_training(point_cloud, bn_decay, num_class, params: VariableStore, levels=None, head=None):
    """Training-mode forward of the classifier; the trainer (buffers, flat parameter bucket) is cached on `params`."""
    key = (tuple(point_cloud.shape), num_class)
    cache = params.__dict__.setdefault("_trainers", {})
    if key not in cache:
        cache[key] = PointNet2ClsTrainer(params, point_cloud.shape[0], point_cloud.shape[1], num_class, levels=levels, head=head,
                                         device=point_cloud.device)
    tr = cache[key]
    tr.fp.flat.requires_grad_(True)
    tr.draw_dropout()
    return _TrainFn.apply(tr.fp.flat, tr, point_cloud, 0.5 if bn_decay is None else float(bn_decay)), tr
