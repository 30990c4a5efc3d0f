"""The optimisation step of the skeleton-matching training loop on the B200 path (SURVEY.md 8f-3, the part after the forward).

Reference: skeleton_matching/train_skeleton_matching.py:163-184 - per batch of `dgl.batch`-ed training graphs: GAT2 forward
(gat2.py:137-149), nn.MSELoss on the edge-node scores (:37, :176-178), `loss.backward()` (torch autograd through
gat2.py:50-88) and torch.optim.Adam(lr=1e-4, weight_decay=1e-20).step() (:150).

`GatGrad` keeps the parameters in one flat fp32 buffer (weight rows padded to a multiple of 4 floats), runs the forward on the
product kernels while keeping what the backward needs (per layer: input planes, activated fc1 planes, z = [ft2 | a1 | a2]) and
the backward on csrc/train.cu + the split-bf16 tensor-core GEMM (dW = G^T X and dX = G W as `b200pose_linear` calls on
transposed planes). `GatTrainer` adds the loss and Adam kernels: one `step()` = the reference's loop body. The drop-in
`gat2.GAT2` uses `GatGrad` under a `torch.autograd.Function`, so the reference's own loop (`loss.backward()`,
`optimizer.step()`) trains the drop-in model unmodified.

`MlpGrad` / `MlpTrainer` do the same for the pose-estimator MLP (utils/mlp.py:8-31: 9 linear layers, LeakyReLU(0.1) between),
with a loss the caller writes in torch: the backward runs on the same GEMM and plane kernels, Adam and the refresh of every
operand plane run as one fused launch (b200pose_mlp_adam_planes). The drop-in `mlp.PoseEstimatorMLP` uses `MlpGrad` under a
`torch.autograd.Function`.
"""
from __future__ import annotations

import collections
import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _lib
from ._lib import check, ptr
from .pipeline import Planes, PosePipeline, round_up
from .weights import GAT_ALPHA, GAT_ACT_SLOPE, MLP_SLOPE


def _ld4(n: int) -> int:
    return round_up(n, 4)


class _Buf:
    """Grow-only device buffers of a trainer, keyed by tag (training batches change size every step)."""

    def __init__(self, device):
        self.device = device
        self.f32 = {}
        self.planes = {}
        self.gen = 0            # bumped on every (re)allocation: captured CUDA graphs hold the old addresses

    def f(self, tag, rows, cols):
        t = self.f32.get(tag)
        if t is None or t.shape[0] < rows or t.shape[1] != cols:
            cap = max(rows, int(t.shape[0] * 1.25) if t is not None and t.shape[1] == cols else rows, 1)
            t = torch.zeros((cap, cols), dtype=torch.float32, device=self.device)
            self.f32[tag] = t
            self.gen += 1
        return t

    def p(self, tag, rows, cols) -> Planes:
        """planes [rows, ld >= round_up(cols, 64)]; both extents grow-only. A view with the requested logical shape."""
        ws = self.planes.get(tag)
        need_ld = round_up(max(cols, 1), 64)
        if ws is None or ws.hi.shape[0] < rows or ws.ld < need_ld:
            r = max(rows, int(ws.hi.shape[0] * 1.25) if ws is not None else rows, 1)
            c = max(need_ld, round_up(int(ws.ld * 1.25), 64) if ws is not None and ws.ld < need_ld else need_ld,
                    ws.ld if ws is not None else 0)
            ws = Planes(r, c, self.device)
            self.planes[tag] = ws
            self.gen += 1
        view = Planes.__new__(Planes)
        view.rows, view.cols, view.ld, view.hi, view.lo = rows, cols, ws.ld, ws.hi, ws.lo
        return view


class _FlatParams:
    """Parameters in one flat fp32 buffer `theta` (gradients in `grad`), addressed through `slots`: key -> (offset, rows, cols, ld)."""

    def view(self, flat: torch.Tensor, key: str, padded: bool = False) -> torch.Tensor:
        off, rows, cols, ld = self.slots[key]
        t = flat[off: off + rows * ld].view(rows, ld)
        return t if padded else t[:, :cols]

    def _shape(self, key, t):
        """the reference's tensor shapes: biases [n], weights [out, in]"""
        return t.reshape(-1) if key.endswith('bias') else t

    def load_state(self, state: Dict[str, torch.Tensor]):
        for key in self.slots:
            src = state[key].detach().to(self.device, torch.float32)
            self.view(self.theta, key).copy_(src.reshape(self.slots[key][1], self.slots[key][2]))
        self.refresh_weights()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {key: self._shape(key, self.view(self.theta, key)).clone() for key in self.slots}

    def grads(self) -> Dict[str, torch.Tensor]:
        return {key: self._shape(key, self.view(self.grad, key)) for key in self.slots}

    def _linear(self, a: Planes, m, w: Planes, n, k, out: torch.Tensor):
        """out [m, n] fp32 = A W^T without bias or activation: the dW and dX products of a backward"""
        self.launches += 1
        check(self.L.b200pose_linear(ptr(a.hi), ptr(a.lo), a.ld, ptr(w.hi), ptr(w.lo), w.ld, None, m, n, k, 1.0, 1.0,
                                     ptr(out), out.stride(0), None, None, 0, 0, self.pipe._stream()), 'linear (backward)')


class _StepGraphs:
    """Captured optimisation steps of a trainer, one CUDA graph per input shape key, least recently used first and at most
    `max_cached` of them. A workspace re-allocation (buf.gen changed) drops them all: the graphs hold the old addresses."""

    def _init_graphs(self, max_cached: int = 64):
        self._graphs = collections.OrderedDict()
        self.max_cached = max_cached

    def _cached_step(self, key, buf: _Buf):
        ent = self._graphs.get(key)
        if ent is not None and ent['gen'] != buf.gen:
            self._graphs.clear()
            ent = None
        if ent is not None:
            self._graphs.move_to_end(key)
        return ent

    def _capture_step(self, key, ent: dict, buf: _Buf, device, enqueue):
        """Captures enqueue() (whose workspaces an eager run has already sized) on a side stream into ent['graph']."""
        ent['gen'] = buf.gen
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                enqueue()
        torch.cuda.current_stream(device).wait_stream(side)
        if ent['gen'] != buf.gen:
            raise RuntimeError('%s.step_captured: a workspace was allocated during the capture' % type(self).__name__)
        ent['graph'] = graph
        self._graphs[key] = ent
        while len(self._graphs) > self.max_cached:
            self._graphs.popitem(last=False)
        return ent


def param_layout(shapes: Dict[str, tuple], residual: bool = False):
    """Flat fp32 layout of the GAT's parameters from the shapes of a reference state dict (gat2.py:25-48 key names).
    Returns (layers, slots, n_floats): per layer its sizes (din, heads, dim, hd, n2 = hd + 2 heads, ldz), and per key
    (offset, rows, cols, ld) with ld = cols rounded up to 4 floats - every row, and so every slot, starts 16-byte aligned, which
    is what lets the dW GEMMs store straight into the gradient buffer (TMA store pitch) and Adam run over one flat range (padding
    elements have zero gradients and stay zero). residual: GAT2 built with residual=True - every layer after the first either
    has `res_fc.*` entries (in_dim != out_dim) or, without them, adds its input broadcast over the heads (gat2.py:43-48)."""
    n_layers = len([k for k in shapes if k.endswith('fc1.weight')])
    layers, slots, off = [], {}, 0

    def slot(key, rows, cols):
        nonlocal off
        ld = _ld4(cols)
        slots[key] = (off, rows, cols, ld)
        off += rows * ld

    for l in range(n_layers):
        pre = 'layers.%d.' % l
        if (pre + 'fc1.bias') not in shapes:
            raise NotImplementedError('GatGrad: the training configuration has biases (train_skeleton_matching.py:148: bias=True)')
        has_res_fc = (pre + 'res_fc.weight') in shapes
        if has_res_fc and not (residual and l > 0):
            raise ValueError('GatGrad: layer %d has res_fc weights but the model is not declared residual (or it is the first layer)' % l)
        H, D = shapes[pre + 'attn_l'][:2]
        din = shapes[pre + 'fc1.weight'][1]
        if shapes[pre + 'fc1.weight'] != (din, din) or shapes[pre + 'fc2.weight'] != (H * D, din):
            raise ValueError('GatGrad: layer %d has shapes fc1 %s, fc2 %s for %d heads x %d' % (l, shapes[pre + 'fc1.weight'], shapes[pre + 'fc2.weight'], H, D))
        res = None
        if residual and l > 0:
            if has_res_fc:
                if shapes[pre + 'res_fc.weight'] != (H * D, din) or (pre + 'res_fc.bias') not in shapes:
                    raise ValueError('GatGrad: layer %d res_fc has shape %s for %d heads x %d (bias required)' % (l, shapes[pre + 'res_fc.weight'], H, D))
                res = 'fc'
            elif din == D:
                res = 'identity'
            else:
                raise ValueError('GatGrad: residual layer %d has in_dim %d != out_dim %d but no res_fc weights' % (l, din, D))
        layers.append(dict(din=din, heads=H, dim=D, hd=H * D, n2=H * D + 2 * H, ldz=round_up(H * D + 2 * H, 4), res=res))
        slot(pre + 'attn_l', 1, H * D)
        slot(pre + 'attn_r', 1, H * D)
        slot(pre + 'fc1.weight', din, din)
        slot(pre + 'fc1.bias', 1, din)
        slot(pre + 'fc2.weight', H * D, din)
        slot(pre + 'fc2.bias', 1, H * D)
        if res == 'fc':
            slot(pre + 'res_fc.weight', H * D, din)
            slot(pre + 'res_fc.bias', 1, H * D)
    return layers, slots, off


class GatGrad(_FlatParams):
    """Forward with saved activations + backward of the skeleton-matching GAT (no dropout: train_skeleton_matching.py:46-48).
    residual=True: the model was built with residual connections (gat2.py:43-48, 70-75; the shipped configuration has none)."""

    def __init__(self, pipe: PosePipeline, state: Dict[str, torch.Tensor], alpha: float = GAT_ALPHA,
                 act_slope: float = GAT_ACT_SLOPE, residual: bool = False):
        self.pipe = pipe
        self.L = pipe.L
        self.device = pipe.device
        self.alpha, self.act_slope = float(alpha), float(act_slope)
        self.layers, self.slots, off = param_layout({k: tuple(v.shape) for k, v in state.items()}, residual)
        self.n_flat = off
        with torch.cuda.device(self.device):
            self.theta = torch.zeros(off, dtype=torch.float32, device=self.device)
            self.grad = torch.zeros(off, dtype=torch.float32, device=self.device)
            self.buf = _Buf(self.device)
            for l, lay in enumerate(self.layers):
                din, hd, n2 = lay['din'], lay['hd'], lay['n2']
                lay['w1'] = Planes(din, din, self.device)
                lay['w1t'] = Planes(din, din, self.device)
                lay['b2e'] = torch.zeros(n2, dtype=torch.float32, device=self.device)
                lay['w2'] = Planes(n2, din, self.device)
                lay['w2t'] = Planes(din, hd, self.device)
                if lay['res'] == 'fc':
                    lay['res_w'] = Planes(hd, din, self.device)
                    lay['res_wt'] = Planes(din, hd, self.device)
        self.cache = None
        self.launches = 0
        self.load_state(state)

    # ------------------------------------------------------------------ parameters
    def _shape(self, key, t):
        """the reference's tensor shapes: attn_* [H, D, 1], biases [n], weights [out, in]"""
        if key.endswith('attn_l') or key.endswith('attn_r'):
            l = int(key.split('.')[1])
            return t.reshape(self.layers[l]['heads'], self.layers[l]['dim'], 1)
        return super()._shape(key, t)

    def refresh_weights(self):
        """The operand planes of every projection, from the flat parameters: W1, W1^T, [W2 ; attention folds] and W2^T
        (after every optimiser step)."""
        L, s = self.L, self.pipe._stream()
        for l, lay in enumerate(self.layers):
            pre = 'layers.%d.' % l
            W1 = self.view(self.theta, pre + 'fc1.weight', padded=True)
            W2 = self.view(self.theta, pre + 'fc2.weight', padded=True)
            check(L.b200pose_gat_prepare_layer(ptr(W1), ptr(W2), W1.stride(0), ptr(self.view(self.theta, pre + 'fc2.bias')),
                                               ptr(self.view(self.theta, pre + 'attn_l')), ptr(self.view(self.theta, pre + 'attn_r')),
                                               lay['heads'], lay['dim'], lay['din'],
                                               ptr(lay['w1'].hi), ptr(lay['w1'].lo), lay['w1'].ld, ptr(lay['w1t'].hi), ptr(lay['w1t'].lo), lay['w1t'].ld,
                                               ptr(lay['w2'].hi), ptr(lay['w2'].lo), lay['w2'].ld, ptr(lay['w2t'].hi), ptr(lay['w2t'].lo), lay['w2t'].ld,
                                               ptr(lay['b2e']), s), 'gat_prepare_layer')
            self.launches += 1
            if lay['res'] == 'fc':
                Wr = self.view(self.theta, pre + 'res_fc.weight', padded=True)
                check(L.b200pose_grad_planes(ptr(Wr), lay['hd'], lay['din'], Wr.stride(0), None, 0, 1.0, None, 0,
                                             ptr(lay['res_w'].hi), ptr(lay['res_w'].lo), lay['res_w'].ld,
                                             ptr(lay['res_wt'].hi), ptr(lay['res_wt'].lo), lay['res_wt'].ld, s), 'grad_planes')
                self.launches += 1

    # ------------------------------------------------------------------ forward
    def forward(self, db, g, x0: Planes) -> torch.Tensor:
        """GAT2.forward (gat2.py:137-149) on a dense feature matrix x0 [N, F] (planes); returns the scores [N] and keeps the
        per-layer tensors for backward()."""
        pipe, N = self.pipe, db.n_nodes
        cache = []
        x = x0
        scores = self.buf.f('scores', N, 1)
        for l, lay in enumerate(self.layers):
            last = l == len(self.layers) - 1
            pre = 'layers.%d.' % l
            h2 = self.buf.p('h2_%d' % l, N, lay['din'])
            z = self.buf.f('z_%d' % l, N, lay['ldz'])
            pipe.linear(x, N, lay['w1'], self.view(self.theta, pre + 'fc1.bias'), lay['din'], lay['din'], self.alpha, out_planes=h2)
            pipe.linear(h2, N, lay['w2'], lay['b2e'], lay['n2'], lay['din'], 1.0, out_f32=z)
            act = None if last else self.buf.p('act_%d' % l, N, lay['hd'])
            res = None
            if lay['res'] == 'fc':                                   # gat2.py:72: res_fc(h)
                res = self.buf.f('res_%d' % l, N, _ld4(lay['hd']))
                pipe.linear(x, N, lay['res_w'], self.view(self.theta, pre + 'res_fc.bias'), lay['hd'], lay['din'], 1.0, out_f32=res)
            elif lay['res'] == 'identity':                           # gat2.py:74: the input itself, broadcast over the heads
                res = x.to_f32()[:N, : lay['din']].repeat(1, lay['heads']).contiguous()
            pipe.aggregate(db, g, z, lay, layer0=False, raw=None, act=act, scores=scores if last else None,
                           alpha=self.alpha, act_slope=self.act_slope, res=res)
            cache.append(dict(x=x, h2=h2, z=z))
            x = act
        self.cache = dict(layers=cache, N=N, g=g, scores=scores)        # (the forward's launches are counted by the pipeline)
        return scores[:N, 0]

    # ------------------------------------------------------------------ backward
    def backward(self, dlogit: torch.Tensor):
        """dlogit [N] fp32 = gradient of the loss w.r.t. the last layer's output (before the sigmoid). Fills self.grad."""
        if self.cache is None:
            raise RuntimeError('GatGrad.backward without a forward')
        L, s = self.L, self.pipe._stream()
        N, g = self.cache['N'], self.cache['g']
        d, ld_d = dlogit, 1
        for l in range(len(self.layers) - 1, -1, -1):
            lay, c = self.layers[l], self.cache['layers'][l]
            pre = 'layers.%d.' % l
            din, hd, H, D, ldz = lay['din'], lay['hd'], lay['heads'], lay['dim'], lay['ldz']
            z, h2, x = c['z'], c['h2'], c['x']
            dz = self.buf.f('dz_%d' % ldz, N, ldz)
            stats = self.buf.f('stats_%d' % H, N, 3 * H)
            check(L.b200pose_gat_aggregate_bwd(N, ptr(g.row_ptr), ptr(g.col), ptr(z), z.stride(0), H, D, self.alpha, ptr(d), ld_d,
                                               ptr(self.view(self.theta, pre + 'attn_l')), ptr(self.view(self.theta, pre + 'attn_r')),
                                               ptr(stats), ptr(dz), dz.stride(0), s), 'gat_aggregate_bwd')
            check(L.b200pose_gat_attn_bias_grad(ptr(z), z.stride(0), ptr(dz), dz.stride(0), N, H, D, ptr(self.view(self.grad, pre + 'attn_l')),
                                                ptr(self.view(self.grad, pre + 'attn_r')), ptr(self.view(self.grad, pre + 'fc2.bias')), s), 'gat_attn_bias_grad')
            G2 = self.buf.p('G2_%d' % l, N, hd)
            G2T = self.buf.p('G2T_%d' % l, hd, N)
            check(L.b200pose_grad_planes(ptr(dz), N, hd, dz.stride(0), None, 0, 1.0, None, 0, ptr(G2.hi), ptr(G2.lo), G2.ld,
                                         ptr(G2T.hi), ptr(G2T.lo), G2T.ld, s), 'grad_planes')
            h2T = self.buf.p('h2T_%d' % l, din, N)
            check(L.b200pose_transpose_planes(ptr(h2.hi), ptr(h2.lo), N, din, h2.ld, ptr(h2T.hi), ptr(h2T.lo), h2T.ld, s), 'transpose_planes')
            self._linear(G2T, hd, h2T, din, N, self.view(self.grad, pre + 'fc2.weight', padded=True))          # dW2 = G2^T h2
            dh2 = self.buf.f('dh2_%d' % _ld4(din), N, _ld4(din))
            self._linear(G2, N, lay['w2t'], din, hd, dh2)                                                       # dh2 = G2 W2
            G1 = self.buf.p('G1_%d' % l, N, din)
            G1T = self.buf.p('G1T_%d' % l, din, N)
            check(L.b200pose_grad_planes(ptr(dh2), N, din, dh2.stride(0), ptr(h2.hi), h2.ld, self.alpha, ptr(dh2), dh2.stride(0),
                                         ptr(G1.hi), ptr(G1.lo), G1.ld, ptr(G1T.hi), ptr(G1T.lo), G1T.ld, s), 'grad_planes')
            check(L.b200pose_colsum(ptr(dh2), N, din, dh2.stride(0), None, 0, 1, ptr(self.view(self.grad, pre + 'fc1.bias')), s), 'colsum')
            xT = self.buf.p('xT_%d' % l, din, N)
            check(L.b200pose_transpose_planes(ptr(x.hi), ptr(x.lo), N, din, x.ld, ptr(xT.hi), ptr(xT.lo), xT.ld, s), 'transpose_planes')
            self._linear(G1T, din, xT, din, N, self.view(self.grad, pre + 'fc1.weight', padded=True))          # dW1 = G1^T x
            dxr = None
            if lay['res'] == 'fc':                                   # the same output gradient d also flows through res_fc(x)
                check(L.b200pose_colsum(ptr(d), N, hd, ld_d, None, 0, 1, ptr(self.view(self.grad, pre + 'res_fc.bias')), s), 'colsum')
                Gr = self.buf.p('Gr_%d' % l, N, hd)
                GrT = self.buf.p('GrT_%d' % l, hd, N)
                check(L.b200pose_grad_planes(ptr(d), N, hd, ld_d, None, 0, 1.0, None, 0, ptr(Gr.hi), ptr(Gr.lo), Gr.ld,
                                             ptr(GrT.hi), ptr(GrT.lo), GrT.ld, s), 'grad_planes')
                self._linear(GrT, hd, xT, din, N, self.view(self.grad, pre + 'res_fc.weight', padded=True))    # dWres = d^T x
                dxr = self.buf.f('dxr_%d' % _ld4(din), N, _ld4(din))
                self._linear(Gr, N, lay['res_wt'], din, hd, dxr)                                              # d Wres
                self.launches += 2
            self.launches += 8          # kernels of the calls above other than the GEMMs (counted by _linear)
            if l > 0:
                dx = self.buf.f('dx_l%d' % l, N, _ld4(din))              # per layer: layer l+1's dx is this layer's d, read until the end
                self._linear(G1, N, lay['w1t'], din, din, dx)                                                   # dx = G1 W1
                if lay['res'] == 'fc':
                    check(L.b200pose_residual_bwd_add(ptr(dx), dx.stride(0), ptr(dxr), dxr.stride(0), N, din, 1, s), 'residual_bwd_add')
                    self.launches += 1
                elif lay['res'] == 'identity':
                    check(L.b200pose_residual_bwd_add(ptr(dx), dx.stride(0), ptr(d), ld_d, N, din, H, s), 'residual_bwd_add')
                    self.launches += 1
                # through the inter-layer LeakyReLU (GAT2.forward :141-142): x is the activated output of layer l-1
                check(L.b200pose_grad_planes(ptr(dx), N, din, dx.stride(0), ptr(x.hi), x.ld, self.act_slope, ptr(dx), dx.stride(0),
                                             None, None, 0, None, None, 0, s), 'grad_planes')
                self.launches += 1
                d, ld_d = dx, dx.stride(0)


class GatTrainer(_StepGraphs):
    """One `step()` = the loop body of train_skeleton_matching.py:166-181 on a batch of training graphs.

    `step()` enqueues the ~125 launches of a step one by one; `step_captured()` replays the same step as ONE CUDA graph per batch
    shape (the reference's DataLoader does not shuffle, :143, so every epoch presents the same batches): the inputs are copied
    into the capture's static buffers, the Adam step count lives on the device."""

    def __init__(self, pipe: PosePipeline, state: Dict[str, torch.Tensor], lr: float = 1e-4, betas: Sequence[float] = (0.9, 0.999),
                 eps: float = 1e-8, weight_decay: float = 1e-20, alpha: float = GAT_ALPHA, act_slope: float = GAT_ACT_SLOPE,
                 residual: bool = False):
        self.pipe = pipe
        self.net = GatGrad(pipe, state, alpha, act_slope, residual)
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        dev = pipe.device
        self.m = torch.zeros(self.net.n_flat, dtype=torch.float32, device=dev)
        self.v = torch.zeros(self.net.n_flat, dtype=torch.float32, device=dev)
        self.t = 0                                                            # host mirror of the device-side step count
        self.t_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.adam_scalars = torch.zeros(2, dtype=torch.float32, device=dev)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self.last_scores = None
        self._init_graphs()

    def features(self, db) -> Planes:
        """ndata['h'] of the batch as GEMM operand planes (the reference feeds the dense N x F matrix, :171-176)"""
        return Planes.from_f32(self.pipe.node_features_f32(db), self.pipe._stream())

    def _enqueue(self, db, g, indices, labels, x0, update):
        net, L, s = self.net, self.pipe.L, self.pipe._stream()
        scores = net.forward(db, g, x0)
        self.last_scores = scores
        N, M = db.n_nodes, int(indices.shape[0])
        dlogit = net.buf.f('dlogit', N, 1)
        check(L.b200pose_mse_sigmoid(ptr(scores), N, ptr(indices), ptr(labels), M, ptr(self.loss), ptr(dlogit), s), 'mse_sigmoid')
        net.backward(dlogit)
        net.launches += 1
        if update:
            check(L.b200pose_adam_step_dev(ptr(net.theta), ptr(net.grad), ptr(self.m), ptr(self.v), net.n_flat, self.lr, self.betas[0],
                                           self.betas[1], self.eps, self.weight_decay, ptr(self.t_dev), ptr(self.adam_scalars), s), 'adam_step_dev')
            net.refresh_weights()
            net.launches += 2

    def step(self, db, g, indices: torch.Tensor, labels: torch.Tensor, x0: Optional[Planes] = None, update: bool = True):
        """indices [M] int32 (edge-node ids of the batched graph), labels [M] fp32, both on the device. Returns the loss as a
        device scalar (read it with .item() when it is needed: the step itself does not synchronise)."""
        if x0 is None:
            x0 = self.features(db)
        self._enqueue(db, g, indices, labels, x0, update)
        if update:
            self.t += 1
        return self.loss

    def step_captured(self, db, g, indices: torch.Tensor, labels: torch.Tensor, x0: Optional[Planes] = None):
        """step() as one CUDA-graph replay. The first call for a batch shape (frames, heads, nodes, edges, labelled edge-nodes,
        in-degree bounds) runs one eager forward + backward to size the workspaces and captures the step on static copies of
        the inputs; later calls copy their inputs there and replay. A workspace re-allocation (a larger batch) drops the graphs."""
        from .pipeline import DeviceBatch
        if x0 is None:
            x0 = self.features(db)
        M = int(indices.shape[0])
        key = (db.n_frames, db.n_heads, db.n_nodes, db.n_edges, M, db.max_heads, db.max_enodes, bool(getattr(g, 'general', False)), x0.ld)
        ent = self._cached_step(key, self.net.buf)
        if ent is None:
            self.pipe.wait_graph(g)
            self._enqueue(db, g, indices, labels, x0, update=False)                 # sizes every workspace; no parameter changes
            clone = lambda t: t.clone()
            sdb = DeviceBatch(db.n_frames, db.n_heads, db.n_nodes, db.max_heads, db.max_enodes, db.sk_xy, db.sk_vp, db.sk_mask, db.sk_cam,
                              clone(db.head_off), clone(db.node_off), host_offsets=db.host_offsets)
            sg = type('StaticGraph', (), {})()
            sg.row_ptr, sg.col, sg.general, sg.pending = clone(g.row_ptr), clone(g.col), bool(getattr(g, 'general', False)), None
            sx = Planes.__new__(Planes)
            sx.rows, sx.cols, sx.ld, sx.hi, sx.lo = x0.rows, x0.cols, x0.ld, clone(x0.hi), clone(x0.lo)
            ent = dict(db=sdb, g=sg, x0=sx, idx=clone(indices), lab=clone(labels))
            self._capture_step(key, ent, self.net.buf, self.pipe.device,
                               lambda: self._enqueue(sdb, sg, ent['idx'], ent['lab'], sx, update=True))
        else:
            ent['db'].head_off.copy_(db.head_off, non_blocking=True)
            ent['db'].node_off.copy_(db.node_off, non_blocking=True)
            ent['g'].row_ptr.copy_(g.row_ptr, non_blocking=True)
            ent['g'].col.copy_(g.col, non_blocking=True)
            ent['x0'].hi.copy_(x0.hi, non_blocking=True)
            ent['x0'].lo.copy_(x0.lo, non_blocking=True)
            ent['idx'].copy_(indices, non_blocking=True)
            ent['lab'].copy_(labels, non_blocking=True)
        ent['graph'].replay()
        self.t += 1
        self.last_scores = self.net.cache['scores'][: db.n_nodes, 0]
        return self.loss


# ====================================================================================================== pose-estimator MLP
MLP_LAYER_INDICES = tuple(range(1, 18, 2))          # nn.Sequential positions of the 9 projections (utils/mlp.py:10-28)


def mlp_param_layout(shapes: Dict[str, tuple]):
    """Flat fp32 layout of PoseEstimatorMLP's parameters from the shapes of a reference state dict (keys
    `layers.{1,3,...,17}.{weight,bias}`). Returns (layers, slots, n_floats): per layer its widths (n out, k in), and per key
    (offset, rows, cols, ld) with ld = cols rounded up to 4 floats, each weight slot followed by its layer's bias slot: every row
    starts 16-byte aligned, so the dW GEMMs store straight into the gradient buffer, and one flat range covers the optimiser
    step. The widths come from the weights, so any input width (252 * cameras) works; they must chain layer to layer."""
    want = {'layers.%d.%s' % (j, w) for j in MLP_LAYER_INDICES for w in ('weight', 'bias')}
    extra = sorted(set(shapes) - want)
    if extra:
        raise ValueError('MlpGrad: keys outside layers.{1,3,...,17}.{weight,bias}: %s' % extra)
    layers, slots, off = [], {}, 0
    for i, j in enumerate(MLP_LAYER_INDICES):
        pre = 'layers.%d.' % j
        if pre + 'weight' not in shapes or pre + 'bias' not in shapes:
            raise ValueError('MlpGrad: layer %s needs a weight and a bias (utils/mlp.py builds nn.Linear with bias=True)' % pre)
        w, b = tuple(shapes[pre + 'weight']), tuple(shapes[pre + 'bias'])
        if len(w) != 2 or b != (w[0],) or (layers and w[1] != layers[-1]['n']):
            raise ValueError('MlpGrad: %sweight %s, bias %s do not chain to the previous layer' % (pre, w, b))
        n, k = w
        slots[pre + 'weight'] = (off, n, k, _ld4(k))
        off += n * _ld4(k)
        slots[pre + 'bias'] = (off, 1, n, _ld4(n))
        off += _ld4(n)
        layers.append(dict(n=n, k=k))
    return layers, slots, off


class MlpGrad(_FlatParams):
    """Forward with saved activations + backward of PoseEstimatorMLP (utils/mlp.py:8-31). The forward keeps every layer's input
    as operand planes in a buffer of its own; the backward goes layer by layer from the last: G = dY * LeakyReLU'(Y) (the sign
    of the stored activated planes; the last layer is linear) as planes in both layouts, d bias = column sums of G,
    dW = G^T X into the gradient slot, dX = G W on the W^T planes (not for the first layer)."""

    def __init__(self, pipe: PosePipeline, state: Dict[str, torch.Tensor], slope: float = MLP_SLOPE):
        self.pipe = pipe
        self.L = pipe.L
        self.device = pipe.device
        self.slope = float(slope)
        self.layers, self.slots, self.n_flat = mlp_param_layout({k: tuple(v.shape) for k, v in state.items()})
        with torch.cuda.device(self.device):
            self.theta = torch.zeros(self.n_flat, dtype=torch.float32, device=self.device)
            self.grad = torch.zeros(self.n_flat, dtype=torch.float32, device=self.device)
            self.buf = _Buf(self.device)
            for i, lay in enumerate(self.layers):
                lay['w'] = Planes(lay['n'], lay['k'], self.device)
                lay['wt'] = Planes(lay['k'], lay['n'], self.device) if i > 0 else None         # dX of the first layer is not needed
        table = []
        for i, lay in enumerate(self.layers):
            off, n, k, ld = self.slots['layers.%d.weight' % MLP_LAYER_INDICES[i]]
            w, wt = lay['w'], lay['wt']
            table.append(_lib.MlpLayer(off, n, k, ld, w.hi.data_ptr(), w.lo.data_ptr(), w.ld,
                                       wt.hi.data_ptr() if wt else None, wt.lo.data_ptr() if wt else None, wt.ld if wt else 0))
        self._table = (_lib.MlpLayer * len(table))(*table)
        self.cache = None
        self.cache_token = None
        self.launches = 0
        self.load_state(state)

    @property
    def n_out(self) -> int:
        return self.layers[-1]['n']

    def adam_planes(self, grad, m=None, v=None, lr=0.0, betas=(0.0, 0.0), eps=0.0, weight_decay=0.0, t_dev=None, scalars=None):
        """b200pose_mlp_adam_planes: one Adam step over theta with `grad` and the refresh of every operand plane, in one launch
        after the scalar kernel; grad=None rebuilds the planes from theta only."""
        check(self.L.b200pose_mlp_adam_planes(ptr(self.theta), ptr(grad), ptr(m), ptr(v), self.n_flat, self._table, len(self.layers),
                                              lr, betas[0], betas[1], eps, weight_decay, ptr(t_dev), ptr(scalars), self.pipe._stream()),
              'mlp_adam_planes')
        self.launches += 1 if grad is None else 2

    def refresh_weights(self):
        self.adam_planes(None)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [P, in] fp32 (contiguous rows) -> the MLP output [P, n_out] (a view of a workspace); keeps what backward() needs."""
        pipe, P = self.pipe, int(x.shape[0])
        if P < 1 or x.dim() != 2 or x.shape[1] != self.layers[0]['k'] or x.stride(1) != 1 or x.dtype != torch.float32:
            raise ValueError('MlpGrad.forward: x must be fp32 [P >= 1, %d] with unit column stride, got %s %s'
                             % (self.layers[0]['k'], x.dtype, tuple(x.shape)))
        xp = self.buf.p('x0', P, x.shape[1])
        check(self.L.b200pose_split_planes(ptr(x), P, x.shape[1], x.stride(0), ptr(xp.hi), ptr(xp.lo), xp.ld, pipe._stream()), 'split_planes')
        self.launches += 1
        xs = [xp]
        for i, lay in enumerate(self.layers):
            bias = self.view(self.theta, 'layers.%d.bias' % MLP_LAYER_INDICES[i])
            if i == len(self.layers) - 1:
                out = self.buf.f('out', P, _ld4(lay['n']))
                pipe.linear(xs[-1], P, lay['w'], bias, lay['n'], lay['k'], 1.0, out_f32=out)
            else:
                y = self.buf.p('a_%d' % i, P, lay['n'])
                pipe.linear(xs[-1], P, lay['w'], bias, lay['n'], lay['k'], self.slope, out_planes=y)
                xs.append(y)
        self.cache = dict(xs=xs, P=P)                     # (the projections' launches are counted by the pipeline)
        return out[:P, : self.n_out]

    def backward(self, dy: torch.Tensor):
        """dy [P, n_out] fp32 (unit column stride) = gradient of the loss w.r.t. the output of the last forward. Fills self.grad."""
        if self.cache is None:
            raise RuntimeError('MlpGrad.backward without a forward')
        L, s, P, xs = self.L, self.pipe._stream(), self.cache['P'], self.cache['xs']
        if tuple(dy.shape) != (P, self.n_out) or dy.stride(1) != 1 or dy.dtype != torch.float32:
            raise ValueError('MlpGrad.backward: dy must be fp32 [%d, %d] with unit column stride' % (P, self.n_out))
        d, ld_d = dy, dy.stride(0)
        for i in range(len(self.layers) - 1, -1, -1):
            lay, pre = self.layers[i], 'layers.%d.' % MLP_LAYER_INDICES[i]
            n, k, x = lay['n'], lay['k'], xs[i]
            mask = xs[i + 1] if i + 1 < len(self.layers) else None              # the activated output of this layer
            G = self.buf.p('G_%d' % i, P, n) if i > 0 else None
            GT = self.buf.p('GT_%d' % i, n, P)
            check(L.b200pose_grad_planes(ptr(d), P, n, ld_d, ptr(mask.hi) if mask else None, mask.ld if mask else 0, self.slope,
                                         ptr(d) if mask else None, ld_d if mask else 0,
                                         ptr(G.hi) if G else None, ptr(G.lo) if G else None, G.ld if G else 0,
                                         ptr(GT.hi), ptr(GT.lo), GT.ld, s), 'grad_planes')
            check(L.b200pose_colsum(ptr(d), P, n, ld_d, None, 0, 1, ptr(self.view(self.grad, pre + 'bias')), s), 'colsum')
            xT = self.buf.p('xT_%d' % i, k, P)
            check(L.b200pose_transpose_planes(ptr(x.hi), ptr(x.lo), P, k, x.ld, ptr(xT.hi), ptr(xT.lo), xT.ld, s), 'transpose_planes')
            self.launches += 3
            self._linear(GT, n, xT, k, P, self.view(self.grad, pre + 'weight', padded=True))       # dW = G^T X
            if i > 0:
                dx = self.buf.f('dx_%d' % i, P, _ld4(k))
                self._linear(G, P, lay['wt'], k, n, dx)                                           # dX = G W
                d, ld_d = dx, dx.stride(0)


def _rows(x: torch.Tensor, device) -> torch.Tensor:
    """nn.Flatten + fp32 + contiguous rows on the device (the MLP's input as the GEMM reads it)"""
    return x.reshape(x.shape[0], -1).to(device, torch.float32).contiguous()


class MlpTrainer(_StepGraphs):
    """One `step()` = forward, the caller's torch loss on the joints and its gradient, backward, Adam, operand-plane refresh.
    Adam's defaults are torch.optim.Adam's. `step_captured()` replays the same step, the caller's loss included, as ONE CUDA
    graph per input shape (and loss function / arguments signature)."""

    def __init__(self, pipe: PosePipeline, state: Dict[str, torch.Tensor], lr: float = 1e-3, betas: Sequence[float] = (0.9, 0.999),
                 eps: float = 1e-8, weight_decay: float = 0.0, slope: float = MLP_SLOPE):
        self.pipe = pipe
        self.net = MlpGrad(pipe, state, slope)
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        dev = pipe.device
        self.m = torch.zeros(self.net.n_flat, dtype=torch.float32, device=dev)
        self.v = torch.zeros(self.net.n_flat, dtype=torch.float32, device=dev)
        self.t = 0                                                            # host mirror of the device-side step count
        self.t_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.adam_scalars = torch.zeros(2, dtype=torch.float32, device=dev)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self.last_joints = None
        self._init_graphs()

    def _enqueue(self, x, loss_fn, args, update):
        net = self.net
        out = net.forward(x)
        joints = out.detach().requires_grad_(True)
        with torch.enable_grad():
            loss = loss_fn(joints, *args)
            (dj,) = torch.autograd.grad(loss, joints)
        self.loss.copy_(loss.detach().reshape(1))
        net.backward(dj.contiguous())
        if update:
            net.adam_planes(net.grad, self.m, self.v, self.lr, self.betas, self.eps, self.weight_decay, self.t_dev, self.adam_scalars)
        self.last_joints = out

    def step(self, x: torch.Tensor, loss_fn, *args, update: bool = True):
        """x [P, ...] MLP inputs (flattened per row); loss_fn(joints [P, n_out], *args) -> scalar tensor, plain torch code.
        Returns the loss as a device scalar (the step itself does not synchronise)."""
        self._enqueue(_rows(x, self.pipe.device), loss_fn, args, update)
        if update:
            self.t += 1
        return self.loss

    def step_captured(self, x: torch.Tensor, loss_fn, *args):
        """step() as one CUDA-graph replay. The first call for a key (input shape, loss function, tensor arguments' shapes and
        dtypes, other arguments by value) runs one eager forward + backward to size the workspaces and captures the step on
        static copies of x and the tensor arguments; later calls copy their inputs there and replay. loss_fn must be capturable
        (no host synchronisation). A workspace re-allocation (a larger batch) drops the graphs."""
        x = _rows(x, self.pipe.device)
        sig = lambda a: ('tensor', tuple(a.shape), a.dtype, a.device) if torch.is_tensor(a) else \
            (a if isinstance(a, (int, float, str, bool, type(None))) else ('object', id(a)))
        key = (tuple(x.shape), id(loss_fn)) + tuple(sig(a) for a in args)
        ent = self._cached_step(key, self.net.buf)
        if ent is None:
            self._enqueue(x, loss_fn, args, update=False)                        # sizes every workspace; no parameter changes
            sx = x.clone()
            sargs = [a.clone() if torch.is_tensor(a) else a for a in args]
            ent = dict(x=sx, args=sargs, fn=loss_fn, held=args)                  # holding fn / args keeps their ids unique
            self._capture_step(key, ent, self.net.buf, self.pipe.device, lambda: self._enqueue(sx, loss_fn, sargs, update=True))
        else:
            ent['x'].copy_(x, non_blocking=True)
            for st, a in zip(ent['args'], args):
                if torch.is_tensor(a):
                    st.copy_(a, non_blocking=True)
        ent['graph'].replay()
        self.t += 1
        self.last_joints = self.net.buf.f('out', x.shape[0], _ld4(self.net.n_out))[: x.shape[0], : self.net.n_out]
        return self.loss
