"""Batched inference pipeline: packed frames -> person proposals -> 3D joints, all on one B200.

This is the frame-batched replacement of the per-frame glue the reference repeats in its drivers
(test/metrics_from_model.py:178-300): graph build -> GAT -> clustering -> MLP-input encoding -> MLP.
Host code is PyTorch (allocation, streams); every computation is a kernel of libb200pose.so called
through the C ABI (include/b200pose.h). There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import collections
import dataclasses
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib
from ._lib import Cameras, check, ptr
from .config import CameraConfig, N_JOINTS
from .pack import PackedBatch
from .weights import GAT_ALPHA, GAT_ACT_SLOPE, MLP_SLOPE, gat_layer_dims


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def person_capacity(n_heads: int, min_views: int) -> int:
    """Upper bound on the persons of a batch: disjoint components of >= min_views heads each."""
    return max(n_heads // max(int(min_views), 1), 1)


def capture_capacity(seen: int, p_bound: int) -> int:
    """Rows the encoder and the MLP of a captured step are sized for: the persons a shape showed, with head-room, in
    multiples of 8 rows (the weight-stream kernel's step), at most p_bound (person_capacity of the shape). A replay that
    finds more persons than that is redone eagerly and re-captured."""
    return min(p_bound, max(8, (int(seen * 1.25) + 7) // 8 * 8))


# the arrays of a packed batch that go to the device, in upload order (the tensor fields of HostBatch and DeviceBatch)
INPUT_NAMES = ('sk_xy', 'sk_vp', 'sk_mask', 'sk_cam', 'head_off', 'node_off')


def pinned_results(n_frames: int, rows: int, n_cameras: int, n_out: int) -> dict:
    """Pinned host buffers for the results of a batch: per-frame person counts and offsets, and `rows` person rows."""
    mk = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
    return dict(n_persons=mk((n_frames,), torch.int32), person_off=mk((n_frames + 1,), torch.int32),
                person_sk=mk((rows, n_cameras), torch.int32), joints=mk((rows, max(n_out, 1)), torch.float32),
                valid=mk((rows,), torch.uint8))


def copy_person_rows(out: dict, res: dict, P: int, p0: int = 0):
    """Enqueues the device->host copies of the first P person rows of a result (person list, and joints and valid when
    the result has them) into rows p0.. of a pinned_results() set, on the current stream."""
    out['person_sk'][p0:p0 + P].copy_(res['person_sk'][:P], non_blocking=True)
    if 'joints' in res:
        out['joints'][p0:p0 + P].copy_(res['joints'][:P], non_blocking=True)
        out['valid'][p0:p0 + P].copy_(res['valid'][:P], non_blocking=True)


def host_results(bufs: dict, P: int, with_mlp: bool) -> dict:
    """The host result of a batch with P persons, as views of a pinned_results() set."""
    out = dict(n_persons=bufs['n_persons'], person_off=bufs['person_off'], person_sk=bufs['person_sk'][:P], n_persons_total=P)
    if with_mlp:
        out['joints'] = bufs['joints'][:P]
        out['valid'] = bufs['valid'][:P]
    return out


class Planes:
    """An fp32 matrix stored as hi/lo bf16 planes [rows, ld] (ld multiple of 64), zero padded."""

    def __init__(self, rows: int, cols: int, device):
        self.rows, self.cols = rows, cols
        self.ld = round_up(max(cols, 1), 64)
        self.hi = torch.zeros((max(rows, 1), self.ld), dtype=torch.bfloat16, device=device)
        self.lo = torch.zeros((max(rows, 1), self.ld), dtype=torch.bfloat16, device=device)

    @staticmethod
    def from_f32(x: torch.Tensor, stream) -> "Planes":
        x = x.contiguous().float()
        p = Planes(x.shape[0], x.shape[1], x.device)
        check(_lib.lib().b200pose_split_planes(ptr(x), x.shape[0], x.shape[1], x.shape[1], ptr(p.hi), ptr(p.lo), p.ld, stream),
              'split_planes')
        return p

    def to_f32(self) -> torch.Tensor:
        return (self.hi.float() + self.lo.float())[: self.rows, : self.cols]


class DeviceCameras:
    """Camera tables uploaded once per configuration (b200pose_cameras)."""

    def __init__(self, cfg: CameraConfig, device):
        self.cfg = cfg
        Cn = cfg.n_cameras
        sm_slot = np.full(Cn, -1, np.int32)
        pe_slot = np.full(Cn, -1, np.int32)
        for s, c in enumerate(cfg.used_sm):
            sm_slot[c] = s
        for s, c in enumerate(cfg.used_pe):
            pe_slot[c] = s
        kinv = np.stack([cfg.Kinv32(cfg.sm_table_camera(c)) for c in range(Cn)]).astype(np.float32)
        tinv = np.stack([cfg.T_cam2root32(c) for c in range(Cn)]).astype(np.float32)
        tinv_sm = np.stack([cfg.T_cam2root32(cfg.sm_table_camera(c)) for c in range(Cn)]).astype(np.float32)
        k64 = np.stack([[cfg.K64_from32(c)[0, 0], cfg.K64_from32(c)[1, 1], cfg.K64_from32(c)[0, 2], cfg.K64_from32(c)[1, 2]]
                        for c in range(Cn)]).astype(np.float64)
        dist = np.stack([cfg.dist64(c) for c in range(Cn)]).astype(np.float64)
        p64 = np.stack([cfg.P64(c) for c in range(Cn)]).astype(np.float64)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
        self.t = dict(sm_slot=up(sm_slot), pe_slot=up(pe_slot), kinv=up(kinv), tinv=up(tinv), k64=up(k64), dist=up(dist), p64=up(p64),
                      tinv_sm=up(tinv_sm))
        self.struct = Cameras(Cn, cfg.V_sm, cfg.V_pe, float(cfg.image_width), float(cfg.image_height),
                              self.t['sm_slot'].data_ptr(), self.t['pe_slot'].data_ptr(), self.t['kinv'].data_ptr(),
                              self.t['tinv'].data_ptr(), self.t['k64'].data_ptr(), self.t['dist'].data_ptr(),
                              self.t['p64'].data_ptr(), self.t['tinv_sm'].data_ptr())

    @property
    def ref(self):
        return C.byref(self.struct)


@dataclasses.dataclass
class DeviceBatch:
    """A PackedBatch resident in HBM."""
    n_frames: int
    n_heads: int
    n_nodes: int
    max_heads: int
    max_enodes: int
    sk_xy: torch.Tensor
    sk_vp: torch.Tensor
    sk_mask: torch.Tensor
    sk_cam: torch.Tensor
    head_off: torch.Tensor
    node_off: torch.Tensor
    host_offsets: Optional[tuple] = None      # (head_off, node_off) numpy copies, when the batch came from a PackedBatch

    @property
    def n_enodes(self):
        return self.n_nodes - self.n_heads

    @property
    def n_edges(self):
        return self.n_heads + 5 * self.n_enodes


class HostBatch:
    """Pinned host copy of a PackedBatch, so host->device copies are asynchronous DMA."""

    def __init__(self, pb: PackedBatch, pinned: bool = True):
        # pinned=False: plain host tensors (page-locking six small arrays costs more than a live frame's copy saves;
        # infer_host_graph stages through its own pinned buffers anyway)
        pin = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).pin_memory() if pinned and torch.cuda.is_available() \
            else torch.from_numpy(np.ascontiguousarray(a)).to(dt)
        self.pb = pb
        pb.validate()
        self.sk_xy = pin(pb.sk_xy, torch.float64)
        self.sk_vp = pin(pb.sk_vp, torch.float32)
        self.sk_mask = pin(pb.sk_mask.view(np.int32), torch.int32)
        self.sk_cam = pin(pb.sk_cam, torch.int32)
        self.head_off = pin(pb.head_off, torch.int32)
        self.node_off = pin(pb.node_off, torch.int32)

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.sk_xy, self.sk_vp, self.sk_mask, self.sk_cam, self.head_off, self.node_off))

    frame_range = None       # (first, last+1) frame of the parent batch, set on chunks
    head_range = None

    def split(self, n_chunks: int):
        """Contiguous runs of frames as HostBatch views that share this batch's pinned memory (offset arrays are
        rebased copies). Cached: the split is part of packing, not of inference."""
        n_chunks = max(1, min(int(n_chunks), max(self.pb.n_frames, 1)))
        cache = self.__dict__.setdefault('_splits', {})
        if n_chunks in cache:
            return cache[n_chunks]
        B = self.pb.n_frames
        out = []
        for k in range(n_chunks):
            f0, f1 = (B * k) // n_chunks, (B * (k + 1)) // n_chunks
            if n_chunks == 1:
                ch = self
            else:
                sub = self.pb.slice(f0, f1)
                h0, h1 = int(self.pb.head_off[f0]), int(self.pb.head_off[f1])
                ch = HostBatch.__new__(HostBatch)
                ch.pb = sub
                ch.sk_xy, ch.sk_vp = self.sk_xy[h0:h1], self.sk_vp[h0:h1]
                ch.sk_mask, ch.sk_cam = self.sk_mask[h0:h1], self.sk_cam[h0:h1]
                pin = (lambda t: t.pin_memory()) if torch.cuda.is_available() else (lambda t: t)
                ch.head_off = pin(torch.from_numpy(np.ascontiguousarray(sub.head_off)))
                ch.node_off = pin(torch.from_numpy(np.ascontiguousarray(sub.node_off)))
            ch.frame_range = (f0, f1)
            ch.head_range = (int(self.pb.head_off[f0]), int(self.pb.head_off[f1]))
            out.append(ch)
        cache[n_chunks] = out
        return out

    def result_buffers(self, n_cameras: int, n_out: int, min_views: int = 2):
        """Pinned host buffers for the results of this batch. A person is a connected component of at least `min_views`
        heads (parameters.min_number_of_views, skeleton_matching_utils.py:120) and components are disjoint, so there are at
        most heads // min_views persons."""
        key = (n_cameras, n_out, min_views)
        cache = self.__dict__.setdefault('_results', {})
        if key not in cache:
            cache[key] = pinned_results(self.pb.n_frames, person_capacity(self.pb.n_heads, min_views), n_cameras, n_out)
        return cache[key]

    def to_device(self, device) -> DeviceBatch:
        pb = self.pb
        cp = lambda t: t.to(device, non_blocking=True)
        return DeviceBatch(pb.n_frames, pb.n_heads, pb.n_nodes, pb.max_heads, pb.max_enodes,
                           cp(self.sk_xy), cp(self.sk_vp), cp(self.sk_mask), cp(self.sk_cam), cp(self.head_off), cp(self.node_off),
                           host_offsets=(np.asarray(pb.head_off, dtype=np.int64), np.asarray(pb.node_off, dtype=np.int64)))

    def upload(self, device, copy_stream, consumer):
        """to_device() enqueued on `copy_stream` for compute on `consumer`: returns the DeviceBatch and an event recorded
        after its copies, which the consumer waits for."""
        with torch.cuda.stream(copy_stream):
            db = self.to_device(device)
            for n in INPUT_NAMES:
                getattr(db, n).record_stream(consumer)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return db, ev

    def static_copy(self, device):
        """(h_in, db) for a captured step that uploads its own inputs (copy_inputs): pinned staging buffers holding this
        batch's arrays, and a DeviceBatch of device buffers of the same shapes. The graph bakes in the addresses of both, so
        a replay takes new frames of the shape through h_in."""
        h_in = {n: torch.empty_like(getattr(self, n)).pin_memory() for n in INPUT_NAMES}
        d_in = [torch.empty_like(getattr(self, n), device=device) for n in INPUT_NAMES]
        for n in INPUT_NAMES:
            h_in[n].copy_(getattr(self, n))
        pb = self.pb
        return h_in, DeviceBatch(pb.n_frames, pb.n_heads, pb.n_nodes, pb.max_heads, pb.max_enodes, *d_in)


def copy_inputs(db: DeviceBatch, h_in: dict):
    """Enqueues the host->device copies of a batch's inputs from the staging buffers of HostBatch.static_copy()."""
    for n in INPUT_NAMES:
        getattr(db, n).copy_(h_in[n], non_blocking=True)


class GraphArrays:
    """Output of stage 1a (b200pose_build_graph)."""

    def __init__(self, db: DeviceBatch, device, with_coo=True):
        i32 = dict(dtype=torch.int32, device=device)
        E = db.n_edges
        self.src = torch.empty(max(E, 1), **i32) if with_coo else None
        self.dst = torch.empty(max(E, 1), **i32) if with_coo else None
        self.row_ptr = torch.empty(db.n_nodes + 1, **i32)
        self.col = torch.empty(max(E, 1), **i32)
        self.pairs = torch.empty((max(db.n_enodes, 1), 2), **i32)
        self.node_cam = torch.empty(max(db.n_nodes, 1), **i32)
        # True: built from an explicit edge-node list (b200pose_build_graph_pairs: training-side topology, dgl.batch
        # members) - clustering then takes the first-seen head order from the list instead of the test-mode closed form.
        # The aggregation kernels only need what both builders guarantee: heads first, three in-edges (h1, h2, self) per
        # edge-node, in-edges of a node in ascending edge id.
        self.general = False
        self.pending = None       # side stream the builder was launched on (build_graph(overlap=True)), until wait_graph() joins it


def _on_own_device(fn):
    """Public entry points run with the pipeline's device current: the kernels launch on that device's current stream and
    cudaFuncSetAttribute is per device, so a PosePipeline('cuda:1') must not depend on what the caller left selected."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        if torch.cuda.current_device() == self._device_index():
            return fn(self, *a, **k)
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)
    return wrapper


class _Owned:
    """The streams and caches of one pipeline. A twin() gets a fresh set, so two lanes share nothing but the read-only
    camera tables and weight planes."""

    def __init__(self):
        self.ws = {}                                 # activation workspaces (planes_ws, f32_ws)
        self.streams = {}                            # auxiliary streams by role, created on first use (_aux_stream)
        self.lanes = None                            # lanes(): (weights generation, pipelines, streams)
        self.graphs = collections.OrderedDict()      # infer_host_graph: captured step per batch shape
        self.graph_person_hint = {}                  # infer_host_graph: the largest person count a shape has shown
        self.stream_results = {}                     # infer_host_stream: rotating pinned result sets per batch size
        self.person_stage = {}                       # encode_person_dicts: pinned + device staging buffers per size


class PosePipeline:
    """Weights + camera tables resident on one GPU; `infer()` runs a whole batch of frames.

    gat_state / mlp_state: state dicts with the reference's key names
    (GAT `layers.{l}.{attn_l,attn_r,fc1.*,fc2.*}`, MLP `layers.{1,3,..,17}.{weight,bias}`).
    """

    def __init__(self, cfg: CameraConfig, gat_state: Optional[Dict[str, torch.Tensor]] = None,
                 mlp_state: Optional[Dict[str, torch.Tensor]] = None,
                 device=None, gemm_impl: int = 0, threshold: float = 0.5):
        if not torch.cuda.is_available():
            raise RuntimeError('PosePipeline needs a CUDA device (sm_100a); there is no CPU fallback')
        self.device = torch.device(device if device is not None else 'cuda')
        self._dev_index = None
        self.cfg = cfg
        self.L = _lib.lib()
        self.gemm_impl = gemm_impl
        self.agg_impl = 0          # 0 = frame-resident aggregation kernel when it fits, 1 = gather kernel
        self.fuse_small_fc2 = True  # last GAT layer: fc2 (3 columns) inside fc1's epilogue (False: two launches, for A/B runs)
        self.threshold = float(threshold)
        self.launches = 0
        self._own = _Owned()
        with torch.cuda.device(self.device):
            self.cams = DeviceCameras(cfg, self.device)
            self.gat = self.prepare_gat(gat_state) if gat_state is not None else None
            self.mlp = self.prepare_mlp(mlp_state) if mlp_state is not None else None
            torch.cuda.synchronize()

    # the prepared weight planes; replacing them invalidates every captured CUDA graph (they hold the old plane addresses)
    @property
    def gat(self):
        return self._gat

    @gat.setter
    def gat(self, layers):
        self._gat = layers
        self._weights_gen = getattr(self, '_weights_gen', 0) + 1

    @property
    def mlp(self):
        return self._mlp

    @mlp.setter
    def mlp(self, layers):
        self._mlp = layers
        self._weights_gen = getattr(self, '_weights_gen', 0) + 1

    def _device_index(self) -> int:
        if self._dev_index is None:
            self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        return self._dev_index

    def _aux_stream(self, role: str):
        """This pipeline's stream for `role` ('side', 'copy', 'd2h', 'counts'), created on first use. Streams map
        round-robin onto the hardware queues, so one created before it is needed can alias a stream that is in use."""
        s = self._own.streams.get(role)
        if s is None:
            s = self._own.streams[role] = torch.cuda.Stream(self.device)
        return s

    # ------------------------------------------------------------------ compute lanes
    def twin(self) -> "PosePipeline":
        """A second pipeline on the same device that SHARES this one's camera tables and weight planes (read-only) and has its
        own workspaces, streams and caches: two independent batches can then be in flight on two CUDA streams. A step
        has ~0.26 ms of latency-bound phases (graph build + features, clustering, person list, encoder: 8-26 % warps
        active) that fit beside another batch's tensor-core GEMMs on the same SMs."""
        t = PosePipeline.__new__(PosePipeline)
        t.__dict__.update(self.__dict__)
        t._own = _Owned()
        t.launches = 0
        return t

    def lanes(self, n: int):
        """[self, twin, ...] and one compute stream per extra lane (lane 0 runs on the caller's current stream); cached.
        A lane whose weights were replaced on `self` since it was made is rebuilt."""
        have = self._own.lanes
        gen = getattr(self, '_weights_gen', 0)
        if have is None or have[0] != gen or len(have[1]) < n:
            pipes = [self] + [self.twin() for _ in range(n - 1)]
            streams = [None] + [torch.cuda.Stream(self.device) for _ in range(n - 1)]
            have = self._own.lanes = (gen, pipes, streams)
        return have[1][:n], have[2][:n]

    # ------------------------------------------------------------------ workspace
    def planes_ws(self, tag: str, rows: int, cols: int) -> Planes:
        """Activation planes from a per-pipeline workspace. They are zero-initialised once; kernels write
        every valid column and only ever write zeros into the K padding, so reuse needs no memset."""
        key = (tag, round_up(max(cols, 1), 64))
        ws = self._own.ws.get(key)
        if ws is None or ws.hi.shape[0] < rows:
            cap = max(rows, int(ws.hi.shape[0] * 1.25) if ws is not None else rows)
            ws = Planes(cap, cols, self.device)
            self._own.ws[key] = ws
        view = Planes.__new__(Planes)
        view.rows, view.cols, view.ld, view.hi, view.lo = rows, cols, ws.ld, ws.hi, ws.lo
        return view

    def f32_ws(self, tag: str, rows: int, cols: int) -> torch.Tensor:
        key = (tag, cols)
        t = self._own.ws.get(key)
        if t is None or t.shape[0] < rows:
            t = torch.empty((max(rows, 1), cols), dtype=torch.float32, device=self.device)
            self._own.ws[key] = t
        return t

    # ------------------------------------------------------------------ weights
    def _stream(self):
        # the raw cudaStream_t of torch's current stream on this device; the public torch.cuda.current_stream() costs
        # ~17 us per call (device-index resolution), which at 30 launches is most of a live frame's host time
        return C.c_void_p(torch._C._cuda_getCurrentRawStream(self._device_index()))

    def prepare_gat(self, st, residual: bool = False):
        """Split every projection into planes; fold the attention vectors into fc2 as 2*heads extra output
        rows: a1[n,h] = sum_d ft2[n,h,d]*attn_l[h,d] = h2[n,:] . (sum_d attn_l[h,d]*W2[hD+d,:]) + bias term
        (gat2.py:55-58), so one GEMM yields [ft2 | a1 | a2]."""
        layers = []
        n_layers = len([k for k in st if k.endswith('fc1.weight')])
        for l in range(n_layers):
            g = lambda k: st['layers.%d.%s' % (l, k)].detach().to('cpu', torch.float64)
            W1, W2 = g('fc1.weight'), g('fc2.weight')
            din = W1.shape[1]
            has_bias = ('layers.%d.fc1.bias' % l) in st
            b1 = g('fc1.bias') if has_bias else torch.zeros(W1.shape[0], dtype=torch.float64)
            b2 = g('fc2.bias') if has_bias else torch.zeros(W2.shape[0], dtype=torch.float64)
            al, ar = g('attn_l')[:, :, 0], g('attn_r')[:, :, 0]          # [H, D]
            H, D = al.shape
            W2h = W2.reshape(H, D, din)
            Wl = torch.einsum('hd,hdk->hk', al, W2h)
            Wr = torch.einsum('hd,hdk->hk', ar, W2h)
            bl = (al * b2.reshape(H, D)).sum(1)
            br = (ar * b2.reshape(H, D)).sum(1)
            W2e = torch.cat([W2, Wl, Wr], 0).float().to(self.device)
            b2e = torch.cat([b2, bl, br], 0).float().to(self.device)
            s = self._stream()
            lay = dict(
                din=din, heads=H, dim=D, hd=H * D, n2=H * D + 2 * H, ldz=round_up(H * D + 2 * H, 4),
                w1=Planes.from_f32(W1.float().to(self.device), s), b1=b1.float().to(self.device),
                w2=Planes.from_f32(W2e, s), b2=b2e)
            if lay['n2'] <= 4 and din <= 256:
                # a few output columns (the last layer: ft2 | a1 | a2 = 3): fc2 is evaluated in fc1's epilogue
                # (b200pose_linear_fused2) from fp32 weight rows padded to a multiple of 64 columns
                w2f = torch.zeros((lay['n2'], round_up(din, 64)), dtype=torch.float32, device=self.device)
                w2f[:, :din] = W2e
                lay['w2_f32'] = w2f
            if residual and l > 0:
                # gat2.py:43-48, 70-75: res_fc(h) when the layer changes the width, the input itself (broadcast over the
                # attention heads) when in_dim == out_dim; the first layer is always built without a residual (:108)
                if ('layers.%d.res_fc.weight' % l) in st:
                    Wr_ = g('res_fc.weight')
                    lay['res_w'] = Planes.from_f32(Wr_.float().to(self.device), s)
                    lay['res_b'] = (g('res_fc.bias') if ('layers.%d.res_fc.bias' % l) in st
                                    else torch.zeros(Wr_.shape[0], dtype=torch.float64)).float().to(self.device)
                elif din == D:
                    lay['res_identity'] = True
                else:
                    raise ValueError('prepare_gat: residual layer %d has in_dim %d != out_dim %d but no res_fc weights' % (l, din, D))
            layers.append(lay)
        return layers

    def prepare_mlp(self, st):
        layers = []
        s = self._stream()
        for l in range(1, 18, 2):
            W = st['layers.%d.weight' % l].detach().float().to(self.device)
            b = st['layers.%d.bias' % l].detach().float().to(self.device)
            layers.append(dict(w=Planes.from_f32(W, s), b=b, n=W.shape[0], k=W.shape[1]))
        return layers

    # ------------------------------------------------------------------ kernels
    def linear(self, a: Planes, m: int, w: Planes, bias, n: int, k: int, slope: float, scale: float = 1.0,
               out_f32: Optional[torch.Tensor] = None, out_planes: Optional[Planes] = None, m_dev: Optional[torch.Tensor] = None):
        """out = act(A W^T + b). With `m_dev` (an int32 device scalar) `m` is only the capacity of the buffers: the kernel reads
        the number of valid rows from the device, so no host round trip is needed to size the launch."""
        self.launches += 1
        tail = (ptr(out_f32), out_f32.stride(0) if out_f32 is not None else 0,
                ptr(out_planes.hi) if out_planes else None, ptr(out_planes.lo) if out_planes else None,
                out_planes.ld if out_planes else 0, self.gemm_impl, self._stream())
        if m_dev is None:
            check(self.L.b200pose_linear(ptr(a.hi), ptr(a.lo), a.ld, ptr(w.hi), ptr(w.lo), w.ld, ptr(bias), m, n, k, slope, scale, *tail), 'linear')
        else:
            check(self.L.b200pose_linear_n(ptr(a.hi), ptr(a.lo), a.ld, ptr(w.hi), ptr(w.lo), w.ld, ptr(bias), m, ptr(m_dev), n, k, slope, scale,
                                           *tail), 'linear_n')

    def build_graph(self, db: DeviceBatch, with_coo=True, overlap: bool = False) -> GraphArrays:
        """overlap=True launches the builder on a side stream: nothing reads the graph before the first aggregation, so it
        runs beside the head features and the two layer-0 projections; `wait_graph(g)` joins it."""
        g = GraphArrays(db, self.device, with_coo)
        self.launches += 1
        if overlap:
            cur = torch.cuda.current_stream(self.device)
            side = self._aux_stream('side')
            side.wait_stream(cur)                               # the packed batch (and, in a capture, the fork point)
            with torch.cuda.stream(side):
                check(self.L.b200pose_build_graph(db.n_frames, ptr(db.head_off), ptr(db.node_off), ptr(db.sk_cam), self.cams.ref,
                                                  ptr(g.src), ptr(g.dst), ptr(g.row_ptr), ptr(g.col), ptr(g.pairs), ptr(g.node_cam),
                                                  self._stream()), 'build_graph')
            g.pending = side
            return g
        check(self.L.b200pose_build_graph(db.n_frames, ptr(db.head_off), ptr(db.node_off), ptr(db.sk_cam), self.cams.ref,
                                          ptr(g.src), ptr(g.dst), ptr(g.row_ptr), ptr(g.col), ptr(g.pairs), ptr(g.node_cam),
                                          self._stream()), 'build_graph')
        return g

    def wait_graph(self, g: GraphArrays):
        side = getattr(g, 'pending', None)
        if side is not None:
            torch.cuda.current_stream(self.device).wait_stream(side)
            g.pending = None

    def build_graph_pairs(self, db: DeviceBatch, pairs, with_coo=True) -> GraphArrays:
        """Graphs of a block-diagonal batch from explicit edge-node lists (process_training topology,
        graph_generator.py:672-810; dgl.batch members): `pairs` [M_tot, 2] int32 graph-local (head1, head2) per
        edge-node, graph after graph, node_off already counting them. db.max_heads must cover the largest in-degree
        (1 + edge-nodes touching a head), which sizes the aggregation scratch."""
        g = GraphArrays(db, self.device, with_coo)
        g.general = True
        pairs = torch.as_tensor(pairs, dtype=torch.int32).reshape(-1, 2)
        if pairs.shape[0] != db.n_enodes:
            raise ValueError('build_graph_pairs: %d pairs for %d edge-nodes' % (pairs.shape[0], db.n_enodes))
        if db.n_enodes:
            g.pairs[: db.n_enodes].copy_(pairs.to(self.device, non_blocking=True))
        self.launches += 1
        check(self.L.b200pose_build_graph_pairs(db.n_frames, ptr(db.head_off), ptr(db.node_off), ptr(db.sk_cam), self.cams.ref,
                                                ptr(g.pairs), db.max_heads, ptr(g.src), ptr(g.dst), ptr(g.row_ptr), ptr(g.col),
                                                ptr(g.node_cam), self._stream()), 'build_graph_pairs')
        return g

    def node_features_f32(self, db: DeviceBatch) -> torch.Tensor:
        F = self.cfg.n_features_sm
        out = torch.empty((max(db.n_nodes, 1), F), dtype=torch.float32, device=self.device)
        self.launches += 1
        check(self.L.b200pose_node_features(db.n_frames, db.n_heads, db.n_nodes, ptr(db.head_off), ptr(db.node_off),
                                            ptr(db.sk_xy), ptr(db.sk_vp), ptr(db.sk_mask), ptr(db.sk_cam), self.cams.ref,
                                            ptr(out), F, None, None, 0, self._stream()), 'node_features')
        return out[: db.n_nodes]

    def head_feature_planes(self, db: DeviceBatch) -> Planes:
        p = self.planes_ws('x0', db.n_heads + 1, self.cfg.n_features_sm)
        self.launches += 1
        check(self.L.b200pose_node_features(db.n_frames, db.n_heads, db.n_nodes, ptr(db.head_off), ptr(db.node_off),
                                            ptr(db.sk_xy), ptr(db.sk_vp), ptr(db.sk_mask), ptr(db.sk_cam), self.cams.ref,
                                            None, 0, ptr(p.hi), ptr(p.lo), p.ld, self._stream()), 'node_features')
        return p

    def aggregate(self, db: DeviceBatch, g: GraphArrays, z: torch.Tensor, layer: dict, layer0: bool,
                  raw: Optional[torch.Tensor], act: Optional[Planes], scores: Optional[torch.Tensor],
                  alpha: float = GAT_ALPHA, act_slope: float = GAT_ACT_SLOPE, res: Optional[torch.Tensor] = None):
        self.launches += 1
        self.wait_graph(g)
        if res is not None:
            check(self.L.b200pose_gat_aggregate_res(db.n_frames, db.n_nodes, db.n_heads, ptr(db.head_off), ptr(db.node_off),
                                                    ptr(g.row_ptr), ptr(g.col), ptr(z), z.stride(0), layer['heads'], layer['dim'],
                                                    db.max_heads, db.max_enodes, alpha, act_slope, ptr(res), res.stride(0), ptr(raw),
                                                    ptr(act.hi) if act else None, ptr(act.lo) if act else None, act.ld if act else 0,
                                                    ptr(scores), self._stream()), 'gat_aggregate_res')
            return
        check(self.L.b200pose_gat_aggregate(db.n_frames, db.n_nodes, db.n_heads, ptr(db.head_off), ptr(db.node_off),
                                            ptr(g.row_ptr), ptr(g.col), ptr(z), z.stride(0), layer['heads'], layer['dim'],
                                            1 if layer0 else 0, db.max_heads, db.max_enodes, alpha, act_slope, ptr(raw),
                                            ptr(act.hi) if act else None, ptr(act.lo) if act else None, act.ld if act else 0,
                                            ptr(scores), self.agg_impl, self._stream()), 'gat_aggregate')

    # ------------------------------------------------------------------ stages
    def gat_forward(self, db: DeviceBatch, g: GraphArrays, x0: Optional[Planes] = None, dense_rows: bool = False,
                    keep_layers: bool = False, layers=None, alpha: float = GAT_ALPHA, act_slope: float = GAT_ACT_SLOPE,
                    final_sigmoid: bool = True):
        """GAT2.forward over the whole batch. By default layer 0 runs on the S+1 compact rows (every head
        plus the one shared edge-node row). With dense_rows=True, x0 holds one row per node (the drop-in
        GAT2.forward path, where the caller hands in an arbitrary feature matrix)."""
        N, S = db.n_nodes, db.n_heads
        raws = []
        if x0 is None:
            x0 = self.head_feature_planes(db)
        x, rows = x0, (N if dense_rows else S + 1)
        scores = torch.empty(max(N, 1), dtype=torch.float32, device=self.device)
        layers = layers if layers is not None else self.gat
        logits = torch.empty(max(N, 1), dtype=torch.float32, device=self.device) if not final_sigmoid else None
        for l, lay in enumerate(layers):
            last = l == len(layers) - 1
            z = self.f32_ws('gat_z', rows, lay['ldz'])
            res = None
            if 'res_w' in lay:
                res = self.f32_ws('gat_res', rows, round_up(lay['hd'], 4))
                self.linear(x, rows, lay['res_w'], lay['res_b'], lay['hd'], lay['din'], 1.0, out_f32=res)
            elif lay.get('res_identity'):
                res = x.to_f32()[:rows, : lay['din']].repeat(1, lay['heads']).contiguous()
            if 'w2_f32' in lay and self.gemm_impl == 0 and rows > 16 and self.fuse_small_fc2:
                self.launches += 1
                w2f = lay['w2_f32']
                check(self.L.b200pose_linear_fused2(ptr(x.hi), ptr(x.lo), x.ld, ptr(lay['w1'].hi), ptr(lay['w1'].lo), lay['w1'].ld, ptr(lay['b1']),
                                                    rows, lay['din'], lay['din'], alpha, ptr(w2f), w2f.stride(0), ptr(lay['b2']), lay['n2'],
                                                    ptr(z), z.stride(0), self._stream()), 'linear_fused2')
            else:
                h = self.planes_ws('gat_h', rows, lay['din'])
                self.linear(x, rows, lay['w1'], lay['b1'], lay['din'], lay['din'], alpha, out_planes=h)
                self.linear(h, rows, lay['w2'], lay['b2'], lay['n2'], lay['din'], 1.0, out_f32=z)
            raw = torch.empty((max(N, 1), lay['hd']), dtype=torch.float32, device=self.device) if keep_layers else None
            act = None if last else self.planes_ws('gat_act%d' % (l & 1), N, lay['hd'])
            if last and not final_sigmoid and raw is None:
                raw = logits.view(-1, 1)
            self.aggregate(db, g, z, lay, layer0=(l == 0 and not dense_rows), raw=raw, act=act,
                           scores=scores if (last and final_sigmoid) else None, alpha=alpha, act_slope=act_slope, res=res)
            if keep_layers:
                raws.append(raw[:N])
            x, rows = act, N
        out = scores[:N] if final_sigmoid else raw.reshape(-1)[:N]
        return (out, raws) if keep_layers else out

    def cluster(self, db: DeviceBatch, g: GraphArrays, scores: torch.Tensor, threshold: Optional[float] = None):
        V = self.cfg.V_sm
        thr = self.threshold if threshold is None else float(threshold)
        person_heads = torch.empty((max(db.n_heads, 1), V), dtype=torch.int32, device=self.device)
        n_persons = torch.empty(max(db.n_frames, 1), dtype=torch.int32, device=self.device)
        self.launches += 1
        fn = self.L.b200pose_cluster_pairs if getattr(g, 'general', False) else self.L.b200pose_cluster
        check(fn(db.n_frames, ptr(db.head_off), ptr(db.node_off), ptr(g.pairs), ptr(g.node_cam), ptr(scores),
                 V, thr, self.cfg.min_number_of_views, db.max_heads, db.max_enodes,
                 ptr(person_heads), ptr(n_persons), self._stream()), 'cluster')
        return person_heads, n_persons[: db.n_frames]

    def person_list(self, db: DeviceBatch, res: dict, rows: int, fill: bool = False):
        """The persons stage_a found as person_sk [rows, C] (skeleton id per camera, -1 = none) and person_frame [rows];
        `rows` must cover the person count. With fill=True the rows past the count are person_sk = -1, person_frame = 0."""
        n, i32 = max(rows, 1), dict(dtype=torch.int32, device=self.device)
        if fill:
            person_sk, person_frame = torch.full((n, self.cfg.n_cameras), -1, **i32), torch.zeros(n, **i32)
        else:
            person_sk, person_frame = torch.empty((n, self.cfg.n_cameras), **i32), torch.empty(n, **i32)
        if rows > 0:
            self.launches += 1
            check(self.L.b200pose_gather_persons(db.n_frames, ptr(db.head_off), ptr(res['person_heads']), ptr(res['n_persons']),
                                                 ptr(res['person_off']), 0, ptr(db.sk_cam), self.cfg.V_sm, self.cams.ref,
                                                 ptr(person_sk), ptr(person_frame), self._stream()), 'gather_persons')
        return person_sk, person_frame

    def encode_persons(self, db: DeviceBatch, P: int, person_sk, want_f32=False, n_dev: Optional[torch.Tensor] = None):
        """MLP input rows of P persons. With `n_dev` (int32 device scalar) P is a capacity and the kernel handles the
        persons the device-side count names."""
        x = self.planes_ws('mlp_x', P, self.cfg.mlp_in)
        valid = torch.empty(max(P, 1), dtype=torch.uint8, device=self.device)
        xf = torch.zeros((max(P, 1), self.cfg.mlp_in), dtype=torch.float32, device=self.device) if want_f32 else None
        self.launches += 1
        args = (ptr(person_sk), ptr(db.sk_xy), ptr(db.sk_vp), ptr(db.sk_mask), self.cams.ref,
                ptr(xf), self.cfg.mlp_in if want_f32 else 0, ptr(x.hi), ptr(x.lo), x.ld, ptr(valid), self._stream())
        if n_dev is None:
            check(self.L.b200pose_encode_persons(P, *args), 'encode_persons')
        else:
            check(self.L.b200pose_encode_persons_n(P, ptr(n_dev), *args), 'encode_persons_n')
        return x, valid[:P], (xf[:P] if want_f32 else None)

    def triangulate(self, db: DeviceBatch, P: int, person_sk):
        xyz = torch.empty((max(P, 1), N_JOINTS, 3), dtype=torch.float64, device=self.device)
        mask = torch.empty((max(P, 1), N_JOINTS), dtype=torch.uint8, device=self.device)
        self.launches += 1
        check(self.L.b200pose_triangulate(P, ptr(person_sk), ptr(db.sk_xy), ptr(db.sk_mask), self.cams.ref, self.cfg.median_axis,
                                          ptr(xyz), ptr(mask), self._stream()), 'triangulate')
        return xyz[:P], mask[:P]

    def encode_person_dicts(self, persons: List[Dict[str, dict]]):
        """MLP input rows for persons given as {camera_name: skeleton dict} (the `raw_input` the reference's
        drivers hand to PoseEstimatorDataset, test/metrics_from_model.py:243-266). Returns (x [P, 252*V] fp32
        on the device, valid [P] bool list)."""
        from .pack import pack_skeleton
        names = self.cfg.camera_names
        xy, vp, mask = [], [], []
        person_sk = np.full((max(len(persons), 1), self.cfg.n_cameras), -1, np.int32)
        for p, person in enumerate(persons):
            for cam, sk in person.items():
                a, b, m = pack_skeleton(sk)
                person_sk[p, names.index(cam)] = len(xy)
                xy.append(a); vp.append(b); mask.append(m)
        S = max(len(xy), 1)
        P = len(persons)
        Pn = max(P, 1)
        # one pinned staging buffer and one host->device copy for the four small inputs (a call per person is how the
        # reference's drivers use this: test/metrics_from_model.py:243-266)
        n_xy, n_vp, n_mask, n_psk = S * N_JOINTS * 2 * 8, S * N_JOINTS * 2 * 4, S * 4, Pn * self.cfg.n_cameras * 4
        offs = [0]
        for nb in (n_xy, n_vp, n_mask, n_psk):                  # every region starts 8-byte aligned
            offs.append((offs[-1] + nb + 7) // 8 * 8)
        total = offs[-1]
        stage = self._own.person_stage
        if total not in stage:
            stage[total] = (torch.empty(total, dtype=torch.uint8).pin_memory(), torch.empty(total, dtype=torch.uint8, device=self.device))
        h_buf, d_buf = stage[total]
        hv = h_buf.numpy()
        hv[offs[0]:offs[0] + n_xy].view(np.float64)[:] = (np.stack(xy) if xy else np.zeros((1, N_JOINTS, 2))).ravel()
        hv[offs[1]:offs[1] + n_vp].view(np.float32)[:] = (np.stack(vp) if vp else np.zeros((1, N_JOINTS, 2), np.float32)).ravel()
        hv[offs[2]:offs[2] + n_mask].view(np.uint32)[:] = np.array(mask if mask else [0], dtype=np.uint32)
        hv[offs[3]:offs[3] + n_psk].view(np.int32)[:] = person_sk.ravel()
        d_buf.copy_(h_buf, non_blocking=True)
        sk_xy = d_buf[offs[0]:offs[0] + n_xy].view(torch.float64)
        sk_vp = d_buf[offs[1]:offs[1] + n_vp].view(torch.float32)
        sk_mask = d_buf[offs[2]:offs[2] + n_mask].view(torch.int32)
        psk = d_buf[offs[3]:offs[3] + n_psk].view(torch.int32)
        valid = torch.empty(Pn, dtype=torch.uint8, device=self.device)
        xf = torch.zeros((Pn, self.cfg.mlp_in), dtype=torch.float32, device=self.device)
        self.launches += 1
        check(self.L.b200pose_encode_persons(P, ptr(psk), ptr(sk_xy), ptr(sk_vp), ptr(sk_mask), self.cams.ref,
                                             ptr(xf), self.cfg.mlp_in, None, None, 0, ptr(valid), self._stream()), 'encode_persons')
        return xf[:P], [bool(v) for v in valid[:P].cpu().tolist()]

    def triangulate_tables(self, k64, dist64, p64, sk_xy, sk_mask, median_axis: int):
        """triangulate() with caller-supplied camera tables (utils/pose_estimator_utils.py:52-75): one person whose
        skeleton in camera i is row i of sk_xy [C,18,2] / sk_mask [C]. Returns ([18,3] float64, [18] mask) on the host."""
        Cn = int(k64.shape[0])
        if Cn > 32:
            raise ValueError('at most 32 cameras')
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(self.device)
        t = dict(k=up(k64, torch.float64), d=up(dist64, torch.float64), p=up(p64, torch.float64),
                 xy=up(sk_xy, torch.float64), m=up(np.asarray(sk_mask, dtype=np.uint32).view(np.int32), torch.int32),
                 psk=torch.arange(Cn, dtype=torch.int32, device=self.device).reshape(1, Cn))
        cams = Cameras(Cn, 0, 0, 0.0, 0.0, None, None, None, None, t['k'].data_ptr(), t['d'].data_ptr(), t['p'].data_ptr())
        xyz = torch.empty((1, N_JOINTS, 3), dtype=torch.float64, device=self.device)
        mask = torch.empty((1, N_JOINTS), dtype=torch.uint8, device=self.device)
        self.launches += 1
        check(self.L.b200pose_triangulate(1, ptr(t['psk']), ptr(t['xy']), ptr(t['m']), C.byref(cams), int(median_axis),
                                          ptr(xyz), ptr(mask), self._stream()), 'triangulate')
        return xyz[0].cpu().numpy(), mask[0].cpu().numpy()

    def mlp_forward(self, x: Planes, P: int, scale: float = 10.0, layers=None, slope: float = MLP_SLOPE,
                    m_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
        """PoseEstimatorMLP.forward (utils/mlp.py:8-31); `scale` is the x10 the callers apply
        (metrics_from_model.py:282), fused into the last epilogue."""
        layers = layers if layers is not None else self.mlp
        n_out = layers[-1]['n']
        out = self.f32_ws('mlp_out', P, round_up(n_out, 4))          # TMA store needs a 16-byte row pitch
        # A live frame's handful of persons: the layers are weight streams (116 MB for 9 layers), served by the kernel that
        # keeps up to 8 rows of A in registers; 9..32 rows go through it 8 at a time - the second pass over a layer's
        # weights (at most 38 MB) comes out of L2
        chunks = [(0, P)] if P <= 8 or P > 32 or m_dev is not None else [(r, min(r + 8, P)) for r in range(0, P, 8)]

        def rows(pl: Planes, r0, r1):
            v = Planes.__new__(Planes)
            v.rows, v.cols, v.ld, v.hi, v.lo = r1 - r0, pl.cols, pl.ld, pl.hi[r0:r1], pl.lo[r0:r1]
            return v
        for i, lay in enumerate(layers):
            last = i == len(layers) - 1
            y = None if last else self.planes_ws('mlp_y%d' % (i & 1), P, lay['n'])
            for r0, r1 in chunks:
                xi = x if len(chunks) == 1 else rows(x, r0, r1)
                if last:
                    self.linear(xi, r1 - r0, lay['w'], lay['b'], lay['n'], lay['k'], 1.0, scale, out_f32=out[r0:r1], m_dev=m_dev)
                else:
                    self.linear(xi, r1 - r0, lay['w'], lay['b'], lay['n'], lay['k'], slope,
                                out_planes=y if len(chunks) == 1 else rows(y, r0, r1), m_dev=m_dev)
            x = y
        return out[:P, :n_out]

    # ------------------------------------------------------------------ whole path
    def stage_a(self, db: DeviceBatch, with_coo: bool = False):
        """Stages 1-2 of a batch, enqueued without any host synchronisation: graph build, GAT, clustering and the
        exclusive scan of the person counts."""
        if db.n_heads == 0:                                     # no detections at all (empty frames only): nothing to launch
            i32 = dict(dtype=torch.int32, device=self.device)
            return dict(graph=None, scores=torch.zeros(1, dtype=torch.float32, device=self.device),
                        person_heads=torch.zeros((1, self.cfg.V_sm), **i32), n_persons=torch.zeros(db.n_frames, **i32),
                        person_off=torch.zeros(db.n_frames + 1, **i32))
        g = self.build_graph(db, with_coo=with_coo, overlap=True)
        scores = self.gat_forward(db, g) if db.n_nodes > 0 else torch.zeros(1, dtype=torch.float32, device=self.device)
        self.wait_graph(g)
        person_heads, n_persons = self.cluster(db, g, scores)
        person_off = torch.empty(db.n_frames + 1, dtype=torch.int32, device=self.device)
        self.launches += 1
        check(self.L.b200pose_gather_persons(db.n_frames, ptr(db.head_off), ptr(person_heads), ptr(n_persons), ptr(person_off), 1,
                                             ptr(db.sk_cam), self.cfg.V_sm, self.cams.ref, None, None, self._stream()), 'scan')
        return dict(graph=g, scores=scores, person_heads=person_heads, n_persons=n_persons, person_off=person_off)

    def stage_b(self, db: DeviceBatch, res: dict, want_triangulation: bool = False):
        """Stage 3 of a batch. Reads the person count back (one 4-byte device->host copy: it sizes the launches),
        then person list, MLP-input encoder and MLP."""
        P = int(res['person_off'][db.n_frames].item()) if db.n_heads > 0 else 0
        person_sk, person_frame = self.person_list(db, res, P)
        res.update(person_sk=person_sk[:P], person_frame=person_frame[:P], n_persons_total=P)
        if self.mlp is not None:
            if P > 0:
                x, valid, _ = self.encode_persons(db, P, res['person_sk'])
                res['valid'] = valid
                res['joints'] = self.mlp_forward(x, P)
            else:
                res['valid'] = torch.zeros(0, dtype=torch.uint8, device=self.device)
                res['joints'] = torch.zeros((0, self.mlp[-1]['n']), dtype=torch.float32, device=self.device)
        if want_triangulation and P > 0:
            res['tri_xyz'], res['tri_mask'] = self.triangulate(db, P, res['person_sk'])
        return res

    def stage_b_nosync(self, db: DeviceBatch, res: dict):
        """Stage 3 enqueued without reading the person count back: person list, encoder and MLP are launched for the
        capacity heads // min_number_of_views and take the real count from the device (person_off[B], written by the scan
        of stage 2). Outputs are capacity-sized; `res['n_persons_dev']` is the count (an int32 device scalar) and
        person_count(res) reads it when the host finally wants it."""
        if db.n_heads == 0 or self.mlp is None:
            return self.stage_b(db, res)
        cap = person_capacity(db.n_heads, self.cfg.min_number_of_views)
        person_sk, person_frame = self.person_list(db, res, cap)
        n_dev = res['person_off'][db.n_frames:db.n_frames + 1]
        x, valid, _ = self.encode_persons(db, cap, person_sk, n_dev=n_dev)
        joints = self.mlp_forward(x, cap, m_dev=n_dev)
        res.update(person_sk=person_sk, person_frame=person_frame, valid=valid, joints=joints, n_persons_dev=n_dev, n_persons_total=None)
        return res

    @staticmethod
    def person_count(res: dict) -> int:
        """Number of persons of a result (reads the device-side count of a sync-free step once)."""
        if res.get('n_persons_total') is None:
            res['n_persons_total'] = int(res['n_persons_dev'].item())
        return res['n_persons_total']

    @_on_own_device
    def infer(self, db: DeviceBatch, with_coo: bool = False, want_triangulation: bool = False, sync: bool = True):
        """graph build -> GAT -> clustering -> encoder -> MLP for every frame of a batch resident in HBM. sync=False enqueues
        the whole step without a host round trip (stage_b_nosync): the rows of person_sk / joints / valid past
        person_count(res) are unspecified."""
        res = self.stage_a(db, with_coo=with_coo)
        if not sync and not want_triangulation:
            return self.stage_b_nosync(db, res)
        return self.stage_b(db, res, want_triangulation=want_triangulation)

    @_on_own_device
    def infer_host(self, hb: HostBatch, n_chunks: int = 1):
        """The public end-to-end call: pinned host buffers in, host results out.

        With n_chunks > 1 the batch is cut into runs of frames: all host->device copies are enqueued up front on a
        copy stream and the compute stream runs stage A of chunk i+1 before it waits for the person count of chunk i.
        Measured on B200 (scripts/e2e_probe.py) this does NOT pay for the reference-sized batch: every extra chunk
        costs ~0.8 ms of fixed work (the MLP re-streams its 116 MB of weights per chunk, persistent GEMMs refill
        their pipelines) against 0.36 ms of copy time to hide, so the default is one chunk; to overlap copies with
        compute use infer_host_stream(), which prefetches the NEXT batch instead. Results are in frame order."""
        chunks = hb.split(n_chunks)
        cur = torch.cuda.current_stream(self.device)
        cs = self._aux_stream('copy')
        cs.wait_stream(cur)
        uploads = [ch.upload(self.device, cs, cur) for ch in chunks]
        out_bufs = hb.result_buffers(self.cfg.n_cameras, self.mlp[-1]['n'] if self.mlp is not None else 0, self.cfg.min_number_of_views)
        parts = []
        p_base = 0

        def finish(i):
            nonlocal p_base
            db, ch = uploads[i][0], chunks[i]
            res = self.stage_b(db, staged[i])
            P = res['n_persons_total']
            f0, f1 = ch.frame_range
            out_bufs['n_persons'][f0:f1].copy_(res['n_persons'], non_blocking=True)
            out_bufs['person_off'][f0:f1 + 1].copy_(res['person_off'], non_blocking=True)
            if P > 0:
                copy_person_rows(out_bufs, res, P, p_base)
            parts.append((f0, f1, p_base, P, ch.head_range[0]))
            p_base += P

        staged = []
        for i, (db, ev) in enumerate(uploads):
            cur.wait_event(ev)
            staged.append(self.stage_a(db))
            if i >= 1:
                finish(i - 1)
        finish(len(uploads) - 1)
        cur.synchronize()
        # chunk-local -> batch-global indices (host side, a few KB)
        P_tot = p_base
        person_off = out_bufs['person_off'].numpy()
        person_sk = out_bufs['person_sk'].numpy()
        for f0, f1, pb0, P, h0 in parts:
            # every chunk wrote its local offsets over [f0, f1]; entry f0 is shared with the previous chunk (its total,
            # then this chunk's 0), so it is set explicitly and only (f0, f1] is shifted
            person_off[f0] = pb0
            person_off[f0 + 1:f1 + 1] += pb0
            if h0:
                blk = person_sk[pb0:pb0 + P]
                blk[blk >= 0] += h0
        return host_results(out_bufs, P_tot, self.mlp is not None)

    # ------------------------------------------------------------------ low-latency path: one CUDA graph per batch shape
    def _stage_b_static(self, db: DeviceBatch, res: dict, p_bound: int, p_max: int):
        """Stage 3 without the person-count readback: the person list is sized for p_bound = heads // min_number_of_views
        persons (disjoint components of at least that many heads), the encoder and the MLP for p_max <= p_bound rows; rows past the real count keep person_sk = -1,
        encode to zero rows with valid = 0 and are dropped on the host. This is what lets the whole step live in one CUDA
        graph."""
        person_sk, person_frame = self.person_list(db, res, p_bound, fill=True)
        x, valid, _ = self.encode_persons(db, p_max, person_sk)
        joints = self.mlp_forward(x, p_max)
        res.update(person_sk=person_sk, person_frame=person_frame, valid=valid, joints=joints)
        return res

    @_on_own_device
    def infer_host_graph(self, hb: HostBatch, max_cached: int = 64):
        """The end-to-end call for live frames (one frame, or a few, per call): same inputs and outputs as infer_host, but
        the ~30 launches, the input copies and the result copies of a batch SHAPE (frames, heads, nodes) are captured once
        into a CUDA graph and replayed, and nothing in the step waits for the host - the person count is read with the
        results. A rig that sees the same number of skeletons per camera from frame to frame replays one graph; a new
        shape costs one eager run plus one capture. Needs the MLP weights (the full path)."""
        if self.mlp is None or self.gat is None:
            raise RuntimeError('infer_host_graph needs both models')
        pb = hb.pb
        if pb.n_heads == 0 or pb.n_nodes == pb.n_heads:          # nothing to match: the eager path handles the degenerate shapes
            return self.infer_host(hb)
        # a captured graph bakes in everything its launches were given: the batch shape, but also the threshold, the
        # kernel choices and the weight planes - all part of the key, so a change re-captures instead of replaying stale values
        key = (pb.n_frames, pb.n_heads, pb.n_nodes, pb.max_heads, pb.max_enodes, self.threshold, self.cfg.min_number_of_views,
               self.agg_impl, self.gemm_impl, self._weights_gen)
        cache = self._own.graphs
        ent = cache.get(key)
        cur = torch.cuda.current_stream(self.device)
        if ent is None:
            warm = self.infer_host(hb)                          # eager warm-up of this shape: workspaces, function attributes
            seen = max(int(warm['n_persons_total']), self._own.graph_person_hint.get(key, 0))
            h_in, db = hb.static_copy(self.device)
            # heads // min_number_of_views bounds the person count and sizes the person list; the encoder and the MLP
            # are captured for the tighter capacity this shape showed
            p_bound = person_capacity(pb.n_heads, self.cfg.min_number_of_views)
            p_max = capture_capacity(seen, p_bound)
            h_out = pinned_results(pb.n_frames, p_max, self.cfg.n_cameras, self.mlp[-1]['n'])
            graph = torch.cuda.CUDAGraph()
            cur.synchronize()
            with torch.cuda.graph(graph):
                copy_inputs(db, h_in)
                res = self._stage_b_static(db, self.stage_a(db), p_bound, p_max)
                h_out['n_persons'].copy_(res['n_persons'], non_blocking=True)
                h_out['person_off'].copy_(res['person_off'], non_blocking=True)
                copy_person_rows(h_out, res, p_max)
            # the graph bakes in device addresses: keep everything it touches alive (workspaces are replaced when a
            # larger batch makes them grow)
            ent = dict(graph=graph, h_in=h_in, h_out=h_out, p_cap=p_max, keep=(db, res, list(self._own.ws.values())))
            cache[key] = ent
            while len(cache) > max_cached:
                cache.popitem(last=False)
        else:
            cache.move_to_end(key)
            for n in INPUT_NAMES:
                ent['h_in'][n].copy_(getattr(hb, n))
        ent['graph'].replay()
        cur.synchronize()
        P = int(ent['h_out']['person_off'][pb.n_frames])
        if P > ent['p_cap']:                                    # more persons than the captured capacity: eager, and a new capture next time
            self._own.graph_person_hint[key] = P
            del cache[key]
            return self.infer_host(hb)
        # copies: the pinned buffers belong to the cached graph and the next replay of this shape overwrites them
        return {k: v.clone() if torch.is_tensor(v) else v for k, v in host_results(ent['h_out'], P, True).items()}

    @_on_own_device
    def infer_frames(self, frames):
        """Live frames as the reference hands them around - a list of `{camera: [json_string, timestamp, ...]}` dicts (or one
        such dict) - to person proposals and joints on the host: native packing of the payload strings, one CUDA-graph
        replay per batch shape (infer_host_graph). Returns what infer_host returns."""
        from .pack import pack_frames_fast
        if isinstance(frames, dict):
            frames = [frames]
        return self.infer_host_graph(HostBatch(pack_frames_fast(frames, self.cfg, keep_json=False), pinned=False))

    def infer_host_stream(self, batches, lanes: Optional[int] = None):
        """Generator over host batches: yields the host results of each batch, in order (the serving loop of a camera rig or
        of a recorded sequence: pack frames -> infer -> consume). In steady state the host->device copy of batch i+1 (copy
        stream), the compute of batch i - enqueued as one sync-free step, so the GPU never waits for the host inside it - and
        the result read-back of batch i-1 (its own stream: first the per-frame person counts, then, once the host knows the
        total, exactly the persons' rows) overlap. With lanes > 1 consecutive batches also alternate between that many compute
        streams (`twin()`: shared weights, own workspaces), so the latency-bound phases of one batch (graph build, clustering,
        person list, encoder: few warps) run beside the projections of another; `lanes` batches stay enqueued behind the one
        whose results the host is reading (measured on 1024-frame Panoptic batches: 2.43 ms per batch with one lane, 2.09 with
        two, 2.05 with three, 2.03 with four). lanes=None: three when the process has 32 hardware stream queues
        (CUDA_DEVICE_MAX_CONNECTIONS, set by this package at import when it can), else two - see the package's
        `_widen_stream_queues`. Results are yielded in order; the last batches are flushed at the end."""
        if lanes is None:
            from . import DEFAULT_LANES
            lanes = DEFAULT_LANES
        cur = torch.cuda.current_stream(self.device)
        cs, ds, dc = [self._aux_stream(role) for role in ('copy', 'd2h', 'counts')]
        pipes, lane_streams = self.lanes(max(1, int(lanes)))
        depth = len(pipes)                                     # batches enqueued ahead of the one whose results the host waits for
        lane_streams = [cur if s is None else s for s in lane_streams]
        for s in lane_streams[1:]:
            s.wait_stream(cur)
        it = iter(batches)
        n_out = self.mlp[-1]['n'] if self.mlp is not None else 0
        count = [0]

        def prefetch():
            try:
                hb = next(it)
            except StopIteration:
                return None
            lane = count[0] % len(pipes)
            count[0] += 1
            return (hb, *hb.upload(self.device, cs, lane_streams[lane]), lane)

        # pinned result buffers: depth + 3 rotating sets per batch size (depth + 1 batches are in flight, and a yielded result
        # stays valid until two more batches have been yielded), owned by the pipeline - the same HostBatch may be streamed
        # repeatedly.
        pool = self._own.stream_results
        turn = [0]

        def result_set(hb):
            B, cap = hb.pb.n_frames, person_capacity(hb.pb.n_heads, self.cfg.min_number_of_views)
            key = (B, cap, n_out, depth + 3)
            sets = pool.get(key)
            if sets is None:
                sets = pool[key] = [pinned_results(B, cap, self.cfg.n_cameras, n_out) for _ in range(depth + 3)]
            turn[0] += 1
            return sets[turn[0] % (depth + 3)]

        def enqueue_compute(hb, db, ev, lane):
            """Compute of one batch on its lane's stream; nothing here waits for the GPU."""
            st = lane_streams[lane]
            with torch.cuda.stream(st):
                st.wait_event(ev)
                res = pipes[lane].infer(db, sync=False)
                if res.get('n_persons_dev') is not None and 'joints' in res:
                    res['joints'] = res['joints'].clone()        # 'mlp_out' is a shared workspace: the lane's next batch overwrites it
                done = torch.cuda.Event()
                done.record(st)
            return hb, res, done

        def enqueue_counts(hb, res, done):
            """Read-back of the batch's per-frame person counts, behind its compute, on the counts stream - NOT the stream the
            rows are read back on: that one runs in order, and rows of an earlier batch queued behind this wait would not move
            (nor would the host, which waits for them, enqueue anything) until this batch's compute has finished."""
            bufs = result_set(hb)
            with torch.cuda.stream(dc):
                dc.wait_event(done)
                bufs['n_persons'].copy_(res['n_persons'], non_blocking=True)
                bufs['person_off'].copy_(res['person_off'], non_blocking=True)
                counts = torch.cuda.Event()
                counts.record(dc)
            return hb, res, bufs, counts

        def finalize(hb, res, bufs, counts):
            counts.synchronize()
            P = int(bufs['person_off'][hb.pb.n_frames]) if hb.pb.n_heads > 0 else 0
            res['n_persons_total'] = P
            if P > 0:
                with torch.cuda.stream(ds):
                    copy_person_rows(bufs, res, P)
                ds.synchronize()
            return host_results(bufs, P, self.mlp is not None)

        nxt = prefetch()
        pending = collections.deque()
        while nxt is not None:
            hb, db, ev, lane = nxt
            nxt = prefetch()                                   # the next batch's copy is in flight during this compute
            pending.append(enqueue_counts(*enqueue_compute(hb, db, ev, lane)))
            if len(pending) > depth:                           # `depth` batches stay enqueued behind the one read back here
                yield finalize(*pending.popleft())
        for s in lane_streams[1:]:
            cur.wait_stream(s)
        while pending:
            yield finalize(*pending.popleft())
