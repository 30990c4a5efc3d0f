"""Live frames: the whole path of ONE frame submitted asynchronously, for the reference's per-frame driver loop.

The reference's drivers (test/metrics_from_model.py:178-300, test/show_results_from_model.py:139-307) walk a frame through
five calls - dataset construction, `model(feats, subgraph)`, `get_person_proposal_from_network_output`, one
`PoseEstimatorDataset` per person, `mlp(input_all)` - and the drop-in modules used to run each of them as its own handful
of eager launches with a host synchronisation in between (3.4 ms per Panoptic frame). Here the drop-in dataset submits the
frame once: three captured CUDA graphs replayed back to back on a side stream,

    G1  input copies, graph build, 5 GAT layers, clustering, person offsets        -> event A (scores, proposals)
    G2  person list, MLP-input encoder (pairwise-DLT hint included)                 -> event B (MLP input rows)
    G3  the 9 MLP projections                                                       -> event C (raw MLP outputs)

and the later calls of the driver are answered from that submission: each waits only for the event it needs, so the
encoder and the MLP run while the driver is still turning proposals into per-person JSON strings. A call the submission
cannot answer - other weights, another threshold, a feature matrix that is not the graph's own, persons that are not the
proposals - takes the eager path as before; nothing is ever served from a stale or mismatching submission.
"""
from __future__ import annotations

import collections
from typing import Optional

import numpy as np
import torch

from .pipeline import (INPUT_NAMES, GraphArrays, HostBatch, PosePipeline, capture_capacity, copy_inputs, person_capacity,
                       pinned_results)


class _Entry:
    """Everything one batch shape needs: static device / pinned buffers and the three captured graphs."""
    pass


class LiveHandle:
    """One submitted frame. Valid until the next frame of the same shape is submitted (`fresh()`)."""

    def __init__(self, live: "LiveFrames", ent: _Entry, pb):
        self.live, self.ent, self.pb = live, ent, pb
        self.gen = ent.gen
        self.key = live.model_key
        self._proposals = None
        self._stage3 = None

    def fresh(self) -> bool:
        return self.ent.gen == self.gen and self.live.model_key == self.key

    # ---- G1
    def scores(self):
        """Device tensor [N] of this frame's scores, ordered after event A on the current stream (a copy: the next
        submission of this shape overwrites the graph's buffer)."""
        if not self.fresh():
            return None
        torch.cuda.current_stream(self.live.pipe.device).wait_event(self.ent.ev_a)
        return self.ent.scores[: self.pb.n_nodes].clone()

    def features(self):
        """ndata['h'] of this frame (device, [N, F] fp32), ordered after event A on the current stream."""
        if not self.fresh():
            return None
        torch.cuda.current_stream(self.live.pipe.device).wait_event(self.ent.ev_a)
        return self.ent.feats[: self.pb.n_nodes]

    def proposals(self):
        """[P, V_sm] frame-local head ids (-1 = no skeleton of that camera), host side."""
        if self._proposals is None:
            if not self.fresh():
                return None
            self.ent.ev_a.synchronize()
            n = int(self.ent.h_out['n_persons'][0])
            self._proposals = self.ent.h_out['person_heads'][:n].numpy().copy()
        return self._proposals

    # ---- G2 / G3
    def stage3(self):
        """(person_sk [P, C] skeleton ids, valid [P], MLP input rows [P, mlp_in] fp32 on the host) of the proposals, or None
        when this submission has no stage 3 (no MLP known yet, more persons than the captured capacity, stale)."""
        if self._stage3 is None:
            if not self.fresh() or not self.ent.has_mlp:
                return None
            props = self.proposals()
            P = len(props)
            if P > self.ent.p_max:
                self.live.person_hint[self.ent.key] = P         # captured too small: a larger capacity next time
                self.live.cache.pop(self.ent.key, None)
                return None
            self.ent.ev_b.synchronize()
            h = self.ent.h_out
            self._stage3 = (h['person_sk'][:P].numpy().copy(), h['valid'][:P].numpy().copy(), h['enc'][:P].clone())
        return self._stage3

    def enc_device(self, P: int):
        return self.ent.xf[:P]

    def mlp_out_raw(self, P: int):
        """Raw MLP outputs [P, n_out] on the device (the reference's `mlp(input_all)`, before its x10), ordered after event C."""
        if not self.fresh() or not self.ent.has_mlp or P > self.ent.p_max:
            return None
        torch.cuda.current_stream(self.live.pipe.device).wait_event(self.ent.ev_c)
        return self.ent.joints[:P].clone()


class LiveFrames:
    def __init__(self, pipe: PosePipeline, max_cached: int = 32):
        self.pipe = pipe
        self.stream = torch.cuda.Stream(pipe.device)
        self.cache = collections.OrderedDict()
        self.person_hint = {}
        self.max_cached = max_cached
        self.model_key = None          # identifies the weights the cached graphs were captured with
        self.last: Optional[LiveHandle] = None

    def set_models(self, key, gat_layers, mlp_layers):
        """(Re)binds the prepared weight planes; a change drops every captured graph (they hold the old plane addresses)."""
        if key != self.model_key:
            self.sync()
            self.cache.clear()
            self.model_key = key
            self.pipe.gat = gat_layers
            self.pipe.mlp = mlp_layers
            self.last = None

    def sync(self):
        """Orders the current stream after everything submitted so far (call before eager work on the same pipeline: the
        graphs and the eager path share its workspaces)."""
        torch.cuda.current_stream(self.pipe.device).wait_stream(self.stream)

    def submit(self, pb) -> Optional[LiveHandle]:
        pipe = self.pipe
        if pipe.gat is None or pb.n_frames != 1 or pb.n_heads == 0 or pb.n_nodes == pb.n_heads:
            return None
        key = (pb.n_heads, pb.n_nodes, pb.max_heads, pb.max_enodes, pipe.threshold, pipe.cfg.min_number_of_views, pipe.agg_impl,
               pipe.gemm_impl, pipe.mlp is not None)
        ent = self.cache.get(key)
        if ent is None:
            pb.validate()
            ent = self._capture(key, pb, HostBatch(pb, pinned=False))
            self.cache[key] = ent
            while len(self.cache) > self.max_cached:
                self.cache.popitem(last=False)
        else:
            self.cache.move_to_end(key)
        # the side stream must not overtake readers of the previous submission's buffers on the current stream
        self.stream.wait_stream(torch.cuda.current_stream(pipe.device))
        for n, view in ent.h_in_np.items():                   # plain memcpy of ~10 KB into the pinned staging buffers
            np.copyto(view, getattr(pb, n).reshape(view.shape), casting='unsafe')
        ent.gen += 1
        with torch.cuda.stream(self.stream):
            ent.g1.replay()
            ent.ev_a.record(self.stream)
            if ent.has_mlp:
                ent.g2.replay()
                ent.ev_b.record(self.stream)
                ent.g3.replay()
                ent.ev_c.record(self.stream)
        self.last = LiveHandle(self, ent, pb)
        return self.last

    def _capture(self, key, pb, hb) -> _Entry:
        pipe, dev = self.pipe, self.pipe.device
        cfg = pipe.cfg
        ent = _Entry()
        ent.key, ent.gen, ent.has_mlp = key, 0, pipe.mlp is not None
        h_in, db = hb.static_copy(dev)
        ent.h_in, ent.db = h_in, db
        ent.h_in_np = {n: h_in[n].numpy() for n in INPUT_NAMES}
        ent.h_in_np['sk_mask'] = ent.h_in_np['sk_mask'].view(np.uint32)
        p_bound = person_capacity(pb.n_heads, cfg.min_number_of_views)
        ent.p_max = p_max = capture_capacity(max(self.person_hint.get(key, 0), p_bound // 2), p_bound)
        mk = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
        n_out = pipe.mlp[-1]['n'] if ent.has_mlp else 0
        ent.h_out = dict(pinned_results(1, p_max, cfg.n_cameras, n_out), person_heads=mk((pb.n_heads, cfg.V_sm), torch.int32),
                         enc=mk((p_max, cfg.mlp_in), torch.float32))
        self.sync()
        cur = torch.cuda.current_stream(dev)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            # eager warm-up of this shape on the side stream: workspaces, function attributes, allocator
            copy_inputs(db, h_in)
            res = pipe.stage_a(db, with_coo=True)
            if ent.has_mlp:
                pipe._stage_b_static(db, res, p_bound, p_max)
            self.stream.synchronize()
            ent.g1, ent.g2, ent.g3 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(ent.g1, stream=self.stream):
                copy_inputs(db, h_in)
                res = pipe.stage_a(db, with_coo=True)
                # the dense N x F feature matrix the reference hands around as `ndata['h']`: nothing on this path reads it
                # (layer 0 runs on the compact rows), but the driver passes it back to the model, so it is kept materialised -
                # 3 us inside the graph instead of an eager launch per frame
                ent.feats = pipe.node_features_f32(db)
                ent.h_out['n_persons'].copy_(res['n_persons'], non_blocking=True)
                ent.h_out['person_heads'].copy_(res['person_heads'][: pb.n_heads], non_blocking=True)
            ent.arrays, ent.scores, ent.res = res['graph'], res['scores'], res
            if ent.has_mlp:
                with torch.cuda.graph(ent.g2, stream=self.stream):
                    person_sk, person_frame = pipe.person_list(db, res, p_bound, fill=True)
                    x, valid, xf = pipe.encode_persons(db, p_max, person_sk, want_f32=True)
                    ent.h_out['person_sk'].copy_(person_sk[:p_max], non_blocking=True)
                    ent.h_out['valid'].copy_(valid, non_blocking=True)
                    ent.h_out['enc'].copy_(xf, non_blocking=True)
                with torch.cuda.graph(ent.g3, stream=self.stream):
                    joints = pipe.mlp_forward(x, p_max, scale=1.0).clone()       # a buffer of its own: the eager path shares 'mlp_out'
                    ent.h_out['joints'][:, :n_out].copy_(joints, non_blocking=True)
                ent.xf, ent.joints, ent.keep3 = xf, joints, (person_sk, person_frame, x, valid)
            ent.ev_a, ent.ev_b, ent.ev_c = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
            ent.keep = list(pipe._own.ws.values())     # the graphs bake in workspace addresses: keep them alive
        return ent
