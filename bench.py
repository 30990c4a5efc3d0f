#!/usr/bin/env python
"""Benchmark of the per-frame inference hot path (BASELINE.json: frames/sec, 5-view, N persons).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]

One step = one pass of the whole path (graph build -> GAT -> clustering -> encoder -> MLP) over one batch
of synthetic frames: Panoptic 5-view, 1024 frames, 4 persons/frame (BASELINE.json configs[1]).
  value : frames/s with the packed inputs already resident in HBM (CUDA events, max over ranks)
  e2e   : frames/s through the public host API (pinned host buffers -> results on the host)
Frames are independent, so N GPUs each process their own 1024 frames (weak scaling); when N > 1 the
per-frame results are gathered with one NCCL all_gather per step.
`--impl reference` times the CPU port of the reference path (oracle/) on a bounded sample instead.
"""
import argparse
import importlib
import json
import os
import sys
import threading
import time

# more hardware stream queues than CUDA's default 8 (read when the CUDA context is created): the job runs on ~10 streams and
# streams that share a queue serialise each other (3d_multi_pose_estimator_b200/__init__.py:_widen_stream_queues)
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
GOLDEN = os.path.join(REPO, 'tests', 'golden')

UNIT = 'frames/s'
RIG_NAMES = {'panoptic': 'Panoptic', 'arp3': 'ARP-lab (tm_arp.pickle, first three cameras)', 'arp6': 'ARP-lab (tm_arp.pickle, as shipped)',
             'ring10': 'stress graph: synthetic ring', 'arp_robot2': 'ARP-lab robot cameras', 'pansub': 'Panoptic camera subset'}


def describe(config, cfg, frames, persons):
    """Metric name and workload description of THIS run (whatever --config / --frames / --persons say)."""
    metric = 'frames/sec (%d-view, %d persons/frame, %d-frame batch)' % (cfg.V_sm, persons, frames)
    workload = '%s %d-view, %d-frame batch, %d persons/frame, skeleton matching + MLP lift' % (
        RIG_NAMES.get(config, config), cfg.V_sm, frames, persons)
    return metric, workload


def load_workload(config, n_frames, n_persons, seed0):
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    cfg = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % config))
    frames = synth.make_frames(cfg, n_frames, n_persons, base_seed=seed0)
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    return cfg, frames


def load_weights(config, cfg):
    """Random-init weights of the reference architectures (seeded) + the stored last-layer calibration."""
    import torch
    W = importlib.import_module('3d_multi_pose_estimator_b200.weights')
    meta = json.load(open(os.path.join(GOLDEN, 'golden_%s.json' % config)))
    npz = np.load(os.path.join(GOLDEN, 'golden_%s.npz' % config))
    gat = W.make_gat_state(cfg.n_features_sm, meta['gat_seed'])
    gat['layers.4.fc2.weight'] = torch.from_numpy(npz['gat_last_fc2_weight'].copy())
    gat['layers.4.fc2.bias'] = torch.from_numpy(npz['gat_last_fc2_bias'].copy())
    mlp = W.make_mlp_state(meta.get('mlp_in_dim', cfg.mlp_in), 54, meta['mlp_seed'])
    return gat, mlp


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                 nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap'}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def _cpu_worker(args):
    """One host process of the CPU arm: runs the oracle port over its share of the frames, one frame at a time like the
    reference's drivers (test/metrics_from_model.py:120-300), single-threaded BLAS (the parallelism is across processes)."""
    config, lo, hi, persons, seed0, weights_path, budget_s = args
    try:                                          # numpy is already loaded in a spawned worker: limit its BLAS pool in place
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    from oracle import pose_oracle as O
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    cfg = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % config))
    tabs = O.CameraTables(cfg)
    W = np.load(weights_path)
    gw = {k[4:]: W[k] for k in W.files if k.startswith('gat/')}
    mw = {k[4:]: W[k] for k in W.files if k.startswith('mlp/')}
    frames = [synth.make_frame(cfg, seed0 + i, persons) for i in range(lo, hi)]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    n, t0 = 0, time.perf_counter()
    while True:                                   # cycle over the share until the time budget is used
        for f in frames:
            O.infer_frame(f, tabs, gw, mw)
            n += 1
            if time.perf_counter() - t0 > budget_s:
                return n, time.perf_counter() - t0
        if not frames:
            return 0, time.perf_counter() - t0


def _cpu_worker_reference(args):
    """One host process of the CPU arm running the UNMODIFIED reference (baseline/_ref or /root/reference, with the dgl /
    pytransform3d shims) through its own driver's call sequence (oracle/ref_runner.py), one torch thread per process."""
    config, lo, hi, persons, seed0, weights_path, budget_s = args
    import contextlib
    import io
    from oracle import ref_runner
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    cfg = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % config))
    W = np.load(weights_path)
    gw = {k[4:]: W[k] for k in W.files if k.startswith('gat/')}
    mw = {k[4:]: W[k] for k in W.files if k.startswith('mlp/')}
    frames = [synth.make_frame(cfg, seed0 + i, persons) for i in range(lo, hi)]
    sink = io.StringIO()
    with contextlib.redirect_stdout(sink):                 # the reference's modules print while they work
        runner = ref_runner.ReferenceRunner(config, gw, mw, threads=1)
        runner.run_frame(frames[0])                        # import-time tables, first-call allocations
        n, t0 = 0, time.perf_counter()
        while True:
            for f in frames:
                runner.run_frame(f)
                n += 1
                if time.perf_counter() - t0 > budget_s:
                    return n, time.perf_counter() - t0


def reference_kind():
    """'reference' when the unmodified reference can be run here (reference tree or its staged copy), else 'port'."""
    try:
        from oracle import ref_runner
        import cv2  # noqa: F401  (the reference needs it; same image on the GPU box)
        import networkx  # noqa: F401
        return 'reference' if ref_runner.available() else 'port'
    except Exception:
        return 'port'


def cpu_reference_run(config, persons, gat_state, mlp_state, budget_s, n_frames=64, seed0=0, procs=None, kind='port', repeats=1):
    """The CPU arm on `procs` host processes (default: every core), each handling its own frames one at a time for
    ~budget_s seconds: kind 'reference' = the unmodified reference under the import shims (oracle/ref_runner.py),
    kind 'port' = the oracle restatement (oracle/pose_oracle.py).
    Returns (frames/s, frames processed, seconds, processes)."""
    import multiprocessing as mp
    import tempfile
    procs = procs or os.cpu_count() or 1
    tmp = tempfile.NamedTemporaryFile(suffix='.npz', delete=False)
    tmp.close()
    np.savez(tmp.name, **{'gat/' + k: v.numpy() for k, v in gat_state.items()}, **{'mlp/' + k: v.numpy() for k, v in mlp_state.items()})
    per = max(1, n_frames // procs)
    jobs = [(config, r * per, (r + 1) * per, persons, seed0, tmp.name, budget_s) for r in range(procs)]
    saved = {k: os.environ.get(k) for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS')}
    try:
        for k in saved:                           # inherited by the workers before they load their BLAS
            os.environ[k] = '1'
        with mp.get_context('spawn').Pool(procs) as pool:                 # one pool for all repeats: workers import torch once
            runs = [pool.map(_cpu_worker_reference if kind == 'reference' else _cpu_worker, jobs) for _ in range(repeats)]
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        os.unlink(tmp.name)
    out = []
    for res in runs:
        n = sum(r[0] for r in res)
        busy = max(r[1] for r in res)             # workers run concurrently for ~budget_s; pool start-up is excluded
        out.append((n / busy, n, busy, procs))
    return out[0] if repeats == 1 else out


def algorithmic_work(pb, pipe_gat_dims, mlp_dims, n_persons):
    """Algorithmic bytes / flops per step (DESIGN.md): edge-softmax compulsory bytes and executed GEMM flops."""
    N, E, S = pb.n_nodes, pb.n_edges, pb.n_heads
    agg_bytes = 0
    gemm_flops = 0
    for l, (din, h, d) in enumerate(pipe_gat_dims):
        rows = (S + 1) if l == 0 else N
        hd = h * d
        gemm_flops += 2 * rows * (din * din + din * (hd + 2 * h))
        agg_bytes += (rows * (hd + 2 * h) + N * hd) * 4 + E * 4 + (N + 1) * 4
    mlp_flops = 0
    for k, n in mlp_dims:
        mlp_flops += 2 * n_persons * k * n
    return agg_bytes, gemm_flops, mlp_flops


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--frames', type=int, default=1024, help='frames per GPU and step')
    ap.add_argument('--persons', type=int, default=4)
    ap.add_argument('--config', default='panoptic')
    ap.add_argument('--total-frames', type=int, default=0,
                    help='size of the whole job (e.g. 1000000 for BASELINE.json configs[2]): sets --steps to ceil(total / (gpus * frames)); '
                         'every rank streams its share in chunks of --frames frames')
    ap.add_argument('--cpu-budget', type=float, default=15.0, help='seconds of CPU work for the cpu_baseline sample')
    ap.add_argument('--gemm-impl', type=int, default=0)
    ap.add_argument('--no-fuse2', action='store_true', help='A/B: run the last GAT layer as two projections instead of the fused launch')
    ap.add_argument('--lanes', type=int, default=0, help='compute lanes (CUDA streams with their own workspaces) the job alternates its steps between; 1 = one stream; 0 = the package default (3 with 32 hardware stream queues, else 2)')
    ap.add_argument('--workload', default='pipeline', choices=['pipeline', 'triangulation', 'train_batch', 'train_step'],
                    help="'triangulation' = BASELINE.json configs[3]: batched pairwise DLT only (not the headline line)")
    ap.add_argument('--chunks', type=int, default=1, help='sub-batches of the end-to-end call (copy/compute overlap)')
    ap.add_argument('--latency-frames', type=int, default=200, help='single-frame calls timed for p50_frame_latency_ms')
    ap.add_argument('--cpu-kind', default='auto', choices=['auto', 'reference', 'port'],
                    help='CPU arm: the unmodified reference under the import shims (needs its staged copy under baseline/_ref) or the oracle port')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed step returned as DIR/<name>.npy (rank 0; see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.workload != 'pipeline'):
        ap.error('--dump-outputs writes the outputs of the GPU pipeline (--impl b200 --workload pipeline)')
    warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.total_frames > 0:
        args.steps = max(1, -(-args.total_frames // (max(world, 1) * args.frames)))

    if args.workload == 'triangulation':
        return triangulation_workload(args, rank, world, local_rank)
    if args.workload == 'train_batch':
        return train_batch_workload(args, rank, world, local_rank)
    if args.workload == 'train_step':
        return train_step_workload(args, rank, world, local_rank)
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    cfg0 = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % args.config))
    METRIC, workload = describe(args.config, cfg0, args.frames, args.persons)
    config_desc = {'workload': workload, 'camera_config': args.config, 'views': cfg0.V_sm, 'frames_per_gpu': args.frames,
                   'persons_per_frame': args.persons, 'weights': 'random-init (seeded) + last-layer bias calibration',
                   'l2': 'L2 flushed (256 MiB write) between timed iterations'}
    if args.total_frames > 0:
        config_desc['job'] = '%d frames in total: %d steps of %d frames on each of %d GPUs (512 distinct frames per GPU, cycled)' % (
            args.steps * world * args.frames, args.steps, args.frames, world)
    if args.lanes != 1:
        config_desc['l2'] = ('job of K steps on %d compute lanes (consecutive steps alternate between CUDA streams with their own workspaces, '
                             'shared weights); no flush between steps: a step\'s working set (1.3 GB of activations at 1024 frames) is ten times '
                             'the 126 MB L2. one_lane = the same steps on one stream with a 256 MiB L2 flush between them' % (args.lanes if args.lanes > 0 else pkg.DEFAULT_LANES))
    kind = reference_kind() if args.cpu_kind == 'auto' else args.cpu_kind
    kind_note = {'reference': 'the unmodified reference (baseline/_ref) under the dgl / pytransform3d import shims, its own driver call sequence '
                              '(test/metrics_from_model.py:178-300), one single-threaded process per host core',
                 'port': 'the numpy restatement of the reference path (oracle/pose_oracle.py), one single-threaded process per host core'}
    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == 'reference':
        if rank != 0:
            return
        import torch
        gat, mlp = load_weights(args.config, cfg0)
        n_steps = args.steps + args.warmup
        budget = max(3.0, min(20.0, 90.0 / n_steps))
        runs = cpu_reference_run(args.config, args.persons, gat, mlp, budget_s=budget, n_frames=4 * (os.cpu_count() or 1), kind=kind,
                                 repeats=n_steps + 1)[1:]           # [0] absorbs the workers' first-call costs
        procs = runs[0][3]
        vals = [(fps, n, dt) for i, (fps, n, dt, _) in enumerate(runs) if i >= args.warmup or len(runs) <= args.warmup]
        value = float(np.mean([v[0] for v in vals]))
        line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': 1e3 * args.frames / value, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f32 (torch CPU), fp64 geometry' if kind == 'reference' else 'f32 (numpy), fp64 geometry',
                'data': 'synthetic', 'config': config_desc,
                'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': procs, 'kind': kind, 'what': kind_note[kind],
                                 'sample': '%d frames per step over %d host processes (one frame at a time each, %.0f s per step, %d steps timed); '
                                           'ms_per_step extrapolated to the %d-frame batch' % (vals[-1][1], procs, budget, len(vals), args.frames)},
                'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    pm = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
    pack = importlib.import_module('3d_multi_pose_estimator_b200.pack')
    W = importlib.import_module('3d_multi_pose_estimator_b200.weights')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    distinct = args.frames if args.total_frames <= 0 else min(args.frames, 512)
    cfg, frames = load_workload(args.config, distinct, args.persons, seed0=rank * args.frames)
    gat, mlp = load_weights(args.config, cfg)
    pb = pack.pack_frames(frames, cfg, keep_json=False)
    if distinct < args.frames:                                   # a long job cycles over its distinct frames
        pb = pb.tile(-(-args.frames // distinct)).slice(0, args.frames)
    hb = pm.HostBatch(pb)
    pipe = pm.PosePipeline(cfg, gat, mlp, device=dev, gemm_impl=args.gemm_impl)
    pipe.fuse_small_fc2 = not args.no_fuse2
    db = hb.to_device(dev)
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    sharding = importlib.import_module('3d_multi_pose_estimator_b200.sharding')
    P_cap = pm.person_capacity(pb.n_heads, cfg.min_number_of_views)
    n_out = pipe.mlp[-1]['n']
    # the job's only exchange: every step's fixed-size record is packed by one kernel behind the step and all-gathered
    # asynchronously; nothing on the compute stream waits for it until the end of the job (SURVEY.md 8e: "final gather")
    gather = sharding.ResultGather(world, args.frames, P_cap, cfg.n_cameras, n_out, dev, depth=4) if world > 1 else None

    n_lanes = args.lanes if args.lanes > 0 else importlib.import_module('3d_multi_pose_estimator_b200').DEFAULT_LANES
    lanes, lane_streams = pipe.lanes(n_lanes)
    main_stream = torch.cuda.current_stream(dev)
    lane_streams = [main_stream if st is None else st for st in lane_streams]

    def step_device(lane=0):
        # the whole step enqueued without a host round trip: stage 3 is launched for the person capacity and reads the
        # count from the device (PosePipeline.stage_b_nosync). Lane k = the k-th pipeline of pipe.lanes() (shared weights,
        # own workspaces) on its own stream.
        with torch.cuda.stream(lane_streams[lane]):
            res = lanes[lane].infer(db, sync=False)
            if gather is not None:
                gather.submit(res, args.frames, head_base=rank * pb.n_heads, stream=lanes[lane]._stream())
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up (also settles the caching allocator)
    for _ in range(warmup):
        for lane in range(n_lanes):
            res = step_device(lane)
        pipe.infer_host(hb, n_chunks=args.chunks)
    if gather is not None:
        gather.finish()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- device-resident timing, one lane: one event pair per step, L2 flushed in between; the wait for the outstanding
    # gathers (the end of the job) is timed as well and counted into the job time
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    tail = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    for p_ in lanes:
        p_.launches = 0
    barrier()
    for a, b in ev:
        flush.fill_(1)
        a.record()
        res = step_device()
        b.record()
    tail[0].record()
    gathered = gather.finish() if gather is not None else None
    tail[1].record()
    barrier()
    launches = pipe.launches // max(1, args.steps) + (1 if gather is not None else 0)
    tail_ms = float(tail[0].elapsed_time(tail[1]))
    ms_one_lane = (float(np.sum([a.elapsed_time(b) for a, b in ev])) + tail_ms) / args.steps
    ms = ms_one_lane
    # ---- the same K steps as a job on n_lanes compute streams: consecutive steps alternate between the lanes, so the
    # latency-bound tail of one step (clustering, person list, encoder) runs beside the projections of the next. One event pair
    # around the whole job (+ the wait for the gathers). No flush: a step's working set (1.3 GB of activations at the
    # headline size) is ten times the L2, and a flush on one lane would only take bandwidth from the step on the other.
    if n_lanes > 1:
        job = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        barrier()
        job[0].record(main_stream)
        for st in lane_streams[1:]:
            st.wait_event(job[0])
        for i in range(args.steps):
            res = step_device(i % n_lanes)
        for st in lane_streams[1:]:
            main_stream.wait_stream(st)
        job[1].record(main_stream)
        tail[0].record()
        gathered = gather.finish() if gather is not None else None
        tail[1].record()
        barrier()
        tail_ms = float(tail[0].elapsed_time(tail[1]))
        ms = (float(job[0].elapsed_time(job[1])) + tail_ms) / args.steps
    if args.dump_outputs and rank == 0:
        # res = the last timed step; rows past the person count, and a frame's person rows past its own count, are unspecified
        P = pm.PosePipeline.person_count(res)
        n_persons, person_off = res['n_persons'].cpu().numpy(), res['person_off'].cpu().numpy()
        person_rows = np.repeat(np.asarray(pb.head_off[:-1], np.int64) - person_off[:-1], n_persons) + np.arange(P)
        dump_outputs(args.dump_outputs, {
            'scores': res['scores'][:pb.n_nodes], 'person_heads': res['person_heads'].cpu().numpy()[person_rows],
            'n_persons': n_persons, 'person_off': person_off, 'person_sk': res['person_sk'][:P],
            'person_frame': res['person_frame'][:P], 'valid': res['valid'][:P], 'joints': res['joints'][:P]})
    gather_ok = None
    if gathered is not None and rank == 0:                       # the gathered records really hold every rank's results
        last = sharding.unpack_records(gathered[-1], [args.frames] * world, args.frames, P_cap, cfg.n_cameras, n_out)
        mine = res['n_persons'].cpu().numpy()
        pm.PosePipeline.person_count(res)
        gather_ok = bool(np.array_equal(last['n_persons'][:args.frames], mine) and len(last['n_persons']) == world * args.frames
                         and np.array_equal(last['joints'][:res['n_persons_total']], res['joints'][:res['n_persons_total']].cpu().numpy()))
    # ---- end-to-end through the public host API: K batches streamed back to back; every step copies its inputs from
    # pinned host memory and reads its results back inside the timed region (the copy of step i+1 overlaps the compute of
    # step i: PosePipeline.infer_host_stream). Per-step activations (1.3 GB) are 10x the L2, so no flush is needed here.
    barrier()
    for _ in pipe.infer_host_stream([hb] * 4, lanes=n_lanes):
        pass
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    n_done = 0
    for out in pipe.infer_host_stream([hb] * args.steps, lanes=n_lanes):
        n_done += 1
    torch.cuda.synchronize()
    e2e_total = time.perf_counter() - t0
    e2e_t = [e2e_total / max(1, n_done)]
    # one isolated call as well (copy not overlapped): reported as e2e.single_call_ms
    single_t = []
    for _ in range(3):
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        pipe.infer_host(hb, n_chunks=args.chunks)
        torch.cuda.synchronize()
        single_t.append(time.perf_counter() - t1)
    single_ms = 1e3 * float(np.median(single_t))
    barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    # ---- single-frame latency: one frame per call through the same public host API (rank 0 only)
    p50_ms = p50_eager_ms = p99_ms = p50_dict_ms = None
    if rank == 0 and args.latency_frames > 0:
        singles = [pm.HostBatch(pb.slice(i, i + 1)) for i in range(min(32, pb.n_frames))]
        lat = []
        for i in range(args.latency_frames + 20):
            h1 = singles[i % len(singles)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipe.infer_host(h1, n_chunks=1)
            if i >= 20:
                lat.append(time.perf_counter() - t0)
        p50_eager_ms = 1e3 * float(np.median(lat))
        lat = []
        for i in range(args.latency_frames + 40):           # the same frames through the CUDA-graph path (one graph per shape)
            h1 = singles[i % len(singles)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipe.infer_host_graph(h1)
            if i >= 40:
                lat.append(time.perf_counter() - t0)
        p50_ms = 1e3 * float(np.median(lat))
        p99_ms = 1e3 * float(np.percentile(lat, 99))
        lat = []
        for i in range(args.latency_frames + 40):           # from the reference's frame dict (JSON strings per camera) to host results
            fr = frames[i % min(32, len(frames))]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipe.infer_frames(fr)
            if i >= 40:
                lat.append(time.perf_counter() - t0)
        p50_dict_ms = 1e3 * float(np.median(lat))
    # ---- the reference driver's own per-frame loop on the drop-in modules (JSON strings in, python dicts out):
    # what an unmodified test/metrics_from_model.py gets with the shadow directory first on sys.path (rank 0 only)
    dropin_fps = dropin_detail = None
    if rank == 0 and args.latency_frames > 0:
        try:
            dropin_detail = dropin_driver_loop(cfg, frames[:48], gat, mlp)
            dropin_fps = dropin_detail['frames_per_s']
        except Exception as e:                                  # an extra line of the report, never the reason a bench fails
            dropin_fps = 'failed: %s' % e
    # ---- host-side ingest: the native JSON packer on the text of 512 of these frames (all host threads; rank 0 only)
    json_fps = None
    if rank == 0:
        try:
            text = json.dumps(frames[:512]).encode()
            best = min(_timed(lambda: pack.pack_json(text, cfg)) for _ in range(3))
            json_fps = len(frames[:512]) / best
        except Exception as e:
            json_fps = 'failed: %s' % e
    e2e_ms = 1e3 * float(np.mean(e2e_t))
    d2h = sum(v.numel() * v.element_size() for v in out.values() if hasattr(v, 'numel'))
    # ---- per-kernel-class timing for the roofline (separate pass, CUDA events around each class)
    kern = profile_classes(pipe, db, pm, torch) if rank == 0 else None
    t = torch.tensor([ms, e2e_ms, ms_one_lane], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_max, one_lane_max = float(t[0]), float(t[1]), float(t[2])
    total_frames = args.frames * world
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = peaks.get('hbm_gbs', 6650.0)
        tc_peak = peaks.get('bf16_tflops_sustained', 1400.0)
        peak_src = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback of B200_PROFILING.md'
        P = pm.PosePipeline.person_count(res)
        gat_dims = W.gat_layer_dims(cfg.n_features_sm)
        mlp_dims = [(l['k'], l['n']) for l in pipe.mlp]
        agg_bytes, gat_flops, mlp_flops = algorithmic_work(pb, gat_dims, mlp_dims, P)
        traffic_all, traffic_tag = load_traffic(args)
        kernels = []
        for name, k_ms in kern.items():
            entry = {'kernel': name, 'ms_per_step': k_ms}
            if name in ('gat_projection_gemm', 'mlp_gemm'):
                fl = gat_flops if name == 'gat_projection_gemm' else mlp_flops
                # executed = the three bf16 MMAs of the split (hi*hi + lo*hi + hi*lo); algorithmic = the fp32 GEMM they stand for
                entry.update(bound='tensor', achieved=3 * fl / k_ms / 1e9, peak=tc_peak, unit='TFLOP/s',
                             achieved_algorithmic=fl / k_ms / 1e9, frac_algorithmic=fl / k_ms / 1e9 / tc_peak)
            elif name == 'edge_softmax_aggregate':
                entry.update(bound='hbm', achieved=agg_bytes / k_ms / 1e6, peak=hbm_peak, unit='GB/s')
            if 'achieved' in entry:
                entry['frac'] = entry['achieved'] / entry['peak']
            if traffic_all is not None and name in traffic_all:
                entry['traffic'] = traffic_all[name]
                entry['dram_gbs'] = traffic_all[name] / k_ms / 1e6
                entry['dram_frac'] = entry['dram_gbs'] / hbm_peak
            kernels.append(entry)
        dominant = max([k for k in kernels if 'frac' in k], key=lambda k: k['ms_per_step'])
        roofline = {'kernel': dominant['kernel'], 'bound': dominant['bound'], 'achieved': dominant['achieved'],
                    'peak': dominant['peak'], 'unit': dominant['unit'], 'frac': dominant['frac'], 'traffic': dominant.get('traffic'),
                    'traffic_note': traffic_tag,
                    'peak_source': peak_src + (' (bf16 sustained; achieved counts the 3 executed split-bf16 MMAs, frac_algorithmic = %.3f)'
                                               % dominant.get('frac_algorithmic', 0.0) if dominant['bound'] == 'tensor' else '')}
        cpu_line = parity = None
        if world == 1:                            # the CPU arm is timed on rank 0 of single-GPU runs only
            n_cpu = 4 * (os.cpu_count() or 1)
            cpu_fps, cpu_n, cpu_dt, cpu_procs = cpu_reference_run(args.config, args.persons, gat, mlp, budget_s=args.cpu_budget,
                                                                   n_frames=n_cpu, kind=kind)
            cpu_line = {'value': cpu_fps, 'unit': UNIT, 'cores': cpu_procs, 'kind': kind, 'what': kind_note[kind],
                        'sample': '%d frames of the same workload over %d host processes, one frame at a time each, %.1f s'
                                  % (cpu_n, cpu_procs, cpu_dt)}
            if kind == 'reference':               # the port next to it (BASELINE.md 3): what the checker itself costs
                p_fps, p_n, p_dt, _ = cpu_reference_run(args.config, args.persons, gat, mlp, budget_s=min(args.cpu_budget, 8.0),
                                                        n_frames=n_cpu, kind='port')
                cpu_line['port_value'] = p_fps
                cpu_line['port_sample'] = '%d frames, %.1f s' % (p_n, p_dt)
            parity = parity_sample(cfg, frames, pb, res, gat, mlp)
        line = {'metric': METRIC, 'value': total_frames / ms_max * 1e3, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': warmup, 'ms_per_step': ms_max, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16x3 split (fp32-accurate), fp32 accumulate; fp64 geometry', 'data': 'synthetic',
                'config': config_desc,
                'lanes': n_lanes, 'cuda_device_max_connections': os.environ.get('CUDA_DEVICE_MAX_CONNECTIONS'),
                'one_lane': {'value': total_frames / one_lane_max * 1e3, 'unit': UNIT, 'ms_per_step': one_lane_max,
                             'how': 'the same K steps one after the other on one stream, one CUDA-event pair per step, L2 flushed (256 MiB '
                                    'write) between them: the figure the per-kernel table below adds up to'},
                'e2e': {'value': total_frames / e2e_max * 1e3, 'unit': UNIT, 'h2d_bytes_per_step': hb.nbytes(),
                        'd2h_bytes_per_step': int(d2h), 'ms_per_step': e2e_max, 'single_call_ms': single_ms,
                        'mode': 'streamed (PosePipeline.infer_host_stream): copy of step i+1 and read-back of step i-1 overlap the compute '
                                'of step i; consecutive steps alternate between %d compute lanes' % n_lanes},
                'gpu_launches': launches, 'clocks': sampler.summary(), 'roofline': roofline, 'kernels': kernels,
                'cpu_baseline': cpu_line, 'parity_sample': parity,
                'final_gather': None if gather is None else {'mode': 'one packing kernel + one asynchronous all-gather per step, waited for once at '
                                                                     'the end of the job', 'tail_ms': tail_ms, 'verified': gather_ok,
                                                             'bytes_per_rank_and_step': 4 * sharding.record_words(args.frames, P_cap, cfg.n_cameras, n_out)},
                'persons_found_per_frame': P / args.frames,
                'dropin_driver_loop_frames_per_s': dropin_fps, 'dropin_driver_loop': dropin_detail, 'json_pack_frames_per_s': json_fps,
                'p50_frame_latency_ms': p50_ms, 'p99_frame_latency_ms': p99_ms, 'p50_frame_latency_eager_ms': p50_eager_ms,
                'p50_frame_latency_from_dict_ms': p50_dict_ms,
                'latency_note': 'one frame per call, host buffers in / host results out: infer_host_graph (CUDA graph per batch '
                                'shape) and, for comparison, the eager infer_host; from_dict = infer_frames, packing of the '
                                'reference frame dict (JSON strings) included'}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def load_traffic(args):
    """DRAM bytes per step and kernel class from the committed ncu --set full capture (profiles/r02_traffic.json), used only
    when it was taken on THIS workload; otherwise traffic is null (a number measured on another configuration or kernel
    revision would be stale)."""
    try:
        t = json.load(open(os.path.join(REPO, 'profiles', 'r02_traffic.json')))
    except Exception:
        return None, 'no ncu capture committed for this workload'
    w = t.get('workload', {})
    if (w.get('config'), w.get('frames'), w.get('persons')) != (args.config, args.frames, args.persons):
        return None, 'the committed ncu capture (%s) is of another workload: traffic not reported' % t.get('source', 'profiles/r02_traffic.json')
    return t.get('classes', {}), 'dram__bytes_read.sum + dram__bytes_write.sum per step and kernel class, ncu --set full (%s, kernel set %s)' % (
        t.get('source', 'profiles/r02_traffic.json'), t.get('kernel_set', '?'))


def parity_sample(cfg, frames, pb, res, gat, mlp, sample=(0, 1, 2, 3)):
    """Four frames of the batch the timed region just processed, checked against the oracle AFTER the timed region (scores
    1e-4 relative, person assignment on the GPU's scores exact, joints 0.5 mm): the benchmark asserts something about its
    own outputs. Part of the cpu_baseline leg (rank 0, N = 1) - the one place bench.py may execute oracle/."""
    try:
        from oracle import check as OC
        scores = res['scores'].cpu().numpy()
        ph, npers = res['person_heads'].cpu().numpy(), res['n_persons'].cpu().numpy()
        poff, joints = res['person_off'].cpu().numpy(), res['joints'].cpu().numpy()
        sample = [i for i in sample if i < pb.n_frames]
        rep = OC.check_frames(cfg, [frames[i % len(frames)] for i in sample], {k: v.numpy() for k, v in gat.items()},
                              {k: v.numpy() for k, v in mlp.items()},
                              [scores[pb.node_off[i]:pb.node_off[i + 1]] for i in sample],
                              [ph[pb.head_off[i]:pb.head_off[i] + npers[i]] for i in sample],
                              [joints[poff[i]:poff[i + 1]] for i in sample])
        return {'status': 'ok', 'frames': rep['frames'], 'persons': rep['persons'], 'worst_score_rel': rep['worst_score_rel'],
                'worst_joint_mm': rep['worst_joint_mm']}
    except AssertionError as e:
        return {'status': 'FAILED', 'why': str(e)}


def triangulation_workload(args, rank, world, local_rank):
    """BASELINE.json configs[3]: triangulation-only path, batched DLT for 5 views x 18 joints x 65536 persons
    (utils/pose_estimator_utils.py:52-75 fed as test/metrics_from_triangulation.py:237-249). Secondary workload:
    its own metric, printed as one JSON line like the headline."""
    import torch
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    pm = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
    cfg = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % args.config))
    P, C = 65536, cfg.n_cameras
    rng = np.random.default_rng(rank)
    people = synth.random_people(cfg, rng, 256)
    xy = np.zeros((256 * C, 18, 2)); mask = np.full(256 * C, (1 << 18) - 1, dtype=np.uint32)
    for p in range(256):
        for c in range(C):
            xy[p * C + c] = synth.project_points(cfg, c, people[p])[0]
    reps = P // 256
    h_xy = torch.from_numpy(np.tile(xy, (reps, 1, 1))).pin_memory()
    h_mask = torch.from_numpy(np.tile(mask, reps).view(np.int32)).pin_memory()
    h_psk = torch.arange(P * C, dtype=torch.int32).reshape(P, C).pin_memory()
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    pipe = pm.PosePipeline(cfg, None, None, device=dev)
    mk = lambda: pm.DeviceBatch(0, P * C, P * C, 0, 0, h_xy.to(dev, non_blocking=True), None, h_mask.to(dev, non_blocking=True), None, None, None)
    db, psk = mk(), h_psk.to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for _ in range(max(3, args.warmup)):
        pipe.triangulate(db, P, psk)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in ev:
        flush.fill_(1); a.record(); xyz, m = pipe.triangulate(db, P, psk); b.record()
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        d2, p2 = mk(), h_psk.to(dev, non_blocking=True)
        xyz, m = pipe.triangulate(d2, P, p2)
        hx, hm = xyz.cpu(), m.cpu()
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    # CPU port on a bounded sample (one process)
    from oracle import pose_oracle as O
    tabs = O.CameraTables(cfg)
    persons = [{cfg.camera_names[c]: {str(j): [j, xy[p * C + c, j, 0], xy[p * C + c, j, 1], 1, 1] for j in range(18)} for c in range(C)} for p in range(64)]
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < min(args.cpu_budget, 10.0):
        O.triangulate_baseline(persons[n % 64], tabs, cfg.median_axis); n += 1
    cpu = n / (time.perf_counter() - t0)
    solves = P * 18 * C * (C - 1) // 2
    in_bytes = P * C * (18 * 16 + 4 + 4); out_bytes = P * 18 * 25
    line = {'metric': 'persons/sec (triangulation-only, %d views x 18 joints, 65536 persons)' % C, 'value': P / ms * 1e3, 'unit': 'persons/s',
            'n_gpus': 1, 'steps': args.steps, 'warmup': max(3, args.warmup), 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64 (fp32 Jacobi start + fp64 Rayleigh-quotient refinement)', 'data': 'synthetic',
            'config': {'workload': 'triangulation-only: batched pairwise DLT, %d views x 18 joints x %d persons' % (C, P), 'camera_config': args.config,
                       'l2': 'L2 flushed (256 MiB write) between timed iterations'},
            'pair_solves_per_s': solves / ms * 1e3,
            'e2e': {'value': P / e2e_ms * 1e3, 'unit': 'persons/s', 'h2d_bytes_per_step': int(h_xy.numel() * 8 + h_mask.numel() * 4 + h_psk.numel() * 4),
                    'd2h_bytes_per_step': int(out_bytes), 'ms_per_step': e2e_ms},
            'gpu_launches': 1,
            'roofline': {'kernel': 'lift_person_kernel<false>', 'bound': 'hbm', 'achieved': (in_bytes + out_bytes) / ms / 1e6, 'peak': 6471.1, 'unit': 'GB/s',
                         'frac': (in_bytes + out_bytes) / ms / 1e6 / 6471.1, 'traffic': None,
                         'note': 'ALU-bound kernel (pairwise 4x4 solves), HBM fraction reported for completeness'},
            'cpu_baseline': {'value': cpu, 'unit': 'persons/s', 'cores': 1, 'kind': 'port', 'sample': '%d persons, one process' % n}}
    if rank == 0:
        print(json.dumps(line))


def train_batch_workload(args, rank, world, local_rank):
    """SURVEY.md 8f-3, forward only: the validation pass of skeleton_matching/train_skeleton_matching.py:88-110 - graphs of
    process_training (graph_generator.py:672-810) merged with dgl.batch (:80) and pushed through GAT2. One step = one
    block-diagonal batch of --frames graphs (the reference batches 15; a batch here is as large as the caller likes):
    edge/CSR build from the explicit edge-node lists, head features, 5 GAT layers. Dataset synthesis (sampling, packing)
    is outside the timed region, as the reference builds its datasets before the loop (:134-141)."""
    import random
    import torch
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    pm = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
    tg = importlib.import_module('3d_multi_pose_estimator_b200.training_graphs')
    cfg = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % args.config))
    gat, mlp = load_weights(args.config, cfg)
    G = args.frames
    n_files, per_file = 4, 24
    files = [[synth.make_frame(cfg, 7000 + 100 * f + t, 1, drop_joint_p=0.1, drop_view_p=0.1) for t in range(per_file)] for f in range(n_files)]
    random.seed(rank)
    inputs, indices = tg.load_inputs(files, 'dev', cfg.used_pe_names, random)          # 'dev': with the view augmentation
    built = []
    for mp in tg.sample_sets(inputs, indices, [0.8, 0.6, 0.7, 0.5], 10 ** 9, random):
        b = tg.training_graph_inputs(mp, cfg)
        if b is not None:
            built.append(b)
        if len(built) >= min(G, 256):
            break
    graphs = [(built[i % len(built)][0], built[i % len(built)][1]) for i in range(G)]   # cycled up to the batch size
    pb, pairs = tg.batch_packed(graphs)
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    pipe = pm.PosePipeline(cfg, gat, mlp, device=dev)
    hb = pm.HostBatch(pb)
    h_pairs = torch.from_numpy(pairs).pin_memory()
    db = hb.to_device(dev)
    d_pairs = h_pairs.to(dev)

    def step(db, d_pairs):
        g = pipe.build_graph_pairs(db, d_pairs, with_coo=False)
        return pipe.gat_forward(db, g)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    warmup = max(3, args.warmup)
    for _ in range(warmup):
        step(db, d_pairs)
    torch.cuda.synchronize()
    l0 = pipe.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    for a, b in ev:
        flush.fill_(1); a.record(); scores = step(db, d_pairs); b.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    launches = (pipe.launches - l0) // args.steps
    ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    # per-class time (CUDA events around the launches of one extra step)
    acc = {}
    orig_linear, orig_agg = pipe.linear, pipe.aggregate

    def timed(name, fn):
        def w(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = fn(*a, **k); e1.record()
            acc.setdefault(name, []).append((e0, e1))
            return r
        return w
    pipe.linear, pipe.aggregate = timed('gat_projection_gemm', orig_linear), timed('edge_softmax_aggregate', orig_agg)
    flush.fill_(1)
    step(db, d_pairs)
    torch.cuda.synchronize()
    pipe.linear, pipe.aggregate = orig_linear, orig_agg
    kern = {k: float(sum(a.elapsed_time(b) for a, b in v)) for k, v in acc.items()}
    # end to end: packed host batch -> device -> scores back on the host
    t0 = time.perf_counter()
    for _ in range(args.steps):
        d2 = hb.to_device(dev)
        s2 = step(d2, h_pairs.to(dev, non_blocking=True))
        host_scores = s2.cpu()
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    # CPU port of the same step on a bounded sample: batches of 15 graphs as the reference's loader makes them
    from oracle import pose_oracle as O
    tabs = O.CameraTables(cfg)
    gat_np = {k: v.numpy() for k, v in gat.items()}
    random.seed(rank)
    inputs, indices = O.load_training_inputs(files, 'dev', cfg.used_pe_names, random)
    sets = []
    for mp in O.training_samples(inputs, indices, [0.8, 0.6, 0.7, 0.5], 10 ** 9, random):
        sets.append(mp)
        if len(sets) >= 60:
            break
    ogs = [g for g in (O.build_training_graph(mp, tabs) for mp in sets) if g is not None]
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < min(args.cpu_budget, 15.0):
        members = [ogs[(n + i) % len(ogs)] for i in range(15)]
        bg = O.batch_graphs(members)
        O.gat_forward(gat_np, bg['feats'], bg['src'], bg['dst'])
        n += 15
    cpu = n / (time.perf_counter() - t0)
    W = importlib.import_module('3d_multi_pose_estimator_b200.weights')
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    agg_bytes, gat_flops, _ = algorithmic_work(pb, W.gat_layer_dims(cfg.n_features_sm), [], 0)
    tc_peak, hbm_peak = peaks.get('bf16_tflops_sustained', 1400.0), peaks.get('hbm_gbs', 6650.0)
    kernels = [{'kernel': 'gat_projection_gemm', 'ms_per_step': kern.get('gat_projection_gemm'), 'bound': 'tensor',
                'achieved': 3 * gat_flops / kern['gat_projection_gemm'] / 1e9, 'peak': tc_peak, 'unit': 'TFLOP/s'},
               {'kernel': 'edge_softmax_aggregate', 'ms_per_step': kern.get('edge_softmax_aggregate'), 'bound': 'hbm',
                'achieved': agg_bytes / kern['edge_softmax_aggregate'] / 1e6, 'peak': hbm_peak, 'unit': 'GB/s'}]
    for k in kernels:
        k['frac'] = k['achieved'] / k['peak']
    dom = max(kernels, key=lambda k: k['ms_per_step'])
    line = {'metric': 'graphs/sec (process_training graphs, dgl.batch + GAT2 forward, %d-graph batch)' % G, 'value': G / ms * 1e3, 'unit': 'graphs/s',
            'n_gpus': 1, 'steps': args.steps, 'warmup': warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'bf16x3 split (fp32-accurate), fp32 accumulate', 'data': 'synthetic',
            'config': {'workload': 'training-side validation batch: %d process_training graphs (%d nodes, %d edges) merged block-diagonally, '
                                   'edge/CSR build + features + 5 GAT layers, forward only' % (G, pb.n_nodes, pb.n_edges),
                       'camera_config': args.config, 'graphs_per_step': G, 'l2': 'L2 flushed (256 MiB write) between timed iterations'},
            'e2e': {'value': G / e2e_ms * 1e3, 'unit': 'graphs/s', 'h2d_bytes_per_step': int(hb.nbytes() + h_pairs.numel() * 4),
                    'd2h_bytes_per_step': int(host_scores.numel() * 4), 'ms_per_step': e2e_ms},
            'gpu_launches': launches, 'clocks': sampler.summary(),
            'roofline': {'kernel': dom['kernel'], 'bound': dom['bound'], 'achieved': dom['achieved'], 'peak': dom['peak'], 'unit': dom['unit'],
                         'frac': dom['frac'], 'traffic': None, 'peak_source': 'measured' if peaks else 'fallback'},
            'kernels': kernels,
            'cpu_baseline': {'value': cpu, 'unit': 'graphs/s', 'cores': 1, 'kind': 'port',
                             'sample': '%d graphs in batches of 15 (the reference loader\'s batch size), one process' % n}}
    if rank == 0:
        print(json.dumps(line))


def train_step_workload(args, rank, world, local_rank):
    """SURVEY.md 8f-3, the optimisation step: the loop body of skeleton_matching/train_skeleton_matching.py:163-184 - GAT2 forward
    on a dgl.batch of process_training graphs, MSE loss on the edge-node scores, backward, Adam - as GatTrainer.step. One step =
    one batch of --frames graphs (the reference's loader makes batches of 15, :42). Dataset synthesis and the graph build are
    outside the timed region (the reference builds its datasets before the loop, :134-141, and its collate runs in the loader)."""
    import random
    import torch
    pkg = importlib.import_module('3d_multi_pose_estimator_b200')
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    pm = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
    tg = importlib.import_module('3d_multi_pose_estimator_b200.training_graphs')
    tr = importlib.import_module('3d_multi_pose_estimator_b200.train')
    W = importlib.import_module('3d_multi_pose_estimator_b200.weights')
    cfg = pkg.CameraConfig.from_npz(os.path.join(GOLDEN, 'cameras_%s.npz' % args.config))
    G = args.frames
    n_files, per_file = 4, 24
    files = [[synth.make_frame(cfg, 7000 + 100 * f + t, 1, drop_joint_p=0.1, drop_view_p=0.1) for t in range(per_file)] for f in range(n_files)]
    random.seed(rank)
    inputs, indices = tg.load_inputs(files, 'train', cfg.used_pe_names, random)
    built = []
    for mp in tg.sample_sets(inputs, indices, [0.8, 0.6, 0.7, 0.5], 10 ** 9, random):
        b = tg.training_graph_inputs(mp, cfg)
        if b is not None:
            built.append(b)
        if len(built) >= min(G, 256):
            break
    members = [built[i % len(built)] for i in range(G)]
    pb, pairs = tg.batch_packed([(m[0], m[1]) for m in members])
    idx, off = [], 0
    for m in members:
        H, N = m[0].n_heads, int(m[0].node_off[-1])
        idx.append(np.arange(off + H, off + N))
        off += N
    idx = np.concatenate(idx).astype(np.int32)
    labels = np.concatenate([m[2].ravel() for m in members]).astype(np.float32)
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    state = W.make_gat_state(cfg.n_features_sm, 0, True)
    pipe = pm.PosePipeline(cfg, None, None, device=dev)
    trainer = tr.GatTrainer(pipe, state)
    hb = pm.HostBatch(pb)
    db = hb.to_device(dev)
    g = pipe.build_graph_pairs(db, torch.from_numpy(pairs).to(dev), with_coo=False)
    d_idx, d_lab = torch.from_numpy(idx).to(dev), torch.from_numpy(labels).to(dev)
    x0 = trainer.features(db)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    warmup = max(3, args.warmup)
    losses = []
    for _ in range(warmup):
        losses.append(float(trainer.step(db, g, d_idx, d_lab, x0=x0).item()))
    torch.cuda.synchronize()
    l0 = trainer.net.launches + pipe.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_losses = []
    # launch by launch first (eager_ms), then the product form: the same step replayed as one CUDA graph
    for a, b in ev:
        flush.fill_(1); a.record(); dev_losses.append(trainer.step(db, g, d_idx, d_lab, x0=x0).clone()); b.record()
    torch.cuda.synchronize()
    launches = (trainer.net.launches + pipe.launches - l0) // args.steps
    eager_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    for _ in range(3):
        trainer.step_captured(db, g, d_idx, d_lab, x0=x0)
    torch.cuda.synchronize()
    for a, b in ev:
        flush.fill_(1); a.record(); dev_losses.append(trainer.step_captured(db, g, d_idx, d_lab, x0=x0).clone()); b.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    losses += [float(x.item()) for x in dev_losses]
    # end to end: host batch (packed skeletons, edge-node list, indices, labels) -> device -> step -> loss on the host
    h_pairs, h_idx, h_lab = torch.from_numpy(pairs).pin_memory(), torch.from_numpy(idx).pin_memory(), torch.from_numpy(labels).pin_memory()
    def e2e_step():
        d2 = hb.to_device(dev)
        g2 = pipe.build_graph_pairs(d2, h_pairs.to(dev, non_blocking=True), with_coo=False)
        return float(trainer.step_captured(d2, g2, h_idx.to(dev, non_blocking=True), h_lab.to(dev, non_blocking=True)).item())
    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_loss = e2e_step()
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    # CPU port of the same step (oracle/train_oracle.py: numpy forward, hand-written backward, Adam) on batches of the same size
    from oracle import pose_oracle as O
    from oracle import train_oracle as TO
    tabs = O.CameraTables(cfg)
    random.seed(rank)
    oin, oidx = O.load_training_inputs(files, 'train', cfg.used_pe_names, random)
    ogs = []
    for mp in O.training_samples(oin, oidx, [0.8, 0.6, 0.7, 0.5], 10 ** 9, random):
        og = O.build_training_graph(mp, tabs)
        if og is not None:
            ogs.append(og)
        if len(ogs) >= min(G, 64):
            break
    ow = {k: v.numpy().copy() for k, v in state.items()}
    oadam = TO.Adam(ow)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < min(args.cpu_budget, 15.0) or n == 0:
        mem = [ogs[(n * G + i) % len(ogs)] for i in range(G)]
        bg = O.batch_graphs(mem)
        oi, o = [], 0
        for m in mem:
            oi.append(np.asarray(m['indices']) + o)
            o += m['n_nodes']
        ol, _, ograds = TO.forward_backward(ow, bg['feats'], bg['src'], bg['dst'], np.concatenate(oi), np.concatenate([m['labels'].ravel() for m in mem]))
        oadam.step(ow, ograds)
        n += 1
    cpu = n * G / (time.perf_counter() - t0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    # executed tensor-core work of a step: forward 2 N (din^2 + din n2), backward dW1 + dW2 + dh2 (+ dx above layer 0), x3 split MMAs
    N = pb.n_nodes
    flops = 0
    for l, (din, H, D) in enumerate(W.gat_layer_dims(cfg.n_features_sm)):
        hd, n2 = H * D, H * D + 2 * H
        flops += 2 * N * (din * din + din * n2)                      # forward
        flops += 2 * N * (hd * din + hd * din + din * din)           # dW2, dh2, dW1
        if l > 0:
            flops += 2 * N * din * din                               # dx
    tc_peak = peaks.get('bf16_tflops_sustained', 1400.0)
    line = {'metric': 'graphs/sec (process_training graphs, one optimisation step per %d-graph batch: forward + MSE + backward + Adam)' % G,
            'value': G / ms * 1e3, 'unit': 'graphs/s', 'n_gpus': 1, 'steps': args.steps, 'warmup': warmup, 'ms_per_step': ms,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16x3 split (fp32-accurate), fp32 accumulate; fp32 optimiser state', 'data': 'synthetic',
            'config': {'workload': 'training step: %d process_training graphs (%d nodes, %d edges, %d labelled edge-nodes) merged block-diagonally; '
                                   'GAT2 forward, MSE, backward, Adam (train_skeleton_matching.py:163-184)' % (G, pb.n_nodes, pb.n_edges, len(idx)),
                       'camera_config': args.config, 'graphs_per_step': G, 'l2': 'L2 flushed (256 MiB write) between timed iterations'},
            'e2e': {'value': G / e2e_ms * 1e3, 'unit': 'graphs/s',
                    'h2d_bytes_per_step': int(hb.nbytes() + h_pairs.numel() * 4 + h_idx.numel() * 4 + h_lab.numel() * 4),
                    'd2h_bytes_per_step': 4, 'ms_per_step': e2e_ms, 'includes': 'graph build from the edge-node list and feature synthesis'},
            'gpu_launches': launches, 'captured_graphs': len(trainer._graphs), 'eager_ms_per_step': eager_ms, 'step_form': 'one CUDA-graph replay per step (GatTrainer.step_captured); eager_ms_per_step = the same launches enqueued one by one',
            'clocks': sampler.summary(),
            'roofline': {'kernel': 'training step (all launches)', 'bound': 'tensor', 'achieved': 3 * flops / ms / 1e9, 'peak': tc_peak, 'unit': 'TFLOP/s',
                         'frac': 3 * flops / ms / 1e9 / tc_peak, 'traffic': None,
                         'note': 'small batches are latency bound (%d dependent launches per step); the fraction is of the whole step' % launches,
                         'peak_source': 'measured' if peaks else 'fallback'},
            'loss_first_last': [losses[0], losses[-1]],
            'cpu_baseline': {'value': cpu, 'unit': 'graphs/s', 'cores': 1, 'kind': 'port',
                             'sample': '%d optimisation steps on batches of %d graphs (numpy restatement oracle/train_oracle.py), one process' % (n, G)}}
    if rank == 0:
        print(json.dumps(line))


def _timed(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


DUMP_BYTES = 60 << 20            # 64 MB in all with room for the .npy headers


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy: integers and float64 as float64 (exact), other floats as float32. The inputs
    of a run are seeded, so two builds run with the same arguments can be compared file for file. When the arrays add up to
    more than DUMP_BYTES, each keeps a fixed, seeded sample of its rows, listed in out_dir/<name>.rows.npy."""
    host = {}
    for name, a in arrays.items():
        a = np.atleast_1d(a.detach().cpu().numpy() if hasattr(a, 'detach') else np.asarray(a))
        host[name] = a.astype(np.float64 if a.dtype.kind in 'biu' or a.dtype == np.float64 else np.float32)
    total = sum(a.nbytes for a in host.values())
    keep = 1.0 if total <= DUMP_BYTES else DUMP_BYTES / (total + 8 * sum(len(a) for a in host.values()))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        if keep < 1.0:
            rows = np.sort(np.random.default_rng(0).choice(len(a), max(1, int(len(a) * keep)), replace=False))
            np.save(os.path.join(out_dir, name + '.rows.npy'), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def dropin_driver_loop(cfg, frames, gat_state, mlp_state):
    """The loop body of the reference's test/metrics_from_model.py:178-300, one frame at a time, on the drop-in modules under
    their reference names (scripts/dropin_steps.py times every step): frames/s, and how much of a frame is the driver script's
    own Python (JSON re-encoding per camera and per person, its host<->device copies) against the drop-in modules' share."""
    sys.path.insert(0, os.path.join(REPO, 'scripts'))
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import dropin_steps
    synth = importlib.import_module('3d_multi_pose_estimator_b200.synth')
    full = [synth.make_frame(cfg, 50000 + i, max(1, len(json.loads(next(iter(f.values()))[0])))) for i, f in enumerate(frames)]
    r = dropin_steps.measure(cfg, full, gat_state, mlp_state)
    r.pop('steps')
    return r


def profile_classes(pipe, db, pm, torch):
    """ms per step spent in each kernel class, measured live with CUDA events on the launching stream."""
    import collections
    acc = collections.OrderedDict()
    orig_linear, orig_agg = pipe.linear, pipe.aggregate
    orig = {n: getattr(pipe, n) for n in ('build_graph', 'head_feature_planes', 'cluster', 'encode_persons')}
    state = {'phase': 'gat'}

    def timed(name, fn):
        def wrapper(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            acc.setdefault(name() if callable(name) else name, []).append((e0, e1))
            return r
        return wrapper
    pipe.linear = timed(lambda: 'gat_projection_gemm' if state['phase'] == 'gat' else 'mlp_gemm', orig_linear)
    pipe.aggregate = timed('edge_softmax_aggregate', orig_agg)
    names = {'build_graph': 'graph_build', 'head_feature_planes': 'node_features', 'cluster': 'cluster',
             'encode_persons': 'encode_dlt'}
    for n, f in orig.items():
        setattr(pipe, n, timed(names[n], f))
    orig_mlp = pipe.mlp_forward

    def mlp_wrapper(*a, **k):
        state['phase'] = 'mlp'
        r = orig_mlp(*a, **k)
        state['phase'] = 'gat'
        return r
    pipe.mlp_forward = mlp_wrapper
    reps = 3
    for _ in range(reps):
        pipe.infer(db)
    torch.cuda.synchronize()
    out = {k: sum(a.elapsed_time(b) for a, b in v) / reps for k, v in acc.items()}
    pipe.linear, pipe.aggregate, pipe.mlp_forward = orig_linear, orig_agg, orig_mlp
    for n, f in orig.items():
        setattr(pipe, n, f)
    return out


if __name__ == '__main__':
    main()
