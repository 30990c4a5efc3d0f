"""GPU: every GAT aggregation kernel variant and the fused last-layer projection against float64 references, at layer shapes
beyond the shipped model (GAT2 / GatTrainer accept any num_hidden / heads, and PosePipeline.prepare_gat hands them to the
C ABI unchanged).

* b200pose_gat_aggregate through the C ABI, one (heads, dim) case per template instantiation the dispatch
  (gat_aggregate_impl, csrc/gat.cu) can pick: the gather, generic frame-resident and large-frame kernels for every column
  vector width (dim % 4 -> 4 / 2 / 1 columns per lane) and column-group count, the shape-specialised kernels of the shipped
  layers, the scalar last-layer kernel. Real frame graphs (a ragged Panoptic batch and a Ring10 batch with more than 32
  heads per frame), both layer-0 row layouts, raw / planes / both outputs, LeakyReLU slopes inside and outside [0, 1].
  Every output buffer starts as NaN: valid elements must match the reference, the K padding of the planes must be exactly
  zero (workspaces are reused across widths) and rows past the batch must stay untouched. The kernel that ran is read
  back from torch.profiler.
* b200pose_linear_fused2 (fc1 + a few-column fc2 in one epilogue) against float64.
* two non-shipped GAT2 architectures end to end (inference and one training step) against the oracles.
* shapes past the compiled limits are refused with an error, not computed.
"""
import ctypes as C
import importlib
import json
import re
import types

import numpy as np
import pytest
import torch

import helpers
from oracle import pose_oracle as O
from oracle import train_oracle as TO

pytestmark = pytest.mark.gpu

pipeline_mod = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
pack_mod = importlib.import_module('3d_multi_pose_estimator_b200.pack')
train_mod = importlib.import_module('3d_multi_pose_estimator_b200.train')
_lib = importlib.import_module('3d_multi_pose_estimator_b200._lib')
ptr, round_up, Planes = _lib.ptr, pipeline_mod.round_up, pipeline_mod.Planes

ALPHA, ACT_SLOPE = 0.15, 0.01              # shipped (weights.GAT_ALPHA, GAT_ACT_SLOPE)
ALPHA_X, ACT_SLOPE_X = 1.6, 1.3            # outside [0, 1]: max(x, slope * x) is no longer LeakyReLU
SHIPPED = [(10, 40), (8, 40), (5, 30)]     # the layers with shape-specialised kernels
NAN = float('nan')

# Tolerance of the aggregation outputs, relative to the largest |ft2| of the layer (every output is a convex combination of
# ft2 rows). The kernels compute the softmax weights with ex2.approx / rcp.approx: a few 1e-7 relative, up to ~2e-6 where
# the large-frame kernel's running softmax reference sits up to 30 below a logit (the rounding of an exp2 argument near 43).
# They sum at most ~100 weighted rows in fp32 (worst case 100 * 2^-24 = 6e-6 relative to the largest row).
RAW_RTOL = 1e-5
PLANE_RTOL = 2.0 ** -16                    # hi + lo bf16 planes hold 16 mantissa bits of the activated value


def msg():
    return (_lib.lib().b200pose_last_error() or b'').decode()


# ------------------------------------------------------------------------------------------------ batches
_batches = {}


def frame_batch(config):
    """A ragged batch of real frame graphs: synthetic frames of several sizes, an empty frame and a frame seen by one camera
    only (heads, no edge-node). 'panoptic': 5 views, at most 20 heads per frame (frame-resident plans fit); 'ring10': 10
    views with 11 persons in one frame (110 heads: past the frame-resident kernels)."""
    if config in _batches:
        return _batches[config]
    cfg = helpers.load_golden(config)[0]
    mk = helpers.synth.make_frame
    if config == 'panoptic':
        frames = [mk(cfg, 4100 + i, 1 + i % 4, drop_view_p=0.1 * (i % 3), drop_joint_p=0.05 * (i % 2)) for i in range(6)]
    else:
        frames = [mk(cfg, 4200, 11), mk(cfg, 4201, 2)]
    frames.insert(1, {})
    frames.append(mk(cfg, 4300, 3, camera_order=[cfg.used_sm[0]]))
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    pb = pack_mod.pack_frames(frames, cfg)
    n_nodes = np.diff(pb.node_off)
    n_heads = np.diff(pb.head_off)
    assert (n_nodes == 0).any() and ((n_heads > 0) & (n_nodes == n_heads)).any()
    pipe = pipeline_mod.PosePipeline(cfg, None, None, device='cuda:0')
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    g = pipe.build_graph(db, with_coo=False)
    torch.cuda.synchronize()
    N, S = db.n_nodes, db.n_heads
    row_ptr = g.row_ptr.cpu().numpy().astype(np.int64)
    col = g.col[: db.n_edges].cpu().numpy().astype(np.int64)
    assert row_ptr[-1] == db.n_edges and (np.diff(row_ptr) >= 1).all()
    # layer 0 reads S + 1 compact rows: a head's own row (h0 + local index), and row S for every edge-node
    zrow0 = np.empty(N, dtype=np.int64)
    for b in range(pb.n_frames):
        n0, n1, h0, h1 = pb.node_off[b], pb.node_off[b + 1], pb.head_off[b], pb.head_off[b + 1]
        zrow0[n0:n0 + (h1 - h0)] = np.arange(h0, h1)
        zrow0[n0 + (h1 - h0):n1] = S
    bt = types.SimpleNamespace(config=config, cfg=cfg, pb=pb, pipe=pipe, db=db, g=g, N=N, S=S, row_ptr=row_ptr, col=col, zrow0=zrow0)
    _batches[config] = bt
    return bt


# ------------------------------------------------------------------------------------------------ references
def leaky(x, s):
    return np.where(x >= 0, x, s * x)


def edge_softmax_ref(z, zrow, src, seg, dst, H, D, alpha):
    """float64: out[v, h, :] = sum_{u -> v} softmax_u(LeakyReLU_alpha(a1[u, h] + a2[v, h])) ft2[u, h, :] for the destinations
    `dst`, whose in-edges are src[seg[i]:seg[i + 1]]; node n reads z row zrow[n] = [ft2 (H*D) | a1 (H) | a2 (H) | padding]."""
    HD = H * D
    deg = np.diff(seg)
    zs, zd = zrow[src], zrow[np.repeat(dst, deg)]
    e = leaky(z[zs, HD:HD + H] + z[zd, HD + H:HD + 2 * H], alpha)
    e = e - np.maximum.reduceat(e, seg[:-1], axis=0)[np.repeat(np.arange(len(dst)), deg)]
    w = np.exp(e)
    w /= np.add.reduceat(w, seg[:-1], axis=0)[np.repeat(np.arange(len(dst)), deg)]
    ft2 = z[:, :HD].reshape(-1, H, D)
    return np.add.reduceat(w[:, :, None] * ft2[zs], seg[:-1], axis=0).reshape(len(dst), HD)


def random_z(rng, rows, H, D):
    """fp32 z rows with a1 / a2 the dots of ft2 with random attention vectors (as the folded projection yields them), the
    row padding NaN (the projection never writes it: no kernel may read it)."""
    HD = H * D
    ldz = round_up(HD + 2 * H, 4)
    ft2 = rng.standard_normal((rows, H, D))
    al, ar = rng.standard_normal((2, H, D)) * (1.5 / np.sqrt(D))
    z = np.full((rows, ldz), np.nan, dtype=np.float32)
    z[:, :HD] = ft2.reshape(rows, HD)
    z[:, HD:HD + H] = np.einsum('nhd,hd->nh', ft2, al)
    z[:, HD + H:HD + 2 * H] = np.einsum('nhd,hd->nh', ft2, ar)
    return z


# ------------------------------------------------------------------------------------------------ the dispatch, restated
def frame_plan_bytes(mh, me, HD, H, ldz):
    """frame_plan() of csrc/gat.cu"""
    hd4 = (HD + 3) & ~3
    e_heads = mh + 2 * me
    r4 = lambda x: (x + 3) & ~3
    return 4 * (4 * 16 * ldz + mh * hd4 + ldz + r4(mh * 2 * H) + r4(me * H) + r4(e_heads * H) + r4(e_heads) + r4(2 * me))


def large_plan_bytes(mh, HD, ldz, vec):
    """large_plan() of csrc/gat.cu"""
    edge_end = 8 * 4 * ldz + 33 * ldz + (mh + 1) // 2 + 1 + 3 * 64
    head_end = 8 * 6 * ldz + 8 * HD + 2 * 8 * (HD // vec) + ldz + 8 * (mh // 2 + 2)
    return 4 * (max(edge_end, head_end) + 4)


def expected_kernel(H, D, impl, bt, raw, planes, ld_planes, alpha, act_slope, layer0):
    """The kernel gat_aggregate_impl launches for these arguments (a name prefix as torch.profiler reports it, spaces
    removed), or the negative status it returns instead."""
    HD = H * D
    if HD == 1:
        return 'gat_aggregate_scalar_kernel'
    ldz = round_up(HD + 2 * H, 4)
    mh, me, nf = bt.db.max_heads, bt.db.max_enodes, bt.db.n_frames
    vec = 4 if D % 4 == 0 else 2 if D % 2 == 0 else 1
    nv = HD // vec
    tiny = impl == 0 and nf * 8 <= 148 and 3 * H <= 32
    frame = ((impl == 0 and not tiny) or impl in (3, 5, 6)) and mh > 0 and me > 0 and mh <= 32 and nv <= 128
    if (frame and impl != 5 and planes and not raw and 0 <= act_slope <= 1 and 0 <= alpha <= 1 and (H, D) in SHIPPED
            and ld_planes == round_up(HD, 64)):
        return 'gat_aggregate_frame_%s_kernel<%d,%d,%s' % ('s' if impl == 6 else 'p', H, D, 'true' if layer0 else 'false')
    if frame and frame_plan_bytes(mh, me, HD, H, ldz) <= 220 * 1024:
        return 'gat_aggregate_frame_kernel<%d,%d>' % (vec, 2 if nv <= 64 and vec != 1 else 4)
    if impl in (3, 5, 6):
        return -3
    large_ok = ((impl == 0 and (mh > 32 or tiny)) or impl == 2) and me > 0 and 3 * H <= 32 and nv <= 128 and ldz <= 640
    kmax = -(-nv // 32)
    if large_ok and large_plan_bytes(max(mh, 1), HD, ldz, vec) <= 113 * 1024 and \
            (vec, kmax) in [(4, 4), (4, 3), (4, 2), (2, 4), (2, 3), (2, 2), (1, 4)]:
        return 'gat_aggregate_large_kernel<%d,%d>' % (vec, kmax)
    if nv > 256:
        return -3
    if vec == 1:
        return 'gat_aggregate_kernel<1,%d>' % (4 if nv <= 128 else 8)
    return 'gat_aggregate_kernel<%d,%d>' % (vec, 2 if nv <= 64 else 4 if nv <= 128 else 8)


def launched_kernels(fn):
    """(fn(), names of the aggregation kernels that ran inside it, spaces removed)"""
    import warnings
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with warnings.catch_warnings():
        warnings.filterwarnings('ignore', message='.*Profiler clears events.*')
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            rc = fn()
            torch.cuda.synchronize()
    names = [re.sub(r'\s+', '', e.name) for e in prof.events() if 'gat_aggregate' in e.name and 'b200pose' in e.name]
    return rc, names


# ------------------------------------------------------------------------------------------------ 1. forward aggregation
# (heads, dim) -> instantiations it reaches (vec from dim % 4, n_vec = heads * dim / vec, kmax = ceil(n_vec / 32)):
#   3x33  vec 1, n_vec  99: gather <1,4>, frame <1,4>, large <1,4>
#   9x25  vec 1, n_vec 225: gather <1,8> (too wide for the frame-resident and large-frame kernels)
#   4x30  vec 2, n_vec  60: gather <2,2>, frame <2,2>, large <2,2>
#   1x250 vec 2, n_vec 125: large <2,4> (gather <2,4>, frame <2,4>)
#   10x30 vec 2, n_vec 150: gather <2,8>
#   6x40  vec 4, n_vec  60: frame <4,2>, large <4,2> (gather <4,2>)
#   6x100 vec 4, n_vec 150: gather <4,8>
#   the shipped 10x40, 8x40, 5x30: the shape-specialised kernels (impl 3: persistent, impl 6: one CTA per frame)
#   1x1: the scalar last-layer kernel with the sigmoid
AGG_SHAPES = [(3, 33), (9, 25), (4, 30), (1, 250), (10, 30), (6, 40), (6, 100)] + SHIPPED


def run_aggregate(bt, z_dev, H, D, layer0, impl, alpha, act_slope, raw, hi, lo, ld_planes, scores=None):
    db, g = bt.db, bt.g
    return _lib.lib().b200pose_gat_aggregate(
        db.n_frames, db.n_nodes, db.n_heads, ptr(db.head_off), ptr(db.node_off), ptr(g.row_ptr), ptr(g.col), ptr(z_dev), z_dev.shape[1],
        H, D, layer0, db.max_heads, db.max_enodes, alpha, act_slope, ptr(raw), ptr(hi), ptr(lo), ld_planes, ptr(scores), impl, None)


class Reference:
    """float64 reference of one layer on one batch (one z per row layout), with its tolerances and a proof that they can fail."""

    def __init__(self, bt, z, H, D, layer0, alpha):
        HD = H * D
        zrow = bt.zrow0 if layer0 else np.arange(bt.N)
        z64 = z.astype(np.float64)
        self.out = edge_softmax_ref(z64, zrow, bt.col, bt.row_ptr, np.arange(bt.N), H, D, alpha)
        self.scale = float(np.abs(z64[:, :HD]).max())
        self.tol = RAW_RTOL * self.scale
        # the tolerance must be able to fail: one in-edge of one node dropped moves the reference far past it
        deg = np.diff(bt.row_ptr)
        v = np.flatnonzero(deg >= 2)[len(np.flatnonzero(deg >= 2)) // 2]
        srcs = bt.col[bt.row_ptr[v] + 1:bt.row_ptr[v + 1]]
        dropped = edge_softmax_ref(z64, zrow, srcs, np.array([0, len(srcs)]), np.array([v]), H, D, alpha)
        moved = float(np.abs(dropped[0] - self.out[v]).max())
        assert moved >= 10 * self.tol, ('a dropped in-edge moves the reference by %g only, tolerance %g' % (moved, self.tol))
        self.moved = moved


def check_outputs(ref, bt, HD, raw, hi, lo, ld_planes, act_slope, what):
    """Valid elements against the reference, plane padding exactly zero, rows past the batch untouched. Returns the worst
    errors relative to the tolerances."""
    N = bt.N
    worst = [0.0, 0.0]
    ref_d = torch.from_numpy(ref.out).cuda()
    if raw is not None:
        err = (raw[:N].double() - ref_d).abs().max().item() if N else 0.0
        assert err <= ref.tol, ('raw', what, err, ref.tol)
        assert torch.isnan(raw[N:]).all(), ('raw rows past the batch written', what)
        worst[0] = err / ref.tol
    if hi is not None:
        act = torch.where(ref_d >= 0, ref_d, ref_d * act_slope)
        got = hi[:N, :HD].double() + lo[:N, :HD].double()
        tol = max(1.0, abs(act_slope)) * ref.tol + PLANE_RTOL * act.abs()
        excess = ((got - act).abs() - tol)
        assert not torch.isnan(got).any() and excess.max().item() <= 0, ('planes', what, excess.max().item())
        worst[1] = ((got - act).abs() / tol).max().item()
        if ld_planes > HD:
            pad_hi, pad_lo = hi[:N, HD:ld_planes], lo[:N, HD:ld_planes]
            assert bool((pad_hi == 0).all()) and bool((pad_lo == 0).all()), ('plane padding not zeroed', what)
        assert torch.isnan(hi[N:].float()).all() and torch.isnan(lo[N:].float()).all(), ('plane rows past the batch written', what)
    return worst


@pytest.mark.parametrize('config', ['panoptic', 'ring10'])
@pytest.mark.parametrize('heads,dim', AGG_SHAPES)
def test_aggregate_forward_vs_fp64(heads, dim, config):
    """b200pose_gat_aggregate against the float64 edge softmax, every impl, both row layouts, every output combination,
    NaN-filled outputs; the kernel that ran is confirmed with torch.profiler once per distinct kernel."""
    bt = frame_batch(config)
    H, D, HD = heads, dim, heads * dim
    N = bt.N
    rng = np.random.default_rng(1000 * H + D)
    impls = [0, 1, 2, 5] + ([3, 6] if (H, D) in SHIPPED else [])
    modes = {'raw': (True, False, 0), 'planes': (False, True, 0), 'both': (True, True, 0), 'planes_wide': (False, True, 64)}
    worst = [0.0, 0.0]
    confirmed, refused = {}, []
    for layer0 in (1, 0):
        z = random_z(rng, bt.S + 1 if layer0 else N, H, D)
        z_dev = torch.from_numpy(z).cuda()
        for alpha, act_slope in ((ALPHA, ACT_SLOPE), (ALPHA_X, ACT_SLOPE_X)):
            ref = Reference(bt, z, H, D, layer0, alpha)
            for impl in impls:
                for mode, (want_raw, want_planes, extra) in modes.items():
                    if (alpha, act_slope) == (ALPHA_X, ACT_SLOPE_X) and mode not in ('planes', 'both'):
                        continue
                    ld_planes = round_up(HD, 64) + extra
                    raw = torch.full((N + 3, HD), NAN, device='cuda') if want_raw else None
                    hi = torch.full((N + 3, ld_planes), NAN, dtype=torch.bfloat16, device='cuda') if want_planes else None
                    lo = torch.full((N + 3, ld_planes), NAN, dtype=torch.bfloat16, device='cuda') if want_planes else None
                    what = '%dx%d %s impl %d layer0 %d %s alpha %g slope %g' % (H, D, config, impl, layer0, mode, alpha, act_slope)
                    expect = expected_kernel(H, D, impl, bt, want_raw, want_planes, ld_planes, alpha, act_slope, layer0)
                    call = lambda: run_aggregate(bt, z_dev, H, D, layer0, impl, alpha, act_slope, raw, hi, lo, ld_planes)
                    if isinstance(expect, str) and expect not in confirmed:
                        rc, names = launched_kernels(call)
                        assert len(names) == 1 and expect in names[0], (what, expect, names)
                        confirmed[expect] = what
                    else:
                        rc = call()
                    torch.cuda.synchronize()
                    if isinstance(expect, int):
                        assert rc == expect and 'impl' in msg(), (what, rc, msg())
                        for t in (raw, hi):
                            assert t is None or torch.isnan(t.float()).all(), ('refused call wrote its output', what)
                        refused.append((impl, layer0))
                        continue
                    assert rc == 0, (what, rc, msg())
                    w = check_outputs(ref, bt, HD, raw, hi, lo, ld_planes, act_slope, what)
                    worst = [max(a, b) for a, b in zip(worst, w)]
    if (H, D) in SHIPPED and config == 'panoptic':
        assert any('frame_p_kernel' in k for k in confirmed) and any('frame_s_kernel' in k for k in confirmed)
    print('%dx%d %s: worst raw error %.3f, worst plane error %.3f of the tolerance (raw tolerance %.2e, a dropped in-edge moves the '
          'reference by %.2e); kernels: %s; refused: %s' % (H, D, config, worst[0], worst[1], ref.tol, ref.moved, sorted(confirmed), sorted(set(refused))))


@pytest.mark.parametrize('config', ['panoptic', 'ring10'])
def test_aggregate_scalar_layer_vs_fp64(config):
    """heads * dim == 1 (the last layer): the scalar kernel with the sigmoid, raw and scores outputs, against float64."""
    bt = frame_batch(config)
    N = bt.N
    rng = np.random.default_rng(11)
    z = random_z(rng, N, 1, 1)
    z_dev = torch.from_numpy(z).cuda()
    worst = 0.0
    for alpha in (ALPHA, ALPHA_X):
        ref = Reference(bt, z, 1, 1, 0, alpha)
        want_scores = torch.from_numpy(1.0 / (1.0 + np.exp(-ref.out[:, 0]))).cuda()
        for want_raw, want_scores_out in ((True, False), (False, True), (True, True)):
            raw = torch.full((N + 3, 1), NAN, device='cuda') if want_raw else None
            scores = torch.full((N + 3,), NAN, device='cuda') if want_scores_out else None
            call = lambda: run_aggregate(bt, z_dev, 1, 1, 0, 0, alpha, ACT_SLOPE, raw, None, None, 0, scores)
            rc, names = launched_kernels(call)
            assert rc == 0, msg()
            assert names == [n for n in names if 'gat_aggregate_scalar_kernel' in n] and len(names) == 1, names
            if raw is not None:
                w = check_outputs(ref, bt, 1, raw, None, None, 0, ACT_SLOPE, 'scalar')
                worst = max(worst, w[0])
            if scores is not None:
                err = (scores[:N].double() - want_scores).abs().max().item()
                assert err <= ref.tol, ('scores', err, ref.tol)
                assert torch.isnan(scores[N:]).all()
                worst = max(worst, err / ref.tol)
    # the scalar layer has no layer-0 form and no planes: refused before any launch
    hi = torch.full((N, 64), NAN, dtype=torch.bfloat16, device='cuda')
    assert run_aggregate(bt, z_dev, 1, 1, 1, 0, ALPHA, ACT_SLOPE, None, None, None, 0, scores) == -1 and 'scalar' in msg()
    assert run_aggregate(bt, z_dev, 1, 1, 0, 0, ALPHA, ACT_SLOPE, None, hi, hi, 64) == -1 and 'scalar' in msg()
    torch.cuda.synchronize()
    assert torch.isnan(hi.float()).all()
    print('1x1 %s: worst error %.3f of the tolerance' % (config, worst))


# ------------------------------------------------------------------------------------------------ 2. fused fc1 + fc2
FUSED_DIN = [1, 32, 64, 150, 200, 250, 256]
FUSED_M = [1, 16, 17, 128, 129, 512, 513, 5000]


def fused2(A, W1, b1, m, n1, k, slope1, w2, ldw2, b2, n2, out, ld_out):
    return _lib.lib().b200pose_linear_fused2(ptr(A.hi), ptr(A.lo), A.ld, ptr(W1.hi), ptr(W1.lo), W1.ld, ptr(b1), m, n1, k, slope1,
                                             w2 if isinstance(w2, C.c_void_p) else ptr(w2), ldw2, ptr(b2), n2, ptr(out), ld_out, None)


@pytest.mark.parametrize('din', FUSED_DIN)
def test_linear_fused2_vs_fp64(din):
    """out2 = LeakyReLU_slope1(A W1^T + b1) W2^T + b2 in one launch (the last GAT layer's fc1 + fc2 + attention dots) against
    float64 from the same split operands: partial and full last panels, m on both sides of the single-CTA / CTA-pair switch at
    512 rows and below the 16 rows the pipeline sends, 1..4 fused columns. Columns [n2, ld_out2) and rows >= m stay untouched."""
    torch.manual_seed(din)
    W1 = Planes.from_f32(torch.randn(din, din, device='cuda') / din ** 0.5, None)
    b1 = torch.randn(din, device='cuda')
    ldw2 = round_up(din, 64)
    worst = 0.0
    for m in FUSED_M:
        A = Planes.from_f32(torch.randn(m, din, device='cuda') * 0.7, None)
        pre = A.to_f32().double() @ W1.to_f32().double().T + b1.double()
        for n2 in (1, 2, 3, 4):
            w2 = torch.zeros(n2, ldw2, device='cuda')
            w2[:, :din] = torch.randn(n2, din, device='cuda') / din ** 0.5
            b2 = torch.randn(n2, device='cuda')
            for slope1 in (0.15, 1.0):
                h = torch.where(pre >= 0, pre, pre * slope1)
                ref = h @ w2[:, :din].double().T + b2.double()
                # first projection as in test_linear_kernels (2e-5 of its largest value), carried through |W2| rows, plus the
                # fp32 dot product of <= 256 terms (256 * 2^-24 of sum |h w2|)
                tol = (2e-5 * max(1.0, h.abs().max().item()) + 256 * 2.0 ** -24 * h.abs().max().item()) * w2.abs().sum(1).max().item()
                out = torch.full((m + 2, 8), NAN, device='cuda')
                rc = fused2(A, W1, b1, m, din, din, slope1, w2, ldw2, b2, n2, out, 8)
                assert rc == 0, (din, m, n2, slope1, rc, msg())
                torch.cuda.synchronize()
                err = (out[:m, :n2].double() - ref).abs().max().item()
                assert err <= tol, (din, m, n2, slope1, err, tol)
                assert torch.isnan(out[:m, n2:]).all() and torch.isnan(out[m:]).all(), ('fused2 wrote outside its output', din, m, n2)
                worst = max(worst, err / tol)
    print('linear_fused2 din %d: worst error %.3f of the tolerance' % (din, worst))


def test_linear_fused2_refusals():
    """Arguments the fused epilogue cannot take are refused with B200POSE_E_INVALID and a message, before any launch."""
    torch.manual_seed(3)
    m, din = 40, 150
    A = Planes.from_f32(torch.randn(m, din, device='cuda'), None)
    W1 = Planes.from_f32(torch.randn(din, din, device='cuda'), None)
    b1 = torch.randn(din, device='cuda')
    w2 = torch.zeros(5, 256, device='cuda')
    b2 = torch.zeros(5, device='cuda')
    out = torch.full((m, 8), NAN, device='cuda')
    cases = {
        'n1 > 256': lambda: fused2(A, W1, b1, m, 257, din, 0.15, w2, 256, b2, 3, out, 8),
        'n2 = 0': lambda: fused2(A, W1, b1, m, din, din, 0.15, w2, 256, b2, 0, out, 8),
        'n2 = 5': lambda: fused2(A, W1, b1, m, din, din, 0.15, w2, 256, b2, 5, out, 8),
        'w2 not 16-byte aligned': lambda: fused2(A, W1, b1, m, din, din, 0.15, C.c_void_p(w2.data_ptr() + 4), 252, b2, 3, out, 8),
        'w2 rows not padded to 64 columns': lambda: fused2(A, W1, b1, m, din, din, 0.15, w2, 152, b2, 3, out, 8),
        'ld_out2 < n2': lambda: fused2(A, W1, b1, m, din, din, 0.15, w2, 256, b2, 3, out, 2),
        'null fused weights': lambda: fused2(A, W1, b1, m, din, din, 0.15, None, 256, b2, 3, out, 8),
    }
    for what, call in cases.items():
        assert call() == -1 and 'linear_fused2' in msg(), (what, msg())
    torch.cuda.synchronize()
    assert torch.isnan(out).all()
    assert fused2(A, W1, b1, m, din, din, 0.15, w2, 256, b2, 3, out, 8) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(out[:, :3]).all()


# ------------------------------------------------------------------------------------------------ 3. other architectures
# 'odd': odd widths (3x33, 7x17: one column per lane), a 1x64 layer, the last layer's fc1 + fc2 fused at din = 64;
# 'wide_last': 6x40 and 3x100 (three column groups), last layer din = 300 > 256 (two launches, no fused epilogue)
ARCHS = {'odd': ([33, 17, 64], [3, 7, 1], 21), 'wide_last': ([40, 100], [6, 3], 22)}


def golden_frames(config):
    cfg, npz, meta = helpers.load_golden(config)
    tags = helpers.graph_cases(config)
    return [{c: meta['frames'][t][c] for c in meta['frames'][t] if json.loads(meta['frames'][t][c][0])} for t in tags]


def fresh_frames(cfg):
    frames = [helpers.synth.make_frame(cfg, 5200 + i, 1 + i % 4, drop_joint_p=0.1 * (i % 2), drop_view_p=0.1 * (i % 3)) for i in range(6)]
    frames += [{}, helpers.synth.make_frame(cfg, 5300, 2, camera_order=[cfg.used_sm[1]])]
    return [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]


def arch_state(cfg, arch):
    """make_gat_state of the architecture with the last layer's output scaled to |logit| <= 3 on the golden frames (fc2 times
    c, the attention vectors divided by c: the softmax is unchanged), so that sigmoid scores are not saturated."""
    hidden, heads, seed = ARCHS[arch]
    state = helpers.weights_mod.make_gat_state(cfg.n_features_sm, seed, True, hidden, heads)
    tabs = O.CameraTables(cfg)
    w = helpers.np_state(state)
    top = 0.0
    for f in golden_frames('panoptic'):
        og = O.build_graph(f, tabs)
        _, layers = O.gat_forward(w, og['feats'], og['src'], og['dst'], heads=tuple(heads) + (1,), return_layers=True)
        top = max(top, float(np.abs(layers[-1]).max()))
    c = 3.0 / top
    last = len(hidden)
    for k in ('fc2.weight', 'fc2.bias'):
        state['layers.%d.%s' % (last, k)] = state['layers.%d.%s' % (last, k)] * c
    for k in ('attn_l', 'attn_r'):
        state['layers.%d.%s' % (last, k)] = state['layers.%d.%s' % (last, k)] / c
    return state, tuple(heads) + (1,)


@pytest.mark.parametrize('arch', sorted(ARCHS))
def test_other_architecture_inference_vs_oracle(arch):
    """GAT2 of a non-shipped architecture through the pipeline (agg_impl 0 / 1 / 2, compact layer-0 rows and the drop-in's
    dense rows) on the golden Panoptic frames and fresh frames, against the oracle: scores 1e-4 relative, every layer 1e-4
    of its largest value."""
    cfg = helpers.load_golden('panoptic')[0]
    state, heads = arch_state(cfg, arch)
    w = helpers.np_state(state)
    pipe = pipeline_mod.PosePipeline(cfg, None, None, device='cuda:0')
    layers = pipe.prepare_gat(state)
    assert ('w2_f32' in layers[-1]) == (arch == 'odd')
    tabs = O.CameraTables(cfg)
    worst_s = worst_l = 0.0
    for frames in (golden_frames('panoptic'), fresh_frames(cfg)):
        pb = pack_mod.pack_frames(frames, cfg)
        db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
        g = pipe.build_graph(db, with_coo=False)
        ogs = [O.build_graph(f, tabs) for f in frames]
        refs = [O.gat_forward(w, og['feats'], og['src'], og['dst'], heads=heads, return_layers=True) if og is not None else None for og in ogs]
        runs = []
        for impl in (0, 1, 2):
            pipe.agg_impl = impl
            try:
                runs.append(pipe.gat_forward(db, g, layers=layers, keep_layers=True))
            finally:
                pipe.agg_impl = 0
        x0 = Planes.from_f32(pipe.node_features_f32(db), pipe._stream())
        runs.append(pipe.gat_forward(db, g, x0=x0, dense_rows=True, layers=layers, keep_layers=True))
        for r, (scores, raws) in enumerate(runs):
            scores = scores.cpu().numpy()
            raws = [x.cpu().numpy() for x in raws]
            for b, ref in enumerate(refs):
                if ref is None:
                    continue
                n0, n1 = pb.node_off[b], pb.node_off[b + 1]
                rel = np.abs(scores[n0:n1] - ref[0]) / np.abs(ref[0])
                assert rel.max() <= 1e-4, (arch, r, b, rel.max())
                worst_s = max(worst_s, rel.max())
                for l, want in enumerate(ref[1]):
                    want = want.reshape(n1 - n0, -1)
                    err = np.abs(raws[l][n0:n1] - want).max() / max(1.0, np.abs(want).max())
                    assert err <= 1e-4, (arch, r, b, l, err)
                    worst_l = max(worst_l, err)
    print('%s: worst relative score error %.2e, worst layer error %.2e of the layer maximum' % (arch, worst_s, worst_l))


@pytest.mark.parametrize('arch', sorted(ARCHS))
def test_other_architecture_training_step_vs_oracle(arch):
    """One GatTrainer.step(update=False) of a non-shipped architecture on the golden Panoptic frames: loss and scores against
    oracle/train_oracle.py, and the backward kernels (gat_prepare_layer's folds, aggregation backward, grad_planes,
    transpose_planes, colsum, attention / bias gradients at these widths) run by the oracle's backward on the forward state
    the device kept: every gradient tensor within 1e-4 of its largest value."""
    cfg = helpers.load_golden('panoptic')[0]
    state, heads = arch_state(cfg, arch)
    w = helpers.np_state(state)
    pipe = pipeline_mod.PosePipeline(cfg, None, None, device='cuda:0')
    pb = pack_mod.pack_frames(golden_frames('panoptic'), cfg)
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    g = pipe.build_graph(db, with_coo=False)
    idx = np.concatenate([np.arange(pb.node_off[b] + (pb.head_off[b + 1] - pb.head_off[b]), pb.node_off[b + 1]) for b in range(pb.n_frames)])
    labels = (np.random.default_rng(7).random(len(idx)) < 0.3).astype(np.float32)
    trainer = train_mod.GatTrainer(pipe, state)
    loss = float(trainer.step(db, g, torch.from_numpy(idx.astype(np.int32)).cuda(), torch.from_numpy(labels).cuda(), update=False).item())
    grads = {k: v.clone().cpu().numpy() for k, v in trainer.net.grads().items()}
    scores = trainer.last_scores.cpu().numpy().copy()
    feats = pipe.node_features_f32(db).cpu().numpy()
    N = db.n_nodes
    row_ptr, src = g.row_ptr.cpu().numpy(), g.col[: db.n_edges].cpu().numpy()
    dst = np.repeat(np.arange(N), np.diff(row_ptr))
    oloss, oscores, _ = TO.forward_backward(w, feats, src, dst, idx, labels, heads=heads)
    assert abs(loss - oloss) <= 1e-5 * oloss, (loss, oloss)
    assert (np.abs(scores - oscores) / np.abs(oscores)).max() <= 1e-4
    cl = trainer.net.cache['layers']
    caches, raws = TO.caches_from_device(w, [c['x'].to_f32()[:N].cpu().numpy() for c in cl], [c['h2'].to_f32()[:N].cpu().numpy() for c in cl],
                                         [c['z'][:N].cpu().numpy() for c in cl], src, dst, heads=heads)
    dl = trainer.net.buf.f('dlogit', N, 1)[:N, 0].cpu().numpy().reshape(-1, 1, 1)
    dgrads = TO.backward(w, caches, raws, src.astype(np.int64), dst.astype(np.int64), dl)
    worst = 0.0
    for k, og in dgrads.items():
        got = grads[k].reshape(og.shape)
        scale, err = np.abs(og).max(), np.abs(got - og).max()
        assert err <= 1e-4 * scale or err <= 1e-9, (arch, k, err, scale)
        worst = max(worst, err / scale if err > 1e-9 else 0.0)
    print('%s: loss %.6f (oracle %.6f); backward kernels on the device forward state: worst %.3g of the tensor maximum' % (arch, loss, oloss, worst))


# ------------------------------------------------------------------------------------------------ 4. limits
def test_aggregate_limits_are_refused():
    """Shapes past the compiled limits give an error status before any launch, and B200PoseError through the pipeline:
    more than 32 attention heads (-1), heads * dim / vec > 256 column vectors per row (-3, 'too large'), the frame-resident
    kernel on frames of more than 32 heads (-3)."""
    pan, ring = frame_batch('panoptic'), frame_batch('ring10')
    rng = np.random.default_rng(5)
    for bt, H, D, impl, rc_want, text in ((pan, 33, 2, 0, -1, 'more than 32'), (pan, 1, 257, 0, -3, 'too large'), (pan, 1, 257, 1, -3, 'too large'),
                                          (pan, 4, 260, 1, -3, 'too large'), (pan, 2, 258, 0, -3, 'too large'), (ring, 10, 40, 3, -3, 'impl 3'),
                                          (ring, 4, 30, 5, -3, 'impl 3')):
        z_dev = torch.from_numpy(random_z(rng, bt.N, H, D)).cuda()
        ld = round_up(H * D, 64)
        raw = torch.full((bt.N, H * D), NAN, device='cuda')
        hi = torch.full((bt.N, ld), NAN, dtype=torch.bfloat16, device='cuda')
        rc = run_aggregate(bt, z_dev, H, D, 0, impl, ALPHA, ACT_SLOPE, raw, hi, hi.clone(), ld)
        assert rc == rc_want and text in msg(), (H, D, impl, rc, msg())
        torch.cuda.synchronize()
        assert torch.isnan(raw).all() and torch.isnan(hi.float()).all()
    cfg = pan.cfg
    for hidden, heads, text in (([2], [33], 'more than 32'), ([257], [1], 'too large')):
        pipe = pan.pipe
        layers = pipe.prepare_gat(helpers.weights_mod.make_gat_state(cfg.n_features_sm, 1, True, hidden, heads))
        with pytest.raises(_lib.B200PoseError, match=text):
            pipe.gat_forward(pan.db, pan.g, layers=layers)
    ring.pipe.agg_impl = 3
    try:
        layers = ring.pipe.prepare_gat(helpers.weights_mod.make_gat_state(ring.cfg.n_features_sm, 1, True))
        with pytest.raises(_lib.B200PoseError, match='impl 3'):
            ring.pipe.gat_forward(ring.db, ring.g, layers=layers)
    finally:
        ring.pipe.agg_impl = 0
    torch.cuda.synchronize()
