"""GPU parity tests: the CUDA path (through the C ABI) against the reference goldens and the oracle.

Tiers (BASELINE.json north_star): graph build / features / clustering / person assignment bit-exact;
edge scores <= 1e-4 relative; 3D joints <= 0.5 mm.
"""
import importlib
import json

import numpy as np
import pytest
import torch

import helpers
from oracle import pose_oracle as O
from oracle import check as OC

pytestmark = pytest.mark.gpu

pipeline_mod = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
pack_mod = importlib.import_module('3d_multi_pose_estimator_b200.pack')

SCORE_RTOL = 1e-4
JOINT_TOL_M = 0.5e-3

_pipes = {}


def get_pipe(config):
    if config not in _pipes:
        cfg, npz, meta = helpers.load_golden(config)
        gat, mlp = helpers.golden_weights(config)
        _pipes[config] = pipeline_mod.PosePipeline(cfg, gat, mlp, device='cuda:0')
    return _pipes[config]


def golden_batch(config, tags=None):
    cfg, npz, meta = helpers.load_golden(config)
    tags = tags or helpers.graph_cases(config)
    frames = []
    for t in tags:
        f = meta['frames'][t]
        frames.append({c: f[c] for c in f if json.loads(f[c][0])})      # metrics_from_model.py:182-191
    pb = pack_mod.pack_frames(frames, cfg)
    return tags, pb, pipeline_mod.HostBatch(pb).to_device('cuda:0')


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_graph_and_features_bit_exact(config):
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    g = pipe.build_graph(db, with_coo=True)
    feats = pipe.node_features_f32(db).cpu().numpy()
    src, dst = g.src.cpu().numpy(), g.dst.cpu().numpy()
    row_ptr, col = g.row_ptr.cpu().numpy(), g.col.cpu().numpy()
    node_cam, pairs = g.node_cam.cpu().numpy(), g.pairs.cpu().numpy()
    for b, tag in enumerate(tags):
        n0, n1 = pb.node_off[b], pb.node_off[b + 1]
        h0, h1 = pb.head_off[b], pb.head_off[b + 1]
        H, M = h1 - h0, (n1 - n0) - (h1 - h0)
        e0 = h0 + 5 * (n0 - h0)
        E = H + 5 * M
        assert n1 - n0 == int(npz[tag + '/n_nodes'])
        assert np.array_equal(src[e0:e0 + E], npz[tag + '/src']), tag
        assert np.array_equal(dst[e0:e0 + E], npz[tag + '/dst']), tag
        assert np.array_equal(node_cam[n0:n1], npz[tag + '/nodes_camera']), tag
        assert np.array_equal(feats[n0:n1], npz[tag + '/feats']), 'features not bit-exact: ' + tag
        # CSR by destination == the COO grouped by dst in edge-id order
        rs, rd = npz[tag + '/src'], npz[tag + '/dst']
        for v in range(n1 - n0):
            want = rs[rd == v] + n0
            got = col[row_ptr[n0 + v]:row_ptr[n0 + v + 1]]
            assert np.array_equal(got, want), (tag, v)
        m0 = n0 - h0
        k = np.arange(M)
        assert np.array_equal(pairs[m0:m0 + M, 0], rs[H + 5 * k]), tag
        assert np.array_equal(pairs[m0:m0 + M, 1], rs[H + 5 * k + 2]), tag
    assert row_ptr[pb.n_nodes] == pb.n_edges


@pytest.mark.parametrize('impl', [4, 5, 7, 0])
def test_linear_kernels(impl):
    """out = act(A W^T + b): the persistent kernel with single CTAs (4) / CTA pairs + cta_group::2 MMAs (5), the few-row
    kernels up to 16 rows (7) and the product dispatch (0) against a float64 reference of the same split operands."""
    pipe = get_pipe('panoptic')
    L = pipe.L
    torch.manual_seed(5)
    shapes = [(1, 54, 1024), (4, 3072, 1260), (8, 1024, 1024), (10, 3072, 3072), (16, 2048, 3072), (13, 54, 1024), (3, 20, 150), (128, 64, 64), (200, 48, 150), (77, 902, 902), (300, 420, 400), (1000, 3, 150), (260, 336, 400),
              (129, 160, 320), (500, 3072, 1260), (64, 54, 1024), (40000, 400, 400), (20481, 902, 902)]
    for (m, n, k) in shapes:
        A = torch.randn(m, k, device='cuda') * 0.7
        W = torch.randn(n, k, device='cuda') / k ** 0.5
        b = torch.randn(n, device='cuda')
        s = pipe._stream()
        Ap, Wp = pipeline_mod.Planes.from_f32(A, s), pipeline_mod.Planes.from_f32(W, s)
        ldo = (n + 3) // 4 * 4                                   # the TMA-store epilogue needs a 16-byte row pitch
        out_buf = torch.full((m, ldo), float('nan'), device='cuda')
        out = out_buf[:, :n]
        outp = pipeline_mod.Planes(m, n, 'cuda')
        outp.hi.fill_(float('nan'))                              # the kernels must write the K padding [n, ld) as zeros
        outp.lo.fill_(float('nan'))
        rc = L.b200pose_linear(pipeline_mod.ptr(Ap.hi), pipeline_mod.ptr(Ap.lo), Ap.ld, pipeline_mod.ptr(Wp.hi),
                               pipeline_mod.ptr(Wp.lo), Wp.ld, pipeline_mod.ptr(b), m, n, k, 0.15, 2.0,
                               pipeline_mod.ptr(out_buf), ldo, pipeline_mod.ptr(outp.hi), pipeline_mod.ptr(outp.lo), outp.ld,
                               impl, s)
        assert rc == 0, ('linear impl %d failed' % impl, rc)
        torch.cuda.synchronize()
        ref = Ap.to_f32().double() @ Wp.to_f32().double().T + b.double()
        ref = torch.where(ref >= 0, ref, ref * 0.15) * 2.0
        err = (out.double() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert err <= 2e-5 * max(scale, 1.0), ('impl %d shape %s: max err %g (scale %g)' % (impl, (m, n, k), err, scale))
        errp = (outp.to_f32().double() - ref).abs().max().item()
        assert errp <= 3e-5 * max(scale, 1.0), ('planes impl %d shape %s: %g' % (impl, (m, n, k), errp))
        if outp.ld > n:
            assert bool((outp.hi[:, n:] == 0).all()) and bool((outp.lo[:, n:] == 0).all()), ('plane padding impl %d shape %s' % (impl, (m, n, k)))


@pytest.mark.parametrize('agg_impl', [0, 1, 2, 3])
@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_gat_scores_vs_reference(config, agg_impl):
    """agg_impl 0: the dispatch (these golden batches are a few frames: large-frame kernel); 1: gather kernel everywhere;
    2: large-frame kernel forced; 3: frame-resident kernel forced (frames of at most 32 heads: panoptic, arp3)."""
    if agg_impl == 3 and config == 'ring10':
        pytest.skip('ring10 golden frames have more than 32 heads: no frame-resident plan')
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    g = pipe.build_graph(db, with_coo=False)
    pipe.agg_impl = agg_impl
    try:
        scores, raws = pipe.gat_forward(db, g, keep_layers=True)
    finally:
        pipe.agg_impl = 0
    scores = scores.cpu().numpy()
    worst = 0.0
    for b, tag in enumerate(tags):
        n0, n1 = pb.node_off[b], pb.node_off[b + 1]
        idx = npz[tag + '/indices']
        ref = npz[tag + '/scores'][idx]
        got = scores[n0:n1][idx]
        rel = np.abs(got - ref) / np.abs(ref)
        worst = max(worst, rel.max())
        assert rel.max() <= SCORE_RTOL, (tag, rel.max())
        for l in range(5):
            key = '%s/gat_l%d' % (tag, l)
            if key in npz:
                a = raws[l][n0:n1].cpu().numpy().reshape(npz[key].shape)
                assert np.abs(a - npz[key]).max() <= 1e-4 * max(1.0, np.abs(npz[key]).max()), (tag, l)
    print('worst relative score error', config, worst)


RESIDUAL_MODELS = {'resfc': ([40, 40, 40, 30], [10, 10, 8, 5], 3), 'ident': ([40, 40], [1, 4], 4)}   # make_golden_residual.py


@pytest.mark.parametrize('dense', [False, True])
@pytest.mark.parametrize('model', sorted(RESIDUAL_MODELS))
def test_gat_residual_vs_reference(model, dense):
    """GAT2 built with residual=True (gat2.py:43-48, 70-75; not the shipped configuration): res_fc projections on the tcgen05
    GEMM, the sum inside the gather aggregation kernel (b200pose_gat_aggregate_res) - against the unmodified reference."""
    import os
    cfg, npz, meta = helpers.load_golden('panoptic')
    res = np.load(os.path.join(helpers.GOLDEN, 'golden_residual.npz'))
    hidden, heads, seed = RESIDUAL_MODELS[model]
    state = helpers.weights_mod.make_gat_state(cfg.n_features_sm, seed, True, hidden, heads, residual=True)
    pipe = get_pipe('panoptic')
    layers = pipe.prepare_gat(state, residual=True)
    assert any('res_w' in l or l.get('res_identity') for l in layers)
    tags, pb, db = golden_batch('panoptic', ['p3', 'rag1'])
    g = pipe.build_graph(db, with_coo=False)
    x0 = pipeline_mod.Planes.from_f32(pipe.node_features_f32(db), pipe._stream()) if dense else None
    scores, raws = pipe.gat_forward(db, g, x0=x0, dense_rows=dense, layers=layers, keep_layers=True)
    scores = scores.cpu().numpy()
    worst = 0.0
    for b, tag in enumerate(tags):
        n0, n1 = pb.node_off[b], pb.node_off[b + 1]
        ref = res['%s/%s/scores' % (model, tag)]
        rel = np.abs(scores[n0:n1] - ref) / np.abs(ref)
        worst = max(worst, rel.max())
        assert rel.max() <= SCORE_RTOL, (model, tag, rel.max())
        for l in range(len(layers)):
            want = res['%s/%s/layer%d' % (model, tag, l)]
            a = raws[l][n0:n1].cpu().numpy().reshape(want.shape)
            assert np.abs(a - want).max() <= 1e-4 * max(1.0, np.abs(want).max()), (model, tag, l)
    print('worst relative score error, residual model', model, worst)


@pytest.mark.parametrize('config', ['panoptic', 'arp3', 'arp6', 'pansub'])
def test_aggregation_kernels_agree_bitwise(config):
    """The frame-resident kernels (shape-specialised product kernel and its generic form) and the gather kernel sum every
    output element in the same order (ascending reference edge id) with the same arithmetic, so their outputs are
    bit-identical: the final scores of the product path (planes out: the specialised kernel) and, with the fp32 layer
    outputs requested (the generic kernels), every layer."""
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    g = pipe.build_graph(db, with_coo=False)
    outs, finals = [], []
    for impl in (3, 6, 5, 1):           # 3 = frame-resident: persistent shape-specialised kernel where the shape is compiled in (a batch this
        pipe.agg_impl = impl            # small would otherwise take the large-frame kernel); 6 = its one-CTA-per-frame form; 5 = generic; 1 = gather
        try:
            finals.append(pipe.gat_forward(db, g).cpu().numpy().copy())
            scores, raws = pipe.gat_forward(db, g, keep_layers=True)
        finally:
            pipe.agg_impl = 0
        outs.append([r.cpu().numpy() for r in raws] + [scores.cpu().numpy()])
    for layer in zip(*outs):
        assert all(np.array_equal(layer[0], x) for x in layer[1:])
    assert all(np.array_equal(finals[0], x) for x in finals[1:])
    assert np.array_equal(finals[0], outs[0][-1])


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_gat_dense_rows_path(config):
    """GAT2.forward as the drop-in calls it: an explicit N x F feature matrix."""
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    g = pipe.build_graph(db, with_coo=False)
    feats = pipe.node_features_f32(db)
    x0 = pipeline_mod.Planes.from_f32(feats, pipe._stream())
    scores = pipe.gat_forward(db, g, x0=x0, dense_rows=True).cpu().numpy()
    for b, tag in enumerate(tags):
        n0, n1 = pb.node_off[b], pb.node_off[b + 1]
        ref = npz[tag + '/scores']
        rel = np.abs(scores[n0:n1] - ref) / np.abs(ref)
        assert rel.max() <= SCORE_RTOL, (tag, rel.max())


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_cluster_on_reference_scores_bit_exact(config):
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    g = pipe.build_graph(db, with_coo=False)
    scores = torch.from_numpy(np.concatenate([npz[t + '/scores'] for t in tags])).cuda()
    ph, npers = pipe.cluster(db, g, scores)
    ph, npers = ph.cpu().numpy(), npers.cpu().numpy()
    for b, tag in enumerate(tags):
        want = npz[tag + '/proposals']
        got = ph[pb.head_off[b]:pb.head_off[b] + npers[b]]
        assert np.array_equal(got, want), (tag, got, want)


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_cluster_fuzz_bit_exact(config):
    """Fuzzed score vectors (ties, all-pass, bimodal, ...) against the reference's own outputs."""
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    fuzz_tags = meta['fuzz_tags']
    tags, pb, db = golden_batch(config, tags=fuzz_tags)
    g = pipe.build_graph(db, with_coo=False)
    scores = torch.from_numpy(np.concatenate([npz['fuzz/%d/scores' % i] for i in range(len(fuzz_tags))])).cuda()
    ph, npers = pipe.cluster(db, g, scores)
    ph, npers = ph.cpu().numpy(), npers.cpu().numpy()
    dup = 0
    for i in range(len(fuzz_tags)):
        want = npz['fuzz/%d/proposals' % i]
        got = ph[pb.head_off[i]:pb.head_off[i] + npers[i]]
        assert np.array_equal(got, want), (i, fuzz_tags[i])
    assert len(fuzz_tags) >= 60


@pytest.mark.parametrize('prefix', ['', 'forced_'])
@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_encoder_mlp_triangulation_vs_reference(config, prefix):
    """Stage 3 on the reference's own proposals ('') and on the forced assignment of the goldens (k-th head of every camera
    = person k: covers every frame, e.g. the narrow-baseline stereo frames of arp6 / arp_robot2 whatever the clustering
    made of them, single-view persons, and cameras that are matched but not used by the pose estimator)."""
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    g = pipe.build_graph(db, with_coo=False)
    rows, owner = [], []
    for b, tag in enumerate(tags):
        if tag + '/' + prefix + 'mlp_in' not in npz:
            continue
        for p, person in enumerate(npz[tag + '/' + prefix + 'proposals']):
            r = np.full(cfg.n_cameras, -1, np.int32)
            for s, h in enumerate(person):
                if h >= 0:
                    r[cfg.used_sm[s]] = pb.head_off[b] + h
            rows.append(r); owner.append((tag, p))
    person_sk = torch.from_numpy(np.stack(rows)).cuda()
    P = len(rows)
    x, valid, xf = pipe.encode_persons(db, P, person_sk, want_f32=True)
    xf = xf.cpu().numpy()
    joints = pipe.mlp_forward(x, P).cpu().numpy()
    # triangulate() works on the views its caller hands it (metrics_from_triangulation.py:237-247); the goldens fed it the
    # pose-estimator cameras of each person
    tri_sk = person_sk.clone()
    tri_sk[:, [c for c in range(cfg.n_cameras) if c not in cfg.used_pe]] = -1
    xyz, mask = pipe.triangulate(db, P, tri_sk)
    xyz, mask = xyz.cpu().numpy(), mask.cpu().numpy()
    valid = valid.cpu().numpy()
    x32 = x.to_f32().cpu().numpy()
    worst_j = worst_t = worst_x = 0.0
    for i, (tag, p) in enumerate(owner):
        key = tag + '/' + prefix
        # the reference raises for a row with sum|v| <= 1 (dataset.py:287-298); the batched path flags it instead
        assert bool(valid[i]) == bool(npz[key + 'enc_ok'][p]), (tag, p)
        if valid[i]:
            ref_in = npz[key + 'mlp_in'][p]
            worst_x = max(worst_x, np.abs(xf[i] - ref_in).max())
            assert np.abs(xf[i] - ref_in).max() <= 1e-6, (tag, p, np.abs(xf[i] - ref_in).max())
            assert (np.abs(x32[i] - ref_in) <= 1e-6 + 2.0 ** -16 * np.abs(ref_in)).all()      # hi + lo bf16 planes: 16 mantissa bits
            ref_j = npz[key + 'mlp_out'][p] * np.float32(10.)
            worst_j = max(worst_j, np.abs(joints[i] - ref_j).max())
            assert np.abs(joints[i] - ref_j).max() <= JOINT_TOL_M, (tag, p)
        assert np.array_equal(mask[i], npz[key + 'tri_mask'][p]), (tag, p)
        d = np.abs(xyz[i] - npz[key + 'tri'][p]).max()
        worst_t = max(worst_t, d)
        assert d <= 1e-7, (tag, p, d)
    assert len(owner) > 0
    print('stage 3 %s%s: %d persons, worst MLP-input deviation %.2e, worst joint deviation %.4f mm, worst triangulation deviation %.2e m'
          % (config, ' (forced)' if prefix else '', len(owner), worst_x, worst_j * 1e3, worst_t))


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_end_to_end_vs_reference(config):
    """Whole path on a ragged batch of the golden frames. Person assignment must equal the reference's; a frame where it
    does not is accepted only with a full attribution (oracle.check.explain_assignment_mismatch): scores within tolerance,
    the oracle clustering of the GPU's scores IS the GPU's assignment, and the reference's sorted matchings hold a gap the
    score tolerance cannot resolve (SURVEY.md 7-2). Everything else fails."""
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    tags, pb, db = golden_batch(config)
    res = pipe.infer(db)
    ph, npers = res['person_heads'].cpu().numpy(), res['n_persons'].cpu().numpy()
    poff = res['person_off'].cpu().numpy()
    joints = res['joints'].cpu().numpy()
    scores = res['scores'].cpu().numpy()
    tabs = O.CameraTables(cfg)
    explained = []
    for b, tag in enumerate(tags):
        want = npz[tag + '/proposals']
        got = ph[pb.head_off[b]:pb.head_off[b] + npers[b]]
        if not np.array_equal(got, want):
            f = meta['frames'][tag]
            og = O.build_graph({c: f[c] for c in f if json.loads(f[c][0])}, tabs)
            why = OC.explain_assignment_mismatch(npz[tag + '/scores'], scores[pb.node_off[b]:pb.node_off[b + 1]], og, cfg, got)
            explained.append((tag, why))
            continue
        if len(want):
            ref_j = npz[tag + '/mlp_out'] * np.float32(10.)
            assert np.abs(joints[poff[b]:poff[b + 1]] - ref_j).max() <= JOINT_TOL_M, tag
    print('end-to-end %s: %d of %d frames equal the reference assignment; explained near-ties: %s' % (config, len(tags) - len(explained), len(tags), explained))
    assert len(explained) < len(tags)


def test_against_oracle_on_fresh_frames():
    """Seeded frames the goldens do not contain: CUDA path vs the oracle on the same inputs."""
    config = 'panoptic'
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    gat_w, mlp_w = helpers.golden_weights(config)
    gat_w, mlp_w = helpers.np_state(gat_w), helpers.np_state(mlp_w)
    tabs = O.CameraTables(cfg)
    frames = [helpers.synth.make_frame(cfg, 500 + i, 2 + i % 4, drop_joint_p=0.1 * (i % 3), drop_view_p=0.1 * (i % 2))
              for i in range(12)]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    pb = pack_mod.pack_frames(frames, cfg)
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    res = pipe.infer(db)
    scores = res['scores'].cpu().numpy()
    ph, npers = res['person_heads'].cpu().numpy(), res['n_persons'].cpu().numpy()
    g = res['graph']
    for b, f in enumerate(frames):
        og = O.build_graph(f, tabs)
        n0, n1 = pb.node_off[b], pb.node_off[b + 1]
        if og is None:
            assert npers[b] == 0
            continue
        os_ = O.gat_forward(gat_w, og['feats'], og['src'], og['dst'])
        idx = og['indices']
        rel = np.abs(scores[n0:n1][idx] - os_[idx]) / np.abs(os_[idx])
        assert rel.max() <= SCORE_RTOL, (b, rel.max())
        # clustering on the GPU's own scores must equal the oracle clustering on the same scores
        props = O.cluster(scores[n0:n1], og['pairs'], og['nodes_camera'][:og['n_heads']], cfg.V_sm, og['n_heads'])
        assert np.array_equal(ph[pb.head_off[b]:pb.head_off[b] + npers[b]], props), b


def test_full_size_properties():
    """BASELINE config 2 size (1024 frames x 4 persons x 5 views): frame-order permutation and batch
    splitting must not change any per-frame result (frames are independent)."""
    config = 'panoptic'
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    base = [helpers.synth.make_frame(cfg, 2000 + i, 4) for i in range(64)]
    base = [{c: f[c] for c in f if json.loads(f[c][0])} for f in base]
    pb64 = pack_mod.pack_frames(base, cfg, keep_json=False)
    pb = pb64.tile(16)
    assert pb.n_frames == 1024
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    res = pipe.infer(db)
    scores = res['scores'].cpu().numpy()
    npers = res['n_persons'].cpu().numpy()
    joints = res['joints'].cpu().numpy()
    poff = res['person_off'].cpu().numpy()
    N64 = pb64.n_nodes
    # every repetition of the 64 frames gives bit-identical scores, counts and joints
    for r in range(1, 16):
        assert np.array_equal(scores[r * N64:(r + 1) * N64], scores[:N64])
        assert np.array_equal(npers[r * 64:(r + 1) * 64], npers[:64])
    P64 = poff[64]
    for r in range(1, 16):
        assert np.array_equal(joints[r * P64:(r + 1) * P64], joints[:P64])
    # a split batch gives the same results as the whole
    half = pipe.infer(pipeline_mod.HostBatch(pb.slice(512, 1024)).to_device('cuda:0'))
    assert np.array_equal(half['scores'].cpu().numpy(), scores[pb.node_off[512]:])
    assert np.array_equal(half['n_persons'].cpu().numpy(), npers[512:])
    assert np.isfinite(joints).all() and npers.sum() > 0
    # the composed full-size run against the oracle: 16 frames spread over the batch (scores, assignment on the GPU's
    # scores, joints) - the kernels the 1024-frame step dispatches, not the small-batch ones
    gat_w, mlp_w = helpers.golden_weights(config)
    gat_w, mlp_w = helpers.np_state(gat_w), helpers.np_state(mlp_w)
    ph = res['person_heads'].cpu().numpy()
    sample = [0, 63, 64, 130, 197, 264, 331, 398, 465, 511, 512, 600, 777, 901, 1000, 1023]
    rep = OC.check_frames(cfg, [base[i % 64] for i in sample], gat_w, mlp_w,
                          [scores[pb.node_off[i]:pb.node_off[i + 1]] for i in sample],
                          [ph[pb.head_off[i]:pb.head_off[i] + npers[i]] for i in sample],
                          [joints[poff[i]:poff[i + 1]] for i in sample])
    print('full-size batch vs oracle:', rep)
    assert rep['persons'] > 0


def test_empty_and_degenerate_batches():
    config = 'panoptic'
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    # frames with all detections in one camera (no graph in the reference) and an empty frame
    f1 = meta['frames']['onecam']
    frames = [{c: f1[c] for c in f1 if json.loads(f1[c][0])}, {}]
    pb = pack_mod.pack_frames(frames, cfg)
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    res = pipe.infer(db)
    assert res['n_persons'].cpu().numpy().tolist() == [0, 0]
    assert res['n_persons_total'] == 0


def test_triangulation_full_size_properties():
    """BASELINE config 4 (triangulation-only: 5 views x 18 joints x 65536 persons): exact projections of known 3D
    points must come back (pairwise DLT is exact for consistent rays), a sample must equal the oracle's cv2-equivalent
    result, and the result must not depend on the position of a person in the batch."""
    config = 'panoptic'
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    rng = np.random.default_rng(7)
    P, C = 65536, cfg.n_cameras
    people = helpers.synth.random_people(cfg, rng, 64)                       # [64,18,3] metres
    xy = np.zeros((64 * C, 18, 2))
    mask = np.zeros(64 * C, dtype=np.uint32)
    for p in range(64):
        for c in range(C):
            uv, z = helpers.synth.project_points(cfg, c, people[p])
            xy[p * C + c] = uv
            mask[p * C + c] = (1 << 18) - 1 if p % 5 else 0x3FFFE                # every 5th person lacks joint 0 in all views
    reps = P // 64
    sk_xy = torch.from_numpy(np.tile(xy, (reps, 1, 1))).cuda()
    sk_mask = torch.from_numpy(np.tile(mask, reps).view(np.int32)).cuda()
    person_sk = torch.arange(P * C, dtype=torch.int32, device='cuda').reshape(P, C)
    # every 7th person is seen by cameras 1 and 3 only, every 11th by one camera only (no triangulation)
    person_sk[::7, 0] = -1; person_sk[::7, 2] = -1; person_sk[::7, 4] = -1
    person_sk[::11, 1:] = -1
    db = pipeline_mod.DeviceBatch(0, P * C, P * C, 0, 0, sk_xy, None, sk_mask, None, None, None)
    xyz, m = pipe.triangulate(db, P, person_sk)
    xyz, m = xyz.cpu().numpy(), m.cpu().numpy()
    psk = person_sk.cpu().numpy()
    n_views = (psk >= 0).sum(1)
    assert np.array_equal(m[n_views < 2], np.zeros_like(m[n_views < 2]))
    seen = n_views >= 2
    want_mask = np.ones((P, 18), np.uint8)
    want_mask[np.arange(P) % 64 % 5 == 0, 0] = 0
    assert np.array_equal(m[seen], want_mask[seen])
    truth = np.tile(people, (reps, 1, 1))
    err = np.abs(xyz - truth)[m.astype(bool)]
    assert err.max() < 1e-4, err.max()                  # limited by the 5 fixed-point undistortion iterations (cv2 behaviour), not by the DLT
    # position independence: identical persons give bit-identical joints
    same = [i for i in range(64, P, 64 * 77) if np.array_equal(psk[i] >= 0, psk[i % 64] >= 0)]
    for i in same[:50]:
        assert np.array_equal(xyz[i], xyz[i % 64])
    # a sample against the oracle
    tabs = O.CameraTables(cfg)
    for p in (1, 7, 14, 33):
        person = {cfg.camera_names[c]: {str(j): [j, xy[(p % 64) * C + c, j, 0], xy[(p % 64) * C + c, j, 1], 1, 1]
                                        for j in range(18) if (mask[(p % 64) * C + c] >> j) & 1}
                  for c in range(C) if psk[p, c] >= 0}
        ref, rm = O.triangulate_baseline(person, tabs, cfg.median_axis)
        assert np.array_equal(rm, m[p])
        assert np.abs(ref - xyz[p]).max() < 1e-9


def test_stress_frame_10_views_16_persons():
    """BASELINE config 5 shape: one 10-view frame with 16 persons (160 heads, 11520 edge-nodes, 57760 edges) next to
    small frames in the same batch - exercises the gather aggregation kernel and the large-frame clustering plan."""
    config = 'ring10'
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    gat_w, mlp_w = helpers.golden_weights(config)
    gat_w, mlp_w = helpers.np_state(gat_w), helpers.np_state(mlp_w)
    tabs = O.CameraTables(cfg)
    frames = [helpers.synth.make_frame(cfg, 4242, 16), helpers.synth.make_frame(cfg, 4243, 2)]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    pb = pack_mod.pack_frames(frames, cfg)
    assert pb.max_heads >= 140 and pb.max_enodes >= 9000
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    res = pipe.infer(db, with_coo=True)
    scores = res['scores'].cpu().numpy()
    ph, npers = res['person_heads'].cpu().numpy(), res['n_persons'].cpu().numpy()
    g = res['graph']
    src, dst = g.src.cpu().numpy(), g.dst.cpu().numpy()
    for b, f in enumerate(frames):
        og = O.build_graph(f, tabs)
        n0, n1 = pb.node_off[b], pb.node_off[b + 1]
        e0 = pb.head_off[b] + 5 * (n0 - pb.head_off[b])
        assert np.array_equal(src[e0:e0 + len(og['src'])], og['src']) and np.array_equal(dst[e0:e0 + len(og['dst'])], og['dst'])
        ref = O.gat_forward(gat_w, og['feats'], og['src'], og['dst'])
        idx = og['indices']
        rel = np.abs(scores[n0:n1][idx] - ref[idx]) / np.abs(ref[idx])
        assert rel.max() <= SCORE_RTOL, (b, rel.max())
        props = O.cluster(scores[n0:n1], og['pairs'], og['nodes_camera'][:og['n_heads']], cfg.V_sm, og['n_heads'])
        assert np.array_equal(ph[pb.head_off[b]:pb.head_off[b] + npers[b]], props), b
    assert np.isfinite(res['joints'].cpu().numpy()).all()


@pytest.mark.parametrize('config,persons,impls', [('ring10', (16, 9, 6, 2, 12), (0, 1)), ('arp6', (8, 6, 7, 3), (0, 1)), ('panoptic', None, (2, 3)), ('arp3', None, (2, 1))])
def test_large_frame_aggregation_agrees_with_other_kernels(config, persons, impls):
    """The large-frame aggregation kernel (staged head rows, cp.async row rings, fixed-reference softmax for heads with
    many in-edges) against the gather / frame-resident kernels, layer by layer: ragged batches of 160-, 90-, 60-,
    20- and 120-head frames where the dispatch picks it (impl 0), and the golden Panoptic / ARP frames with it forced
    (impl 2). It reassociates the heads' sums, so the comparison is to fp32 rounding, not bitwise."""
    pipe = get_pipe(config)
    cfg = pipe.cfg
    if persons is None:
        tags, pb, db = golden_batch(config)
    else:
        frames = [helpers.synth.make_frame(cfg, 777 + i, n) for i, n in enumerate(persons)]
        frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
        pb = pack_mod.pack_frames(frames, cfg)
        assert pb.max_heads > 32                                  # beyond the frame-resident kernels: the dispatch takes the large-frame kernel
        db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    g = pipe.build_graph(db, with_coo=False)
    outs = []
    for impl in impls:
        pipe.agg_impl = impl
        try:
            scores, raws = pipe.gat_forward(db, g, keep_layers=True)
        finally:
            pipe.agg_impl = 0
        outs.append([r.cpu().numpy() for r in raws] + [scores.cpu().numpy()])
    for l, (a, b) in enumerate(zip(*outs)):
        scale = np.abs(b).max()
        assert np.isfinite(a).all()
        assert np.abs(a - b).max() <= 1e-4 * scale, (l, np.abs(a - b).max(), scale)      # 5 layers of fp32 reassociation noise (observed up to 6e-5)
    sa, sb = outs[0][-1], outs[1][-1]
    assert (np.abs(sa - sb) / np.abs(sb)).max() <= 2e-5


def test_cluster_fuzz_large_frames_vs_oracle():
    """Clustering of 160- and 90-head frames (1024-thread plan: compaction, CTA-wide sort, 32-at-a-time rejection tests
    with re-test after a group absorption, parallel link scan) on fuzzed score vectors - uniform, bimodal, all-pass,
    heavy ties, sparse - bit-exact against the oracle's restatement of get_person_proposal_from_network_output."""
    config = 'ring10'
    pipe = get_pipe(config)
    cfg = pipe.cfg
    tabs = O.CameraTables(cfg)
    frames = [helpers.synth.make_frame(cfg, 99, 16), helpers.synth.make_frame(cfg, 100, 9)]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    pb = pack_mod.pack_frames(frames, cfg)
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    g = pipe.build_graph(db, with_coo=False)
    ogs = [O.build_graph(f, tabs) for f in frames]
    rng = np.random.default_rng(5)
    N = int(pb.node_off[-1])
    cases = {
        'uniform': rng.random(N),
        'bimodal': np.where(rng.random(N) < 0.1, 0.5 + 0.5 * rng.random(N), 0.4 * rng.random(N)),
        'all_pass': 0.5 + 0.5 * rng.random(N),
        'ties': np.round(rng.random(N) * 8) / 8,
        'sparse': np.where(rng.random(N) < 0.01, 0.9, 0.1),
        'none': np.full(N, 0.5),
    }
    for name, sc in cases.items():
        sc = sc.astype(np.float32)
        ph, npers = pipe.cluster(db, g, torch.from_numpy(sc).cuda())
        ph, npers = ph.cpu().numpy(), npers.cpu().numpy()
        for b, og in enumerate(ogs):
            n0, n1 = pb.node_off[b], pb.node_off[b + 1]
            props = O.cluster(sc[n0:n1], og['pairs'], og['nodes_camera'][:og['n_heads']], cfg.V_sm, og['n_heads'])
            got = ph[pb.head_off[b]:pb.head_off[b] + npers[b]]
            assert np.array_equal(got, props), (name, b, len(got), len(props))


def test_host_api_variants_agree():
    """The public host entry points - infer_host (one chunk and several), infer_host_stream, and the native JSON packer
    feeding them - return exactly what infer() computes on the same frames, in frame order with batch-global indices."""
    config = 'panoptic'
    cfg, npz, meta = helpers.load_golden(config)
    pipe = get_pipe(config)
    frames = [helpers.synth.make_frame(cfg, 7000 + i, 1 + i % 5, drop_view_p=0.15 * (i % 3)) for i in range(37)]
    frames[5] = {}                                                          # an empty frame in the middle
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    pb = pack_mod.pack_frames(frames, cfg, keep_json=False)
    hb = pipeline_mod.HostBatch(pb)
    ref = pipe.infer(hb.to_device('cuda:0'))
    want = dict(n_persons=ref['n_persons'].cpu().numpy(), person_off=ref['person_off'].cpu().numpy(),
                person_sk=ref['person_sk'].cpu().numpy(), joints=ref['joints'].cpu().numpy(), valid=ref['valid'].cpu().numpy())

    def check(out, exact=True):
        assert out['n_persons_total'] == ref['n_persons_total']
        for k, v in want.items():
            if k == 'joints' and not exact:      # few-person chunks take the small-m projection kernel: other summation order
                assert np.abs(np.asarray(out[k]) - v).max() <= 1e-5, k
            else:
                assert np.array_equal(np.asarray(out[k]), v), k

    check(pipe.infer_host(hb))
    for n_chunks in (2, 3, 37):
        check(pipe.infer_host(hb, n_chunks=n_chunks), exact=False)
    outs = list(pipe.infer_host_stream([hb, hb, hb]))
    assert len(outs) == 3
    check(outs[-1])
    # native packer + pinned buffers
    pb2 = pack_mod.pack_json(json.dumps(frames), cfg, pinned=True)
    check(pipe.infer_host(pipeline_mod.HostBatch(pb2)))
    # a stream of different batches comes back in order
    halves = [pipeline_mod.HostBatch(pb.slice(0, 20)), pipeline_mod.HostBatch(pb.slice(20, 37))]
    a, b2 = [dict(n_persons=np.asarray(o['n_persons']).copy(), joints=np.asarray(o['joints']).copy()) for o in pipe.infer_host_stream(halves)]
    assert np.array_equal(np.concatenate([a['n_persons'], b2['n_persons']]), want['n_persons'])
    assert np.abs(np.concatenate([a['joints'], b2['joints']]) - want['joints']).max() <= 1e-5


def test_stream_lanes_keep_order_and_results():
    """infer_host_stream over eleven DIFFERENT batches (ragged sizes, one of them a single frame) with 1, 2, 3 and 4 compute
    lanes: the yielded results come back in order and equal infer_host of each batch - counts and assignments exactly, joints
    to 1e-5 m (a few-person batch takes the small-m projection kernel in infer_host and the capacity-sized launch in the
    stream: other summation order) and bit-for-bit between lane counts - also when the caller holds on to yielded results
    while the stream runs ahead (results stay valid for two further batches)."""
    config = 'panoptic'
    pipe = get_pipe(config)
    cfg = pipe.cfg
    rng = np.random.default_rng(9)
    sizes = [int(x) for x in rng.integers(2, 24, size=10)] + [1]
    frames = [helpers.synth.make_frame(cfg, 900 + i, 1 + i % 5, drop_view_p=0.1 * (i % 3)) for i in range(sum(sizes))]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    hbs, o = [], 0
    for n in sizes:
        hbs.append(pipeline_mod.HostBatch(pack_mod.pack_frames(frames[o:o + n], cfg)))
        o += n
    want = []
    for hb in hbs:
        r = pipe.infer_host(hb)
        want.append({k: np.asarray(r[k]).copy() for k in ('n_persons', 'person_sk', 'joints', 'valid')})
    first = None
    for lanes in (1, 2, 3, 4):
        got = []
        for out in pipe.infer_host_stream(hbs, lanes=lanes):
            got.append({k: np.asarray(out[k]).copy() for k in ('n_persons', 'person_sk', 'joints', 'valid')})
        assert len(got) == len(want)
        for i, (g, w) in enumerate(zip(got, want)):
            for k in w:
                if k == 'joints':
                    assert g[k].shape == w[k].shape and (g[k].size == 0 or np.abs(g[k] - w[k]).max() <= 1e-5), (lanes, i, k)
                else:
                    assert np.array_equal(g[k], w[k]), (lanes, i, k)
        if first is None:
            first = got
        else:
            assert all(np.array_equal(a['joints'], b['joints']) for a, b in zip(first, got)), lanes
    held = list(pipe.infer_host_stream(hbs[:3], lanes=3))                 # three results held without copying
    for g, w in zip(held[-2:], first[1:3]):
        assert np.array_equal(np.asarray(g['joints']), w['joints'])
    # a twin owns its streams: one made after the stream ran does not share the pipeline's counts stream
    assert pipe.twin()._aux_stream('counts') is not pipe._aux_stream('counts')


def test_cuda_graph_host_path_matches_eager():
    """infer_host_graph (one CUDA graph per batch shape, no host wait inside the step) against infer_host: same persons,
    same skeleton assignment, same joints - on first sight of a shape (capture), on replays with other frames of the same
    shape, on a multi-frame batch, and on the degenerate shapes it hands to the eager path."""
    config = 'panoptic'
    pipe = get_pipe(config)
    cfg = pipe.cfg
    frames = [helpers.synth.make_frame(cfg, 600 + i, 4) for i in range(6)] + [helpers.synth.make_frame(cfg, 700, 3, drop_view_p=0.3)]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    batches = [pack_mod.pack_frames([f], cfg) for f in frames] + [pack_mod.pack_frames(frames[:3], cfg),
                                                                   pack_mod.pack_frames([{}], cfg)]
    keys = set()
    for rep in range(2):                                                # second round: every shape replays its graph
        for pb in batches:
            hb = pipeline_mod.HostBatch(pb)
            want = {k: (v.clone() if hasattr(v, 'clone') else v) for k, v in pipe.infer_host(hb).items()}
            got = pipe.infer_host_graph(hb)
            keys.add((pb.n_frames, pb.n_heads, pb.n_nodes))
            assert got['n_persons_total'] == want['n_persons_total']
            assert torch.equal(got['n_persons'], want['n_persons']) and torch.equal(got['person_off'], want['person_off'])
            assert torch.equal(got['person_sk'], want['person_sk'])
            if want['n_persons_total']:
                assert torch.equal(got['valid'].bool(), want['valid'].bool())
                assert (got['joints'] - want['joints']).abs().max().item() <= 1e-5
    graphs = pipe._own.graphs
    assert len(graphs) >= 2 and len(graphs) <= len(keys)
    # a replay that finds more persons than the captured capacity falls back to the eager path and re-captures next time
    hb = pipeline_mod.HostBatch(batches[0])
    want = {k: (v.clone() if hasattr(v, 'clone') else v) for k, v in pipe.infer_host(hb).items()}
    key = next(k for k in graphs if k[0] == 1 and k[1] == batches[0].n_heads and k[2] == batches[0].n_nodes)
    assert want['n_persons_total'] > 0
    graphs[key]['p_cap'] = 0
    got = pipe.infer_host_graph(hb)
    assert key not in graphs and got['n_persons_total'] == want['n_persons_total']
    assert torch.equal(got['person_sk'], want['person_sk']) and torch.equal(got['joints'], want['joints'])
    got = pipe.infer_host_graph(hb)                                     # captured again, capacity from the remembered count
    assert key in graphs and graphs[key]['p_cap'] >= want['n_persons_total']
    assert torch.equal(got['person_sk'], want['person_sk']) and (got['joints'] - want['joints']).abs().max().item() <= 1e-5


def test_cabi_argument_errors_on_device():
    """Error behaviour of the C ABI with real device buffers: a bad argument is a negative status with a message that
    names the call, nothing is launched, and the next valid call works (no sticky state)."""
    import ctypes as C
    pipe = get_pipe('panoptic')
    L, ptr = pipe.L, pipeline_mod.ptr
    tags, pb, db = golden_batch('panoptic')
    g = pipe.build_graph(db, with_coo=False)
    lay = pipe.gat[1]
    z = torch.zeros(db.n_nodes, lay['ldz'], device='cuda')
    act = pipe.planes_ws('err_act', db.n_nodes, lay['hd'])
    st = pipe._stream()

    def agg(ldz=None, impl=0, ld_planes=None, z_t=z):
        return L.b200pose_gat_aggregate(db.n_frames, db.n_nodes, db.n_heads, ptr(db.head_off), ptr(db.node_off), ptr(g.row_ptr), ptr(g.col),
                                        ptr(z_t), lay['ldz'] if ldz is None else ldz, lay['heads'], lay['dim'], 0, db.max_heads, db.max_enodes,
                                        0.15, 0.01, None, ptr(act.hi), ptr(act.lo), act.ld if ld_planes is None else ld_planes, None, impl, st)
    msg = lambda: (L.b200pose_last_error() or b'').decode()
    assert agg(ldz=lay['ldz'] + 1) == -1 and 'gat_aggregate' in msg()                 # row pitch not a multiple of 4
    assert agg(ld_planes=act.ld + 8) == -1 and 'ld_planes' in msg()
    assert agg(impl=9) == -1 and 'impl' in msg()
    assert agg(z_t=None) == -1
    assert agg() == 0
    scores = torch.rand(db.n_nodes, device='cuda')
    ph = torch.empty((db.n_heads, pipe.cfg.V_sm), dtype=torch.int32, device='cuda')
    npers = torch.empty(db.n_frames, dtype=torch.int32, device='cuda')
    cl = lambda v_sm, pairs: L.b200pose_cluster(db.n_frames, ptr(db.head_off), ptr(db.node_off), pairs, ptr(g.node_cam), ptr(scores), v_sm,
                                                 0.5, 2, db.max_heads, db.max_enodes, ptr(ph), ptr(npers), st)
    assert cl(33, ptr(g.pairs)) == -1 and 'v_sm' in msg()
    assert cl(pipe.cfg.V_sm, None) == -1 and 'null' in msg()
    assert cl(pipe.cfg.V_sm, ptr(g.pairs)) == 0
    # a frame plan beyond the compiled limits is "unsupported", not a crash: 40000 heads in one frame
    big = L.b200pose_cluster(1, ptr(db.head_off), ptr(db.node_off), ptr(g.pairs), ptr(g.node_cam), ptr(scores), pipe.cfg.V_sm, 0.5, 2,
                             40000, 1 << 24, ptr(ph), ptr(npers), st)
    assert big == -3 and 'too large' in msg()
    assert L.b200pose_build_graph_pairs(1, ptr(db.head_off), ptr(db.node_off), ptr(db.sk_cam), pipe.cams.ref, None, db.max_heads,
                                        None, None, ptr(g.row_ptr), ptr(g.col), ptr(g.node_cam), st) == -1
    A = pipeline_mod.Planes.from_f32(torch.randn(4, 64, device='cuda'), st)
    out = torch.empty(4, 8, device='cuda')
    lin = lambda ldo: L.b200pose_linear(ptr(A.hi), ptr(A.lo), A.ld, ptr(A.hi), ptr(A.lo), A.ld, None, 200, 8, 64, 1.0, 1.0, ptr(out), ldo,
                                        None, None, 0, 4, st)
    assert lin(7) == -1 and 'linear' in msg()                                            # TMA store needs a 16-byte row pitch
    torch.cuda.synchronize()
    assert pipe.infer(db)['n_persons_total'] >= 0


def test_infer_frames_from_reference_dicts():
    """infer_frames (reference frame dicts -> native packing -> CUDA-graph replay) returns what infer_host returns for the
    same frames packed by the Python packer."""
    pipe = get_pipe('panoptic')
    cfg = pipe.cfg
    frames = [helpers.synth.make_frame(cfg, 820 + i, 4, drop_joint_p=0.1) for i in range(4)]
    for batch in ([frames[0]], [frames[1]], frames, frames[2]):
        want_frames = batch if isinstance(batch, list) else [batch]
        want = pipe.infer_host(pipeline_mod.HostBatch(pack_mod.pack_frames([{c: f[c] for c in f} for f in want_frames], cfg)))
        want = {k: (v.clone() if hasattr(v, 'clone') else v) for k, v in want.items()}
        got = pipe.infer_frames(batch)
        assert got['n_persons_total'] == want['n_persons_total']
        assert torch.equal(got['person_sk'], want['person_sk']) and torch.equal(got['person_off'], want['person_off'])
        if want['n_persons_total']:
            assert (got['joints'] - want['joints']).abs().max().item() <= 1e-5


def test_result_record_kernel_matches_host_packing():
    """The multi-GPU result record written by one kernel behind the step (b200pose_pack_record, person count read on the
    device) holds what the eager packing (sharding.pack_record: the layout the gloo tests exchange) writes, and unpacks to
    the step's results; ResultGather keeps `depth` records in flight."""
    sharding = importlib.import_module('3d_multi_pose_estimator_b200.sharding')
    pipe = get_pipe('panoptic')
    cfg = pipe.cfg
    tags, pb, db = golden_batch('panoptic')
    res = pipe.infer(db)
    P = res['n_persons_total']
    assert P > 0
    F, Fcap, Pcap = pb.n_frames, pb.n_frames + 3, pipeline_mod.person_capacity(pb.n_heads, cfg.min_number_of_views)
    want = sharding.pack_record(res['n_persons'], res['person_sk'], res['joints'], Fcap, Pcap, cfg.n_cameras, 54, head_base=1000)
    words = sharding.record_words(Fcap, Pcap, cfg.n_cameras, 54)
    got = torch.full((words,), -7, dtype=torch.int32, device='cuda')
    sharding.pack_record_device(res, F, Fcap, Pcap, cfg.n_cameras, 54, got, head_base=1000, stream=pipe._stream())
    torch.cuda.synchronize()
    a = sharding.unpack_records(got.reshape(1, -1), [F], Fcap, Pcap, cfg.n_cameras, 54)
    b = sharding.unpack_records(want.reshape(1, -1), [F], Fcap, Pcap, cfg.n_cameras, 54)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a['joints'], res['joints'].cpu().numpy()) and a['n_persons'].tolist() == res['n_persons'].cpu().tolist()
    g = sharding.ResultGather(1, Fcap, Pcap, cfg.n_cameras, 54, 'cuda', depth=2)
    for i in range(5):
        g.submit(res, F, head_base=i, stream=pipe._stream())
    outs = g.finish()
    torch.cuda.synchronize()
    assert len(outs) == 2
    last = sharding.unpack_records(outs[-1], [F], Fcap, Pcap, cfg.n_cameras, 54)
    sk = res['person_sk'].cpu().numpy()
    assert np.array_equal(last['person_sk'], np.where(sk >= 0, sk + 4, sk))


def test_persistent_aggregation_ragged_batch_bitwise():
    """The persistent aggregation kernel walks several frames per CTA (more frames than SMs) with the table sets of
    consecutive frames double-buffered: a ragged batch - 1 to 6 persons, missing views, frames without detections or with one
    camera only in between - must give bit for bit the scores of the gather kernel and of the one-CTA-per-frame kernel."""
    pipe = get_pipe('panoptic')
    cfg = pipe.cfg
    base = []
    for i in range(61):
        if i % 13 == 5:
            base.append({})                                                 # no detections at all
        elif i % 17 == 3:
            base.append(helpers.synth.make_frame(cfg, 3000 + i, 3, camera_order=[i % 5]))      # one camera: heads but no edge-node
        else:
            base.append(helpers.synth.make_frame(cfg, 3000 + i, 1 + i % 6, drop_view_p=0.1 * (i % 4), drop_joint_p=0.05 * (i % 3)))
    base = [{c: f[c] for c in f if json.loads(f[c][0])} for f in base]
    pb = pack_mod.pack_frames(base, cfg, keep_json=False).tile(9)            # 549 frames: 3.7 per SM, uneven
    db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
    g = pipe.build_graph(db, with_coo=False)
    outs = []
    for impl in (3, 6, 1):
        pipe.agg_impl = impl
        try:
            outs.append(pipe.gat_forward(db, g).cpu().numpy().copy())
        finally:
            pipe.agg_impl = 0
    assert np.isfinite(outs[0]).all()
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    again = pipe.gat_forward(db, g).cpu().numpy()                          # the dispatch (549 frames: persistent kernel), run to run
    assert np.array_equal(again, outs[0])


def test_sync_free_step_matches_the_synchronous_one():
    """infer(sync=False) launches stage 3 for the person capacity and lets the kernels read the count from the device
    (b200pose_encode_persons_n / b200pose_linear_n): same persons, same assignment and - bit for bit - the same joints as the
    step that reads the count back, on a ragged batch, on a batch without any person, and at the full 1024-frame size."""
    pipe = get_pipe('panoptic')
    cfg = pipe.cfg
    frames = [helpers.synth.make_frame(cfg, 9100 + i, 1 + i % 5, drop_view_p=0.1 * (i % 3)) for i in range(40)] + [{}]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    small = pack_mod.pack_frames(frames, cfg, keep_json=False)
    none = pack_mod.pack_frames([{c: v for c, v in frames[0].items() if c == list(frames[0])[0]}], cfg, keep_json=False)   # one camera: no person
    for pb in (small, none, small.tile(25)):
        db = pipeline_mod.HostBatch(pb).to_device('cuda:0')
        want = pipe.infer(db)
        got = pipe.infer(db, sync=False)
        P = pipeline_mod.PosePipeline.person_count(got)
        assert P == want['n_persons_total']
        assert torch.equal(got['n_persons'], want['n_persons']) and torch.equal(got['person_off'], want['person_off'])
        if P:
            assert torch.equal(got['person_sk'][:P], want['person_sk'])
            assert torch.equal(got['valid'][:P], want['valid'])
            assert torch.equal(got['joints'][:P], want['joints'])
