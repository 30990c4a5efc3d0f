"""CPU: the C-ABI library loads and exports every symbol include/b200pose.h declares; host-side packer."""
import ctypes
import importlib
import json
import os
import re

import numpy as np
import pytest

import helpers
from oracle import pose_oracle as O

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
libmod = importlib.import_module('3d_multi_pose_estimator_b200._lib')
pack = importlib.import_module('3d_multi_pose_estimator_b200.pack')


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(REPO, 'include', 'b200pose.h')).read()
    declared = set(re.findall(r'\b(b200pose_[a-z0-9_]+)\s*\(', header))
    assert len(declared) >= 10
    if not os.path.exists(libmod.LIB_PATH):
        importlib.import_module('3d_multi_pose_estimator_b200.build').build()
    L = ctypes.CDLL(libmod.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), 'missing export ' + name
    assert declared == set(libmod.EXPORTS)
    L.b200pose_last_error.restype = ctypes.c_char_p
    assert L.b200pose_version() >= 100


def test_argument_errors_are_reported_not_fatal():
    L = libmod.lib()
    # null operands: must return an error code and a message, never abort (no GPU needed for validation)
    rc = L.b200pose_linear(None, None, 64, None, None, 64, None, 1, 1, 1, 1.0, 1.0, None, 0, None, None, 0, 0, None)
    assert rc == -1
    assert b'null' in L.b200pose_last_error()
    with pytest.raises(libmod.B200PoseError):
        libmod.check(rc, 'linear')


@pytest.mark.parametrize('impl', [1, 2, 3, 6, 9])
def test_linear_refuses_unknown_impl(impl):
    """b200pose_linear takes impl 0 (dispatch), 4, 5 or 7 only. Anything else is refused before any launch, so the dummy
    pointers below are never dereferenced, with or without a GPU."""
    L = libmod.lib()
    p = ctypes.c_void_p(0x1000)                  # non-null, 16-byte aligned
    rc = L.b200pose_linear(p, p, 64, p, p, 64, p, 4, 64, 64, 1.0, 1.0, p, 64, p, p, 64, impl, None)
    assert rc == -1
    assert re.search(rb'impl must be 0 .*4 .*5 .*or 7 ', L.b200pose_last_error())


def test_pipeline_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip('has a GPU')
    pm = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
    cfg, npz, meta = helpers.load_golden('panoptic')
    with pytest.raises(RuntimeError):
        pm.PosePipeline(cfg, {}, None)


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_packer_matches_oracle_graph_sizes(config):
    cfg, npz, meta = helpers.load_golden(config)
    tabs = O.CameraTables(cfg)
    frames = [meta['frames'][t] for t in meta['cases']]
    frames = [{c: f[c] for c in f if json.loads(f[c][0])} for f in frames]
    pb = pack.pack_frames(frames, cfg)
    assert pb.n_frames == len(frames)
    for b, (tag, f) in enumerate(zip(meta['cases'], frames)):
        g = O.build_graph(f, tabs)
        H = pb.head_off[b + 1] - pb.head_off[b]
        N = pb.node_off[b + 1] - pb.node_off[b]
        if g is None:
            assert N == H                     # no edge-node: the reference builds no graph
            continue
        assert (H, N) == (g['n_heads'], g['n_nodes'])
        cams = pb.sk_cam[pb.head_off[b]:pb.head_off[b + 1]]
        assert np.array_equal([cfg.used_sm.index(c) for c in cams], g['nodes_camera'][:H])
        for h in range(H):
            sk = g['heads_json'][h]
            m = 0
            for j, v in sk.items():
                m |= 1 << int(j)
                assert pb.sk_xy[pb.head_off[b] + h, int(j), 0] == v[1]
            assert pb.sk_mask[pb.head_off[b] + h] == m
            assert pb.skeleton_index[b][h] == g['skeleton_index'][h]
    t = pb.tile(3)
    assert t.n_frames == 3 * pb.n_frames and t.n_nodes == 3 * pb.n_nodes
    s = t.slice(pb.n_frames, 2 * pb.n_frames)
    assert np.array_equal(s.head_off, pb.head_off) and np.array_equal(s.sk_xy, pb.sk_xy)


def test_package_import_widens_the_stream_queues():
    """Importing the package before any CUDA context exists sets CUDA_DEVICE_MAX_CONNECTIONS=32 (the streamed path runs on more
    streams than the default 8 hardware queues) and then defaults to three compute lanes; a value the user chose is kept, and
    with fewer than 16 queues the default falls back to two lanes."""
    import subprocess
    import sys
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import importlib, os; p = importlib.import_module('3d_multi_pose_estimator_b200'); "
            "print(os.environ.get('CUDA_DEVICE_MAX_CONNECTIONS'), p.lanes_ok, p.DEFAULT_LANES)")
    for preset, want in ((None, '32 True 3'), ('8', '8 False 2'), ('64', '64 True 3')):
        env = {k: v for k, v in os.environ.items() if k != 'CUDA_DEVICE_MAX_CONNECTIONS'}
        if preset is not None:
            env['CUDA_DEVICE_MAX_CONNECTIONS'] = preset
        out = subprocess.run([sys.executable, '-c', code], cwd=repo, env=env, stdout=subprocess.PIPE, check=True).stdout.decode().strip()
        assert out.splitlines()[-1] == want, (preset, out)
