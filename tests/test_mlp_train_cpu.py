"""CPU: host logic of the pose-estimator MLP's training step - the flat parameter layout (3d_multi_pose_estimator_b200/train.py,
mlp_param_layout) against the reference's state-dict keys (utils/mlp.py via weights.make_mlp_state) and its refusals - and the
fp64 oracle the GPU tests differentiate: an nn.Sequential restatement of utils/mlp.py that reproduces what the unmodified
reference recorded, so its autograd gives the reference's gradients."""
import importlib

import numpy as np
import pytest
import torch

import helpers

train_mod = importlib.import_module('3d_multi_pose_estimator_b200.train')


def oracle_mlp(state, dtype=torch.float64):
    """utils/mlp.py:8-31 as a plain nn.Sequential (Flatten, Linear, LeakyReLU(0.1) x 8, Linear) holding `state`."""
    dims = [state['layers.1.weight'].shape[1]] + [state['layers.%d.weight' % j].shape[0] for j in train_mod.MLP_LAYER_INDICES]
    mods = [torch.nn.Flatten()]
    for i in range(9):
        mods.append(torch.nn.Linear(dims[i], dims[i + 1]))
        if i < 8:
            mods.append(torch.nn.LeakyReLU(0.1))
    net = torch.nn.Sequential(*mods).to(dtype)
    net.load_state_dict({k[len('layers.'):]: v.to(dtype) for k, v in state.items()})     # nn.Sequential keys: '1.weight', ...
    return net


def _in_dims():
    return sorted({helpers.load_golden(c)[2]['mlp_in_dim'] for c in helpers.CONFIGS})


@pytest.mark.parametrize('in_dim', _in_dims())
def test_mlp_param_layout_covers_the_reference_state_dict(in_dim):
    state = helpers.weights_mod.make_mlp_state(in_dim, 54, 1)
    shapes = {k: tuple(v.shape) for k, v in state.items()}
    layers, slots, n = train_mod.mlp_param_layout(shapes)
    assert sorted(slots) == sorted(shapes)
    assert [(l['k'], l['n']) for l in layers] == list(zip((in_dim,) + helpers.weights_mod.MLP_HIDDEN, helpers.weights_mod.MLP_HIDDEN + (54,)))
    spans = []
    for key, (off, rows, cols, ld) in slots.items():
        assert off % 4 == 0 and ld % 4 == 0 and ld >= cols and ld - cols < 4, key          # 16-byte aligned rows (TMA store pitch)
        assert rows * cols == int(np.prod(shapes[key])), key
        spans.append((off, off + rows * ld, key))
    spans.sort()
    assert spans[0][0] == 0 and spans[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))                                # contiguous, no overlap
    # each weight slot is followed by its own bias (the fused optimiser kernel updates the floats after a weight slot element-wise)
    assert [k for _, _, k in spans] == ['layers.%d.%s' % (j, w) for j in train_mod.MLP_LAYER_INDICES for w in ('weight', 'bias')]
    n_params = sum(int(np.prod(s)) for s in shapes.values())
    assert n_params <= n <= n_params + 4 * sum(r for _, r, _, _ in slots.values())
    if in_dim == 1260:
        assert n_params == 29106230                                                           # the Panoptic model: 29.1 M parameters


def test_mlp_param_layout_refusals():
    shapes = {k: tuple(v.shape) for k, v in helpers.weights_mod.make_mlp_state(756, 54, 1).items()}
    with pytest.raises(ValueError):                                        # a missing bias
        train_mod.mlp_param_layout({k: v for k, v in shapes.items() if k != 'layers.5.bias'})
    with pytest.raises(ValueError):                                        # a missing layer
        train_mod.mlp_param_layout({k: v for k, v in shapes.items() if not k.startswith('layers.17.')})
    bad = dict(shapes)
    bad['layers.3.weight'] = (3072, 3000)                                  # widths that do not chain
    with pytest.raises(ValueError):
        train_mod.mlp_param_layout(bad)
    bad = dict(shapes)
    bad['layers.5.bias'] = (2047,)                                         # a bias of the wrong width
    with pytest.raises(ValueError):
        train_mod.mlp_param_layout(bad)
    for extra in ('layers.19.weight', 'layers.2.weight', 'head.weight'):   # keys outside the pattern
        with pytest.raises(ValueError):
            train_mod.mlp_param_layout(dict(shapes, **{extra: (54, 54)}))


@pytest.mark.parametrize('config', helpers.CONFIGS)
def test_fp64_oracle_reproduces_the_reference_mlp(config):
    """The fp64 nn.Sequential with the golden weights gives the unmodified reference's recorded MLP outputs on every golden frame
    (own and forced proposals), to 0.5 mm on the x10 joints the drivers report."""
    cfg, npz, meta = helpers.load_golden(config)
    net = oracle_mlp(helpers.golden_weights(config)[1])
    checked = 0
    for key in npz.files:
        if not key.endswith('mlp_in'):
            continue
        x = torch.from_numpy(npz[key].astype(np.float64))
        want = npz[key[: -len('mlp_in')] + 'mlp_out'].astype(np.float64)
        with torch.no_grad():
            got = net(x).numpy()
        assert np.abs(got - want).max() * 10 < 5e-4, (config, key, np.abs(got - want).max())
        checked += x.shape[0]
    assert checked > 0


def test_reference_module_gives_the_oracle_gradients():
    """With the reference tree staged, its own utils/mlp.py (PoseEstimatorMLP) under fp64 autograd gives the oracle's output and
    every gradient of a seeded loss."""
    from oracle import ref_env
    if not ref_env.reference_available():
        pytest.skip('reference tree not staged')
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location('_reference_mlp', os.path.join(ref_env.REFERENCE_ROOT, 'utils', 'mlp.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    state = helpers.weights_mod.make_mlp_state(504, 54, 12)
    ref = mod.PoseEstimatorMLP(504, 54).double()
    ref.load_state_dict({k: v.double() for k, v in state.items()})
    ora = oracle_mlp(state)
    g = torch.Generator().manual_seed(2)
    x, dy = torch.randn(6, 504, generator=g, dtype=torch.float64), torch.randn(6, 54, generator=g, dtype=torch.float64)
    outs = []
    for net in (ref, ora):
        out = net(x)
        (out * dy).sum().backward()
        outs.append(out.detach())
    assert torch.allclose(outs[0], outs[1], rtol=1e-12, atol=1e-14)
    ora_grads = {'layers.' + k: p.grad for k, p in ora.named_parameters()}
    for k, p in ref.named_parameters():
        assert torch.allclose(p.grad, ora_grads[k], rtol=1e-12, atol=1e-14), k
