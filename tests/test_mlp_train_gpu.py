"""GPU: the training step of the pose-estimator MLP (utils/mlp.py:8-31) on the B200 path.

* MlpGrad's backward (csrc/train.cu plane / column-sum kernels + the split-bf16 tensor-core GEMM) against the fp64 oracle of
  tests/test_mlp_train_cpu.py over batch sizes that exercise the few-row kernels, tile edges and CTA pairs, at three input widths;
* the fused optimiser kernel b200pose_mlp_adam_planes against b200pose_adam_step_dev + b200pose_split_planes, bit for bit;
* MlpTrainer against fp64 torch autograd + torch.optim.Adam, the captured step against the eager one;
* the drop-in PoseEstimatorMLP under the reference-style loop (loss.backward(), Adam.step()) against an fp32 nn.Sequential twin.
"""
import functools
import importlib

import numpy as np
import pytest
import torch

import dropin_env
import helpers
from test_mlp_train_cpu import oracle_mlp

pytestmark = pytest.mark.gpu

pipeline_mod = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
train_mod = importlib.import_module('3d_multi_pose_estimator_b200.train')
_lib = importlib.import_module('3d_multi_pose_estimator_b200._lib')
SLOPE = 0.1


@functools.lru_cache(maxsize=None)
def _pipe():
    cfg, _, _ = helpers.load_golden('panoptic')
    return pipeline_mod.PosePipeline(cfg, None, None, device='cuda:0')


@functools.lru_cache(maxsize=None)
def _net(width):
    state = helpers.weights_mod.make_mlp_state(width, 54, 7)
    return state, train_mod.MlpGrad(_pipe(), state), oracle_mlp(state).cuda()


def _oracle_on_device_state(state, xs, dy):
    """The oracle's backward in fp64 with the forward state pinned to what the device kept (every layer's input and the sign of
    every activated output): autograd of utils/mlp.py layer by layer. This is the fp64 oracle's gradient with no LeakyReLU mask
    flipped by the forward's ~1e-5 differences, so what remains to compare is the arithmetic of the backward."""
    grads = {}
    d = dy.double()
    for i in range(8, -1, -1):
        j = train_mod.MLP_LAYER_INDICES[i]
        W = state['layers.%d.weight' % j].double().cuda()
        if i < 8:
            d = d * torch.where(xs[i + 1] > 0, 1.0, SLOPE)
        grads['layers.%d.weight' % j] = d.t() @ xs[i]
        grads['layers.%d.bias' % j] = d.sum(0)
        d = d @ W
    return grads


@pytest.mark.parametrize('width', [504, 1260, 2520])
@pytest.mark.parametrize('P', [1, 8, 9, 16, 17, 255, 256, 257, 1000])
def test_mlp_backward_vs_fp64_oracle(width, P):
    state, net, ora = _net(width)
    g = torch.Generator().manual_seed(1000 * P + width)
    x = torch.randn(P, width, generator=g).cuda()
    dy = torch.randn(P, 54, generator=g).cuda()
    out = net.forward(x)
    net.backward(dy)
    torch.cuda.synchronize()
    grads = {k: v.double() for k, v in net.grads().items()}
    xs = [p.to_f32()[:P].double() for p in net.cache['xs']]
    # forward: the fp64 oracle's output within the inference bar (0.5 mm on the x10 joints)
    with torch.no_grad():
        assert (out.double() - ora(x.double())).abs().max().item() * 10 < 5e-4
    worst = 0.0
    for k, ref in _oracle_on_device_state(state, xs, dy).items():
        err, scale = (grads[k] - ref).abs().max().item(), ref.abs().max().item()
        assert err <= 1e-4 * scale, (k, err, scale)
        worst = max(worst, err / scale)
    # end to end against plain fp64 autograd (masks from the oracle's own forward): a pre-activation within the forward's ~1e-5
    # difference of zero flips its LeakyReLU mask, which changes that row's gradient by (1 - slope) times a dense vector in every
    # layer below it. The first layer collects all of them: at a few rows its relative L2 error reaches a few per cent (3.4e-2 for
    # layers.1.weight at P = 9, width 504, on a B200), where a wrong backward would be off by O(1); with no flip, ~1e-5
    xd = x.double()
    ora.zero_grad()
    (ora(xd) * dy.double()).sum().backward()
    worst_l2 = 0.0
    for name, p in ora.named_parameters():
        k = 'layers.' + name
        l2 = ((grads[k] - p.grad).norm() / p.grad.norm()).item()
        assert l2 <= 1e-1, (k, l2)
        worst_l2 = max(worst_l2, l2)
    print('width %d, P = %d: worst gradient error on the device forward state %.3g of the tensor maximum; end to end worst relative L2 %.3g'
          % (width, P, worst, worst_l2))


def _split(x, rows, cols, ld_in, ld):
    hi = torch.full((rows, ld), float('nan'), dtype=torch.bfloat16, device='cuda')
    lo = hi.clone()
    _lib.check(_lib.lib().b200pose_split_planes(_lib.ptr(x), rows, cols, ld_in, _lib.ptr(hi), _lib.ptr(lo), ld, None), 'split_planes')
    return hi, lo


@pytest.mark.parametrize('wd', [0.0, 1e-2])
def test_fused_adam_planes_bit_identical(wd):
    """b200pose_mlp_adam_planes over 3 steps: theta, m, v and the step count bit-identical to b200pose_adam_step_dev; every
    plane bit-identical to b200pose_split_planes of the updated weight (W) and of its transpose (W^T), paddings included (the
    planes are filled with NaN before each call); grad = null rebuilds the planes and leaves theta, m, v untouched."""
    state = helpers.weights_mod.make_mlp_state(504, 54, 3)
    net = train_mod.MlpGrad(_pipe(), state)
    L, ptr = _lib.lib(), _lib.ptr
    n = net.n_flat
    gen = torch.Generator(device='cuda').manual_seed(11)
    m, v = torch.zeros(n, device='cuda'), torch.zeros(n, device='cuda')
    t_dev, scal = torch.zeros(1, dtype=torch.int32, device='cuda'), torch.zeros(2, device='cuda')
    th_r, m_r, v_r = net.theta.clone(), m.clone(), v.clone()
    t_r, scal_r = t_dev.clone(), scal.clone()
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=wd)
    for step in range(3):
        grad = torch.randn(n, generator=gen, device='cuda') * 1e-3
        for lay in net.layers:
            for p in (lay['w'], lay['wt']):
                if p is not None:
                    p.hi.fill_(float('nan')); p.lo.fill_(float('nan'))
        net.adam_planes(grad, m, v, t_dev=t_dev, scalars=scal, **hp)
        _lib.check(L.b200pose_adam_step_dev(ptr(th_r), ptr(grad), ptr(m_r), ptr(v_r), n, hp['lr'], 0.9, 0.999, 1e-8, wd, ptr(t_r), ptr(scal_r), None),
                   'adam_step_dev')
        torch.cuda.synchronize()
        assert torch.equal(net.theta, th_r) and torch.equal(m, m_r) and torch.equal(v, v_r), step
        assert int(t_dev.item()) == int(t_r.item()) == step + 1 and torch.equal(scal, scal_r)
        for i, lay in enumerate(net.layers):
            W = net.view(net.theta, 'layers.%d.weight' % train_mod.MLP_LAYER_INDICES[i])
            nn_, k = lay['n'], lay['k']
            hi, lo = _split(W, nn_, k, W.stride(0), lay['w'].ld)
            assert torch.equal(lay['w'].hi.view(torch.int16), hi.view(torch.int16)) and torch.equal(lay['w'].lo.view(torch.int16), lo.view(torch.int16)), (step, i)
            if i == 0:
                assert lay['wt'] is None
                continue
            WT = W.t().contiguous()
            hi, lo = _split(WT, k, nn_, nn_, lay['wt'].ld)
            assert torch.equal(lay['wt'].hi.view(torch.int16), hi.view(torch.int16)) and torch.equal(lay['wt'].lo.view(torch.int16), lo.view(torch.int16)), (step, i)
            assert lay['wt'].ld == pipeline_mod.round_up(nn_, 64)
    th0, m0, v0, t0 = net.theta.clone(), m.clone(), v.clone(), t_dev.clone()
    w_before = net.layers[3]['wt'].hi.clone()
    net.layers[3]['wt'].hi.zero_()
    net.refresh_weights()
    torch.cuda.synchronize()
    assert torch.equal(net.theta, th0) and torch.equal(m, m0) and torch.equal(v, v0) and torch.equal(t_dev, t0)
    assert torch.equal(net.layers[3]['wt'].hi.view(torch.int16), w_before.view(torch.int16))


def test_fused_adam_planes_rejects_bad_tables():
    _, net, _ = _net(504)
    L, ptr = _lib.lib(), _lib.ptr
    T = _lib.MlpLayer * 2
    t = T(net._table[0], net._table[1])
    assert L.b200pose_mlp_adam_planes(ptr(net.theta), None, None, None, net.n_flat, t, 17, 0, 0, 0, 0, 0, None, None, None) != 0
    assert L.b200pose_mlp_adam_planes(ptr(net.theta), ptr(net.grad), None, None, net.n_flat, t, 2, 0, 0, 0, 0, 0, None, None, None) != 0
    t[1].offset = 0                                                                        # overlapping slots
    assert L.b200pose_mlp_adam_planes(ptr(net.theta), None, None, None, net.n_flat, t, 2, 0, 0, 0, 0, 0, None, None, None) != 0
    t = T(net._table[0], net._table[1])
    t[1].ld_wt = 100                                                                       # not a multiple of 64
    assert L.b200pose_mlp_adam_planes(ptr(net.theta), None, None, None, net.n_flat, t, 2, 0, 0, 0, 0, 0, None, None, None) != 0
    assert b'mlp_adam_planes' in L.b200pose_last_error()


def _mse(joints, target):
    return torch.nn.functional.mse_loss(joints, target)


def test_trainer_vs_fp64_autograd_adam():
    """5 steps of MlpTrainer against fp64 torch autograd + torch.optim.Adam (same defaults) on the same batches. The losses agree
    to 1e-4. Parameters: Adam moves each element by about lr * m / sqrt(v), whatever the gradient's magnitude, so an element whose
    gradient is tiny (within the forward's ~1e-5 relative noise of the larger ones) can take a step of a different size or sign.
    The LeakyReLU masks flipped by the forward's ~1e-5 differences (see test_mlp_backward_vs_fp64_oracle) add to that in the first
    layer. The bar is therefore on the update of each tensor as a whole (relative L2 of theta - theta_0 within 0.15; 7.8e-2 observed
    at worst on a B200, where a wrong gradient gives O(1)) and on the outliers (every element within 2 lr * steps of the
    reference, the largest difference two independent Adam paths allow)."""
    width, P, steps, lr = 504, 64, 5, 1e-3
    state = helpers.weights_mod.make_mlp_state(width, 54, 5)
    trainer = train_mod.MlpTrainer(_pipe(), state, lr=lr)
    ref = oracle_mlp(state).cuda()
    opt = torch.optim.Adam(ref.parameters(), lr=lr)
    g = torch.Generator().manual_seed(3)
    batches = [(torch.randn(P, width, generator=g).cuda(), torch.randn(P, 54, generator=g).cuda() * 0.1) for _ in range(steps)]
    for s, (x, y) in enumerate(batches):
        loss = float(trainer.step(x, _mse, y).item())
        opt.zero_grad()
        rl = torch.nn.functional.mse_loss(ref(x.double()), y.double())
        rl.backward()
        opt.step()
        assert abs(loss - rl.item()) <= 1e-4 * rl.item(), (s, loss, rl.item())
    got = trainer.net.state_dict()
    worst = 0.0
    for name, p in ref.named_parameters():
        k = 'layers.' + name
        d_ref = p.detach() - state[k].double().cuda()
        d_got = got[k].double() - state[k].double().cuda()
        l2 = ((d_got - d_ref).norm() / d_ref.norm()).item()
        assert l2 <= 0.15, (k, l2)
        assert (d_got - d_ref).abs().max().item() <= 2 * lr * steps, k
        worst = max(worst, l2)
    assert trainer.t == steps and int(trainer.t_dev.item()) == steps
    print('MlpTrainer vs fp64 autograd + Adam after %d steps: worst relative L2 of a tensor update %.3g' % (steps, worst))


def test_captured_step_is_the_eager_step():
    """step_captured against step over two alternating shapes: same losses and bit-identical parameters after every step; a
    larger batch re-allocates the workspaces and re-captures; the cache of graphs stays bounded."""
    width = 504
    state = helpers.weights_mod.make_mlp_state(width, 54, 9)
    eager, captured = train_mod.MlpTrainer(_pipe(), state), train_mod.MlpTrainer(_pipe(), state)
    g = torch.Generator().manual_seed(4)
    batches = [(torch.randn(P, width, generator=g).cuda(), torch.randn(P, 54, generator=g).cuda()) for P in (48, 32)]
    for it in range(6):
        x, y = batches[it % 2]
        le = float(eager.step(x, _mse, y).item())
        lc = float(captured.step_captured(x, _mse, y).item())
        assert le == lc, (it, le, lc)
        assert torch.equal(eager.net.theta, captured.net.theta), it
        assert torch.equal(eager.m, captured.m) and torch.equal(eager.v, captured.v), it
    assert len(captured._graphs) == 2 and int(captured.t_dev.item()) == 6
    assert torch.equal(captured.last_joints, eager.last_joints)
    xb, yb = torch.randn(300, width, generator=g).cuda(), torch.randn(300, 54, generator=g).cuda()
    le, lc = float(eager.step(xb, _mse, yb).item()), float(captured.step_captured(xb, _mse, yb).item())
    assert le == lc and torch.equal(eager.net.theta, captured.net.theta)
    gen = captured.net.buf.gen                                         # the larger batch grew the workspaces: the older graphs are
    assert sum(e['gen'] == gen for e in captured._graphs.values()) == 1   # stale, and the next lookup of one drops them all
    x, y = batches[0]
    assert float(eager.step(x, _mse, y).item()) == float(captured.step_captured(x, _mse, y).item())
    assert len(captured._graphs) == 1 and torch.equal(eager.net.theta, captured.net.theta)
    captured.max_cached = 2
    for P in (200, 100, 250):
        x, y = torch.randn(P, width, generator=g).cuda(), torch.randn(P, 54, generator=g).cuda()
        assert float(eager.step(x, _mse, y).item()) == float(captured.step_captured(x, _mse, y).item())
    assert len(captured._graphs) == 2 and torch.equal(eager.net.theta, captured.net.theta)


def test_reprojection_loss_inside_captured_step():
    """A loss in the style of the reference's training script: the predicted joints, placed in front of a camera, projected with
    the shadow's camera_matrix and apply_distortion (pose_estimator_utils.py) and compared with 2D targets - run inside the
    captured step, bit-identical to the eager step."""
    cfg, _, _ = helpers.load_golden('panoptic')
    mods = dropin_env.activate(cfg)
    pu = mods['pose_estimator_utils']
    K = pu.camera_matrix(0)
    kd = pu.get_distortion_coefficients(0)
    offset = torch.tensor([0.0, 0.0, 4.0], device='cuda').reshape(3, 1)

    def reprojection(joints, K, kd, target):
        X = joints.reshape(-1, 3).t() + offset                        # [3, P * 18], metres in front of the camera
        v = pu.apply_distortion(kd, X / X[2:3])
        uv = (K @ v)[:2]
        return ((uv - target) ** 2).mean()

    width = cfg.n_cameras * 18 * 14
    state = helpers.weights_mod.make_mlp_state(width, 54, 2)
    eager, captured = train_mod.MlpTrainer(_pipe(), state, lr=1e-4), train_mod.MlpTrainer(_pipe(), state, lr=1e-4)
    g = torch.Generator().manual_seed(8)
    x = torch.randn(24, width, generator=g).cuda()
    target = (torch.rand(2, 24 * 18, generator=g) * 500 + 200).cuda()
    for it in range(3):
        le = eager.step(x, reprojection, K, kd, target).item()
        lc = captured.step_captured(x, reprojection, K, kd, target).item()
        assert np.isfinite(le) and le == lc, (it, le, lc)
        assert torch.equal(eager.net.theta, captured.net.theta)
    assert len(captured._graphs) == 1


def test_dropin_reference_loop_against_fp32_twin():
    """The loop of a torch training script on the drop-in PoseEstimatorMLP (to(cuda), Adam, zero_grad, forward, loss, backward,
    step) beside an fp32 nn.Sequential twin: gradients at every step, eval() outputs after the steps within the inference bar
    (0.5 mm on the x10 joints), the reference's state-dict keys; the two refused uses raise. Gradients: relative L2 within 1e-1 per
    tensor - the twin's fp32 forward flips a few LeakyReLU masks against the split-bf16 one and the first layer collects them (see
    test_mlp_backward_vs_fp64_oracle; 5.2e-2 observed at worst on a B200)."""
    cfg, npz, meta = helpers.load_golden('panoptic')
    mods = dropin_env.activate(cfg)
    width = meta['mlp_in_dim']
    state = helpers.weights_mod.make_mlp_state(width, 54, 4)
    device = torch.device('cuda')
    with torch.enable_grad():
        model = mods['mlp'].PoseEstimatorMLP(input_dimensions=width, output_dimensions=54)
        model.load_state_dict(state)
        model = model.to(device)
        optimizer = torch.optim.Adam(model.parameters(), lr=1e-4)
        twin = oracle_mlp(state, torch.float32).to(device)
        opt_twin = torch.optim.Adam(twin.parameters(), lr=1e-4)
        g = torch.Generator().manual_seed(6)
        x = torch.randn(40, width, generator=g).to(device)
        y = (torch.randn(40, 54, generator=g) * 0.1).to(device)
        with torch.no_grad():
            out_ng = model(x)
        model.train()
        worst = worst_l2 = 0.0
        for step in range(3):
            optimizer.zero_grad()
            opt_twin.zero_grad()
            out = model(x)
            assert out.requires_grad and out.shape == (40, 54)
            if step == 0:
                assert (out.detach() - out_ng).abs().max().item() * 10 < 5e-4
            loss = torch.nn.functional.mse_loss(out, y)
            loss.backward()
            torch.nn.functional.mse_loss(twin(x), y).backward()
            for (name, p), (_, q) in zip(model.named_parameters(), twin.named_parameters()):
                assert p.grad is not None and p.grad.shape == p.shape and p.grad.dtype == p.dtype and p.grad.device == p.device, name
                l2 = ((p.grad - q.grad).norm() / q.grad.norm()).item()
                err = (p.grad - q.grad).abs().max().item() / q.grad.abs().max().item()
                assert l2 <= 1e-1, (step, name, l2, err)
                worst = max(worst, err)
                worst_l2 = max(worst_l2, l2)
            optimizer.step()
            opt_twin.step()
        model.eval()
        with torch.no_grad():
            assert (model(x) - twin(x)).abs().max().item() * 10 < 5e-4
        assert sorted(model.state_dict()) == sorted(state)
        # the refused uses
        with pytest.raises(NotImplementedError):
            model(x.clone().requires_grad_(True))
        out1 = model(x)
        model(x[:8])
        with pytest.raises(RuntimeError):
            out1.sum().backward()
    print('drop-in vs fp32 twin: worst gradient element %.3g of the tensor maximum, worst relative L2 %.3g' % (worst, worst_l2))
