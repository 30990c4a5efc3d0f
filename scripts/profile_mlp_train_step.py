"""Training step of the pose-estimator MLP at the Panoptic width (in = 1260, 29.1 M parameters): native MlpTrainer (captured and
launch by launch) against torch fp32 on the same GPU (identical nn.Sequential, autograd, torch.optim.Adam(fused=True), TF32 off -
torch's default; a TF32 row for information), and an A/B of the fused optimiser kernel (b200pose_mlp_adam_planes) against the
unfused pair (b200pose_adam_step_dev + one b200pose_grad_planes refresh per layer). Arms alternate, 3 repeats, median and spread.
The optimiser's working set (theta, grad, m, v: 466 MB) is far larger than the 126 MB L2, so no cache flush is needed between
timed passes. Card name and power limit are read in the same run.

    python scripts/profile_mlp_train_step.py [--out profiles/r03_mlp_train_step.json] [--steps 20]
    python scripts/profile_mlp_train_step.py --profile P --out DIR/trace.txt    (a torch.profiler table of both steps at batch P)
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
pm = importlib.import_module('3d_multi_pose_estimator_b200.pipeline')
tr = importlib.import_module('3d_multi_pose_estimator_b200.train')
W = importlib.import_module('3d_multi_pose_estimator_b200.weights')
_lib = importlib.import_module('3d_multi_pose_estimator_b200._lib')
pkg = importlib.import_module('3d_multi_pose_estimator_b200')

WIDTH, PEAK_BW = 1260, 7.7e12


def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=30).stdout.decode().strip()
        info['power_limit'], info['sm_max_clock'] = [s.strip() for s in q.split(',')]
    except Exception as e:                                  # the numbers stay unlabelled rather than guessed
        info['power_limit'] = 'not read (%s)' % type(e).__name__
    return info


def torch_twin(state):
    dims = [WIDTH] + list(W.MLP_HIDDEN) + [54]
    mods = [torch.nn.Flatten()]
    for i in range(9):
        mods.append(torch.nn.Linear(dims[i], dims[i + 1]))
        if i < 8:
            mods.append(torch.nn.LeakyReLU(W.MLP_SLOPE))
    net = torch.nn.Sequential(*mods)
    net.load_state_dict({k[len('layers.'):]: v for k, v in state.items()})
    return net.cuda()


def mse(j, y):
    return torch.nn.functional.mse_loss(j, y)


def timed(fn, n):
    """ms per call over n calls, CUDA events, after the caller's warm-up"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def stats(v):
    return {'median_ms': float(np.median(v)), 'min_ms': float(min(v)), 'max_ms': float(max(v)), 'runs_ms': [float(x) for x in v]}


def unfused_pair(net, tm):
    L, s = net.L, net.pipe._stream()

    def run():
        _lib.check(L.b200pose_adam_step_dev(_lib.ptr(net.theta), _lib.ptr(net.grad), _lib.ptr(tm.m), _lib.ptr(tm.v), net.n_flat, tm.lr,
                                            tm.betas[0], tm.betas[1], tm.eps, tm.weight_decay, _lib.ptr(tm.t_dev), _lib.ptr(tm.adam_scalars), s),
                   'adam_step_dev')
        for i, lay in enumerate(net.layers):
            Wv = net.view(net.theta, 'layers.%d.weight' % tr.MLP_LAYER_INDICES[i], padded=True)
            w, wt = lay['w'], lay['wt']
            _lib.check(L.b200pose_grad_planes(_lib.ptr(Wv), lay['n'], lay['k'], Wv.stride(0), None, 0, 1.0, None, 0, _lib.ptr(w.hi), _lib.ptr(w.lo), w.ld,
                                              _lib.ptr(wt.hi) if wt else None, _lib.ptr(wt.lo) if wt else None, wt.ld if wt else 0, s), 'grad_planes')
    return run


def optimiser_bytes(net):
    planes = sum(4 * (l['n'] * l['w'].ld + (l['k'] * l['wt'].ld if l['wt'] is not None else 0)) for l in net.layers)
    adam = 7 * 4 * net.n_flat                               # read theta, g, m, v; write theta, m, v
    weights = sum(4 * l['n'] * l['k'] for l in net.layers)  # the unfused refresh reads theta again
    return adam + planes, adam + planes + weights


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(REPO, 'profiles', 'r03_mlp_train_step.json'))
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--batches', default='32,256,1024,4096')
    ap.add_argument('--profile', type=int, default=0, help='batch size: write a torch.profiler table instead of the timings')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    cfg = pkg.CameraConfig.from_npz(os.path.join(REPO, 'tests', 'golden', 'cameras_panoptic.npz'))
    pipe = pm.PosePipeline(cfg, None, None, device='cuda:0')
    state = W.make_mlp_state(WIDTH, 54, 1)
    tm = tr.MlpTrainer(pipe, state)
    twin = torch_twin(state)
    opt = torch.optim.Adam(twin.parameters(), lr=1e-3, fused=True)

    def torch_step(x, y):
        opt.zero_grad(set_to_none=False)
        loss = mse(twin(x), y)
        loss.backward()
        opt.step()
        return loss

    g = torch.Generator().manual_seed(0)
    if a.profile:
        from torch.profiler import profile, ProfilerActivity
        P = a.profile
        x, y = torch.randn(P, WIDTH, generator=g).cuda(), (torch.randn(P, 54, generator=g) * 0.1).cuda()
        for _ in range(3):
            tm.step(x, mse, y); torch_step(x, y)
        torch.cuda.synchronize()
        out = []
        for name, fn in (('native step (launch by launch)', lambda: tm.step(x, mse, y)), ('torch fp32', lambda: torch_step(x, y))):
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    fn()
                torch.cuda.synchronize()
            out.append('==== %s, P = %d, 5 steps, %s\n%s' % (name, P, json.dumps(card()), prof.key_averages().table(sort_by='cuda_time_total', row_limit=25)))
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, 'w').write('\n\n'.join(out))
        print('\n\n'.join(out))
        return

    res = {'card': card(), 'width': WIDTH, 'n_params': sum(int(v.numel()) for v in state.values()), 'steps_per_timing': a.steps,
           'repeats': a.repeats, 'loss': 'mse_loss(joints, target)', 'adam': 'lr 1e-3, betas (0.9, 0.999), eps 1e-8, no weight decay',
           'timing': 'CUDA events around steps_per_timing steps after 3 warm-up steps per arm; arms alternate within each repeat',
           'batches': {}}
    for P in [int(p) for p in a.batches.split(',')]:
        x, y = torch.randn(P, WIDTH, generator=g).cuda(), (torch.randn(P, 54, generator=g) * 0.1).cuda()
        # parity first (one gradient from the same parameters): the native backward against torch fp32 autograd
        tm.net.load_state(state)
        twin.load_state_dict({k[len('layers.'):]: v for k, v in state.items()})
        tm.step(x, mse, y, update=False)
        opt.zero_grad()
        mse(twin(x), y).backward()
        worst_max, worst_l2 = 0.0, 0.0
        for name, p in twin.named_parameters():
            d = tm.net.grads()['layers.' + name] - p.grad
            worst_max = max(worst_max, (d.abs().max() / p.grad.abs().max()).item())
            worst_l2 = max(worst_l2, (d.norm() / p.grad.norm()).item())
        l0 = tm.net.launches + pipe.launches
        tm.step(x, mse, y)
        launches = tm.net.launches + pipe.launches - l0
        arms = {'native step_captured': lambda: tm.step_captured(x, mse, y), 'native step': lambda: tm.step(x, mse, y),
                'torch fp32': lambda: torch_step(x, y)}
        for fn in arms.values():
            for _ in range(3):
                fn()
        tf32_prev = torch.backends.cuda.matmul.allow_tf32
        runs = {k: [] for k in list(arms) + ['torch tf32 (information)']}
        for r in range(a.repeats):
            for k, fn in arms.items():
                runs[k].append(timed(fn, a.steps))
            torch.backends.cuda.matmul.allow_tf32 = True
            if r == 0:
                torch_step(x, y); torch_step(x, y)
            runs['torch tf32 (information)'].append(timed(lambda: torch_step(x, y), a.steps))
            torch.backends.cuda.matmul.allow_tf32 = tf32_prev
        ent = {k: stats(v) for k, v in runs.items()}
        ent['launches_per_step'] = launches
        ent['captured_graphs_per_step'] = 1
        ent['parity_vs_torch_fp32'] = {'worst_max_error_of_tensor_max': worst_max, 'worst_relative_l2': worst_l2}
        ent['gemm_gflop'] = 3 * 2 * res['n_params'] * P / 1e9
        ent['native_captured_vs_torch_fp32'] = ent['torch fp32']['median_ms'] / ent['native step_captured']['median_ms']
        res['batches'][str(P)] = ent
        print(P, json.dumps({k: (v['median_ms'] if isinstance(v, dict) and 'median_ms' in v else v) for k, v in ent.items()}), flush=True)
    # ---- optimiser: fused kernel vs the unfused pair, same call, alternating
    fused_b, unfused_b = optimiser_bytes(tm.net)
    net = tm.net
    fused = lambda: net.adam_planes(net.grad, tm.m, tm.v, tm.lr, tm.betas, tm.eps, tm.weight_decay, tm.t_dev, tm.adam_scalars)
    unfused = unfused_pair(net, tm)
    for fn in (fused, unfused):
        for _ in range(3):
            fn()
    ab = {'fused b200pose_mlp_adam_planes': [], 'unfused adam_step_dev + 9 grad_planes': []}
    for _ in range(a.repeats):
        ab['fused b200pose_mlp_adam_planes'].append(timed(fused, 50))
        ab['unfused adam_step_dev + 9 grad_planes'].append(timed(unfused, 50))
    opt_res = {}
    for (k, v), nbytes in zip(ab.items(), (fused_b, unfused_b)):
        s = stats(v)
        s['bytes'] = nbytes
        s['GB_per_s'] = nbytes / (s['median_ms'] * 1e-3) / 1e9
        s['share_of_7.7_TB_per_s'] = nbytes / (s['median_ms'] * 1e-3) / PEAK_BW
        opt_res[k] = s
    opt_res['note'] = ('bytes from shapes: Adam reads theta, grad, m, v and writes theta, m, v (7 x 4 B x n_flat); planes: hi + lo bf16 of W '
                       '[n, round_up(k, 64)] and of W^T [k, round_up(n, 64)] (none for layer 1); the unfused refresh reads theta again. '
                       'The 466 MB working set exceeds the 126 MB L2: no flush between passes. Both paths include the scalar kernel.')
    opt_res['fused_speedup'] = float(np.median(ab['unfused adam_step_dev + 9 grad_planes']) / np.median(ab['fused b200pose_mlp_adam_planes']))
    res['optimiser_ab'] = opt_res
    print(json.dumps(opt_res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, 'w'), indent=1)
    print('wrote', a.out)


if __name__ == '__main__':
    main()
