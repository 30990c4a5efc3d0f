"""Drop-in for the reference's utils/mlp.py (PoseEstimatorMLP :3-31): same module tree, so checkpoints with keys
`layers.{1,3,...,17}.{weight,bias}` load unchanged; forward runs the 9 projections on the B200 tensor cores. Under autograd
(grad enabled, trainable parameters) the output is differentiable: `loss.backward()` runs the hand-written backward of
3d_multi_pose_estimator_b200/train.py (MlpGrad) and fills every parameter's .grad, so a torch optimiser trains the module."""
import torch
from torch import nn

import _b200pose_runtime as rt

class _MlpTrainFunction(torch.autograd.Function):
    """PoseEstimatorMLP.forward under autograd: the forward keeps its activations inside an MlpGrad, `loss.backward()` lands
    here and the parameter gradients come from csrc/train.cu + the tensor-core GEMM."""

    @staticmethod
    def forward(ctx, inputs, holder, *params):
        net, x2, _ = holder
        out = net.forward(x2).clone()
        ctx.holder = holder
        return out

    @staticmethod
    def backward(ctx, dout):
        net, _, named = ctx.holder
        if net.cache_token is not ctx.holder:
            raise RuntimeError('B200 PoseEstimatorMLP: backward() after another forward of the same model (the drop-in keeps one set '
                               'of activations)')
        net.backward(dout.to(net.device, torch.float32).contiguous())
        grads = net.grads()
        return (None, None) + tuple(grads[k].reshape(p.shape).to(p.device, p.dtype, copy=True) for k, p in named)


HIDDEN_WIDTHS = (3072, 3072, 2048, 2048, 1024, 1024, 1024, 1024)     # the reference's layer widths (utils/mlp.py:11-27)


class PoseEstimatorMLP(nn.Module):
    def __init__(self, input_dimensions, output_dimensions):
        super().__init__()
        print('MLP input size', input_dimensions)
        self.negative_slope = 0.1                                   # LeakyReLU slope of every hidden layer (utils/mlp.py:7)
        widths = (input_dimensions,) + HIDDEN_WIDTHS + (output_dimensions,)
        modules = [nn.Flatten()]                                    # index 0, so the projections sit at 1, 3, ..., 17
        for i in range(len(widths) - 1):
            modules.append(nn.Linear(widths[i], widths[i + 1]))
            if i < len(widths) - 2:
                modules.append(nn.LeakyReLU(negative_slope=self.negative_slope))
        self.layers = nn.Sequential(*modules)
        self._prepared = None
        self._prepared_key = None

    def _forward_train(self, x, ctx):
        """Grad mode with trainable parameters: only the parameters are trained (the input gets no gradient)."""
        if x.requires_grad:
            raise NotImplementedError('B200 PoseEstimatorMLP: gradients with respect to the input are not computed (only the '
                                      'parameters are trained)')
        named = list(self.named_parameters())
        key = tuple((p.data_ptr(), p._version) for _, p in named)
        net = self.__dict__.get('_grad_net')
        rt.sync_live()
        if net is None:
            train_mod = rt.importlib.import_module('3d_multi_pose_estimator_b200.train')
            net = train_mod.MlpGrad(ctx, {k: v for k, v in self.state_dict().items()}, self.negative_slope)
            self.__dict__['_grad_net'] = net
        elif key != self.__dict__.get('_grad_key'):
            net.load_state({k: v for k, v in self.state_dict().items()})       # optimizer.step() changed them: planes rebuilt
        self.__dict__['_grad_key'] = key
        x2 = x.reshape(x.shape[0], -1).to(ctx.device, torch.float32).contiguous()
        holder = (net, x2, named)
        net.cache_token = holder
        return _MlpTrainFunction.apply(x, holder, *[p for _, p in named]).to(x.device)

    def forward(self, x):
        ctx = rt.context()
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return self._forward_train(x, ctx)
        plist = self.__dict__.get('_plist')
        if plist is None:                       # the module-tree walk of parameters() is done once
            plist = list(self.parameters())
            self.__dict__['_plist'] = plist
        key = tuple((p.data_ptr(), p._version) for p in plist)
        if self._prepared is None or key != self._prepared_key:
            rt.sync_live()
            self._prepared = ctx.prepare_mlp({k: v for k, v in self.state_dict().items()})
            self._prepared_key = key
        if abs(self.negative_slope - rt.pipeline.MLP_SLOPE) < 1e-12:
            rt.note_model('mlp', self, key, self._prepared)      # the dataset drop-in submits whole frames with these weights from now on
        x2 = x.reshape(x.shape[0], -1).to(ctx.device).float()
        # the rows are the MLP inputs of the proposals of the frame submitted as a whole, in the order its persons were asked
        # for: the submission already ran these 9 projections (checked by value, not assumed)
        lv = rt.last_live()
        served = getattr(lv, 'served', None) if lv is not None else None
        if served and lv.fresh() and lv.key[2] == (id(self), key) and len(served) == x2.shape[0]:
            mine = lv.enc_device(max(served) + 1)
            mine = mine if served == list(range(len(served))) else mine[served]
            torch.cuda.current_stream(ctx.device).wait_event(lv.ent.ev_b)
            if mine.shape == x2.shape and torch.equal(mine, x2):
                out = lv.mlp_out_raw(max(served) + 1)
                if out is not None:
                    lv.served = []
                    out = out if served == list(range(len(served))) else out[served]
                    return out.to(x.device)
        rt.sync_live()
        planes = rt.pipeline.Planes.from_f32(x2, ctx._stream())
        out = ctx.mlp_forward(planes, x2.shape[0], scale=1.0, layers=self._prepared, slope=self.negative_slope)
        return out.clone().to(x.device)
