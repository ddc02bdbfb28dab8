"""ORACLE — test infrastructure / CPU baseline only (never imported by the product path).

Plain-PyTorch restatement of the reference's WHOLE training step on stock torch ops — the
"port" that is timed as the CPU baseline on the GPU box's host cores (where /root/reference does
not exist) and that serves as the end-to-end parity reference for the full network.

  block forward         models/mobilenet_base.py:446-451 (unfused), :330-342 (fused)
  step sequence         train.py:64-114 (zero_grad, forward_loss, cal_l2_loss, backward,
                        optimizer.step, EMA loop) and common.py:67-80 (the two host syncs)
  RMSprop               utils/rmsprop.py:67-129 (per-tensor Python loop)
  EMA                   utils/optim.py:53-64
  L2 ('mnas')           utils/optim.py:177-200
  label-smooth CE       utils/optim.py:150-158

`as_reference(model)` deep-copies a model built from the package's boundary modules (identical
module tree / state_dict to the reference's) and rebinds the two block classes' forward to the
reference's stock-torch graph, so it runs on CPU (or on a GPU through cuDNN/ATen: the
"stock PyTorch eager" context row).  Validated against three steps of the live reference
(oracle/make_golden.py --step -> tests/golden/ref_step.pt) by tests/test_oracle_step_vs_reference.py.
"""
import copy
import types

import torch
from torch import nn


def _unfused_forward(self, x):
    out = sum(op(x) for op in self.ops)          # mobilenet_base.py:447
    out = self.pw_bn(out)                        # :448
    return x + out if self.use_res_connect else out


def _fused_forward(self, x):
    h = self.expand_conv(x)                      # :331
    parts = [op(h) for op in self.depth_ops]     # :332
    h = parts[0] if len(parts) == 1 else torch.cat(parts, dim=1)
    h = self.se_op(h)
    h = self.project_conv(h)
    h = self.nl_op(h)
    return x + h if self.use_res_connect else h


def _model_forward(self, x):
    x = self.features(x)                         # mobilenet_supernet.py:169-173
    x = x.squeeze(3).squeeze(2)
    return self.classifier(x)


def as_reference(model):
    """Copy of `model` whose forward is the reference's stock-torch graph."""
    ref = copy.deepcopy(model)
    for m in ref.modules():
        if isinstance(m, nn.Sequential) and type(m).forward is not nn.Sequential.forward:
            # ConvBNReLU of the boundary package routes BatchNorm+activation to the sm_100a
            # kernels on CUDA; the reference's ConvBNReLU (:181-203) is a plain nn.Sequential
            m.forward = types.MethodType(nn.Sequential.forward, m)
        if hasattr(m, "pw_bn") and hasattr(m, "ops"):
            m.forward = types.MethodType(_unfused_forward, m)
        elif hasattr(m, "project_conv") and hasattr(m, "depth_ops"):
            m.forward = types.MethodType(_fused_forward, m)
    if hasattr(ref, "features") and hasattr(ref, "classifier"):   # a whole network, not a block
        ref.forward = types.MethodType(_model_forward, ref)
    return ref


def label_smooth_ce(logits, target, smoothing):
    """Per-sample loss of CrossEntropyLabelSmooth(reduction='none') (utils/optim.py:150-158)."""
    logp = torch.log_softmax(logits, 1)
    t = torch.zeros_like(logp).scatter_(1, target.unsqueeze(1), 1)
    t = (1 - smoothing) * t + smoothing / logits.size(1)
    return torch.sum(-t * logp, 1)


def l2_loss_mnas(model, weight_decay):
    """cal_l2_loss(method='mnas') (utils/optim.py:177-200)."""
    loss = 0.0
    for name, p in model.named_parameters():
        if p.dim() in (4, 2) or "classifier" in name:
            loss = loss + weight_decay * (p ** 2).sum()
    return loss * 0.5


class RefRMSprop:
    """utils/rmsprop.py:67-129, non-centered, as a per-tensor Python loop (the reference's
    launch pattern), state in plain dicts."""

    def __init__(self, params, lr, alpha, eps, eps_inside_sqrt, momentum, weight_decay=0.0):
        self.params = list(params)
        self.lr, self.alpha, self.eps = lr, alpha, eps
        self.eps_inside_sqrt, self.momentum, self.weight_decay = eps_inside_sqrt, momentum, \
            weight_decay
        self.state = {}

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    @torch.no_grad()
    def step(self):
        for p in self.params:
            if p.grad is None:
                continue
            g = p.grad
            st = self.state.setdefault(id(p), {})
            if not st:
                st["square_avg"] = torch.zeros_like(p)
                if self.momentum > 0:
                    st["momentum_buffer"] = torch.zeros_like(p)
            sq = st["square_avg"]
            if self.weight_decay != 0:
                g = g.add(p, alpha=self.weight_decay)
            sq.mul_(self.alpha).addcmul_(g, g, value=1 - self.alpha)
            avg = sq.add(self.eps).sqrt_() if self.eps_inside_sqrt else sq.sqrt().add_(self.eps)
            if self.momentum > 0:
                buf = st["momentum_buffer"]
                buf.mul_(self.momentum).addcdiv_(g, avg)
                p.add_(buf, alpha=-self.lr)
            else:
                p.addcdiv_(g, avg, value=-self.lr)


class RefEMA:
    """ExponentialMovingAverage (utils/optim.py:15-128) restricted to register/forward."""

    def __init__(self, momentum):
        self.momentum = momentum
        self.shadow = {}

    def register(self, name, val):
        self.shadow[name] = val.detach().clone()

    @torch.no_grad()
    def __call__(self, name, x, num_updates=None):
        m = self.momentum if num_updates is None else min(
            self.momentum, (1.0 + num_updates) / (10.0 + num_updates))
        return self.shadow[name].mul_(m).add_(x.detach(), alpha=1.0 - m)


class RefTrainer:
    """One object = the reference's training state for the step of train.py:64-114."""

    def __init__(self, model, batch_size_global, base_lr=0.016, base_total_batch=256, alpha=0.9,
                 momentum=0.9, eps=1e-3, weight_decay=1e-5, label_smoothing=0.1,
                 ema_decay=0.9999, ema_base_batch=4096, autocast=None):
        self.model = model
        # None: the reference as written (fp32).  A dtype: the same stock-torch graph under
        # torch.autocast — "the reference's own bf16 path", the parity yardstick of SURVEY §8c(ii)
        self.autocast = autocast
        self.lr = base_lr * batch_size_global / base_total_batch      # common.py:204-205
        self.opt = RefRMSprop(model.parameters(), self.lr, alpha, eps, True, momentum)
        self.wd = weight_decay
        self.smoothing = label_smoothing
        decay = ema_decay ** (batch_size_global / ema_base_batch)     # common.py:47-57
        self.ema = RefEMA(decay)
        for n, p in model.named_parameters():
            self.ema.register(n, p)
        for n, b in model.named_buffers():                            # common.py:61-63
            if "running_var" in n or "running_mean" in n:
                self.ema.register(n, b)
        self.global_step = 0

    def step(self, x, target):
        model = self.model
        model.train()
        self.opt.zero_grad()                                          # train.py:66
        if self.autocast is not None:
            with torch.autocast(x.device.type, dtype=self.autocast):
                out = model(x).float()
        else:
            out = model(x)
        loss_vec = label_smooth_ce(out, target, self.smoothing)
        _ = loss_vec.tolist()                                         # common.py:71 host sync #1
        _, pred = out.topk(5)
        correct = pred.t().eq(target.view(1, -1).expand_as(pred.t()))
        for k in (1, 5):
            _ = correct[:k].float().sum(0).cpu().numpy()              # common.py:73-79 sync #2
        loss = loss_vec.mean() + l2_loss_mnas(model, self.wd)         # train.py:68-70
        loss.backward()
        self.opt.step()                                               # train.py:102
        self.global_step += 1
        named = dict(model.named_parameters())
        named.update({n: b for n, b in model.named_buffers()})
        for n in self.ema.shadow:                                     # train.py:109-114
            self.ema(n, named[n], self.global_step)
        return float(loss.detach())
