"""ORACLE tooling — generates tests/golden/*.pt by running the LIVE reference
(/root/reference, imported unmodified) on seeded inputs.  Run in the build container only:

    python oracle/make_golden.py            # blocks.pt, optim.pt
    python oracle/make_golden.py --nl       # blocks_nl.pt
    python oracle/make_golden.py --step     # ref_step.pt

The fixtures travel to the GPU box; /root/reference does not.
Reference entry points exercised:
  models/mobilenet_base.py:352-458 InvertedResidualChannels, :206-349 InvertedResidualChannelsFused,
  :510-537 init_weights_mnas;  utils/rmsprop.py:6-129 RMSprop;
  utils/optim.py:15-128 ExponentialMovingAverage, :161-200 cal_l2_loss, :131-158 CrossEntropyLabelSmooth
"""
import os
import sys
import warnings

import torch

REF = os.environ.get("YAMB_REFERENCE", "/root/reference")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")

BLOCK_CASES = [
    # name, class, (inp, oup, stride, channels, kernel_sizes, expand), act, extra, input NCHW shape
    ("v2_s2_relu", "InvertedResidualChannels", (16, 24, 2, [96], [3], True), "nn.ReLU", {},
     (4, 16, 16, 16)),
    ("v2_res_relu6", "InvertedResidualChannels", (24, 24, 1, [144], [3], True), "nn.ReLU6", {},
     (3, 24, 10, 10)),
    ("v2_noexpand", "InvertedResidualChannels", (32, 16, 1, [32], [3], False), "nn.ReLU", {},
     (4, 32, 12, 12)),
    ("multi_k357", "InvertedResidualChannels", (24, 24, 1, [48, 32, 16], [3, 5, 7], True),
     "nn.ReLU6", {}, (2, 24, 12, 12)),
    ("fused_se_swish", "InvertedResidualChannelsFused", (24, 24, 1, [48, 32, 16], [3, 5, 7], True),
     "nn.Swish", {"se_ratio": 0.5}, (2, 24, 12, 12)),
    ("fused_s2_k5", "InvertedResidualChannelsFused", (24, 40, 2, [72, 24], [5, 3], True),
     "nn.Swish", {"se_ratio": 0.25}, (2, 24, 14, 14)),
    ("fused_plain", "InvertedResidualChannelsFused", (16, 16, 1, [64], [3], True), "nn.ReLU", {},
     (2, 16, 8, 8)),
]


NL_CASES = [
    # non-local blocks (Nonlocal, models/mobilenet_base.py:131-178); "A"/"B" = the association
    # order the reference's MAC test (:164-170) picks for that shape
    ("nl_B_res", "InvertedResidualChannelsFused", (24, 24, 1, [72], [3], True), "nn.Swish",
     {"se_ratio": 0.25, "nl_c": 0.25, "nl_s": 1}, (2, 24, 12, 12)),
    ("nl_A_small_map", "InvertedResidualChannelsFused", (64, 64, 1, [128], [3], True), "nn.Swish",
     {"nl_c": 0.25, "nl_s": 1}, (2, 64, 4, 4)),
    ("nl_sub2_odd_map", "InvertedResidualChannelsFused", (40, 40, 1, [120], [5], True), "nn.Swish",
     {"se_ratio": 0.25, "nl_c": 0.25, "nl_s": 2}, (2, 40, 7, 7)),
    ("nl_s2_nores", "InvertedResidualChannelsFused", (16, 24, 2, [48], [5], True), "nn.ReLU6",
     {"nl_c": 0.25, "nl_s": 2}, (2, 16, 12, 12)),
]


def _block_records(mb, cases, bnk):
    blocks = {}
    for name, cls, args, act, extra, xshape in cases:
        torch.manual_seed(1995)
        blk = getattr(mb, cls)(*args, active_fn=mb.get_active_fn(act), batch_norm_kwargs=bnk,
                               **extra)
        blk.apply(mb.init_weights_mnas)
        g = torch.Generator().manual_seed(7)
        for m in blk.modules():  # pattern of tests/models/mobilenet_base_test.py:7-10
            if isinstance(m, torch.nn.BatchNorm2d):   # ZeroInitBN included: gamma != 0
                m.weight.data.uniform_(0.5, 1.5, generator=g)
                m.bias.data.normal_(0, 0.3, generator=g)
                m.running_mean.normal_(0, 0.2, generator=g)
                m.running_var.uniform_(0.5, 1.5, generator=g)
        state0 = {k: v.clone() for k, v in blk.state_dict().items()}
        x = torch.randn(*xshape, generator=g)
        rec = {"cls": cls, "args": args, "act": act, "extra": extra, "bn": bnk, "state": state0,
               "x": x}
        for mode in ("train", "eval"):
            blk.load_state_dict(state0)
            blk.train(mode == "train")
            blk.zero_grad()
            xi = x.clone().requires_grad_(True)
            y = blk(xi)
            dy = torch.randn(y.shape, generator=g)
            y.backward(dy)
            rec[mode] = {
                "y": y.detach().clone(), "dy": dy, "dx": xi.grad.clone(),
                "grads": {k: p.grad.clone() for k, p in blk.named_parameters()},
                "state_after": {k: v.clone() for k, v in blk.state_dict().items()},
            }
        blocks[name] = rec
    return blocks


def main_nl():
    """tests/golden/blocks_nl.pt: non-local blocks.  Nonlocal.__init__ imports the reference's
    FLAGS singleton (models/mobilenet_base.py:151), which parses sys.argv at import
    (utils/config.py:216): give it the AutoNL yml."""
    os.environ.setdefault("ARNOLD_OUTPUT", "/tmp/yamb_out")
    os.environ.setdefault("DATA_LMDB", "/tmp/yamb_lmdb")
    sys.argv = ["make_golden", "app:" + os.path.join(REF, "apps/searched/autonl/autonl_l.yml")]
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)
    import logging
    import models.mobilenet_base as mb
    logging.disable(logging.CRITICAL)
    os.chdir(cwd)
    warnings.simplefilter("ignore")
    blocks = _block_records(mb, NL_CASES, {"momentum": 0.01, "eps": 1e-3})
    torch.save(blocks, os.path.join(OUT, "blocks_nl.pt"))
    print("blocks_nl.pt", os.path.getsize(os.path.join(OUT, "blocks_nl.pt")), "bytes")


STEP_ROWS = [[1, 16, 1, 1, [3]], [6, 24, 1, 2, [3]], [6, 32, 1, 2, [3, 5]], [3, 40, 1, 2, [5]],
             [3, 48, 2, 2, [3]]]
STEP_KW = dict(inverted_residual_setting=STEP_ROWS, active_fn="nn.ReLU", batch_norm_momentum=0.01,
               batch_norm_epsilon=1e-3, input_size=64, num_classes=10, last_channel=64)


def _digest(tensors, k, g):
    """Per named tensor: a tensor of at most one dimension in full (fp32); a larger one as float64
    sum, sum of |x| and sum of x^2 of every output channel (dim 0) plus `k` elements at seeded flat
    indices.  Everything is concatenated in `names` order; `count` splits the samples."""
    names = list(tensors)
    full, ch_sum, ch_abs, ch_sq, idx, val, count = [], [], [], [], [], [], []
    for n in names:
        t = tensors[n].detach()
        if t.dim() <= 1:
            full.append(t.float().flatten())
            continue
        rows = t.double().flatten(1)
        ch_sum.append(rows.sum(1))
        ch_abs.append(rows.abs().sum(1))
        ch_sq.append(rows.square().sum(1))
        v = t.float().flatten()
        i = torch.randperm(v.numel(), generator=g)[:k].sort().values
        idx.append(i.to(torch.int32))
        val.append(v[i])
        count.append(len(i))
    return {"names": names, "numel": torch.tensor([tensors[n].numel() for n in names]),
            "full": torch.cat(full), "ch_sum": torch.cat(ch_sum), "ch_abs": torch.cat(ch_abs),
            "ch_sq": torch.cat(ch_sq), "count": torch.tensor(count), "idx": torch.cat(idx),
            "val": torch.cat(val)}


def main_step(k=64):
    """tests/golden/ref_step.pt: three training steps of the reference (train.py:64-114 with the
    live model, RMSprop, label-smoothed CE, 'mnas' L2 and EMA classes) on a small MobileNetV2 at
    64x64, dropout off.  Per step the loss and a few input values (to pin the seeded batches);
    after the last step every tensor of the state_dict and every EMA shadow as _digest()."""
    sys.path.insert(0, REF)
    warnings.simplefilter("ignore")
    import models.mobilenet_base as rmb
    import models.mobilenet_supernet as rsup
    from utils.rmsprop import RMSprop
    from utils import optim as roptim
    B, steps, seed, data_seed = 8, 3, 1995, 0
    torch.manual_seed(seed)
    ref = rsup.Model(**STEP_KW)
    ref.apply(rmb.init_weights_mnas)
    for m in ref.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    opt = RMSprop(ref.parameters(), lr=0.016 * B / 256, alpha=0.9, momentum=0.9, eps=1e-3,
                  eps_inside_sqrt=True, weight_decay=0)
    crit = roptim.CrossEntropyLabelSmooth(STEP_KW["num_classes"], 0.1)
    ema = roptim.ExponentialMovingAverage(0.9999 ** (B / 4096.0))
    for n, p in ref.named_parameters():
        ema.register(n, p)
    for n, b in ref.named_buffers():
        if "running_var" in n or "running_mean" in n:
            ema.register(n, b)
    g = torch.Generator().manual_seed(data_seed)
    losses, x_head, targets = [], [], []
    for step in range(1, steps + 1):
        x = torch.randn(B, 3, STEP_KW["input_size"], STEP_KW["input_size"], generator=g)
        t = torch.randint(0, STEP_KW["num_classes"], (B,), generator=g)
        ref.train()
        opt.zero_grad()
        loss = crit(ref(x), t).mean() + roptim.cal_l2_loss(ref, 1e-5, "mnas")
        loss.backward()
        opt.step()
        named = dict(ref.named_parameters())
        named.update(dict(ref.named_buffers()))
        for n in ema.average_names():
            ema(n, named[n], step)
        losses.append(float(loss))
        x_head.append(x.flatten()[:16].clone())
        targets.append(t.clone())
    gs = torch.Generator().manual_seed(11)
    rec = {"kw": STEP_KW, "batch": B, "steps": steps, "seed": seed, "data_seed": data_seed,
           "losses": losses, "x_head": torch.stack(x_head), "targets": torch.stack(targets),
           "state": _digest(ref.state_dict(), k, gs),
           "ema": _digest({n: ema.average(n) for n in ema.average_names()}, k, gs)}
    path = os.path.join(OUT, "ref_step.pt")
    torch.save(rec, path)
    print("ref_step.pt", os.path.getsize(path), "bytes")


def main():
    sys.path.insert(0, REF)
    import models.mobilenet_base as mb
    from utils.rmsprop import RMSprop
    from utils import optim as roptim
    os.makedirs(OUT, exist_ok=True)
    warnings.simplefilter("ignore")
    bnk = {"momentum": 0.01, "eps": 1e-3}

    blocks = {}
    for name, cls, args, act, extra, xshape in BLOCK_CASES:
        torch.manual_seed(1995)
        blk = getattr(mb, cls)(*args, active_fn=mb.get_active_fn(act), batch_norm_kwargs=bnk,
                               **extra)
        blk.apply(mb.init_weights_mnas)
        g = torch.Generator().manual_seed(7)
        for m in blk.modules():  # pattern of tests/models/mobilenet_base_test.py:7-10
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.data.uniform_(0.5, 1.5, generator=g)
                m.bias.data.normal_(0, 0.3, generator=g)
                m.running_mean.normal_(0, 0.2, generator=g)
                m.running_var.uniform_(0.5, 1.5, generator=g)
        state0 = {k: v.clone() for k, v in blk.state_dict().items()}
        x = torch.randn(*xshape, generator=g)
        rec = {"cls": cls, "args": args, "act": act, "extra": extra, "bn": bnk, "state": state0,
               "x": x}
        for mode in ("train", "eval"):
            blk.load_state_dict(state0)
            blk.train(mode == "train")
            blk.zero_grad()
            xi = x.clone().requires_grad_(True)
            y = blk(xi)
            dy = torch.randn(y.shape, generator=g)
            y.backward(dy)
            rec[mode] = {
                "y": y.detach().clone(), "dy": dy, "dx": xi.grad.clone(),
                "grads": {k: p.grad.clone() for k, p in blk.named_parameters()},
                "state_after": {k: v.clone() for k, v in blk.state_dict().items()},
            }
        blocks[name] = rec
    torch.save(blocks, os.path.join(OUT, "blocks.pt"))

    # ---- optimizer / EMA / L2 / loss sequences from the live reference classes ----
    torch.manual_seed(3)
    opt_rec = {}
    for tag, kw in {
        "mnas": dict(lr=0.016, alpha=0.9, momentum=0.9, eps=1e-3, eps_inside_sqrt=True),
        "plain": dict(lr=0.01, alpha=0.99, momentum=0.0, eps=1e-8, eps_inside_sqrt=False),
        "wd": dict(lr=0.01, alpha=0.95, momentum=0.5, eps=1e-5, eps_inside_sqrt=False,
                   weight_decay=1e-2),
    }.items():
        p = torch.nn.Parameter(torch.randn(257))
        p0 = p.detach().clone()
        opt = RMSprop([p], **kw)
        grads, ps = [], []
        for step in range(12):
            gr = torch.randn(257) * (0.5 + step * 0.1)
            p.grad = gr.clone()
            opt.step()
            grads.append(gr)
            ps.append(p.detach().clone())
        st = opt.state[p]
        opt_rec[tag] = {"kw": kw, "p0": p0, "grads": torch.stack(grads), "ps": torch.stack(ps),
                        "square_avg": st["square_avg"].clone(),
                        "momentum_buffer": st.get("momentum_buffer", torch.zeros(0)).clone()}
    # EMA with the num_updates rule (train.py:109-114 passes FLAGS._global_step)
    ema = roptim.ExponentialMovingAverage(0.9999 ** (256 / 4096.0))
    v = torch.randn(33)
    ema.register("v", v)
    xs, shadows = [], []
    for t in range(1, 15):
        xnew = torch.randn(33)
        ema("v", xnew, t)
        xs.append(xnew)
        shadows.append(ema.average("v").clone())
    opt_rec["ema"] = {"decay": 0.9999 ** (256 / 4096.0), "v0": v, "xs": torch.stack(xs),
                      "shadows": torch.stack(shadows)}
    # L2 ('mnas') gradient on a toy model with conv / dw conv / bn / classifier
    class Toy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = torch.nn.Conv2d(4, 8, 1, bias=False)
            self.dw = torch.nn.Conv2d(8, 8, 3, groups=8, bias=False)
            self.bn = torch.nn.BatchNorm2d(8)
            self.classifier = torch.nn.Linear(8, 5)
    toy = Toy()
    l2 = roptim.cal_l2_loss(toy, 1e-5, "mnas")
    l2.backward()
    opt_rec["l2"] = {"wd": 1e-5, "loss": l2.detach(),
                     "params": {k: p.detach().clone() for k, p in toy.named_parameters()},
                     "grads": {k: (p.grad.clone() if p.grad is not None else torch.zeros_like(p))
                               for k, p in toy.named_parameters()}}
    # label-smoothed CE (utils/optim.py:150-158)
    crit = roptim.CrossEntropyLabelSmooth(10, 0.1)
    logits = torch.randn(6, 10)
    tgt = torch.randint(0, 10, (6,))
    opt_rec["ce"] = {"logits": logits, "target": tgt, "loss": crit(logits, tgt)}
    torch.save(opt_rec, os.path.join(OUT, "optim.pt"))
    for f in ("blocks.pt", "optim.pt"):
        print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__":
    if "--nl" in sys.argv:          # separate process: FLAGS of the reference is a singleton
        main_nl()
    elif "--step" in sys.argv:
        main_step()
    else:
        main()
