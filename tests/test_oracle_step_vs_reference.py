"""CPU: pin oracle/torch_model.py (the CPU-baseline port of the whole training step) against three
training steps of the reference's own model, RMSprop, loss, L2 and EMA classes, recorded by
oracle/make_golden.py --step in tests/golden/ref_step.pt: the losses, every one-dimensional tensor
in full and every output channel of the larger ones."""
import os
import warnings

import torch


def _check(got, rec, what, rtol=1e-5, atol=1e-6):
    """`got` (name -> tensor) against a record of oracle.make_golden._digest: tensors of at most one
    dimension elementwise; larger ones on their seeded elements, and per output channel the sum and
    the sum of squares within the bounds that elementwise closeness (|x - y| <= atol + rtol |y|)
    implies."""
    assert sorted(got) == sorted(rec["names"]), what
    idx = iter(rec["idx"].long().split(rec["count"].tolist()))
    val = iter(rec["val"].split(rec["count"].tolist()))
    f = c = 0                                   # cursors into "full" and the per-channel sums
    for j, n in enumerate(rec["names"]):
        t = got[n].detach()
        assert t.numel() == int(rec["numel"][j]), (what, n)
        if t.dim() <= 1:
            want = rec["full"][f:f + t.numel()]
            f += t.numel()
            assert torch.allclose(t.float().flatten(), want, rtol=rtol, atol=atol), (what, n)
            continue
        assert torch.allclose(t.float().flatten()[next(idx)], next(val), rtol=rtol, atol=atol), \
            (what, n)
        rows = t.double().flatten(1)
        k = rows.shape[1]
        s1, s2 = rec["ch_abs"][c:c + len(rows)], rec["ch_sq"][c:c + len(rows)]
        d_sum = (rows.sum(1) - rec["ch_sum"][c:c + len(rows)]).abs()
        d_sq = (rows.square().sum(1) - s2).abs()
        c += len(rows)
        bad_sum = (d_sum > atol * k + rtol * s1).nonzero().flatten().tolist()
        bad_sq = (d_sq > atol * atol * k + 2 * atol * (1 + rtol) * s1 + (2 * rtol + rtol * rtol) * s2)
        assert not bad_sum and not bad_sq.any(), (what, n, "channels", bad_sum,
                                                 bad_sq.nonzero().flatten().tolist())
    assert f == rec["full"].numel() and c == rec["ch_sum"].numel(), what


def test_port_step_equals_reference_step(golden_dir):
    warnings.simplefilter("ignore")
    from yet_another_mobilenet_series_b200 import mobilenet_base as mb, mobilenet_supernet as sup
    from oracle import torch_model as tm

    rec = torch.load(os.path.join(golden_dir, "ref_step.pt"), weights_only=False)
    kw, B = rec["kw"], rec["batch"]
    torch.manual_seed(rec["seed"])
    ours = sup.Model(**kw)
    ours.apply(mb.init_weights_mnas)
    port = tm.as_reference(ours)
    for m in port.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    trainer = tm.RefTrainer(port, B)
    g = torch.Generator().manual_seed(rec["data_seed"])
    for step in range(rec["steps"]):
        x = torch.randn(B, 3, kw["input_size"], kw["input_size"], generator=g)
        t = torch.randint(0, kw["num_classes"], (B,), generator=g)
        assert torch.equal(x.flatten()[:16], rec["x_head"][step])   # the recorded batches
        assert torch.equal(t, rec["targets"][step])
        lp = trainer.step(x, t)
        want = rec["losses"][step]
        assert abs(lp - want) < 1e-5 * max(1.0, abs(want)), (step, lp, want)
    _check({k: v.float() for k, v in port.state_dict().items()}, rec["state"], "state_dict")
    _check(trainer.ema.shadow, rec["ema"], "EMA shadow")
