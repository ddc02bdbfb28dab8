"""GPU driver: how far apart two runs of the training step land with the same inputs, and what
`bench.py --dump-outputs` writes in two runs with the same arguments (profiles/r03_dump_spread.txt).

  python tests/gpu_dump_spread.py [--steps 20 --warmup 5]

1. Two identically seeded MobileNetV2 models (dropout off) take five steps on the same batch, one
   after the other in one process: rel-L2 distance of their weights after every step.
2. bench.py --dump-outputs twice as separate processes: per file max |a - b|, rel-L2 and whether
   the two are bit-identical, plus each run's ms/step."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def chain(steps=5, batch=256):
    import torch
    import bench
    from yet_another_mobilenet_series_b200.trainer import TrainStep
    dev = torch.device("cuda", 0)

    def make():
        m = bench.build_model()
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
        return TrainStep(m.to(dev), batch)

    g = torch.Generator().manual_seed(0)
    x = torch.randn(batch, 3, 224, 224, generator=g).to(torch.bfloat16).contiguous(
        memory_format=torch.channels_last)
    t = torch.randint(0, 1000, (batch,), generator=g)
    a, b = make(), make()
    a.load(x, t)
    b.load(x, t)
    for s in range(1, steps + 1):
        a.run()
        b.run()
        torch.cuda.synchronize()
        pa = torch.cat([p.detach().double().flatten() for p in a.model.parameters()])
        pb = torch.cat([p.detach().double().flatten() for p in b.model.parameters()])
        print("chain step %d: loss %.6f / %.6f, weights rel-L2 %.3e, max |a - b| %.3e" % (
            s, float(a.loss), float(b.loss), float((pa - pb).norm() / pb.norm()),
            float((pa - pb).abs().max())))


def dumps(steps, warmup):
    tmp = tempfile.mkdtemp()
    for r in ("a", "b"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1",
                            "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
                            "--no-gpu-context", "--dump-outputs", os.path.join(tmp, r)],
                           capture_output=True, text=True, check=True)
        line = json.loads(p.stdout.strip().splitlines()[-1])
        print("bench run %s: --steps %d --warmup %d, %.3f ms/step" % (r, steps, warmup,
                                                                     line["ms_per_step"]))
    for n in sorted(os.listdir(os.path.join(tmp, "a"))):
        a = np.load(os.path.join(tmp, "a", n)).astype(np.float64)
        b = np.load(os.path.join(tmp, "b", n)).astype(np.float64)
        print("%-20s %-12s max |a - b| %.3e  rel-L2 %.3e  bit-identical %s" % (
            n, a.shape, float(np.abs(a - b).max()),
            float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)), bool(np.array_equal(a, b))))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print("GPU:", q.stdout.strip() or "unknown")
    import __graft_entry__ as ge
    ge.build()
    chain()
    dumps(args.steps, args.warmup)
