"""Training-step time with the two attention-dropout masks (model.temporal.dropout_rng = "philox" / "torch"), on one GPU.

The loop body of train/ucf_train.py:60-106 through the drop-in in train() mode (attention dropout 0.1): forward, the
caller's torch objective, backward, AdamW; 768-d model, B clips x T = 256 of config 4.  The two modes alternate step by
step in one process after a warm-up of each; ms per step from CUDA events, median and spread over the reps.  Both modes
make one Philox call per 4 attention weights; torch mode adds the element -> (thread, iteration) division.

python scripts/train_dropout_rng_bench.py [--out FILE] [--batch B] [--reps N]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import iefvad_b200  # noqa: E402
from iefvad_b200 import synth  # noqa: E402
from train_objective_bench import card, torch_objective  # noqa: E402

MODES = ("philox", "torch")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    m = synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda().train()
    opt = torch.optim.AdamW(m.parameters(), lr=2e-5)
    img, ev, lengths, labels = (t.cuda() for t in synth.make_c4_batch(a.batch))
    nu = float(m.temporal.nu)

    def one_step(mode):
        m.temporal.dropout_rng = mode
        out = m(img, ev, None, None, lengths)
        loss = torch_objective(out, labels, lengths, nu)
        opt.zero_grad()
        loss.backward()
        opt.step()

    for mode in MODES:
        for _ in range(a.warmup):
            one_step(mode)
    torch.cuda.synchronize()
    times = {mode: [] for mode in MODES}
    for _ in range(a.reps):
        for mode in MODES:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one_step(mode)
            e1.record()
            e1.synchronize()
            times[mode].append(e0.elapsed_time(e1))
    res = {"batch": a.batch, "T": 256, "D": 768, "reps": a.reps, "card": card(),
           "ms_per_step": {k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in times.items()}}
    res["torch_over_philox"] = res["ms_per_step"]["torch"]["median"] / res["ms_per_step"]["philox"]["median"]
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
