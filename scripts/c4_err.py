"""Score error of every precision plan on config 4 (64 zero-padded clips) against the reference's golden logits,
for the default-init and the perturbed weight set.  Usage (GPU box): python scripts/c4_err.py [plan ...]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import load_golden  # noqa: E402
from iefvad_b200 import synth  # noqa: E402
from iefvad_b200.imf_vad import MMFMIL  # noqa: E402

plans = sys.argv[1:] or ["fp32", "HH", "B"]
img, ev, lengths, labels = synth.make_c4_batch()
valid = (np.arange(256)[None, :] < lengths.numpy()[:, None])
sig = lambda a: 1 / (1 + np.exp(-a.astype(np.float64)))  # noqa: E731
for wset in ("full_default", "full_perturbed"):
    z = load_golden(wset + ".npz")
    m = synth.build_model(MMFMIL, seed=0)
    if wset == "full_perturbed":
        synth.perturb_(m)
    m = m.cuda().eval()
    ref = sig(z["c4:logits"])
    for plan in plans:
        m.temporal.precision = plan
        with torch.no_grad():
            out = m(img.cuda(), ev.cuda(), None, None, None)["logits"].cpu().numpy().reshape(64, 256)
        e = np.abs(sig(out) - ref) / ref
        print(wset, plan, "valid rows %.2e   pad rows %.2e" % (e[valid].max(), e[~valid].max()), flush=True)
    # valid-rows mode with pad de-duplication (the evaluation default) against the same golden logits
    if "HH" in plans:
        m.temporal.precision = "HH"
        lens = [int(x) for x in lengths]
        rowmap = torch.cat([torch.arange(n) + c * 256 for c, n in enumerate(lens)]).to(torch.int32).cuda()
        with torch.no_grad():
            out = m.temporal.scores(img.cuda().half(), ev.cuda().half(), None, lens, rowmap)["logits"].cpu().numpy()
        e = np.abs(sig(out) - ref[valid]) / ref[valid]
        print(wset, "HH valid-rows + pad de-duplication (fp16 inputs): valid rows %.2e" % e.max(), flush=True)
