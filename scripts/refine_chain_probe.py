"""Times the refinement chain alone (fused persistent kernel vs per-step GEMMs) on the bench-size valid-row count through
the evaluation forward's profile classes."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from iefvad_b200 import _lib, synth
from iefvad_b200.evaluate import Evaluator
from iefvad_b200.imf_vad import MMFMIL

dev = torch.device("cuda:0")
model = synth.build_model(MMFMIL, seed=0).to(dev).eval()
wl = bench.build_workload("ucf", 1, synth)
ev = Evaluator(model, wl["lengths"], wl["classes"], wl["gt"], device=dev)
img_c, ev_c = bench.make_features(ev, wl["video_ids"], wl["lengths"], synth, 768)
ev.set_device_features(img_c, ev_c)
with torch.no_grad():
    for mode in (False, True):
        model.temporal.refine_fused = mode
        for _ in range(3):
            ev.step()
        _lib.lib.iefvad_profile_enable(1)
        ev.step(with_metrics=False)
        torch.cuda.synchronize()
        ms, work, n = bench.read_kernel_profile(_lib)
        _lib.lib.iefvad_profile_enable(0)
        tot = {k: round(ms[i], 4) for i, k in enumerate(bench.KERNEL_CLASSES) if n[i]}
        print("refine_fused =", mode, tot, "sum", round(sum(ms), 4))
