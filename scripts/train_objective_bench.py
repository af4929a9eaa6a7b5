"""The training objective of train/ucf_train.py:73-102 (CLAS2 + cosine / norm regulariser + StudentT KL) with its
backward: the native kernels (iefvad_b200.loss.train_loss, csrc/train_loss.cu) against the caller's torch composition
(the package's CLAS2 + stock torch ops, as bench.py's train_step_measure builds it), on one GPU.

  1. Objective forward + backward alone at B = 64 and 128 clips x T = 256 x D = 768 (inputs of 200 / 400 MB, larger than
     the 126 MB L2): CUDA events per rep over alternating reps after a warm-up; median ms and achieved GB/s against the
     traffic floor (forward reads 16 D bytes per row; backward reads 16 D and writes 16 D).
  2. The training step of bench.py's loop (forward, loss, backward, AdamW; B = 64, train() mode) with each objective,
     alternating in one process: ms per step (CUDA events), library launches per step (iefvad_launch_count) and all
     device operations per step (kernels, memsets and copies seen by the torch profiler, in a separate pass).

python scripts/train_objective_bench.py [--out FILE] [--reps N] [--step-reps N]"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import iefvad_b200  # noqa: E402
from iefvad_b200 import _lib, synth  # noqa: E402
from iefvad_b200.loss import CLAS2, train_loss  # noqa: E402

T, D = 256, 768


def torch_objective(out, labels, lengths, nu):
    """train/ucf_train.py:73-102 as the caller writes it."""
    mu_i, mu_e, lv_i, lv_e = out["image_mu"], out["event_mu"], out["image_logvar"], out["event_logvar"]
    loss_c = CLAS2(out["logits"], labels, lengths, mu_i.device)
    cos = F.cosine_similarity(F.normalize(mu_i, p=2, dim=-1), F.normalize(mu_e, p=2, dim=-1), dim=-1)
    loss_reg = (1 - cos).mean() + torch.abs(torch.norm(mu_i, p=2, dim=-1) - torch.norm(mu_e, p=2, dim=-1)).mean()
    eli, ele = lv_i + math.log(nu / (nu + 1)), lv_e + math.log(nu / (nu + 1))
    return (loss_c + loss_reg - 0.5 * torch.mean(1 + eli - mu_i.pow(2) - eli.exp())
            - 0.5 * torch.mean(1 + ele - mu_e.pow(2) - ele.exp()))


def native_objective(out, labels, lengths, nu):
    return train_loss(out, labels, lengths, nu).total


OBJECTIVES = {"native": native_objective, "torch": torch_objective}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True)
    return {"nvidia_smi": q.stdout.strip(), "torch_device": torch.cuda.get_device_name()}


def objective_alone(B, reps):
    g = torch.Generator(device="cuda").manual_seed(B)
    xs = [torch.randn(B, T, D, device="cuda", generator=g) for _ in range(4)]
    xs[2].mul_(0.5)
    xs[3].mul_(0.5)
    logits = torch.randn(B, T, 1, device="cuda", generator=g)
    lengths = torch.randint(1, T + 1, (B,), device="cuda", generator=g)
    labels = torch.zeros(B, 14, device="cuda")
    labels[::2, 0] = 1.0
    leaves = [t.requires_grad_(True) for t in (logits, *xs)]
    out = dict(zip(("logits", "image_mu", "event_mu", "image_logvar", "event_logvar"), leaves))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    times = {k: {"fwd": [], "bwd": []} for k in OBJECTIVES}

    def once(name):
        for t in leaves:
            t.grad = None
        ev[0].record()
        loss = OBJECTIVES[name](out, labels, lengths, 8.0)
        ev[1].record()
        loss.backward()
        ev[2].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), float(loss)

    for _ in range(5):
        for name in OBJECTIVES:
            once(name)
    losses = {}
    for _ in range(reps):
        for name in OBJECTIVES:
            f, b, losses[name] = once(name)
            times[name]["fwd"].append(f)
            times[name]["bwd"].append(b)
    M = B * T
    floor = {"fwd": 16 * D * M, "bwd": 32 * D * M}
    res = {"B": B, "T": T, "D": D, "reps": reps, "input_MB": round(4 * M * D * 4 / 1e6, 1),
           "traffic_floor_MB": {k: round(v / 1e6, 1) for k, v in floor.items()}, "loss": losses}
    for name in OBJECTIVES:
        r = {}
        for part in ("fwd", "bwd"):
            ms = statistics.median(times[name][part])
            r[part + "_ms"] = round(ms, 4)
            r[part + "_GBps_vs_floor"] = round(floor[part] / ms / 1e6, 1)
        tot = [f + b for f, b in zip(times[name]["fwd"], times[name]["bwd"])]
        r["fwd_bwd_ms"] = round(statistics.median(tot), 4)
        r["fwd_bwd_ms_min_max"] = [round(min(tot), 4), round(max(tot), 4)]
        res[name] = r
    res["saving_ms"] = round(res["torch"]["fwd_bwd_ms"] - res["native"]["fwd_bwd_ms"], 4)
    return res


def training_step(B, reps):
    img, ev_, lengths, labels = (t.cuda() for t in synth.make_c4_batch(B))
    m = synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda().train()
    opt = torch.optim.AdamW(m.parameters(), lr=2e-5)
    nu = m.temporal.nu

    def step(name):
        loss = OBJECTIVES[name](m(img, ev_, None, None, lengths), labels, lengths, nu)
        opt.zero_grad()
        loss.backward()
        opt.step()

    for _ in range(3):
        for name in OBJECTIVES:
            step(name)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in OBJECTIVES}
    lib = {}
    for _ in range(reps):
        for name in OBJECTIVES:
            l0 = _lib.lib.iefvad_launch_count()
            e0.record()
            step(name)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
            lib[name] = _lib.lib.iefvad_launch_count() - l0
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for name in OBJECTIVES:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(name)
            torch.cuda.synchronize()
        kernels[name] = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    res = {"B": B, "T": T, "reps": reps, "mode": "train() (attention dropout 0.1), AdamW lr 2e-5"}
    for name in OBJECTIVES:
        res[name] = {"ms_per_step": round(statistics.median(times[name]), 3),
                     "ms_min_max": [round(min(times[name]), 3), round(max(times[name]), 3)],
                     "library_launches_per_step": int(lib[name]),
                     "device_ops_per_step": int(kernels[name]),
                     "torch_device_ops_per_step": int(kernels[name] - lib[name])}
    res["saving_ms"] = round(res["torch"]["ms_per_step"] - res["native"]["ms_per_step"], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--step-reps", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"card": card(), "objective": [objective_alone(B, a.reps) for B in (64, 128)],
           "training_step": training_step(64, a.step_reps)}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
