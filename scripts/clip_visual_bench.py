"""CLIP ViT-L/14 @ 224 image encoder (extracting/clip/model.py:206-241, the encoder of the feature-extraction step):
iefvad_b200.clip.VisionTransformer (default fp16 plan, one libiefvad.so call) against OpenAI's fp16 forward as
oracle/clip_visual.clip_visual_torch restates it, in eager torch fp16 on the same GPU.

Seeded random weights; fp16 inputs resident in device memory, N = 64 and 256 images per call.  The two arms alternate
rep by rep after a warm-up; each rep is timed with CUDA events, the median is reported.  The library arm converts its
weights on every call (it is stateless); the torch arm is handed weights already in fp16, as `clip.load` keeps them.
An N = 1 call of each arm shows the per-call overhead, weight conversion included.  FLOPs per image:
2 G^2 3P^2 W + layers (24 T W^2 + 4 T^2 W) + 2 W out, T = G^2 + 1; TFLOP/s are algorithmic (that count over time).

python scripts/clip_visual_bench.py [--out FILE] [--reps N]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from iefvad_b200.clip import VisionTransformer  # noqa: E402
from oracle import iefvad_oracle as O  # noqa: E402
from oracle import clip_visual as CV  # noqa: E402

R, P, W, LAYERS, HEADS, OUT = 224, 14, 1024, 24, 16, 768


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True)
    return {"nvidia_smi": q.stdout.strip(), "torch_device": torch.cuda.get_device_name()}


BURST_TFLOPS = 1671.1     # BASELINE.md: burst bf16 dense matmul (torch.matmul 8192^3) on one B200 at 1000 W


def burst_peak():
    """The burst dense 16-bit peak bench.py reports shares of: MEASURED_PEAKS.json where present, else BASELINE.md's."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["bf16_tflops"]), "MEASURED_PEAKS.json"
    except (OSError, KeyError, ValueError):
        return BURST_TFLOPS, "BASELINE.md (1 671.1 TFLOP/s burst bf16, one B200)"


def flops_per_image():
    G = R // P
    T = G * G + 1
    return 2 * G * G * 3 * P * P * W + LAYERS * (24 * T * W * W + 4 * T * T * W) + 2 * W * OUT


def timed(fn, x):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn(x)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    sd = {k: torch.from_numpy(v).float() for k, v in CV.clip_visual_params(R, P, W, LAYERS, OUT, seed=0).items()}
    m = VisionTransformer(R, P, W, LAYERS, HEADS, OUT)
    m.load_state_dict(sd)
    m = m.cuda().eval().requires_grad_(False)
    # clip.load's fp16 model: LayerNorm parameters stay fp32, everything else fp16
    sd16 = {k: (v if (".ln_" in k or k.startswith("ln_")) else v.half()).cuda() for k, v in sd.items()}
    del sd
    arms = {"iefvad": lambda x: m(x), "torch_fp16": lambda x: CV.clip_visual_torch(x, sd16, HEADS, torch.float16)}
    fl = flops_per_image()
    peak, peak_src = burst_peak()
    res = {"card": card(), "config": {"R": R, "P": P, "width": W, "layers": LAYERS, "heads": HEADS, "output_dim": OUT,
                                      "input_dtype": "float16", "plan": m.precision},
           "gflop_per_image": round(fl / 1e9, 2), "peak_tflops": peak, "peak_source": peak_src, "runs": []}
    g = torch.Generator("cpu").manual_seed(1)
    with torch.no_grad():
        for N in (1, 64, 256):
            x = torch.randn((N, 3, R, R), generator=g).half().cuda()
            for fn in arms.values():             # warm-up: module loads, allocator pools, library algorithm choices
                fn(x)
                fn(x)
            torch.cuda.synchronize()
            times = {k: [] for k in arms}
            outs = {}
            for _ in range(a.reps):
                for k, fn in arms.items():
                    t, outs[k] = timed(fn, x)
                    times[k].append(t)
            row = {"N": N, "reps": a.reps,
                   "max_norm_err_iefvad_vs_torch_fp16": O.max_norm_err(outs["iefvad"].float().cpu().numpy(),
                                                                        outs["torch_fp16"].float().cpu().numpy())}
            for k, ts in times.items():
                ms = statistics.median(ts)
                tf = fl * N / (ms * 1e-3) / 1e12
                row[k] = {"ms": round(ms, 3), "ms_min_max": [round(min(ts), 3), round(max(ts), 3)],
                          "images_per_s": round(N / (ms * 1e-3), 1), "tflops": round(tf, 1),
                          "share_of_peak": round(tf / peak, 4)}
            row["speedup_vs_torch_fp16"] = round(row["torch_fp16"]["ms"] / row["iefvad"]["ms"], 3)
            res["runs"].append(row)
            print(json.dumps(row), flush=True)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
