"""Row N3 - the training step against float64 references built here, at shapes and configurations the reference goldens
of tests/test_gpu_train.py do not reach.

- Training attention (csrc/train_attn_mma.cu; the FFMA kernels of csrc/train.cu under IEFVAD_TRAIN_ATTN=simt): out, lse,
  dq, dk, dv against float64 autograd of (softmax(q k^T / sqrt(dh)) * keep) v, with `keep` the documented Philox mask
  (oracle.iefvad_oracle.attention_keep), so train-mode gradients are checked exactly, not statistically.
- The whole step (train.ForwardFn + train.Clas2Fn) against float64 autograd of oracle/torch_port.py with the same
  per-layer masks: loss, the 8 outputs, every parameter gradient and the gradients of the image / event features.
- The elementwise backward operators (fuse_bwd, layernorm_bwd, colsum, clas2_bwd) at their edges.

Errors are max |got - ref| / max |ref| per tensor.  Worst measured on an NVIDIA B200 (1000 W power limit):
    attention, mma.sync 3xTF32 (bound 2e-5)   dh 32: 4.3e-6   dh 64: 4.1e-6   dh 96: 4.8e-6   dh 128: 6.7e-6
    attention, SIMT FFMA (bound 2e-5)         1.2e-6;  a wrong mask (words permuted, query / key swapped, seed's high
                                              word lost) leaves 0.55 - 0.86 on out, dq, dk and dv
    whole step, D = 128 (bound 1e-3)          H 4: 2.9e-5   H 2: 2.2e-5   H 1: 2.3e-5 (eval and train alike); fp16 inputs
                                              2.8e-4 (their gradient is rounded to fp16)
    whole step, D = 768, train mode           90 % quantile 4.6e-4, worst entry 0.10 (one ReLU gate flip, see the test)
    fuse_bwd 2.8e-7 (bound 2e-5), layernorm_bwd 1.3e-6 (bound 1e-5), colsum 1.5e-7 of sum |a| (bound 1e-6),
    clas2_bwd 4.3e-7 (bound 1e-5).
The whole file runs in about 15 s.  Needs a B200."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import iefvad_oracle as O
from oracle import torch_port
from test_gpu_train import reference_loss

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEEDS = (0, (0x00000007 << 32) | 0xDEADBEEF, 2 ** 62 - 77)      # low word only; distinct high / low words; near 2^62


@pytest.fixture(scope="module")
def pkg():
    assert torch.cuda.is_available()
    import iefvad_b200
    from iefvad_b200 import ops, synth
    return iefvad_b200, ops, synth


def rel_err(got, ref, scale=None) -> float:
    got = got.detach().double().cpu() if torch.is_tensor(got) else torch.as_tensor(got, dtype=torch.float64)
    ref = ref.detach().double().cpu() if torch.is_tensor(ref) else torch.as_tensor(ref, dtype=torch.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if scale is None:
        scale = float(ref.abs().max())
    return float((got - ref).abs().max()) / max(scale, 1e-300)


# ------------------------------------------------------------------------------------------------ training attention
def attention_ref(qkv, dout, B, T, H, keep=None):
    """float64 autograd of the training attention on the [B*T, 3D] qkv layout -> (out, lse, dq, dk, dv)."""
    qkv = qkv.detach().double().cpu().requires_grad_(True)
    D = qkv.shape[1] // 3
    dh = D // H
    q, k, v = (t.reshape(B, T, H, dh).transpose(1, 2) for t in qkv.split(D, dim=-1))
    s = (q / math.sqrt(dh)) @ k.transpose(-1, -2)
    lse = torch.logsumexp(s, dim=-1)
    p = torch.softmax(s, dim=-1)
    if keep is not None:
        p = p * torch.as_tensor(keep)
    out = (p @ v).transpose(1, 2).reshape(B * T, D)
    out.backward(dout.detach().double().cpu())
    g = qkv.grad
    return out.detach(), lse.detach(), g[:, :D], g[:, D:2 * D], g[:, 2 * D:]


def attention_inputs(B, T, H, dh, seed):
    g = torch.Generator("cpu").manual_seed(seed)
    D = H * dh
    qkv = torch.randn(B * T, 3 * D, generator=g)
    qkv[:, :2 * D] *= 1.5                          # scores of std ~2.2: peaked rows, not a flat average
    qkv[:, :D] += 0.3 * torch.randn(D, generator=g)  # a shared query offset (a bias of the in-projection)
    dout = torch.randn(B * T, D, generator=g)
    return qkv, dout


def attention_errors(got, ref, T):
    """-> {name: error}; dq and dk vanish at T = 1 (one key: the weights do not depend on the scores), so there they are
    measured against the scale of dv."""
    names = ("out", "lse", "dq", "dk", "dv")
    errs = {}
    for n, a, r in zip(names, got, ref):
        scale = float(ref[4].abs().max()) if (T == 1 and n in ("dq", "dk")) else None
        errs[n] = rel_err(a, r, scale)
    return errs


def run_attention(ops, qkv, dout, B, T, H, p, seed):
    D = qkv.shape[1] // 3
    qkv_d, dout_d = qkv.cuda(), dout.cuda()
    out, lse = ops.attention_train_fwd(qkv_d, B, T, H, p, seed)
    dqkv = ops.attention_train_bwd(qkv_d, out, dout_d, lse, B, T, H, p, seed)
    dqkv = dqkv.cpu()
    return out.cpu(), lse.cpu(), dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:]


ATTN_CASES = sorted(
    {(dh, T, 0.1, SEEDS[(i + j) % 3]) for i, dh in enumerate((32, 64, 96, 128))
     for j, T in enumerate((1, 31, 32, 33, 64, 65, 129, 300))}
    | {(96, 129, p, s) for p in (0.0, 0.1, 0.5) for s in SEEDS}
    | {(dh, T, p, SEEDS[1]) for dh in (32, 64, 128) for T in (65, 300) for p in (0.0, 0.5)})


@pytest.mark.parametrize("dh, T, p, seed", ATTN_CASES, ids=[f"dh{c[0]}-T{c[1]}-p{c[2]}-s{c[3]:x}" for c in ATTN_CASES])
def test_train_attention_matches_float64_with_the_exact_mask(pkg, dh, T, p, seed):
    _, ops, _ = pkg
    B, H = 2, 3                                   # b * H + h is not a power-of-two pattern
    qkv, dout = attention_inputs(B, T, H, dh, 1000 * dh + T)
    keep = O.attention_keep(seed, B, H, T, p) if p > 0 else None
    got = run_attention(ops, qkv, dout, B, T, H, p, seed)
    errs = attention_errors(got, attention_ref(qkv, dout, B, T, H, keep), T)
    print(f"attention dh {dh} T {T} p {p} seed {seed:#x}:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) <= 2e-5, errs


def test_train_attention_distinguishes_the_documented_mask_from_wrong_ones(pkg):
    """Non-vacuity: the 2e-5 bound above is far below what a mask with permuted words, (query, key) swapped in the counter
    or the seed's high word lost would leave."""
    _, ops, _ = pkg
    B, H, T, dh, p, seed = 2, 3, 128, 64, 0.1, SEEDS[1]
    qkv, dout = attention_inputs(B, T, H, dh, 7)
    got = run_attention(ops, qkv, dout, B, T, H, p, seed)
    keep = O.attention_keep(seed, B, H, T, p)
    right = attention_errors(got, attention_ref(qkv, dout, B, T, H, keep), T)
    assert max(right.values()) <= 2e-5, right
    k = np.arange(T)
    wrong = {
        "words permuted": keep[..., (k & ~3) | ((k + 1) & 3)],        # key k decided by word (k + 1) & 3 of its call
        "query / key swapped": keep.transpose(0, 1, 3, 2),
        "high word lost": O.attention_keep(seed & 0xFFFFFFFF, B, H, T, p),
    }
    for name, bad in wrong.items():
        errs = attention_errors(got, attention_ref(qkv, dout, B, T, H, bad), T)
        print(f"wrong mask ({name}):", {k: f"{v:.2e}" for k, v in errs.items()})
        assert errs["out"] > 1e-2 and errs["dv"] > 1e-2, (name, errs)       # >= 500x the bound


_SIMT_SCRIPT = r"""
import sys
import numpy as np
import torch
sys.path.insert(0, sys.argv[1])
from iefvad_b200 import ops
z = np.load(sys.argv[2])
res = {}
for name in z.files:
    if not name.startswith("qkv:"):
        continue
    case = name[4:]
    B, T, H, _, pm, seed = (int(v) for v in case.split("_"))
    qkv, dout = torch.from_numpy(z["qkv:" + case]).cuda(), torch.from_numpy(z["dout:" + case]).cuda()
    out, lse = ops.attention_train_fwd(qkv, B, T, H, pm / 1000, seed)
    dqkv = ops.attention_train_bwd(qkv, out, dout, lse, B, T, H, pm / 1000, seed)
    res["out:" + case], res["lse:" + case], res["dqkv:" + case] = out.cpu().numpy(), lse.cpu().numpy(), dqkv.cpu().numpy()
try:                                  # head dim 128 exists only on the mma.sync path: refused here proves the SIMT path ran
    ops.attention_train_fwd(torch.zeros(4, 3 * 128, device="cuda"), 1, 4, 1)
    res["dh128_refused"] = np.array(0)
except RuntimeError:
    res["dh128_refused"] = np.array(1)
np.savez(sys.argv[3], **res)
"""


def test_simt_train_attention_matches_float64_with_the_exact_mask(pkg, tmp_path):
    """The FFMA kernels of csrc/train.cu, selected by IEFVAD_TRAIN_ATTN=simt (read once per process, hence a child
    process with a timeout)."""
    B, H, seed = 2, 3, SEEDS[1]
    cases, data = [], {}
    for dh in (32, 64, 96):
        for T in (1, 33, 129):
            for p in (0.0, 0.1):
                qkv, dout = attention_inputs(B, T, H, dh, 31 * dh + T)
                case = f"{B}_{T}_{H}_{dh}_{int(round(p * 1000))}_{seed}"
                data[f"qkv:{case}"], data[f"dout:{case}"] = qkv.numpy(), dout.numpy()
                cases.append((dh, T, p, qkv, dout, case))
    np.savez(tmp_path / "in.npz", **data)
    env = dict(os.environ, IEFVAD_TRAIN_ATTN="simt")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-c", _SIMT_SCRIPT, ROOT, str(tmp_path / "in.npz"), str(tmp_path / "out.npz")]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-4000:]
    z = np.load(tmp_path / "out.npz")
    assert int(z["dh128_refused"]) == 1
    worst = 0.0
    for dh, T, p, qkv, dout, case in cases:
        D = H * dh
        keep = O.attention_keep(seed, B, H, T, p) if p > 0 else None
        d = torch.from_numpy(z["dqkv:" + case])
        got = (torch.from_numpy(z["out:" + case]), torch.from_numpy(z["lse:" + case]), d[:, :D], d[:, D:2 * D], d[:, 2 * D:])
        errs = attention_errors(got, attention_ref(qkv, dout, B, T, H, keep), T)
        worst = max(worst, max(errs.values()))
        assert max(errs.values()) <= 2e-5, (dh, T, p, errs)
    print("SIMT attention worst error:", worst)


# ------------------------------------------------------------------------------------------------ the whole training step
def clas2_64(logits, labels, lengths, device=None):
    """train/loss.py:18-30 in torch (differentiable): BCE of the mean of the int(len / 16 + 1) largest sigmoids per row."""
    B = logits.shape[0]
    p = torch.sigmoid(logits.reshape(B, -1))
    v = torch.stack([torch.topk(p[i, :n], int(n / 16 + 1)).values.mean() for i, n in enumerate(lengths.tolist())])
    return F.binary_cross_entropy(v, (1 - labels[:, 0]).to(v.dtype))


def train_step_pair(CLAS2, m, img, ev, lengths, labels, call_seed=None):
    """One `loss.backward()` through the CUDA module and the same step in float64 autograd of oracle/torch_port.py.
    img / ev: CUDA tensors (they may require grad).  In train() mode the module draws its Philox seed from torch's CPU
    generator (imf_vad.py: _forward_train); `call_seed` seeds that generator, and the reference redraws the same value.
    -> (got, ref): dicts of the loss, the 8 outputs, 'grad:<param>' and 'grad:img' / 'grad:ev'."""
    t = m.temporal
    B, T, _ = img.shape
    keep = None
    if m.training and t.dropout > 0:
        torch.manual_seed(call_seed)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        keep = {(mod, i): torch.from_numpy(O.attention_keep(seed + 1000 * mi + i, B, t.num_heads, T, float(t.dropout)))
                for mi, mod in enumerate(("image", "event")) for i in range(t.num_layers)}
        torch.manual_seed(call_seed)
    outs = {}

    def gpu_model(i, e, *_):
        outs.update(m(i, e, None, None, None))
        return outs
    loss, _ = reference_loss(gpu_model, CLAS2, img, ev, lengths, labels, float(t.nu))
    loss.backward()
    got = {"loss": loss.detach(), **{k: v.detach() for k, v in outs.items()}}
    for k, p in m.named_parameters():
        if p.requires_grad:
            got["grad:" + k] = p.grad
    P = {k: p.detach().double().cpu().requires_grad_(p.requires_grad) for k, p in m.named_parameters()}
    x64 = {n: x.detach().double().cpu().requires_grad_(x.requires_grad) for n, x in (("img", img), ("ev", ev))}
    ref_outs = {}

    def ref_model(i, e, *_):
        ref_outs.update(torch_port.forward(P, i, e, heads=t.num_heads, lambda_ref=float(t.lambda_ref),
                                           noise_model=t.noise_model, nu=float(t.nu), epsilon=float(t.epsilon), keep=keep,
                                           dtype=torch.float64))
        ref_outs["logits"].retain_grad()             # relu_flip_allowance starts from it
        return ref_outs
    ref_loss, _ = reference_loss(ref_model, clas2_64, x64["img"], x64["ev"], lengths.cpu(), labels.double().cpu(),
                                 float(t.nu))
    ref_loss.backward()
    ref = {"loss": ref_loss.detach(), **{k: v.detach() for k, v in ref_outs.items()}, "g_logits": ref_outs["logits"].grad}
    ref.update({"grad:" + k: p.grad for k, p in P.items() if p.requires_grad})
    for n, x in (("img", img), ("ev", ev)):
        if x.requires_grad:
            got["grad:" + n], ref["grad:" + n] = x.grad, x64[n].grad
    return got, ref


def small_model(iefvad_b200, synth, H, L, R, noise, train, seed=0):
    args = synth.default_args(visual_head=H, visual_layers=L, num_refinement_steps=R, noise_model=noise, nu=5)
    torch.manual_seed(seed)
    m = iefvad_b200.MMFMIL(14, 128, 256, 128, H, L, 8, 10, 10, "cuda", args)
    synth.perturb_(m, seed=seed + 1)             # nonzero biases and LayerNorm affines
    return m.cuda().train(train)


def small_batch(dtype=torch.float32):
    """B = 3 clips of T = 47 rows, lengths 47 (= T), 9 (< 16, k = 1) and 30; one normal and two abnormal labels."""
    g = torch.Generator("cpu").manual_seed(5)
    img, ev = (torch.randn(3, 47, 128, generator=g).to(dtype).cuda().requires_grad_(True) for _ in range(2))
    lengths = torch.tensor([47, 9, 30]).cuda()
    labels = torch.zeros(3, 14)
    labels[0, 0], labels[1, 3], labels[2, 7] = 1.0, 1.0, 1.0
    return img, ev, lengths, labels.cuda()


def assert_all_close(got, ref, bound, what):
    ref = {k: v for k, v in ref.items() if k != "g_logits"}
    assert set(got) == set(ref), (what, sorted(set(got) ^ set(ref)))
    errs = {k: rel_err(got[k], ref[k]) for k in ref}
    worst = max(errs, key=errs.get)
    print(f"{what}: worst {worst} {errs[worst]:.2e}, loss {errs['loss']:.2e}")
    bad = {k: v for k, v in errs.items() if not v < bound}
    assert not bad, (what, bad)
    return errs


STEP_CASES = [(H, L, R, noise, train) for H in (4, 2, 1) for L in (1, 2) for R in (0, 3)
              for noise in ("StudentT", "Gaussian") for train in (False, True)]


@pytest.mark.parametrize("H, L, R, noise, train", STEP_CASES,
                         ids=[f"H{c[0]}-L{c[1]}-R{c[2]}-{c[3]}-{'train' if c[4] else 'eval'}" for c in STEP_CASES])
def test_small_train_step_matches_float64_autograd(pkg, H, L, R, noise, train):
    """D = 128 (head dims 32 / 64 / 128), every parameter and both input gradients, eval and train (p = 0.1) mode."""
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = small_model(iefvad_b200, synth, H, L, R, noise, train)
    got, ref = train_step_pair(CLAS2, m, *small_batch(), call_seed=17)
    assert len([k for k in got if k.startswith("grad:")]) == len(list(m.parameters())) + 2
    assert_all_close(got, ref, 1e-3, f"D=128 H{H} L{L} R{R} {noise} {'train' if train else 'eval'}")


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_input_gradients_reach_the_features(pkg, dtype):
    """loss.backward() fills img.grad / ev.grad (in the inputs' dtype) and torch.autograd.grad sees the inputs as used."""
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = small_model(iefvad_b200, synth, 4, 2, 3, "StudentT", True)
    img, ev, lengths, labels = small_batch(dtype)
    got, ref = train_step_pair(CLAS2, m, img, ev, lengths, labels, call_seed=3)
    assert img.grad is not None and img.grad.dtype == dtype and ev.grad.dtype == dtype
    assert_all_close(got, ref, 1e-3, f"input gradients {dtype}")
    torch.manual_seed(3)
    loss, _ = reference_loss(lambda i, e, *_: m(i, e), CLAS2, img, ev, lengths, labels, float(m.temporal.nu))
    gi, ge = torch.autograd.grad(loss, (img, ev))
    assert torch.equal(gi, img.grad) and torch.equal(ge, ev.grad)      # same seed, same mask: the same gradients


def test_input_gradients_with_frozen_parameters(pkg):
    """Parameters frozen with requires_grad_(False), only the features require grad (e.g. attribution maps)."""
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = small_model(iefvad_b200, synth, 2, 2, 3, "Gaussian", False).requires_grad_(False)
    got, ref = train_step_pair(CLAS2, m, *small_batch(), call_seed=None)
    assert all(p.grad is None for p in m.parameters())
    assert sorted(k for k in got if k.startswith("grad:")) == ["grad:ev", "grad:img"]
    assert_all_close(got, ref, 1e-3, "frozen parameters")


def relu_flip_allowance(m, ref, tau=2.0 ** -16):
    """The ReLU gates of the refinement MLPs whose float64 pre-activation z[r, j] lies within tau * sum_k |W1[j, k] x[r, k]|
    of zero may go either way in the kernels (the split-bf16 GEMM keeps ~16 mantissa bits and the chain's input carries the
    encoder's ~1e-5 error).  A flipped gate moves dW1[j, :] by dh[r, j] x[r, :] and db1[j] by dh[r, j] (dh = gradient of
    the gate's output).  -> ({gradient key: per-entry sum of those moves over the ambiguous gates}, fraction of gates
    that are ambiguous); the float64 chain is recomputed from the reference's fusion outputs and logits gradient."""
    t = m.temporal
    D = t.embed_dim
    P = {k: p.detach().double().cpu() for k, p in m.named_parameters()}
    pre = "temporal.refinement_blocks."
    x = (ref["w_i"] * ref["image_mu"] + ref["w_e"] * ref["event_mu"]).reshape(-1, D).requires_grad_(True)
    taps = []
    with torch.enable_grad():
        for s in range(t.num_refinement_steps):
            W1, b1, W2, b2 = (P[f"{pre}{s}.{n}"] for n in ("0.weight", "0.bias", "2.weight", "2.bias"))
            z = x @ W1.T + b1
            h = torch.relu(z)
            h.retain_grad()
            taps.append((s, x.detach(), z.abs() < tau * (x.detach().abs() @ W1.abs().T + b1.abs()), h))
            x = x - float(t.lambda_ref) * (h @ W2.T + b2)
        logits = x @ P["temporal.classifier.weight"].T + P["temporal.classifier.bias"]
        assert float((logits.detach() - ref["logits"].reshape(-1, 1)).abs().max()) < 1e-9
        logits.backward(ref["g_logits"].reshape(-1, 1))
    allow, n_amb, n = {}, 0, 0
    for s, xs, amb, h in taps:
        moved = amb * h.grad.abs()
        allow[f"grad:{pre}{s}.0.weight"] = moved.T @ xs.abs()
        allow[f"grad:{pre}{s}.0.bias"] = moved.sum(0)
        n_amb, n = n_amb + int(amb.sum()), n + amb.numel()
    return allow, n_amb / n


def test_full_size_train_step_matches_float64_autograd(pkg):
    """The 768-d model (synth.build_model) in train() mode on 4 config-4 clips of T = 256 (fp16 features requiring grad),
    every entry of every gradient, with the rule of test_gpu_train.test_full_size_gradients_match_the_reference_autograd:
    norm within 2e-3, 90 % of the entries within 1e-3 of the tensor's scale and none beyond 5e-2 - plus, in the refinement
    MLPs' first-layer gradients, what flipping the ReLU gates that sit within rounding of zero would move (measured: one
    flip, unit 574 of step 0 at row 774, z = 4.6e-7 of sum |W x|, moves its dW1 row by up to 0.10 of the scale and db1 by
    0.058 - exactly the difference observed)."""
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda().train()
    img, ev, lengths, labels = synth.make_c4_batch(4)
    img, ev = img.cuda().requires_grad_(True), ev.cuda().requires_grad_(True)
    got, ref = train_step_pair(CLAS2, m, img, ev, lengths.cuda(), labels.cuda(), call_seed=29)
    assert abs(float(got["loss"]) - float(ref["loss"])) < 2e-4 * abs(float(ref["loss"]))
    allow, amb_frac = relu_flip_allowance(m, ref)
    assert amb_frac < 1e-3, amb_frac                 # the allowance covers a few gates, not the tensors
    worst_q, worst_max, n = 0.0, 0.0, 0
    for k in ref:
        if k in ("loss", "g_logits"):
            continue
        g = got[k].detach().double().cpu().reshape(-1)
        r = ref[k].reshape(-1)
        norm_ref = float(r.norm())
        assert abs(float(g.norm()) - norm_ref) < 2e-3 * norm_ref + 1e-12, k
        scale = max(norm_ref / math.sqrt(r.numel()), float(r.abs().max())) + 1e-20
        err = (g - r).abs() / scale
        q = float(np.quantile(err.numpy(), 0.9))
        excess = err - (5e-2 + allow[k].reshape(-1) / scale if k in allow else 5e-2)
        worst_q, worst_max = max(worst_q, q), max(worst_max, float(err.max()))
        assert q < 1e-3 and float(excess.max()) < 0, (k, q, float(err.max()), float(excess.max()))
        n += k.startswith("grad:")
    assert n == 78 + 2
    print(f"D=768 train step: worst 90 % quantile {worst_q:.2e}, worst entry {worst_max:.2e}, "
          f"ambiguous ReLU gates {amb_frac:.2e}")


# ------------------------------------------------------------------------------------------------ elementwise backward ops
def test_fuse_bwd_at_logvar_extremes_against_float64(pkg):
    """Gaussian and StudentT 5 / 8; logvar pairs from {-80, -30, 0, 30, 80} (weights saturating at 0 / 1, epsilon
    dominating the denominator) next to ordinary values; every upstream gradient absent and present.  Checked over the
    whole tensor and over the extreme entries alone."""
    _, ops, _ = pkg
    g = torch.Generator("cpu").manual_seed(11)
    n_rows, D = 40, 96
    mu = [torch.randn(n_rows, D, generator=g) for _ in range(2)]
    lv = [2 * torch.randn(n_rows, D, generator=g) for _ in range(2)]
    ext = torch.tensor([-80.0, -30.0, 0.0, 30.0, 80.0])
    grid_i, grid_e = ext.repeat_interleave(5), ext.repeat(5)              # all 25 pairs
    lv[0][:8] = grid_i.repeat(8 * D // 25 + 1)[:8 * D].view(8, D)
    lv[1][:8] = grid_e.repeat(8 * D // 25 + 1)[:8 * D].view(8, D)
    # upstream gradients of fused, w_i, w_e, mu_i, mu_e, logvar_i, logvar_e: all, all but one, one alone
    ups = [torch.randn(n_rows, D, generator=g) for _ in range(7)]
    patterns = [tuple(range(7))] + [tuple(j for j in range(7) if j != i) for i in range(7)] + [(i,) for i in range(7)]
    worst = 0.0
    for noise, nu in (("Gaussian", 8.0), ("StudentT", 5.0), ("StudentT", 8.0)):
        factor = 1.0 if noise == "Gaussian" else (nu + 1) / nu
        for present in patterns:
            gs = [ups[j] if j in present else None for j in range(7)]
            x = [t.double().requires_grad_(True) for t in (mu[0], mu[1], lv[0], lv[1])]
            wi, we = factor * torch.exp(-x[2]), factor * torch.exp(-x[3])
            den = wi + we + 1e-8
            nwi, nwe = wi / den, we / den
            fused = nwi * x[0] + nwe * x[1]
            terms = (fused, nwi, nwe, x[0], x[1], x[2], x[3])
            sum((t * u.double()).sum() for t, u in zip(terms, gs) if u is not None).backward()
            got = ops.fuse_bwd(*(t.cuda() for t in (mu[0], mu[1], lv[0], lv[1])),
                               *(u.cuda() if u is not None else None for u in gs), noise, nu)
            for name, a, t in zip(("d_mu_i", "d_mu_e", "d_lv_i", "d_lv_e"), got, x):
                a = a.cpu()
                ref = t.grad if t.grad is not None else torch.zeros_like(t)      # None: no upstream path reaches it
                assert torch.isfinite(a).all(), (noise, nu, present, name)
                for part in (slice(None), slice(0, 8)):
                    if float(ref[part].abs().max()) == 0.0:
                        assert float(a[part].abs().max()) == 0.0, (noise, nu, present, name)
                        continue
                    e = rel_err(a[part], ref[part])
                    worst = max(worst, e)
                    assert e < 2e-5, (noise, nu, present, name, part, e)
    print(f"fuse_bwd worst error: {worst:.2e}")


@pytest.mark.parametrize("D", [128, 768, 1024])
@pytest.mark.parametrize("rows", [1, 333, 16384])
def test_layernorm_bwd_with_large_means_against_float64(pkg, D, rows):
    """Rows whose mean is up to 30x their standard deviation (the mean is cancelled in fp32)."""
    _, ops, _ = pkg
    g = torch.Generator("cpu").manual_seed(D + rows)
    std = 0.5 + 1.5 * torch.rand(rows, 1, generator=g)
    mean = 30 * std * (2 * torch.rand(rows, 1, generator=g) - 1)
    mean[0] = 30 * std[0]
    x = mean + std * torch.randn(rows, D, generator=g)
    w = 1 + 0.2 * torch.randn(D, generator=g)
    b = 0.1 * torch.randn(D, generator=g)
    dy = torch.randn(rows, D, generator=g)
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
    F.layer_norm(x64, (D,), w64, b64).backward(dy.double())
    got = ops.layernorm_bwd(x.cuda(), w.cuda(), dy.cuda())
    errs = {n: rel_err(a, r.grad) for n, a, r in zip(("dx", "dweight", "dbias"), got, (x64, w64, b64))}
    print(f"layernorm_bwd D {D} rows {rows}:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) < 1e-5, errs


@pytest.mark.parametrize("rows", [1, 63, 64, 65, 16384, 100000])
@pytest.mark.parametrize("weighted", [False, True])
def test_colsum_against_float64(pkg, rows, weighted):
    """Row counts across the 64-row slabs and the 4 * num_sms cap on the slab count (csrc/train.cu: train_colsum_blocks),
    300 columns (more than one pass of the 256-thread block).  Bound relative to sum_r |a[r, c] w[r]| per column: fp32
    sums of zero-mean terms in this fixed two-level order stay ~1e-8 of it; 1e-6 still catches one row lost or doubled."""
    _, ops, _ = pkg
    g = torch.Generator("cpu").manual_seed(rows + weighted)
    a = torch.randn(rows, 300, generator=g)
    w = torch.randn(rows, generator=g) if weighted else None
    a64 = a.double() * (w.double()[:, None] if weighted else 1.0)
    ref, mag = a64.sum(0), a64.abs().sum(0)
    got = ops.colsum(a.cuda(), w.cuda() if weighted else None).cpu().double()
    err = float(((got - ref).abs() / mag).max())
    print(f"colsum rows {rows} weighted {weighted}: {err:.2e} of sum |a|")
    assert err < 1e-6, err


def test_clas2_bwd_against_float64_autograd(pkg):
    """Lengths 1, 15 (k = 1), 16, 17 (k = 2) and T (k = 7), both labels, upstream gradient 0.37; logits free of ties in
    [-3, 3] (the fp32 rounding of the top-k mean v is amplified by at most 1 / min(v, 1 - v) < 21)."""
    _, ops, _ = pkg
    T = 100
    lengths = torch.tensor([1, 15, 16, 17, T] * 2)
    B = lengths.numel()
    g = torch.Generator("cpu").manual_seed(4)
    logits = (torch.randperm(B * T, generator=g).view(B, T).float() / (B * T) * 6 - 3)
    labels = torch.zeros(B, 14)
    labels[:5, 0] = 1.0                             # normal: target 0
    labels[5:, 4] = 1.0                             # abnormal: target 1
    x64 = logits.double().requires_grad_(True)
    (0.37 * clas2_64(x64, labels.double(), lengths)).backward()
    lg, lb, ln = logits.cuda(), labels.cuda(), lengths.cuda()
    means, idx = ops.mil_topk_mean(lg, ln, apply_sigmoid=True, return_indices=True)
    got = ops.clas2_bwd(lg, means, lb, idx, torch.tensor(0.37).cuda()).cpu()
    ref = x64.grad
    assert torch.equal(got == 0, ref == 0)          # exactly the chosen positions carry a gradient
    err = rel_err(got, ref)
    print(f"clas2_bwd error: {err:.2e}")
    assert err < 1e-5, err
