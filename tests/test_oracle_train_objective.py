"""oracle.train_objective.train_objective (the training loss of train/ucf_train.py:73-102 and its gradient, float64) against
float64 torch autograd of the loop's own torch ops, including their edge rules: zero rows (the normalize / cosine clamps),
equal norms (|x| at 0), parallel and anti-parallel rows and large log-variances.  CPU only."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.train_objective import train_objective


def torch_objective(logits, labels, lengths, mu_i, mu_e, lv_i, lv_e, nu, reg_weight=1.0, kl_weight=1.0):
    """train/ucf_train.py:73-102 verbatim (CLAS2 of train/loss.py:18-30 in torch) -> (total, cls, reg, kl)."""
    B = logits.shape[0]
    p = torch.sigmoid(logits.reshape(B, -1))
    v = torch.stack([torch.topk(p[i, :n], int(n / 16 + 1)).values.mean() for i, n in enumerate(lengths.tolist())])
    loss_cls = F.binary_cross_entropy(v, (1 - labels[:, 0]).to(v.dtype))
    cos_sim = F.cosine_similarity(F.normalize(mu_i, p=2, dim=-1), F.normalize(mu_e, p=2, dim=-1), dim=-1)
    loss_reg = (1 - cos_sim).mean() + torch.abs(torch.norm(mu_i, p=2, dim=-1) - torch.norm(mu_e, p=2, dim=-1)).mean()
    eli = lv_i + math.log(nu / (nu + 1))
    ele = lv_e + math.log(nu / (nu + 1))
    loss_kl = -0.5 * torch.mean(1 + eli - mu_i.pow(2) - eli.exp()) - 0.5 * torch.mean(1 + ele - mu_e.pow(2) - ele.exp())
    return loss_cls + reg_weight * loss_reg + kl_weight * loss_kl, loss_cls, loss_reg, loss_kl


NAMES = ("total", "classification", "regulariser", "kl")
GRADS = ("d_logits", "d_mu_i", "d_mu_e", "d_lv_i", "d_lv_e")


def torch_reference(inputs, labels, lengths, nu, reg_weight=1.0, kl_weight=1.0, upstream=(1.0, 0.0, 0.0, 0.0),
                    dtype=torch.float64, device="cpu"):
    """The four scalars and the five input gradients of sum_i upstream[i] * scalar_i by torch autograd."""
    xs = [torch.as_tensor(np.asarray(t)).to(device, dtype).requires_grad_(True) for t in inputs]
    outs = torch_objective(xs[0], torch.as_tensor(np.asarray(labels)).to(device, dtype),
                           torch.as_tensor(np.asarray(lengths)).to(device), *xs[1:], nu, reg_weight, kl_weight)
    sum(g * o for g, o in zip(upstream, outs) if g != 0).backward()
    res = {n: o.detach() for n, o in zip(NAMES, outs)}
    res.update({n: x.grad if x.grad is not None else torch.zeros_like(x) for n, x in zip(GRADS, xs)})
    return res


def objective_inputs(B, T, D, seed, edge=False):
    """Seeded fp32 (logits, mu_i, mu_e, lv_i, lv_e), labels, lengths.  edge=True plants, in clip 0: a zero mu_i row, an
    anti-parallel pair (mu_e = -mu_i: equal norms, cos = -1), a parallel pair (mu_e = 3 mu_i, cos = 1) and rows of
    log-variance -80, -30, 0, 30, 80."""
    g = np.random.default_rng(seed)
    logits = g.standard_normal((B, T, 1)).astype(np.float32)
    mu_i, mu_e = (g.standard_normal((B, T, D)).astype(np.float32) for _ in range(2))
    lv_i, lv_e = ((0.5 * g.standard_normal((B, T, D))).astype(np.float32) for _ in range(2))
    if edge:
        mu_i[0, 0] = 0.0
        mu_e[0, 1] = -mu_i[0, 1]
        mu_e[0, 2] = 3.0 * mu_i[0, 2]
        for j, lv in enumerate((-80.0, -30.0, 0.0, 30.0, 80.0)):
            lv_i[0, 3 + j] = lv
            lv_e[0, 3 + j, : D // 2] = lv
    labels = np.zeros((B, 14), dtype=np.float32)
    labels[::2, 0] = 1.0
    labels[1::2, 3] = 1.0
    lengths = np.array([T, 1, 9] + [int(x) for x in g.integers(1, T + 1, size=max(B - 3, 0))], dtype=np.int64)[:B]
    return (logits, mu_i, mu_e, lv_i, lv_e), labels, lengths


def rel(got, ref):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return float(np.max(np.abs(got - ref))) / max(float(np.max(np.abs(ref))), 1e-300)


CASES = [(3, 47, 128, False), (2, 20, 768, False), (3, 47, 128, True), (3, 20, 768, True)]


@pytest.mark.parametrize("B, T, D, edge", CASES, ids=[f"{c[0]}x{c[1]}x{c[2]}{'-edge' if c[3] else ''}" for c in CASES])
@pytest.mark.parametrize("weights, upstream", [((1.0, 1.0), (1.0, 0.0, 0.0, 0.0)), ((0.01, 0.01), (0.5, 2.0, -1.0, 3.0)),
                                               ((0.0, 1.0), (0.0, 0.0, 1.0, 0.0))])
def test_train_objective_matches_float64_autograd(B, T, D, edge, weights, upstream):
    inputs, labels, lengths = objective_inputs(B, T, D, seed=B * T + D, edge=edge)
    nu = 5.0
    got = train_objective(inputs[0], labels, lengths, *inputs[1:], nu, *weights, upstream=upstream)
    ref = torch_reference(inputs, labels, lengths, nu, *weights, upstream=upstream)
    for n in NAMES:
        assert abs(float(got[n]) - float(ref[n])) <= 1e-12 * abs(float(ref[n])) + 1e-15, (n, float(got[n]), float(ref[n]))
    for n in GRADS:
        assert got[n].shape == tuple(ref[n].shape), n
        assert rel(got[n], ref[n]) <= 1e-12, (n, rel(got[n], ref[n]))


def test_edge_rows_take_torch_values():
    """The zero row gets torch's very large normalize-clamp gradient, the anti-parallel pair the zero subgradient of |x|
    at 0, and the parallel pair cos = 1."""
    B, T, D = 1, 8, 128
    inputs, labels, lengths = objective_inputs(B, T, D, seed=3, edge=True)
    got = train_objective(inputs[0], labels, lengths, *inputs[1:], 8.0)
    row0 = np.abs(got["d_mu_i"][0, 0]).max()
    assert row0 > 1e17 * max(np.abs(got["d_mu_i"][0, 1:]).max(), 1e-30)      # ~1e20 / M
    a, b = (inputs[1][0, 1].astype(np.float64), inputs[2][0, 1].astype(np.float64))
    assert np.linalg.norm(a) == np.linalg.norm(b)
    ref = torch_reference(inputs, labels, lengths, 8.0)
    assert rel(got["d_mu_i"][0, 1], ref["d_mu_i"][0, 1]) <= 1e-12
