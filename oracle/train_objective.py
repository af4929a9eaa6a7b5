"""CPU restatement of the training objective (test infrastructure only, like oracle/iefvad_oracle.py: nothing in the
product package imports it).  `train_objective` restates, in float64 numpy, the loss the reference's training loop builds
from the module's outputs (train/ucf_train.py:73-102) and its gradient, the arithmetic of csrc/train_loss.cu."""
from __future__ import annotations

import math
from typing import Dict, Sequence

import numpy as np

from oracle.iefvad_oracle import mil_topk, sigmoid


def train_objective(logits, labels, lengths, mu_i, mu_e, lv_i, lv_e, nu: float, reg_weight: float = 1.0,
                    kl_weight: float = 1.0, upstream: Sequence[float] = (1.0, 0.0, 0.0, 0.0)) -> Dict[str, np.ndarray]:
    """The training loss of train/ucf_train.py:73-102 and its gradient, in float64.  mu_* / lv_* [B, T, D], logits [B, T, 1].

        loss_cls = CLAS2(logits, labels, lengths)                                           train/loss.py:18-30
        cos      = cosine_similarity(normalize(mu_i), normalize(mu_e))                      :75-82
        loss_reg = mean(1 - cos) + mean |norm(mu_i) - norm(mu_e)|                           :75-82
        loss_kl  = -0.5 mean(1 + eli - mu_i^2 - exp(eli)) - 0.5 mean(same for e), el = lv + log(nu / (nu + 1))   :93-98
        total    = loss_cls + reg_weight loss_reg + kl_weight loss_kl

    with torch's edge rules: F.normalize divides by max(|x|, 1e-12) (the clamp passes no gradient below it);
    cosine_similarity divides each factor by max(|x|, 1e-8), the clamp applied without autograd, so the gradient
    reaches the norm as if unclamped (torch/.../Distance.cpp); the gradients of |x| at 0 and of a norm at the zero
    vector are 0.  The means run over every row, pad rows included.  `upstream` = (g_total, g_cls, g_reg, g_kl): the
    gradients returned are those of g_total total + g_cls loss_cls + g_reg loss_reg + g_kl loss_kl."""
    f64 = lambda t: np.asarray(t, dtype=np.float64)  # noqa: E731
    a, b, la, lb = (f64(t) for t in (mu_i, mu_e, lv_i, lv_e))
    B, T, D = a.shape
    M, N = B * T, B * T * D
    a, b, la, lb = (t.reshape(M, D) for t in (a, b, la, lb))
    g_total, g_cls, g_reg, g_kl = (float(g) for g in upstream)
    G_reg, G_kl, G_cls = g_total * reg_weight + g_reg, g_total * kl_weight + g_kl, g_total + g_cls
    # CLAS2 and its gradient (the mean-reduced BCE of the mean of the k largest sigmoids of each row)
    p = sigmoid(f64(logits).reshape(B, T))
    y = 1.0 - f64(labels)[:, 0]
    v = np.zeros(B)
    d_logits = np.zeros((B, T))
    for r in range(B):
        n = int(lengths[r])
        k = int(n / 16 + 1)
        vals, idx = mil_topk(p[r, :n], k)
        v[r] = vals.mean()
        dv = (v[r] - y[r]) / max((1.0 - v[r]) * v[r], 1e-12) / B              # ATen binary_cross_entropy_backward
        d_logits[r, idx] = G_cls * dv / k * p[r, idx] * (1.0 - p[r, idx])
    loss_cls = -(y * np.maximum(np.log(v), -100.0) + (1 - y) * np.maximum(np.log1p(-v), -100.0)).mean()
    # regulariser
    sa, sb, sab = (a * a).sum(1), (b * b).sum(1), (a * b).sum(1)
    na, nb = np.sqrt(sa), np.sqrt(sb)
    ca, cb = np.maximum(na, 1e-12), np.maximum(nb, 1e-12)              # F.normalize
    cu, cv = np.maximum(na / ca, 1e-8), np.maximum(nb / cb, 1e-8)      # cosine_similarity of the normalised rows
    cos = sab / (ca * cb * cu * cv)
    loss_reg = (1.0 - cos).mean() + np.abs(na - nb).mean()
    gc = -G_reg / M                                                    # d / d cos_r
    inv = lambda x: np.divide(1.0, x, out=np.zeros_like(x), where=x > 0)  # noqa: E731  (norm gradient at 0 is 0)
    sgn = np.sign(na - nb)

    def d_reg(x, y_, nx, cx, cux, cvy, cy, other_sign):
        # u = x / cx, cos = (u . w) / (cux cvy) with w = y / cy: d cos / d u = w / (cux cvy) - (cos / cux) x / nx,
        # then through normalize: d / dx = g_u / cx - (g_u . x) / cx^2 [nx >= 1e-12] x / nx
        g_u_w = gc / (cux * cvy)
        g_u_x = -gc * cos / cux * inv(nx)
        g_u_dot_x = g_u_w * (x * (y_ / cy[:, None])).sum(1) + g_u_x * (nx * nx)
        alpha = g_u_w / (cy * cx)
        beta = g_u_x / cx - g_u_dot_x / (cx * cx) * (nx >= 1e-12) * inv(nx) + other_sign * G_reg / M * inv(nx)
        return alpha[:, None] * y_ + beta[:, None] * x

    d_a = d_reg(a, b, na, ca, cu, cv, cb, sgn) + G_kl / N * a
    d_b = d_reg(b, a, nb, cb, cv, cu, ca, -sgn) + G_kl / N * b
    # KL term
    c = math.log(nu / (nu + 1))
    ea, eb = la + c, lb + c
    loss_kl = -0.5 * (1 + ea - a * a - np.exp(ea)).mean() - 0.5 * (1 + eb - b * b - np.exp(eb)).mean()
    d_la = 0.5 * G_kl / N * (np.exp(ea) - 1.0)
    d_lb = 0.5 * G_kl / N * (np.exp(eb) - 1.0)
    total = loss_cls + reg_weight * loss_reg + kl_weight * loss_kl
    shape = (B, T, D)
    return {"total": np.float64(total), "classification": np.float64(loss_cls), "regulariser": np.float64(loss_reg),
            "kl": np.float64(loss_kl), "d_logits": d_logits.reshape(B, T, 1), "d_mu_i": d_a.reshape(shape),
            "d_mu_e": d_b.reshape(shape), "d_lv_i": d_la.reshape(shape), "d_lv_e": d_lb.reshape(shape)}
