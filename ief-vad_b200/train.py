"""Training step of the drop-in module (SURVEY 8f row N3): `loss.backward()` of the reference's loops
(train/ucf_train.py:60-106, train/xd_train.py:45-80) through `MMFMIL.forward` and `CLAS2`.

The reference's loop builds its loss in the CALLER from `outputs['logits']` (through CLAS2) and from
`outputs['image_mu' / 'event_mu' / 'image_logvar' / 'event_logvar']` (cosine / norm regulariser, KL term), so the drop-in
contract is: the forward's outputs carry a grad_fn, and backward turns the gradients of those outputs into gradients of
the 78 parameters and, when the image / event features require grad, of those inputs (the gradient reaching each
modality's first attention layer; fp32, cast by autograd to the input's dtype).  `ForwardFn` is that autograd node.
Its forward is the model composed from the library's stand-alone operators (tcgen05 GEMMs with the 3-term bf16 split -
gradients need fp32's exponent range, fp16 operands would flush them - the 3xTF32 tensor-core training attention of
csrc/train_attn.cu, fp32 LayerNorm / fusion kernels) keeping what the backward needs; its backward runs entirely in
libiefvad.so kernels too: dgrad = linear(dY, W^T), wgrad = linear(dY^T, X^T) on the same tcgen05 GEMM, the attention
backward of csrc/train_attn.cu and the LayerNorm / fusion / ReLU backward kernels of csrc/train.cu.  torch only owns the
buffers and the autograd graph.

Attention dropout (p = 0.1, active in train() mode like nn.MultiheadAttention): a counter-based Philox4x32-10 mask,
regenerated, not stored, by the backward (include/iefvad.h: iefvad_dropout).  With `dropout_rng = "philox"` (the default)
it is the library's own mask, a pure function of (seed, layer, batch element, head, query, key), so train-mode runs
match the reference statistically; with `dropout_rng = "torch"` it is torch.native_dropout's mask for the CUDA
generator's state, bit for bit, so train-mode forward and gradients match the reference's autograd to fp32 GEMM
accuracy, as they do in eval() mode (or with dropout = 0)."""
from __future__ import annotations

from typing import List

import torch

from . import ops

_PLAN = "split"          # 3-term bf16 split: ~16 mantissa bits with fp32's exponent range (gradients span 1e-8 .. 1e+1)
_MODS = ("image", "event")


def _lin(x, w, b=None, resid=None, alpha=1.0, act=None):
    return ops.linear(x, w, b, resid=resid, alpha=alpha, act=act, plan=_PLAN)


def _dgrad(dy, w, resid=None, alpha=1.0):
    """dX = alpha * dY . W (+ resid): the forward GEMM with W^T [in, out] as its K-major weight."""
    return _lin(dy, ops.transpose(w), None, resid=resid, alpha=alpha)


def _wgrad(dy, x, alpha=1.0):
    """dW [out, in] = alpha * dY^T . X from row-major dY [M, out], X [M, in] (iefvad_wgrad: both operands transposed straight
    into the GEMM's bf16 hi / lo form, split-K over the rows)."""
    return ops.wgrad(dy, x, alpha)


def _drop(cfg, mi: int, i: int) -> dict:
    """Dropout arguments of attention layer i of modality mi (0 image, 1 event) for ops.attention_train_fwd / _bwd."""
    if cfg["offsets"] is not None:
        return dict(p_drop=cfg["p_drop"], seed=cfg["seed"], rng="torch", offset=cfg["offsets"][mi * cfg["layers"] + i],
                    threads=cfg["threads"])
    return dict(p_drop=cfg["p_drop"], seed=cfg["seed"] + 1000 * mi + i)


def param_list(temporal) -> List[torch.nn.Parameter]:
    """Flat parameter order of the autograd node (any fixed order works; this one follows the forward)."""
    ps = []
    for mod in _MODS:
        for i in range(temporal.num_layers):
            a = getattr(temporal, f"{mod}_attn_layers")[i]
            n = getattr(temporal, f"{mod}_norms")[i]
            ps += [a.in_proj_weight, a.in_proj_bias, a.out_proj.weight, a.out_proj.bias, n.weight, n.bias]
        wh = getattr(temporal, f"whiten_{mod}")
        ps += [wh.weight, wh.bias]
        for kind in ("mu", "logvar"):
            lin = getattr(temporal, f"{mod}_{kind}")
            ps += [lin.weight, lin.bias]
    for i in range(temporal.num_refinement_steps):
        blk = temporal.refinement_blocks[i]
        ps += [blk[0].weight, blk[0].bias, blk[2].weight, blk[2].bias]
    ps += [temporal.classifier.weight, temporal.classifier.bias]
    return ps


class ForwardFn(torch.autograd.Function):
    """(cfg, img, ev, *params) -> (fused, logits, image_mu, event_mu, image_logvar, event_logvar, w_i, w_e)."""

    @staticmethod
    def forward(ctx, cfg, img, ev, *params):
        B, T, D = img.shape
        M = B * T
        L, R, H = cfg["layers"], cfg["steps"], cfg["heads"]
        it = iter(params)
        saved = []                      # tensors for backward, in the order backward pops them
        enc, heads_out = {}, {}
        for mi, (mod, x_in) in enumerate(zip(_MODS, (img, ev))):
            x = x_in.reshape(M, D).float().contiguous()
            for i in range(L):
                w_in, b_in, w_o, b_o, g, bt = (next(it) for _ in range(6))
                qkv = _lin(x, w_in, b_in)
                ctx_, lse = ops.attention_train_fwd(qkv, B, T, H, **_drop(cfg, mi, i))
                y = _lin(ctx_, w_o, b_o, resid=x)                                   # x + MHA(x)        :115-116
                saved += [x, qkv, ctx_, lse, y]
                x = ops.layernorm(y, g, bt)
            g, bt = next(it), next(it)
            saved.append(x)                                                        # input of the whitening LN :117
            e = ops.layernorm(x, g, bt)
            w_mu, b_mu, w_lv, b_lv = (next(it) for _ in range(4))
            enc[mod] = e
            heads_out[mod] = (_lin(e, w_mu, b_mu), _lin(e, w_lv, b_lv))          # :125-128
            saved.append(e)
        mu_i, lv_i = heads_out["image"]
        mu_e, lv_e = heads_out["event"]
        w_i, w_e, fused = ops.fuse(mu_i, mu_e, lv_i, lv_e, cfg["noise_model"], cfg["nu"], cfg["epsilon"])   # :130-144
        x = fused
        for _ in range(R):                                                         # :146-149
            w1, b1, w2, b2 = (next(it) for _ in range(4))
            h = _lin(x, w1, b1, act="relu")
            xn = _lin(h, w2, b2, resid=x, alpha=-cfg["lambda_ref"])
            saved += [x, h]
            x = xn
        w_c, b_c = next(it), next(it)
        logits = ops.classifier(x, w_c, b_c)                                       # :150
        saved += [x, mu_i, mu_e, lv_i, lv_e]
        ctx.cfg = cfg
        ctx.shape = (B, T, D)
        ctx.save_for_backward(*saved, *params)
        ctx.n_saved = len(saved)
        v = lambda t: t.view(B, T, D)  # noqa: E731
        return v(x), logits.view(B, T, 1), v(mu_i), v(mu_e), v(lv_i), v(lv_e), v(w_i), v(w_e)

    @staticmethod
    def backward(ctx, g_fused, g_logits, g_mu_i, g_mu_e, g_lv_i, g_lv_e, g_wi, g_we):
        cfg = ctx.cfg
        B, T, D = ctx.shape
        M = B * T
        L, R, H = cfg["layers"], cfg["steps"], cfg["heads"]
        lam = cfg["lambda_ref"]
        saved = list(ctx.saved_tensors[:ctx.n_saved])
        params = list(ctx.saved_tensors[ctx.n_saved:])
        grads: List[torch.Tensor] = [None] * len(params)
        flat = lambda g: None if g is None else g.reshape(M, -1).float().contiguous()  # noqa: E731
        g_fused, g_logits, g_mu_i, g_mu_e, g_lv_i, g_lv_e, g_wi, g_we = map(
            flat, (g_fused, g_logits, g_mu_i, g_mu_e, g_lv_i, g_lv_e, g_wi, g_we))
        lv_e, lv_i, mu_e, mu_i, x_last = saved.pop(), saved.pop(), saved.pop(), saved.pop(), saved.pop()
        # ---- classifier (:150)
        pi = len(params) - 2
        w_c = params[pi]
        if g_logits is not None:
            dx = ops.outer(g_logits, w_c)
            if g_fused is not None:
                ops.axpy_(dx, g_fused)
            grads[pi] = ops.colsum(x_last, row_weight=g_logits).view(1, D)
            grads[pi + 1] = ops.colsum(g_logits.view(M, 1)).view(1)
        else:
            dx = g_fused.clone() if g_fused is not None else torch.zeros((M, D), dtype=torch.float32, device=x_last.device)
            grads[pi] = torch.zeros_like(w_c)
            grads[pi + 1] = torch.zeros_like(params[pi + 1])
        # ---- refinement chain, last step first (:146-149): x' = x - lam (W2 relu(W1 x + b1) + b2)
        for s in reversed(range(R)):
            pi -= 4
            w1, w2 = params[pi], params[pi + 2]
            h, x = saved.pop(), saved.pop()
            grads[pi + 3] = ops.axpy_(torch.zeros(D, dtype=torch.float32, device=dx.device), ops.colsum(dx), -lam)
            grads[pi + 2] = _wgrad(dx, h, alpha=-lam)
            dz = ops.relu_bwd(_dgrad(dx, w2, alpha=-lam), h)
            grads[pi + 1] = ops.colsum(dz)
            grads[pi] = _wgrad(dz, x)
            dx = _dgrad(dz, w1, resid=dx)
        # ---- fusion (:130-144): dx is the gradient of `fused`
        d_mu_i, d_mu_e, d_lv_i, d_lv_e = ops.fuse_bwd(mu_i, mu_e, lv_i, lv_e, dx, g_wi, g_we, g_mu_i, g_mu_e, g_lv_i, g_lv_e,
                                                     cfg["noise_model"], cfg["nu"], cfg["epsilon"])
        # ---- heads, whitening LN and the attention stacks, event modality first (reverse of the forward)
        d_in = [None, None]                            # gradients of img / ev
        for mi in (1, 0):
            d_mu, d_lv = (d_mu_i, d_lv_i) if mi == 0 else (d_mu_e, d_lv_e)
            base = mi * (6 * L + 6)
            ph = base + 6 * L + 2                      # mu.weight, mu.bias, logvar.weight, logvar.bias
            e = saved.pop()
            grads[ph] = _wgrad(d_mu, e)
            grads[ph + 1] = ops.colsum(d_mu)
            grads[ph + 2] = _wgrad(d_lv, e)
            grads[ph + 3] = ops.colsum(d_lv)
            d_e = _dgrad(d_lv, params[ph + 2], resid=_dgrad(d_mu, params[ph]))
            x_w = saved.pop()
            dxm, grads[ph - 2], grads[ph - 1] = ops.layernorm_bwd(x_w, params[ph - 2], d_e)
            for i in reversed(range(L)):
                p0 = base + 6 * i
                w_in, w_o, g = params[p0], params[p0 + 2], params[p0 + 4]
                y, lse, ctx_, qkv, x = saved.pop(), saved.pop(), saved.pop(), saved.pop(), saved.pop()
                dy, grads[p0 + 4], grads[p0 + 5] = ops.layernorm_bwd(y, g, dxm)
                grads[p0 + 2] = _wgrad(dy, ctx_)
                grads[p0 + 3] = ops.colsum(dy)
                dqkv = ops.attention_train_bwd(qkv, ctx_, _dgrad(dy, w_o), lse, B, T, H, **_drop(cfg, mi, i))
                grads[p0] = _wgrad(dqkv, x)
                grads[p0 + 1] = ops.colsum(dqkv)
                dxm = _dgrad(dqkv, w_in, resid=dy)     # residual path + attention path
            if ctx.needs_input_grad[1 + mi]:
                d_in[mi] = dxm.view(B, T, D)           # fp32; autograd casts it to the input's dtype
        assert not saved
        grads = [g.view_as(p) if g is not None else None for g, p in zip(grads, params)]
        return (None, *d_in, *grads)


class Clas2Fn(torch.autograd.Function):
    """train/loss.py:18-30 with a gradient: (logits [B, T, 1], labels, lengths) -> scalar loss."""

    @staticmethod
    def forward(ctx, logits, labels, lengths):
        means, idx = ops.mil_topk_mean(logits, lengths, apply_sigmoid=True, return_indices=True)
        loss, _ = ops.clas2(logits, labels, lengths)
        ctx.save_for_backward(logits, means, labels, idx)
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        logits, means, labels, idx = ctx.saved_tensors
        d = ops.clas2_bwd(logits, means, labels, idx, g_loss)
        return d.view_as(logits), None, None


class TrainLossFn(torch.autograd.Function):
    """train/ucf_train.py:73-102 with a gradient: (logits, image_mu, event_mu, image_logvar, event_logvar, labels, lengths,
    nu, reg_weight, kl_weight) -> (total, classification, regulariser, kl), 0-dim fp32 device tensors.  Forward and backward
    are the kernels of csrc/train_loss.cu plus CLAS2's; the gradients of the five tensor inputs go on to
    ForwardFn.backward unchanged."""

    @staticmethod
    def forward(ctx, logits, mu_i, mu_e, lv_i, lv_e, labels, lengths, nu, reg_weight, kl_weight):
        scalars, saved = ops.train_loss_fwd(logits, labels, lengths, mu_i, mu_e, lv_i, lv_e, nu, reg_weight, kl_weight)
        ctx.save_for_backward(logits, mu_i, mu_e, lv_i, lv_e, labels, *saved)
        ctx.consts = (nu, reg_weight, kl_weight)
        ctx.set_materialize_grads(False)          # an unused output's gradient stays None: the kernel reads NULL as 0
        return scalars

    @staticmethod
    def backward(ctx, g_total, g_cls, g_reg, g_kl):
        logits, mu_i, mu_e, lv_i, lv_e, labels, *saved = ctx.saved_tensors
        grads = ops.train_loss_bwd(logits, labels, mu_i, mu_e, lv_i, lv_e, saved, *ctx.consts, g_total, g_cls, g_reg, g_kl)
        return (*grads, None, None, None, None, None)
