"""Restatements of the CLIP image encoder (test / benchmark infrastructure only, like oracle/iefvad_oracle.py: nothing in
the product package imports it).  OpenAI's `VisionTransformer.forward`, extracting/clip/model.py:206-241:

    clip_visual(x, params, heads)                  float64 numpy (the yardstick)
    clip_visual_torch(x, P, heads, dtype)          the same in torch ops on any device; dtype float16 follows OpenAI's
                                                   fp16 model (the "reference arithmetic" bar on CUDA)
    clip_visual_params(R, P, W, layers, out, seed) seeded random `visual.state_dict()` (float64)"""
from __future__ import annotations

import math
from typing import Dict

import numpy as np
import torch
import torch.nn.functional as F

from oracle.iefvad_oracle import layer_norm, transformer


def clip_visual_params(R: int, P: int, W: int, layers: int, out_dim: int, seed: int = 0) -> Dict[str, np.ndarray]:
    """Seeded random `visual.state_dict()` of a VisionTransformer (float64): fan-in-scaled weights, LayerNorm gains
    near 1, small biases, embeddings at OpenAI's init scale width^-0.5 (model.py:219-224)."""
    rng = np.random.default_rng(seed)
    n = lambda *s: rng.standard_normal(s)
    sc = W ** -0.5
    sd = {"conv1.weight": n(W, 3, P, P) / math.sqrt(3 * P * P), "class_embedding": sc * n(W),
          "positional_embedding": sc * n((R // P) ** 2 + 1, W), "ln_pre.weight": 1 + 0.1 * n(W), "ln_pre.bias": 0.1 * n(W)}
    for i in range(layers):
        pre = f"transformer.resblocks.{i}."
        sd.update({pre + "ln_1.weight": 1 + 0.1 * n(W), pre + "ln_1.bias": 0.1 * n(W),
                   pre + "attn.in_proj_weight": n(3 * W, W) * sc, pre + "attn.in_proj_bias": 0.02 * n(3 * W),
                   pre + "attn.out_proj.weight": n(W, W) * sc, pre + "attn.out_proj.bias": 0.02 * n(W),
                   pre + "ln_2.weight": 1 + 0.1 * n(W), pre + "ln_2.bias": 0.1 * n(W),
                   pre + "mlp.c_fc.weight": n(4 * W, W) * sc, pre + "mlp.c_fc.bias": 0.02 * n(4 * W),
                   pre + "mlp.c_proj.weight": n(W, 4 * W) * (0.5 * sc), pre + "mlp.c_proj.bias": 0.02 * n(W)})
    sd.update({"ln_post.weight": 1 + 0.1 * n(W), "ln_post.bias": 0.1 * n(W), "proj": sc * n(W, out_dim)})
    return sd


def _layers(P) -> int:
    return len([k for k in P if k.startswith("transformer.resblocks.") and k.endswith(".attn.in_proj_weight")])


def clip_visual(x: np.ndarray, params: Dict[str, np.ndarray], heads: int) -> np.ndarray:
    """CLIP VisionTransformer.forward, extracting/clip/model.py:206-241, in float64.  x [N, 3, R, R] (normalised
    pixels); `params` holds `visual.state_dict()` entries by name.  Conv2d(stride = kernel = P, no bias) as a product
    over non-overlapping patches (:226-228), class token + positional embedding (:229-230), ln_pre (:231), the
    residual blocks (:233-235), ln_post on the class token (:237) and the projection (:239-240).  -> [N, output_dim]."""
    f = np.float64
    x = np.asarray(x, dtype=f)
    P = {k: np.asarray(v, dtype=f) for k, v in params.items()}
    w = P["conv1.weight"]                                          # [W, 3, p, p]
    W, p = w.shape[0], w.shape[-1]
    N, R = x.shape[0], x.shape[-1]
    G = R // p
    col = x.reshape(N, 3, G, p, G, p).transpose(0, 2, 4, 1, 3, 5).reshape(N, G * G, 3 * p * p)
    tok = col @ w.reshape(W, -1).T                                 # [N, G*G, W]
    cls = np.broadcast_to(P["class_embedding"], (N, 1, W))
    tok = np.concatenate([cls, tok], axis=1) + P["positional_embedding"]
    tok = layer_norm(tok, P["ln_pre.weight"], P["ln_pre.bias"])
    blocks = [{k[len(f"transformer.resblocks.{i}."):]: v for k, v in P.items() if k.startswith(f"transformer.resblocks.{i}.")}
              for i in range(_layers(P))]
    tok = transformer(tok.transpose(1, 0, 2), blocks, heads).transpose(1, 0, 2)
    return layer_norm(tok[:, 0, :], P["ln_post.weight"], P["ln_post.bias"]) @ P["proj"]


def clip_visual_torch(x: torch.Tensor, P: Dict[str, torch.Tensor], heads: int, dtype: torch.dtype = torch.float64
                      ) -> torch.Tensor:
    """`clip_visual` on whichever device `x` is on, with `P` = `visual.state_dict()`.  dtype float64 / float32: every
    parameter and the activations in that type.  dtype float16: OpenAI's fp16 model as `clip.load` builds it on CUDA
    (model.py:378-397, `convert_weights`): conv1, the Linear / MHA weights and biases and `proj` in fp16, class /
    positional embeddings cast to fp16 where they are added, LayerNorm computed in fp32 with fp32 affine parameters and
    cast back (:157-163), residual stream and QuickGELU in fp16, attention through `scaled_dot_product_attention` as
    `nn.MultiheadAttention(need_weights=False)` runs it.  Returns [N, output_dim] in `dtype`."""
    half = dtype == torch.float16
    wt = (lambda t: t.to(device=x.device, dtype=dtype))
    ln_t = (lambda t: t.to(device=x.device, dtype=torch.float32 if half else dtype))

    def ln(h, pre):
        w, b = ln_t(P[pre + ".weight"]), ln_t(P[pre + ".bias"])
        return F.layer_norm(h.to(w.dtype), (h.shape[-1],), w, b).to(dtype)

    x = x.to(dtype)
    h = F.conv2d(x, wt(P["conv1.weight"]), stride=P["conv1.weight"].shape[-1])       # [N, W, G, G]
    N, W = h.shape[0], h.shape[1]
    h = h.reshape(N, W, -1).permute(0, 2, 1)
    h = torch.cat([wt(P["class_embedding"]).expand(N, 1, W), h], dim=1) + wt(P["positional_embedding"])
    h = ln(h, "ln_pre")
    dh = W // heads
    for i in range(_layers(P)):
        pre = f"transformer.resblocks.{i}."
        a = ln(h, pre + "ln_1")
        q, k, v = F.linear(a, wt(P[pre + "attn.in_proj_weight"]), wt(P[pre + "attn.in_proj_bias"])).split(W, dim=-1)
        q, k, v = (t.reshape(N, -1, heads, dh).transpose(1, 2) for t in (q, k, v))
        o = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(N, -1, W)
        h = h + F.linear(o, wt(P[pre + "attn.out_proj.weight"]), wt(P[pre + "attn.out_proj.bias"]))
        a = F.linear(ln(h, pre + "ln_2"), wt(P[pre + "mlp.c_fc.weight"]), wt(P[pre + "mlp.c_fc.bias"]))
        a = a * torch.sigmoid(1.702 * a)
        h = h + F.linear(a, wt(P[pre + "mlp.c_proj.weight"]), wt(P[pre + "mlp.c_proj.bias"]))
    return ln(h[:, 0, :], "ln_post") @ wt(P["proj"])
