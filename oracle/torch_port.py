"""CPU port of the oracle on torch CPU tensor ops - TEST / BASELINE INFRASTRUCTURE ONLY.

Same arithmetic as `oracle/iefvad_oracle.py` (which is pinned to the reference's golden outputs), restated with
`torch.nn.functional` primitives so that it runs on the same multi-threaded CPU kernels (MKL / oneDNN GEMM,
vectorised softmax / LayerNorm) the reference's own PyTorch forward uses.  `bench.py` times it as the
`cpu_baseline` ("port") and as the `--impl reference` arm: the reference itself is Python that cannot travel to
the GPU box (`/root/reference` does not exist there).  `tests/test_oracle_golden.py` checks it against the numpy
oracle and the reference goldens.  The product package never imports this file."""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F


def mha(x, in_w, in_b, out_w, out_b, heads: int, keep: Optional[torch.Tensor] = None):
    """nn.MultiheadAttention(batch_first=True)(x, x, x)[0], eval mode, no masks (model/imf_vad.py:115,121;
    torch/nn/functional.py:6244: q scaled by d_h^-1/2 before QK^T, softmax over keys).  keep [B, heads, T, T]: train
    mode, the attention weights times this dropout multiplier (0 or 1 / (1 - p); oracle.iefvad_oracle.attention_keep)."""
    B, T, D = x.shape
    dh = D // heads
    qkv = F.linear(x, in_w, in_b)
    q, k, v = qkv.split(D, dim=-1)
    q = (q * (1.0 / math.sqrt(dh))).view(B, T, heads, dh).transpose(1, 2)
    k = k.view(B, T, heads, dh).transpose(1, 2)
    v = v.view(B, T, heads, dh).transpose(1, 2)
    p = torch.softmax(q @ k.transpose(-1, -2), dim=-1)
    if keep is not None:
        p = p * keep
    o = (p @ v).transpose(1, 2).reshape(B, T, D)
    return F.linear(o, out_w, out_b)


def forward(P: Dict[str, torch.Tensor], img: torch.Tensor, ev: torch.Tensor, *, heads: int = 8,
            lambda_ref: float = 0.5, noise_model: str = "StudentT", nu: float = 8, epsilon: float = 1e-8,
            keep: Optional[Dict[Tuple[str, int], torch.Tensor]] = None, dtype: torch.dtype = torch.float
            ) -> Dict[str, torch.Tensor]:
    """model/imf_vad.py:40-44 + :109-161 with state_dict keys as parameter names.  keep[(modality, layer)]: dropout
    multiplier of that attention layer (see `mha`), None = eval mode.  dtype: the type the inputs are cast to (:41-42
    cast to float32; float64 with float64 parameters gives the high-precision training reference)."""
    D = P["temporal.classifier.weight"].shape[1]
    L = sum(1 for k in P if k.startswith("temporal.image_attn_layers.") and k.endswith("in_proj_weight"))
    R = sum(1 for k in P if k.startswith("temporal.refinement_blocks.") and k.endswith(".0.weight"))
    enc = {}
    for mod, x in (("image", img), ("event", ev)):
        x = x.to(dtype)
        for i in range(L):
            pre = f"temporal.{mod}_attn_layers.{i}."
            a = mha(x, P[pre + "in_proj_weight"], P[pre + "in_proj_bias"], P[pre + "out_proj.weight"],
                    P[pre + "out_proj.bias"], heads, None if keep is None else keep[(mod, i)])
            x = F.layer_norm(x + a, (D,), P[f"temporal.{mod}_norms.{i}.weight"], P[f"temporal.{mod}_norms.{i}.bias"])
        enc[mod] = F.layer_norm(x, (D,), P[f"temporal.whiten_{mod}.weight"], P[f"temporal.whiten_{mod}.bias"])
    image_mu = F.linear(enc["image"], P["temporal.image_mu.weight"], P["temporal.image_mu.bias"])
    event_mu = F.linear(enc["event"], P["temporal.event_mu.weight"], P["temporal.event_mu.bias"])
    image_logvar = F.linear(enc["image"], P["temporal.image_logvar.weight"], P["temporal.image_logvar.bias"])
    event_logvar = F.linear(enc["event"], P["temporal.event_logvar.weight"], P["temporal.event_logvar.bias"])
    if noise_model == "Gaussian":
        wi, we = torch.exp(-image_logvar), torch.exp(-event_logvar)
    elif noise_model == "StudentT":
        f = (nu + 1) / nu
        wi, we = f * torch.exp(-image_logvar), f * torch.exp(-event_logvar)
    else:
        raise ValueError("Unsupported noise_model. Choose 'Gaussian' or 'StudentT'.")
    den = wi + we + epsilon
    nwi, nwe = wi / den, we / den
    x = nwi * image_mu + nwe * event_mu
    for i in range(R):
        h = F.relu(F.linear(x, P[f"temporal.refinement_blocks.{i}.0.weight"], P[f"temporal.refinement_blocks.{i}.0.bias"]))
        x = x - lambda_ref * F.linear(h, P[f"temporal.refinement_blocks.{i}.2.weight"],
                                      P[f"temporal.refinement_blocks.{i}.2.bias"])
    logits = F.linear(x, P["temporal.classifier.weight"], P["temporal.classifier.bias"])
    return {"fused": x, "logits": logits, "image_mu": image_mu, "event_mu": event_mu, "image_logvar": image_logvar,
            "event_logvar": event_logvar, "w_i": nwi, "w_e": nwe}
