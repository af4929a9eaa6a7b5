"""B200 counterpart of the CLIP image encoder that the reference's feature extraction runs (SURVEY row N4):
OpenAI's `VisionTransformer`, extracting/clip/model.py:206-241, with the same constructor arguments and state_dict
layout, so that `load_state_dict(clip_model.visual.state_dict())` of an OpenAI checkpoint works unchanged:

    sd = clip_model.visual.state_dict()
    visual = VisionTransformer.from_state_dict(sd).cuda()
    with torch.no_grad():
        emb = visual(images)                # [N, 3, 224, 224] normalised pixels -> [N, 768] fp32 (ViT-L/14)

The whole forward runs in one libiefvad.so call (`iefvad_clip_visual`).  Inference only."""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .module import LayerNorm, Transformer
from .ops import PLAN_CODES, _stream

_DTYPES = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}


class VisionTransformer(nn.Module):
    """model.py:206-241.  `precision`: "fp16" (default; fp16 GEMM / attention operands with fp32 accumulation, fp32
    LayerNorm, residual stream and projection) or "fp32" (FFMA throughout, the yardstick)."""

    def __init__(self, input_resolution: int, patch_size: int, width: int, layers: int, heads: int, output_dim: int):
        super().__init__()
        self.input_resolution = input_resolution
        self.output_dim = output_dim
        self.heads = heads
        self.conv1 = nn.Conv2d(in_channels=3, out_channels=width, kernel_size=patch_size, stride=patch_size, bias=False)
        scale = width ** -0.5
        self.class_embedding = nn.Parameter(scale * torch.randn(width))
        self.positional_embedding = nn.Parameter(scale * torch.randn((input_resolution // patch_size) ** 2 + 1, width))
        self.ln_pre = LayerNorm(width)
        self.transformer = Transformer(width, layers, heads)
        self.ln_post = LayerNorm(width)
        self.proj = nn.Parameter(scale * torch.randn(width, output_dim))
        self.precision = "fp16"

    @classmethod
    def from_state_dict(cls, sd) -> "VisionTransformer":
        """The configuration as OpenAI's `build_model` infers it (model.py:399-410, without the `visual.` prefix), then
        `load_state_dict(sd)`.  fp16 checkpoints are copied into the fp32 parameters."""
        width = sd["conv1.weight"].shape[0]
        layers = len([k for k in sd if k.startswith("transformer.resblocks.") and k.endswith(".attn.in_proj_weight")])
        patch = sd["conv1.weight"].shape[-1]
        grid = round((sd["positional_embedding"].shape[0] - 1) ** 0.5)
        m = cls(patch * grid, patch, width, layers, width // 64, sd["proj"].shape[1])
        m.load_state_dict(sd)
        return m

    def _params(self):
        blocks = [p for b in self.transformer.resblocks for p in b._params()]
        return [self.conv1.weight, self.class_embedding, self.positional_embedding, self.ln_pre.weight, self.ln_pre.bias,
                *blocks, self.ln_post.weight, self.ln_post.bias, self.proj]

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        params = self._params()
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params)):
            raise RuntimeError("VisionTransformer runs inference only (there is no backward): call it under "
                               "torch.no_grad() or torch.inference_mode()")
        if not x.is_cuda:
            raise RuntimeError(f"VisionTransformer: CUDA tensor required (the B200 path has no CPU fallback), got {x.device}")
        if x.dtype not in _DTYPES:
            raise RuntimeError(f"VisionTransformer: input dtype must be float32, float16 or bfloat16, got {x.dtype}")
        R, P = self.input_resolution, self.conv1.kernel_size[0]
        if x.dim() != 4 or tuple(x.shape[1:]) != (3, R, R):
            raise RuntimeError(f"VisionTransformer: input must be [N, 3, {R}, {R}], got {tuple(x.shape)}")
        xs = x.contiguous()
        keep = [p.detach().to(device=xs.device, dtype=torch.float32).contiguous() for p in params]
        table = (C.c_void_p * len(keep))(*[t.data_ptr() for t in keep])
        width = self.conv1.out_channels
        out = torch.empty((xs.shape[0], self.output_dim), dtype=torch.float32, device=xs.device)
        with torch.cuda.device(xs.device):
            _lib.check(_lib.lib.iefvad_clip_visual(xs.data_ptr(), _DTYPES[xs.dtype], xs.shape[0], R, P, width,
                                                   self.transformer.layers, self.heads, self.output_dim,
                                                   C.cast(table, C.c_void_p), PLAN_CODES[self.precision], out.data_ptr(),
                                                   _stream(xs)))
        return out
