"""PyTorch's own CUDA attention-dropout mask restated in numpy - TEST INFRASTRUCTURE ONLY.

F.multi_head_attention_forward in train() mode with need_weights (the default, and what model/imf_vad.py:115,121 take)
drops the [B*H, T, T] attention weights through torch.native_dropout, whose CUDA kernel (fused_dropout_kernel_vec,
aten/src/ATen/native/cuda/Dropout.cu) draws counter-based Philox4x32-10 through curand: the mask is a pure function of the
generator's (seed, offset), the element index and the launch width.  This is the definition the library's "torch"
dropout mode (include/iefvad.h: iefvad_dropout) reproduces; philox4x32_10 is the one of oracle/iefvad_oracle.py."""
from __future__ import annotations

from typing import Tuple

import numpy as np

from oracle.iefvad_oracle import _M32, philox4x32_10


def torch_dropout_launch(n: int, sms: int, max_threads_per_sm: int = 2048) -> Tuple[int, int]:
    """Launch width and generator advance of torch.native_dropout on n elements: 256-thread blocks,
    grid = min(SMs * (threads per SM / 256), ceil(n / 256)) -> (G = grid * 256 threads, offset increment
    ((n - 1) / (G * 4) + 1) * 4)."""
    grid = min(sms * (max_threads_per_sm // 256), (n + 255) // 256)
    G = grid * 256
    return G, ((n - 1) // (G * 4) + 1) * 4


def torch_dropout_words(seed: int, offset: int, n: int, threads: int, swap_halves: bool = False) -> np.ndarray:
    """The uint32 random word of each of the n elements (uint64 array).  Element e lies in the 4-word group v = e // 4,
    drawn by thread v % G in its iteration v // G: Philox4x32-10 with key (seed & 0xffffffff, seed >> 32) and counter
    (lo64 = offset // 4 + v // G, hi64 = v % G), word e % 4 - curand_init(seed, thread, offset) followed by one
    curand_uniform4 per iteration.  swap_halves exchanges the two 64-bit counter halves (a negative control)."""
    seed, offset, G = int(seed), int(offset), np.uint64(int(threads))
    v = np.arange(n // 4, dtype=np.uint64)
    lo, hi = np.uint64(offset // 4) + v // G, v % G
    if swap_halves:
        lo, hi = hi, lo
    s32 = np.uint64(32)
    words = philox4x32_10((lo & _M32, lo >> s32, hi & _M32, hi >> s32), (seed, seed >> 32))
    return np.stack(words, axis=1).reshape(-1)


def torch_dropout_keep(seed: int, offset: int, B: int, H: int, T: int, p: float, threads: int,
                       swap_halves: bool = False) -> np.ndarray:
    """Multiplier of the attention weights under torch.native_dropout of the [B*H, T, T] weights with generator state
    (seed, offset) and launch width `threads` = G -> float64 [B, H, T, T] indexed (b, h, query, key), element
    e = ((b * H + h) * T + query) * T + key.  Kept when float32(word) * 2^-32 + 2^-33 < float32(1 - p) in float32
    arithmetic (curand_uniform4, then `rand < keep`); kept weights are scaled by float32(1 / float64(float32(1 - p)))."""
    n = B * H * T * T
    if n % 4:
        raise ValueError(f"B*H*T*T = {n} is not a multiple of 4: torch would use a narrower vector width")
    words = torch_dropout_words(seed, offset, n, threads, swap_halves)
    u = words.astype(np.float64).astype(np.float32) * np.float32(2.0 ** -32) + np.float32(2.0 ** -33)
    keep = np.float32(1.0 - float(p))
    scale = np.float64(np.float32(1.0 / np.float64(keep)))
    return np.where(u < keep, scale, 0.0).reshape(B, H, T, T)
