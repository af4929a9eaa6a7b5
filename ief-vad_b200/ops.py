"""torch-tensor wrappers over the stand-alone operators of libiefvad.so (include/iefvad.h).

Every function takes CUDA tensors, allocates its outputs with torch and launches on the current stream.
There is no CPU implementation: a non-CUDA tensor raises."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib

PLAN_CODES = {"fp32": -1, "bf16": 0, "split": 1, "fp16": 2}      # fp16: linear, mha, iefvad_transformer, clip
ACTS = {None: 0, "none": 0, "relu": 1, "quickgelu": 2}


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name}: CUDA tensor required (the B200 path has no CPU fallback), got {t.device}")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def fuse(mu_i, mu_e, logvar_i, logvar_e, noise_model: str = "StudentT", nu: float = 8, epsilon: float = 1e-8
         ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """model/imf_vad.py:130-144 -> (w_i, w_e, fused)."""
    if noise_model == "Gaussian":
        factor = 1.0
    elif noise_model == "StudentT":
        factor = (nu + 1) / nu
    else:
        raise ValueError("Unsupported noise_model. Choose 'Gaussian' or 'StudentT'.")
    a, b, c, d = (_f32c(t, "fuse") for t in (mu_i, mu_e, logvar_i, logvar_e))
    w_i, w_e, fused = torch.empty_like(a), torch.empty_like(a), torch.empty_like(a)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib.iefvad_fuse(a.data_ptr(), b.data_ptr(), c.data_ptr(), d.data_ptr(), a.numel(), factor,
                                        epsilon, w_i.data_ptr(), w_e.data_ptr(), fused.data_ptr(), _stream(a)))
    return w_i, w_e, fused


def layernorm(x, w1, b1, w2=None, b2=None, eps: float = 1e-5) -> torch.Tensor:
    x = _f32c(x, "layernorm")
    D = x.shape[-1]
    out = torch.empty_like(x)
    ws = [_f32c(t, "layernorm") if t is not None else None for t in (w1, b1, w2, b2)]
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_layernorm(x.data_ptr(), x.numel() // D, D, *[_lib.ptr(t) for t in ws], eps,
                                             out.data_ptr(), _stream(x)))
    return out


def outproj_ln(ctx, w, bias, resid, ln_w, ln_b, ln2_w=None, ln2_b=None, eps: float = 1e-5, row_map=None, out_rows=None,
               want_lo: bool = True):
    """LN2?(LN(resid + ctx @ w.T + bias)) of one encoder layer's tail in one launch (plan HH arithmetic, D = 768).
    -> (hi, lo): fp16(result) and fp16(result - hi) (lo is None with a row map or want_lo=False).  row_map (int32 [rows]):
    result row r lands in row row_map[r] of the [out_rows, 768] output, negative entries are dropped."""
    ctx, w, resid = _f32c(ctx, "outproj_ln"), _f32c(w, "outproj_ln"), _f32c(resid, "outproj_ln")
    D = ctx.shape[-1]
    rows = ctx.numel() // D
    vec = [_f32c(t, "outproj_ln") if t is not None else None for t in (bias, ln_w, ln_b, ln2_w, ln2_b)]
    if row_map is not None:
        assert row_map.dtype == torch.int32 and row_map.is_cuda and row_map.numel() == rows
        hi = torch.zeros((int(out_rows), D), dtype=torch.float16, device=ctx.device)
        lo = None
    else:
        hi = torch.empty((rows, D), dtype=torch.float16, device=ctx.device)
        lo = torch.empty_like(hi) if want_lo else None
    with torch.cuda.device(ctx.device):
        _lib.check(_lib.lib.iefvad_outproj_ln(ctx.data_ptr(), w.data_ptr(), vec[0].data_ptr(), resid.data_ptr(),
                                              vec[1].data_ptr(), vec[2].data_ptr(), _lib.ptr(vec[3]), _lib.ptr(vec[4]), eps,
                                              rows, _lib.ptr(row_map), hi.data_ptr(), _lib.ptr(lo), _stream(ctx)))
    return hi, lo


def linear(x, w, bias=None, resid=None, alpha: float = 1.0, act: Optional[str] = None, plan: str = "bf16",
           tile_n: int = 0) -> torch.Tensor:
    """out = (resid or 0) + alpha * act(x @ w.T + bias)."""
    x = _f32c(x, "linear")
    w = _f32c(w, "linear")
    in_f, out_f = x.shape[-1], w.shape[0]
    rows = x.numel() // in_f
    out = torch.empty(x.shape[:-1] + (out_f,), dtype=torch.float32, device=x.device)
    bias = _f32c(bias, "linear") if bias is not None else None
    resid = _f32c(resid, "linear") if resid is not None else None
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_linear(x.data_ptr(), w.data_ptr(), _lib.ptr(bias), _lib.ptr(resid), alpha,
                                          ACTS[act], rows, in_f, out_f, PLAN_CODES[plan], tile_n, out.data_ptr(),
                                          _stream(x)))
    return out


def mha(x, in_w, in_b, out_w, out_b, num_heads: int, attn_mask=None, key_padding_mask=None, plan: str = "bf16"
        ) -> torch.Tensor:
    """nn.MultiheadAttention(batch_first=True)(x, x, x)[0], eval mode.  x [B, T, D]."""
    x = _f32c(x, "mha")
    B, T, D = x.shape
    out = torch.empty_like(x)
    in_w, in_b, out_w, out_b = (_f32c(t, "mha") for t in (in_w, in_b, out_w, out_b))
    am = _f32c(attn_mask, "mha") if attn_mask is not None else None
    kp = key_padding_mask.to(torch.uint8).contiguous() if key_padding_mask is not None else None
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_mha(x.data_ptr(), in_w.data_ptr(), in_b.data_ptr(), out_w.data_ptr(),
                                       out_b.data_ptr(), B, T, D, num_heads, _lib.ptr(am), _lib.ptr(kp),
                                       PLAN_CODES[plan], out.data_ptr(), _stream(x)))
    return out


def attention_core(q, k, vt, attn_mask=None, key_padding_mask=None, row_out=None, items=None, out=None):
    """softmax(q k^T) v on the tensor-core attention kernels (iefvad_attention_core), in their own layouts.
    q, k [B, H, T, dhp] and vt [B, H, dh, Tpad], all fp16 or all bf16 (the kernels run in that format); q is already
    scaled by dh^-1/2.  attn_mask [T, T] additive, key_padding_mask [B, T] (True = ignore), row_out int32 [B*T] (output
    row per query row, < 0 = dropped), items int32 [n_chunks, 4] ragged rows (B = 1).  out: [rows, ldo] tensor of the
    operands' dtype that receives head h in columns [h dh, (h+1) dh), untouched elsewhere; default [B*T, H*dh] zeros."""
    if q.dtype not in (torch.float16, torch.bfloat16) or k.dtype != q.dtype or vt.dtype != q.dtype:
        raise RuntimeError(f"attention_core: q, k and vt must all be fp16 or all bf16, got {q.dtype}, {k.dtype}, {vt.dtype}")
    for name, t in (("q", q), ("k", k), ("vt", vt)):
        if not t.is_cuda or not t.is_contiguous() or t.dim() != 4:
            raise RuntimeError(f"attention_core: {name} must be a contiguous 4-d CUDA tensor")
    B, H, T, dhp = q.shape
    dh, Tpad = vt.shape[2], vt.shape[3]
    if tuple(k.shape) != (B, H, T, dhp) or tuple(vt.shape[:2]) != (B, H):
        raise RuntimeError(f"attention_core: shapes q {list(q.shape)}, k {list(k.shape)}, vt {list(vt.shape)} disagree")
    if out is None:
        out = torch.zeros((B * T, H * dh), dtype=q.dtype, device=q.device)
    if out.dtype != q.dtype or out.dim() != 2 or out.stride(1) != 1:
        raise RuntimeError("attention_core: out must be a [rows, ldo] tensor of the operands' dtype with unit column stride")
    am = _f32c(attn_mask, "attention_core") if attn_mask is not None else None
    kp = key_padding_mask.to(torch.uint8).contiguous() if key_padding_mask is not None else None
    ro = row_out.to(torch.int32).contiguous() if row_out is not None else None
    it = items.to(torch.int32).contiguous() if items is not None else None
    with torch.cuda.device(q.device):
        _lib.check(_lib.lib.iefvad_attention_core(q.data_ptr(), k.data_ptr(), vt.data_ptr(), B, T, H, dh, dhp, Tpad,
                                                  _lib.ptr(am), _lib.ptr(kp), _lib.ptr(ro), _lib.ptr(it),
                                                  0 if it is None else it.shape[0], int(q.dtype == torch.float16),
                                                  out.data_ptr(), out.stride(0), _stream(q)))
    return out


def classifier(x, w, bias, with_scores: bool = False):
    x = _f32c(x, "classifier")
    D = x.shape[-1]
    rows = x.numel() // D
    logits = torch.empty(x.shape[:-1] + (1,), dtype=torch.float32, device=x.device)
    scores = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device) if with_scores else None
    w, bias = _f32c(w, "classifier"), _f32c(bias, "classifier")
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_classifier(x.data_ptr(), rows, D, w.data_ptr(), bias.data_ptr(), logits.data_ptr(),
                                              _lib.ptr(scores), _stream(x)))
    return (logits, scores) if with_scores else logits


def mil_topk_mean(x, lengths=None, apply_sigmoid: bool = False, return_indices: bool = False):
    """train/loss.py:24-27 per row: mean of the int(len/16 + 1) largest of x[row, :len].  x [B, T] (or [B, T, 1]);
    lengths [B] integer tensor (device).  Optionally also the chosen positions [B, kmax] (-1 padded),
    descending value, ties by ascending position."""
    x = _f32c(x, "mil_topk_mean")
    if x.dim() == 3 and x.shape[-1] == 1:
        x = x[..., 0]
    B, T = x.shape
    x = x.contiguous()
    if lengths is not None:
        lengths = lengths.to(device=x.device, dtype=torch.int64).contiguous()
    mean = torch.empty(B, dtype=torch.float32, device=x.device)
    kmax = T // 16 + 1
    idx = torch.empty((B, kmax), dtype=torch.int32, device=x.device) if return_indices else None
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_mil_topk_mean(x.data_ptr(), _lib.ptr(lengths), B, T, int(apply_sigmoid),
                                                 mean.data_ptr(), _lib.ptr(idx), kmax, _stream(x)))
    return (mean, idx) if return_indices else mean


def clas2(logits, labels, lengths):
    """train/loss.py:18-30 -> (loss scalar tensor, per-row means)."""
    x = _f32c(logits, "clas2")
    B, T = x.shape[0], x.shape[1]
    x = x.reshape(B, T).contiguous()
    labels = _f32c(labels.to(x.device), "clas2")
    lengths = lengths.to(device=x.device, dtype=torch.int64).contiguous()
    means = torch.empty(B, dtype=torch.float32, device=x.device)
    loss = torch.empty((), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_clas2(x.data_ptr(), labels.data_ptr(), labels.stride(0), lengths.data_ptr(), B, T,
                                         means.data_ptr(), loss.data_ptr(), _stream(x)))
    return loss, means


def sort_scores(scores) -> torch.Tensor:
    """Stable descending argsort (int32) == np.argsort(-scores, kind='stable')."""
    s = _f32c(scores, "sort_scores").reshape(-1)
    order = torch.empty(s.numel(), dtype=torch.int32, device=s.device)
    with torch.cuda.device(s.device):
        _lib.check(_lib.lib.iefvad_sort_scores(s.data_ptr(), s.numel(), order.data_ptr(), _stream(s)))
    return order


def auc_ap(scores, pos, repeat: int = 16, return_order: bool = False):
    """-> float64 tensor [4] on the device: AUC, AP, #positive frames, #negative frames (train/ucf_test.py:151-152
    on np.repeat(scores, repeat)); pos[j] = positives among segment j's `repeat` frames."""
    s = _f32c(scores, "auc_ap").reshape(-1)
    p = pos.to(device=s.device, dtype=torch.int32).contiguous().reshape(-1)
    if p.numel() != s.numel():
        raise RuntimeError(f"auc_ap: {s.numel()} scores but {p.numel()} label counts")
    out = torch.empty(4, dtype=torch.float64, device=s.device)
    order = torch.empty(s.numel(), dtype=torch.int32, device=s.device) if return_order else None
    with torch.cuda.device(s.device):
        _lib.check(_lib.lib.iefvad_auc_ap(s.data_ptr(), p.data_ptr(), s.numel(), repeat, out.data_ptr(),
                                          _lib.ptr(order), _stream(s)))
    return (out, order) if return_order else out


def auc_ap_multi(scores, pos, member, num_subsets: int, repeat: int = 16):
    """AUC / AP of `num_subsets` (<= 32) subsets of the segments from ONE ranking pass (class-wise AUC / AP and
    Ano-AUC, train/ucf_test.py:164-178, 336-353).  member[j] bit s = segment j is in subset s.
    -> float64 tensor [num_subsets, 4] on the device (AUC, AP, #positive frames, #negative frames)."""
    s = _f32c(scores, "auc_ap_multi").reshape(-1)
    p = pos.to(device=s.device, dtype=torch.int32).contiguous().reshape(-1)
    m = member.to(device=s.device).contiguous().reshape(-1)
    if m.dtype not in (torch.int32, torch.uint32):
        raise RuntimeError("auc_ap_multi: member must be a 32-bit mask tensor")
    if p.numel() != s.numel() or m.numel() != s.numel():
        raise RuntimeError(f"auc_ap_multi: {s.numel()} scores, {p.numel()} label counts, {m.numel()} masks")
    out = torch.empty((num_subsets, 4), dtype=torch.float64, device=s.device)
    with torch.cuda.device(s.device):
        _lib.check(_lib.lib.iefvad_auc_ap_multi(s.data_ptr(), p.data_ptr(), m.data_ptr(), s.numel(), repeat,
                                                num_subsets, out.data_ptr(), None, _stream(s)))
    return out


# ------------------------------------------------------------------------------------------------ training step (row N3)
def torch_dropout_launch(n: int, device=None) -> Tuple[int, int]:
    """Launch width and generator advance of torch's CUDA dropout (torch.native_dropout) on n elements of `device`:
    256-thread blocks, grid = min(SMs * (max threads per SM / 256), ceil(n / 256)) -> (threads G = grid * 256, offset
    increment ((n - 1) / (G * 4) + 1) * 4).  G depends on the SM count, so the mask does too (include/iefvad.h)."""
    props = torch.cuda.get_device_properties(device)
    grid = min(props.multi_processor_count * (props.max_threads_per_multi_processor // 256), (n + 255) // 256)
    G = grid * 256
    return G, (((n - 1) // (G * 4) + 1) * 4 if n > 0 else 0)


def _dropout(rng: str, p_drop: float, seed: int, offset: int, threads: int):
    kind = _lib.DROPOUT_KINDS.get(rng)
    if kind is None:
        raise ValueError(f"unknown dropout rng {rng!r}; choose from {sorted(_lib.DROPOUT_KINDS)}")
    return _lib.Dropout(kind, float(p_drop), int(seed), int(offset), int(threads))


def attention_train_fwd(qkv, B: int, T: int, heads: int, p_drop: float = 0.0, seed: int = 0, rng: str = "philox",
                        offset: int = 0, threads: int = 0):
    """dropout(softmax(q k^T / sqrt(dh))) v of nn.MultiheadAttention in train mode -> (out [B*T, D], lse [B, H, T]).
    rng "philox": the library's own mask keyed by `seed`; "torch": torch.native_dropout's mask for a CUDA generator at
    (seed, offset), launch width `threads` (torch_dropout_launch) - the caller advances the generator."""
    qkv = _f32c(qkv, "attention_train_fwd")
    D = qkv.shape[-1] // 3
    out = torch.empty((B * T, D), dtype=torch.float32, device=qkv.device)
    lse = torch.empty((B, heads, T), dtype=torch.float32, device=qkv.device)
    with torch.cuda.device(qkv.device):
        if rng == "philox":
            _lib.check(_lib.lib.iefvad_attention_train_fwd(qkv.data_ptr(), B, T, heads, D // heads, float(p_drop), int(seed),
                                                           out.data_ptr(), lse.data_ptr(), _stream(qkv)))
        else:
            drop = _dropout(rng, p_drop, seed, offset, threads)
            _lib.check(_lib.lib.iefvad_attention_train_fwd_dropout(qkv.data_ptr(), B, T, heads, D // heads, C.byref(drop),
                                                                   out.data_ptr(), lse.data_ptr(), _stream(qkv)))
    return out, lse


def attention_train_bwd(qkv, out, dout, lse, B: int, T: int, heads: int, p_drop: float = 0.0, seed: int = 0,
                        rng: str = "philox", offset: int = 0, threads: int = 0):
    """dqkv of attention_train_fwd, regenerating the same mask (same p_drop / seed / rng / offset / threads)."""
    qkv, out, dout, lse = (_f32c(t, "attention_train_bwd") for t in (qkv, out, dout, lse))
    D = qkv.shape[-1] // 3
    dqkv = torch.empty_like(qkv)
    with torch.cuda.device(qkv.device):
        if rng == "philox":
            _lib.check(_lib.lib.iefvad_attention_train_bwd(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(),
                                                           B, T, heads, D // heads, float(p_drop), int(seed),
                                                           dqkv.data_ptr(), _stream(qkv)))
        else:
            drop = _dropout(rng, p_drop, seed, offset, threads)
            _lib.check(_lib.lib.iefvad_attention_train_bwd_dropout(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(),
                                                                   lse.data_ptr(), B, T, heads, D // heads, C.byref(drop),
                                                                   dqkv.data_ptr(), _stream(qkv)))
    return dqkv


def dropout_mask(B: int, heads: int, T: int, p_drop: float, seed: int, rng: str = "torch", offset: int = 0,
                 threads: int = 0, device=None) -> torch.Tensor:
    """uint8 [B*heads, T, T] (1 = kept): the keep decisions of the training attention under the given mask, in the layout
    of torch.native_dropout's mask (iefvad_dropout_mask)."""
    drop = _dropout(rng, p_drop, seed, offset, threads)
    device = torch.device("cuda") if device is None else torch.device(device)
    mask = torch.empty((B * heads, T, T), dtype=torch.uint8, device=device)
    with torch.cuda.device(mask.device):
        _lib.check(_lib.lib.iefvad_dropout_mask(C.byref(drop), B, heads, T, mask.data_ptr(), _stream(mask)))
    return mask


def layernorm_bwd(x, weight, dy, eps: float = 1e-5):
    """-> (dx, dweight, dbias) of nn.LayerNorm(x) given dy."""
    x, weight, dy = _f32c(x, "layernorm_bwd"), _f32c(weight, "layernorm_bwd"), _f32c(dy, "layernorm_bwd")
    D = x.shape[-1]
    dx = torch.empty_like(x)
    dw = torch.empty(D, dtype=torch.float32, device=x.device)
    db = torch.empty(D, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_layernorm_bwd(x.data_ptr(), weight.data_ptr(), dy.data_ptr(), x.numel() // D, D, eps,
                                                 dx.data_ptr(), dw.data_ptr(), db.data_ptr(), _stream(x)))
    return dx, dw, db


def colsum(a, row_weight=None):
    """out[c] = sum_r a[r, c] (* row_weight[r]); a [rows, dim]."""
    a = _f32c(a, "colsum")
    D = a.shape[-1]
    rw = _f32c(row_weight, "colsum").reshape(-1) if row_weight is not None else None
    out = torch.empty(D, dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib.iefvad_colsum(a.data_ptr(), _lib.ptr(rw), a.numel() // D, D, out.data_ptr(), _stream(a)))
    return out


def fuse_bwd(mu_i, mu_e, lv_i, lv_e, g_fused=None, g_wi=None, g_we=None, g_mu_i=None, g_mu_e=None, g_lv_i=None,
             g_lv_e=None, noise_model: str = "StudentT", nu: float = 8, epsilon: float = 1e-8):
    """Backward of model/imf_vad.py:130-144 -> total gradients (d_mu_i, d_mu_e, d_logvar_i, d_logvar_e)."""
    factor = 1.0 if noise_model == "Gaussian" else (nu + 1) / nu
    ins = [_f32c(t, "fuse_bwd") for t in (mu_i, mu_e, lv_i, lv_e)]
    gs = [(_f32c(t, "fuse_bwd") if t is not None else None) for t in (g_fused, g_wi, g_we, g_mu_i, g_mu_e, g_lv_i, g_lv_e)]
    outs = [torch.empty_like(ins[0]) for _ in range(4)]
    with torch.cuda.device(ins[0].device):
        _lib.check(_lib.lib.iefvad_fuse_bwd(*[t.data_ptr() for t in ins], *[_lib.ptr(t) for t in gs], ins[0].numel(), factor,
                                            epsilon, *[t.data_ptr() for t in outs], _stream(ins[0])))
    return tuple(outs)


def quickgelu(x):
    """model/module.py:15-17: x * sigmoid(1.702 x)."""
    xs = _f32c(x, "quickgelu")
    out = torch.empty_like(xs)
    with torch.cuda.device(xs.device):
        _lib.check(_lib.lib.iefvad_quickgelu(xs.data_ptr(), xs.numel(), out.data_ptr(), _stream(xs)))
    return out.to(x.dtype)


def relu_bwd(dh, h):
    dh, h = _f32c(dh, "relu_bwd"), _f32c(h, "relu_bwd")
    out = torch.empty_like(dh)
    with torch.cuda.device(dh.device):
        _lib.check(_lib.lib.iefvad_relu_bwd(dh.data_ptr(), h.data_ptr(), dh.numel(), out.data_ptr(), _stream(dh)))
    return out


def axpy_(y, x, alpha: float = 1.0):
    """y += alpha * x in place (y must be a contiguous fp32 CUDA tensor)."""
    if y.dtype != torch.float32 or not y.is_contiguous() or not y.is_cuda:
        raise RuntimeError("axpy_: y must be a contiguous fp32 CUDA tensor")
    x = _f32c(x, "axpy_")
    with torch.cuda.device(y.device):
        _lib.check(_lib.lib.iefvad_axpy(y.data_ptr(), x.data_ptr(), float(alpha), y.numel(), _stream(y)))
    return y


def outer(a, w):
    """out[r, c] = a[r] * w[c]."""
    a, w = _f32c(a, "outer").reshape(-1), _f32c(w, "outer").reshape(-1)
    out = torch.empty((a.numel(), w.numel()), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib.iefvad_outer(a.data_ptr(), w.data_ptr(), a.numel(), w.numel(), out.data_ptr(), _stream(a)))
    return out


def transpose(x, pad_to: int = 1):
    """[rows, cols] -> [cols, ld] with ld = rows rounded up to a multiple of pad_to, the tail zero-filled."""
    x = _f32c(x, "transpose")
    rows, cols = x.shape
    ld = (rows + pad_to - 1) // pad_to * pad_to
    out = torch.empty((cols, ld), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_transpose(x.data_ptr(), rows, cols, out.data_ptr(), ld, _stream(x)))
    return out


def wgrad(dy, x, alpha: float = 1.0):
    """dW [out, in] = alpha * dy^T @ x for dy [rows, out], x [rows, in]."""
    dy, x = _f32c(dy, "wgrad"), _f32c(x, "wgrad")
    rows, out_f = dy.shape
    in_f = x.shape[1]
    dw = torch.empty((out_f, in_f), dtype=torch.float32, device=dy.device)
    with torch.cuda.device(dy.device):
        _lib.check(_lib.lib.iefvad_wgrad(dy.data_ptr(), x.data_ptr(), rows, out_f, in_f, alpha, dw.data_ptr(), _stream(dy)))
    return dw


def clas2_bwd(logits, means, labels, idx, g_loss=None):
    x = _f32c(logits, "clas2_bwd")
    B, T = x.shape[0], x.shape[1]
    x = x.reshape(B, T).contiguous()
    labels = _f32c(labels.to(x.device), "clas2_bwd")
    g = _f32c(g_loss, "clas2_bwd").reshape(1) if g_loss is not None else None
    out = torch.empty((B, T), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_clas2_bwd(x.data_ptr(), means.data_ptr(), labels.data_ptr(), labels.stride(0),
                                             idx.data_ptr(), B, T, idx.shape[1], _lib.ptr(g), out.data_ptr(), _stream(x)))
    return out


def _check_objective_inputs(logits, labels, lengths, wide):
    for name, t in zip(("logits", "labels", "lengths", "image_mu", "event_mu", "image_logvar", "event_logvar"),
                       (logits, labels, lengths, *wide)):
        if not t.is_cuda:
            raise RuntimeError(f"train_loss: {name} must be a CUDA tensor (the B200 path has no CPU fallback), got {t.device}")
    shape = wide[0].shape
    if wide[0].dim() != 3 or any(t.shape != shape for t in wide[1:]):
        raise RuntimeError("train_loss: image_mu, event_mu, image_logvar and event_logvar must share one [B, T, D] shape, "
                           f"got {[tuple(t.shape) for t in wide]}")
    if tuple(logits.shape) != (shape[0], shape[1], 1):
        raise RuntimeError(f"train_loss: logits must be [B, T, 1] = {[shape[0], shape[1], 1]}, got {list(logits.shape)}")
    if labels.dim() != 2 or labels.shape[0] != shape[0] or lengths.numel() != shape[0]:
        raise RuntimeError(f"train_loss: labels must be [B, C] and lengths [B] with B = {shape[0]}, "
                           f"got {list(labels.shape)} and {list(lengths.shape)}")


def train_loss_fwd(logits, labels, lengths, mu_i, mu_e, lv_i, lv_e, nu: float, reg_weight: float = 1.0,
                   kl_weight: float = 1.0):
    """Loss of train/ucf_train.py:73-102 (CLAS2 + cosine / norm regulariser + StudentT KL, iefvad_train_loss_fwd).
    logits [B, T, 1], mu_* / lv_* [B, T, D], labels [B, C], lengths [B] -> (total, classification, regulariser, kl) as
    0-dim fp32 device tensors, and (means, idx, record), what train_loss_bwd needs."""
    _check_objective_inputs(logits, labels, lengths, (mu_i, mu_e, lv_i, lv_e))
    B, T, D = mu_i.shape
    x = _f32c(logits, "train_loss").reshape(B, T)
    labels = _f32c(labels, "train_loss")
    lengths = lengths.to(dtype=torch.int64).contiguous()
    wide = [_f32c(t, "train_loss") for t in (mu_i, mu_e, lv_i, lv_e)]
    kmax = T // 16 + 1
    dev = x.device
    means = torch.empty(B, dtype=torch.float32, device=dev)
    idx = torch.empty((B, kmax), dtype=torch.int32, device=dev)
    record = torch.empty((B * T, 4), dtype=torch.float64, device=dev)
    scalars = [torch.empty((), dtype=torch.float32, device=dev) for _ in range(4)]
    with torch.cuda.device(dev):
        _lib.check(_lib.lib.iefvad_train_loss_fwd(x.data_ptr(), labels.data_ptr(), labels.stride(0), lengths.data_ptr(), B, T,
                                                  *[t.data_ptr() for t in wide], D, float(nu), float(reg_weight),
                                                  float(kl_weight), means.data_ptr(), idx.data_ptr(), kmax, record.data_ptr(),
                                                  *[t.data_ptr() for t in scalars], _stream(x)))
    return tuple(scalars), (means, idx, record)


def train_loss_bwd(logits, labels, mu_i, mu_e, lv_i, lv_e, saved, nu: float, reg_weight: float = 1.0, kl_weight: float = 1.0,
                   g_total=None, g_cls=None, g_reg=None, g_kl=None):
    """Backward of train_loss_fwd: gradients of g_total total + g_cls classification + g_reg regulariser + g_kl kl
    (device scalars, None = 0) -> (d_logits [B, T, 1], d_mu_i, d_mu_e, d_lv_i, d_lv_e [B, T, D]), fp32."""
    means, idx, record = saved
    B, T, D = mu_i.shape
    x = _f32c(logits, "train_loss_bwd").reshape(B, T)
    labels = _f32c(labels, "train_loss_bwd")
    wide = [_f32c(t, "train_loss_bwd") for t in (mu_i, mu_e, lv_i, lv_e)]
    gs = [_f32c(g, "train_loss_bwd").reshape(()) if g is not None else None for g in (g_total, g_cls, g_reg, g_kl)]
    d_logits = torch.empty((B, T, 1), dtype=torch.float32, device=x.device)
    outs = [torch.empty((B, T, D), dtype=torch.float32, device=x.device) for _ in range(4)]
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib.iefvad_train_loss_bwd(x.data_ptr(), means.data_ptr(), labels.data_ptr(), labels.stride(0),
                                                  idx.data_ptr(), B, T, idx.shape[1], *[t.data_ptr() for t in wide], D,
                                                  record.data_ptr(), float(nu), float(reg_weight), float(kl_weight),
                                                  *[_lib.ptr(g) for g in gs], d_logits.data_ptr(),
                                                  *[t.data_ptr() for t in outs], _stream(x)))
    return (d_logits, *outs)
