"""CPU oracle for the IEF-VAD inference hot path (numpy restatement).

TEST INFRASTRUCTURE ONLY.  Nothing in the product package (`ief-vad_b200/`) may
import this file; only `tests/`, `__graft_entry__.smoke()` and the
`cpu_baseline` / `--impl reference` legs of `bench.py` do, and there only as the
checker / the timed CPU baseline, never as the thing shipped.

Every function restates the arithmetic of one reference function and cites the
reference file:line it follows (paths relative to the upstream checkout, or
`torch/...` / `sklearn/...` for the third-party packages the reference calls).

Parity pin: the reference holds no tests, golden vectors or fixtures for this
path (SURVEY.md section 4), so the pin is *outputs of the reference itself run
in the authoring container*: `tests/golden/make_golden.py` imports the
unmodified reference (`model.imf_vad.MMFMIL`, `train.loss.CLAS2`,
`train.ucf_test.test`, `model.layers.*`, `model.module.Transformer`) and
scikit-learn, and commits their outputs as fixtures under `tests/golden/`;
`tests/test_oracle_golden.py` checks this file against every one of them.

All functions take / return numpy arrays.  `dtype` selects the arithmetic type
(np.float32 mirrors the reference, np.float64 is the high-precision yardstick
used to measure both the reference's and the CUDA path's error).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

# --------------------------------------------------------------------------
# Elementary pieces (torch semantics restated)
# --------------------------------------------------------------------------


def linear(x: np.ndarray, w: np.ndarray, b: Optional[np.ndarray]) -> np.ndarray:
    """torch.nn.Linear: y = x W^T + b  (weight stored [out, in])."""
    y = x @ w.T
    if b is not None:
        y = y + b
    return y


def layer_norm(x: np.ndarray, w: np.ndarray, b: np.ndarray, eps: float = 1e-5) -> np.ndarray:
    """torch.nn.LayerNorm over the last axis: biased variance, eps inside the sqrt.
    Call sites: model/imf_vad.py:73,80,83-84 (modules) and :116-117,122-123."""
    mu = x.mean(axis=-1, keepdims=True)
    xc = x - mu
    var = (xc * xc).mean(axis=-1, keepdims=True)
    return xc / np.sqrt(var + x.dtype.type(eps)) * w + b


def softmax(x: np.ndarray, axis: int = -1) -> np.ndarray:
    m = x.max(axis=axis, keepdims=True)
    e = np.exp(x - m)
    return e / e.sum(axis=axis, keepdims=True)


def sigmoid(x: np.ndarray) -> np.ndarray:
    return 1.0 / (1.0 + np.exp(-x))


def multihead_self_attention(x, in_w, in_b, out_w, out_b, heads: int,
                             key_padding_mask: Optional[np.ndarray] = None,
                             attn_mask: Optional[np.ndarray] = None) -> np.ndarray:
    """nn.MultiheadAttention(batch_first=True)(x, x, x)[0] in eval mode.

    model/imf_vad.py:115,121 call it with no mask; the packed in-projection,
    the q * d_h**-0.5 scaling *before* QK^T and the softmax over keys follow
    torch/nn/functional.py:6244 (multi_head_attention_forward; scaling at :6632,
    softmax at :6643) which the eval fast path (torch/nn/modules/activation.py:1431)
    matches.  x: [B, T, D].  key_padding_mask: [B, T] bool (True = ignore) and
    attn_mask: additive [T, T] are only used by the model/module.py block."""
    B, T, D = x.shape
    dh = D // heads
    qkv = linear(x, in_w, in_b)                                   # [B,T,3D]
    q, k, v = qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:]
    q = q * x.dtype.type(1.0 / math.sqrt(dh))
    q = q.reshape(B, T, heads, dh).transpose(0, 2, 1, 3)         # [B,H,T,dh]
    k = k.reshape(B, T, heads, dh).transpose(0, 2, 1, 3)
    v = v.reshape(B, T, heads, dh).transpose(0, 2, 1, 3)
    s = q @ k.transpose(0, 1, 3, 2)                               # [B,H,T,T]
    if attn_mask is not None:
        s = s + attn_mask.astype(x.dtype)
    if key_padding_mask is not None:
        s = np.where(key_padding_mask[:, None, None, :], -np.inf, s).astype(x.dtype)
    p = softmax(s, axis=-1)
    o = (p @ v).transpose(0, 2, 1, 3).reshape(B, T, D)
    return linear(o, out_w, out_b)


# --------------------------------------------------------------------------
# N3: the attention-dropout mask of the training step
# --------------------------------------------------------------------------

_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """Philox4x32-10 (Salmon et al., SC'11; Random123's philox4x32 with 10 rounds) on uint64 arrays holding uint32
    words.  ctr: four broadcastable integer arrays, key: two integers -> the four output words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _M32 for c in ctr)
    k0, k1 = (np.uint64(int(k) & 0xFFFFFFFF) for k in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0                          # exact: both factors < 2^32
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0, c1, c2, c3


def attention_keep(seed: int, B: int, H: int, T: int, p: float) -> np.ndarray:
    """Multiplier of the attention weights under the training step's dropout (include/iefvad.h,
    iefvad_attention_train_fwd) -> float64 [B, H, T, T] indexed (b, h, query, key): Philox4x32-10 with counter
    (key >> 2, query, b * H + h, 0) and key (seed & 0xffffffff, seed >> 32), word key & 3; the weight is dropped when
    that word < uint32(double(float32(p)) * 2^32), kept weights are scaled by 1 / (1 - p) in float32 arithmetic."""
    seed = int(seed)
    q = np.arange(T, dtype=np.uint64)[None, :, None]
    k = np.arange(T, dtype=np.uint64)[None, None, :]
    bh = np.arange(B * H, dtype=np.uint64)[:, None, None]
    words = np.stack(np.broadcast_arrays(*philox4x32_10((k >> np.uint64(2), q, bh, 0), (seed, seed >> 32))))
    word = np.take_along_axis(words, np.broadcast_to(k & np.uint64(3), words.shape[1:])[None].astype(np.int64), 0)[0]
    pf = np.float32(p)
    thresh = int(np.float64(pf) * 4294967296.0) if pf > 0 else 0
    scale = np.float64(np.float32(1) / (np.float32(1) - pf))
    return np.where(word >= np.uint64(thresh), scale, 0.0).reshape(B, H, T, T)


# --------------------------------------------------------------------------
# A1-A6, A9: the MMFMIL forward
# --------------------------------------------------------------------------


def infer_config(params: Dict[str, np.ndarray]) -> Tuple[int, int, int]:
    """(embed_dim, num_layers, num_refinement_steps) from state_dict keys."""
    D = params["temporal.classifier.weight"].shape[1]
    L = 0
    while f"temporal.image_attn_layers.{L}.in_proj_weight" in params:
        L += 1
    R = 0
    while f"temporal.refinement_blocks.{R}.0.weight" in params:
        R += 1
    return D, L, R


def forward(params: Dict[str, np.ndarray], img: np.ndarray, ev: np.ndarray, *,
            heads: int = 8, lambda_ref: float = 0.5, noise_model: str = "StudentT",
            nu: float = 8, epsilon: float = 1e-8, dtype=np.float32) -> Dict[str, np.ndarray]:
    """MMFMIL.forward (model/imf_vad.py:40-44) -> MultiModal_Fusion_Attn_Iter.forward
    (model/imf_vad.py:109-161).  `params` uses the reference's state_dict keys.
    padding_mask / text / lengths are dropped by the reference (:40-44) and so
    have no parameter here."""
    P = {k: np.asarray(v, dtype=dtype) for k, v in params.items()}
    _, L, R = infer_config(P)
    enc = {}
    for mod, x in (("image", img), ("event", ev)):
        x = np.asarray(x).astype(dtype)                           # :41-42 .to(torch.float)
        for i in range(L):                                        # :114-116 / :120-122
            pre = f"temporal.{mod}_attn_layers.{i}."
            a = multihead_self_attention(x, P[pre + "in_proj_weight"], P[pre + "in_proj_bias"],
                                         P[pre + "out_proj.weight"], P[pre + "out_proj.bias"], heads)
            x = layer_norm(x + a, P[f"temporal.{mod}_norms.{i}.weight"], P[f"temporal.{mod}_norms.{i}.bias"])
        enc[mod] = layer_norm(x, P[f"temporal.whiten_{mod}.weight"], P[f"temporal.whiten_{mod}.bias"])  # :117/:123
    image_mu = linear(enc["image"], P["temporal.image_mu.weight"], P["temporal.image_mu.bias"])              # :125
    event_mu = linear(enc["event"], P["temporal.event_mu.weight"], P["temporal.event_mu.bias"])              # :126
    image_logvar = linear(enc["image"], P["temporal.image_logvar.weight"], P["temporal.image_logvar.bias"])  # :127
    event_logvar = linear(enc["event"], P["temporal.event_logvar.weight"], P["temporal.event_logvar.bias"])  # :128
    w_i, w_e, fused = fuse(image_mu, event_mu, image_logvar, event_logvar,
                           noise_model=noise_model, nu=nu, epsilon=epsilon)
    x = fused
    lam = np.asarray(lambda_ref, dtype=dtype)
    for i in range(R):                                            # :147-149
        h = np.maximum(linear(x, P[f"temporal.refinement_blocks.{i}.0.weight"],
                              P[f"temporal.refinement_blocks.{i}.0.bias"]), 0)
        r = linear(h, P[f"temporal.refinement_blocks.{i}.2.weight"], P[f"temporal.refinement_blocks.{i}.2.bias"])
        x = x - lam * r
    logits = linear(x, P["temporal.classifier.weight"], P["temporal.classifier.bias"])   # :150
    return {"fused": x, "logits": logits, "image_mu": image_mu, "event_mu": event_mu,    # :152-161
            "image_logvar": image_logvar, "event_logvar": event_logvar, "w_i": w_i, "w_e": w_e}


def fuse(image_mu, event_mu, image_logvar, event_logvar, *, noise_model="StudentT", nu=8, epsilon=1e-8):
    """Uncertainty-weighted fusion, model/imf_vad.py:130-144, in the reference's op order."""
    dt = image_mu.dtype.type
    if noise_model == "Gaussian":                                 # :130-132
        wi = np.exp(-image_logvar)
        we = np.exp(-event_logvar)
    elif noise_model == "StudentT":                               # :133-136
        factor = dt((nu + 1) / nu)
        wi = factor * np.exp(-image_logvar)
        we = factor * np.exp(-event_logvar)
    else:                                                         # :137-138
        raise ValueError("Unsupported noise_model. Choose 'Gaussian' or 'StudentT'.")
    denom = wi + we + dt(epsilon)                                 # :140
    nwi = wi / denom                                              # :141
    nwe = we / denom                                              # :142
    fused = nwi * image_mu + nwe * event_mu                       # :144
    return nwi, nwe, fused


# --------------------------------------------------------------------------
# A10: MIL top-k loss
# --------------------------------------------------------------------------


def clas2(logits: np.ndarray, labels: np.ndarray, lengths: Sequence[int], dtype=np.float32):
    """train/loss.py:18-30 (CLAS2).  logits [B,T,1] or [B,T]; labels [B,C] (column 0 = normal);
    lengths [B].  Returns (loss, per-row top-k means)."""
    B = logits.shape[0]
    p = sigmoid(np.asarray(logits, dtype=dtype).reshape(B, -1))   # :22
    y = (1 - np.asarray(labels, dtype=dtype)[:, 0]).reshape(B)    # :20
    v = np.zeros(B, dtype=dtype)
    for i in range(B):                                            # :24-27
        n = int(lengths[i])
        k = int(n / 16 + 1)
        row = p[i, :n]
        top = np.sort(row)[::-1][:k]                              # torch.topk values, descending
        v[i] = top.astype(dtype).mean(dtype=dtype)
    # F.binary_cross_entropy, mean reduction; torch clamps each log at -100
    ll = np.maximum(np.log(v), -100.0)
    l1 = np.maximum(np.log1p(-v), -100.0)
    loss = -(y * ll + (1 - y) * l1).mean(dtype=dtype)
    return dtype(loss), v


def mil_topk(p_row: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
    """Top-k of one row with the deterministic order the CUDA path promises:
    descending value, ties by ascending index (== torch.sort(stable=True, descending=True)[:k]).
    torch.topk's own tie order is unspecified and train/loss.py:25 discards the indices."""
    idx = np.argsort(-p_row, kind="stable")[:k]
    return p_row[idx], idx


# --------------------------------------------------------------------------
# Input shaping (what the reference's data layer hands to the path)
# --------------------------------------------------------------------------


def pad_rows(feat: np.ndarray, min_len: int) -> np.ndarray:
    """data/tools.py:81-86."""
    n = feat.shape[0]
    if n <= min_len:
        return np.pad(feat, ((0, min_len - n), (0, 0)), mode="constant", constant_values=0)
    return feat


def process_split(feat: np.ndarray, length: int) -> Tuple[np.ndarray, int]:
    """data/tools.py:100-114: < length -> one zero-padded [length, D] array (2-D!);
    otherwise int(n/length)+1 chunks of exactly `length` rows, the last zero padded -
    an all-zero chunk when n % length == 0."""
    n = feat.shape[0]
    if n < length:
        return pad_rows(feat, length), n
    s = int(n / length) + 1
    out = np.zeros((s, length, feat.shape[1]), dtype=feat.dtype)
    for i in range(s):
        part = feat[i * length:(i + 1) * length]
        out[i, :part.shape[0]] = part
    return out, n


def uniform_extract(feat: np.ndarray, t_max: int) -> np.ndarray:
    """data/tools.py:65-78 (avg=True branch): variable-width mean pooling into t_max bins."""
    out = np.zeros((t_max, feat.shape[1]), dtype=np.float32)
    r = np.linspace(0, len(feat), t_max + 1, dtype=np.int32)
    for i in range(t_max):
        if r[i] != r[i + 1]:
            out[i] = np.mean(feat[r[i]:r[i + 1]], 0)
        else:
            out[i] = feat[r[i]]
    return out


def process_feat(feat: np.ndarray, length: int) -> Tuple[np.ndarray, int]:
    """data/tools.py:89-97 with is_random=False."""
    if feat.shape[0] > length:
        return uniform_extract(feat, length), length
    return pad_rows(feat, length), feat.shape[0]


# --------------------------------------------------------------------------
# A8: frame-level AUC / AP  (scikit-learn restated)
# --------------------------------------------------------------------------


def _binary_clf_curve(y_true: np.ndarray, y_score: np.ndarray):
    """sklearn/metrics/_ranking.py `_binary_clf_curve`: stable descending argsort,
    distinct-score thresholds, cumulative TP / FP at each."""
    y_true = np.asarray(y_true, dtype=np.float64)
    y_score = np.asarray(y_score, dtype=np.float64)
    order = np.argsort(-y_score, kind="stable")
    y_score = y_score[order]
    y_true = y_true[order]
    distinct = np.where(np.diff(y_score))[0]
    thr = np.r_[distinct, y_true.size - 1]
    tps = np.cumsum(y_true, dtype=np.float64)[thr]
    fps = 1 + thr - tps
    return fps, tps, y_score[thr]


def roc_auc_score(y_true: np.ndarray, y_score: np.ndarray) -> float:
    """sklearn.metrics.roc_auc_score for binary labels (train/ucf_test.py:151,170,349):
    roc_curve (drop collinear points, prepend the origin) then the trapezoid rule.
    One class only -> NaN, as sklearn >= 1.6 returns (with a warning)."""
    y_true = np.asarray(y_true)
    if len(np.unique(y_true)) != 2:
        return float("nan")
    fps, tps, _ = _binary_clf_curve(y_true, y_score)
    if len(fps) > 2:                                              # drop_intermediate=True
        keep = np.where(np.r_[True, np.logical_or(np.diff(fps, 2), np.diff(tps, 2)), True])[0]
        fps, tps = fps[keep], tps[keep]
    tps = np.r_[0, tps]
    fps = np.r_[0, fps]
    fpr = fps / fps[-1]
    tpr = tps / tps[-1]
    return float(np.trapezoid(tpr, fpr))


def average_precision_score(y_true: np.ndarray, y_score: np.ndarray) -> float:
    """sklearn.metrics.average_precision_score (train/ucf_test.py:152,171):
    AP = sum_n (R_n - R_{n-1}) P_n over distinct thresholds."""
    fps, tps, _ = _binary_clf_curve(y_true, y_score)
    ps = tps + fps
    precision = np.zeros_like(tps)
    np.divide(tps, ps, out=precision, where=(ps != 0))
    if tps[-1] == 0:
        recall = np.ones_like(tps)
    else:
        recall = tps / tps[-1]
    sl = slice(None, None, -1)
    precision = np.hstack((precision[sl], 1))
    recall = np.hstack((recall[sl], 0))
    return float(max(0.0, -np.sum(np.diff(recall) * np.array(precision)[:-1])))


def auc_ap_segments(scores: np.ndarray, pos: np.ndarray, repeat: int = 16) -> Tuple[float, float]:
    """Closed form the CUDA path implements: each segment score stands for `repeat` frames of
    which pos[j] are positive.  Exact integer tie-group sums; equals roc_auc_score /
    average_precision_score on np.repeat(scores, repeat) (checked in tests)."""
    scores = np.asarray(scores)
    pos = np.asarray(pos, dtype=np.int64)
    neg = repeat - pos
    P, N = int(pos.sum()), int(neg.sum())
    order = np.argsort(-scores, kind="stable")
    s, p, n = scores[order], pos[order], neg[order]
    ends = np.r_[np.where(np.diff(s))[0], s.size - 1]
    tp = np.cumsum(p)[ends]
    fp = np.cumsum(n)[ends]
    tp0 = np.r_[0, tp[:-1]]
    fp0 = np.r_[0, fp[:-1]]
    if P == 0 or N == 0:
        auc = float("nan")
    else:
        num2 = int(np.sum((fp - fp0) * (tp + tp0)))               # 2 x trapezoid area x P x N, exact
        auc = num2 / (2.0 * P * N)
    if P == 0:
        # sklearn: recall := 1 everywhere, so the only non-zero recall step is the (1 -> 0) sentinel,
        # which multiplies the precision of the highest threshold = 0/.. = 0.
        ap = 0.0
    else:
        prec = tp / (tp + fp).astype(np.float64)
        ap = float(np.sum((tp - tp0) / float(P) * prec))
    return auc, ap


# --------------------------------------------------------------------------
# A7 + A8: the evaluation loop (train/ucf_test.py:70-178, 336-353)
# --------------------------------------------------------------------------


def eval_loop(params, videos: List[Tuple[np.ndarray, np.ndarray, str]], gt: np.ndarray, *,
              maxlen: int = 256, normal_keys=("Normal", "normal"), fwd=None, **fwd_kw):
    """videos: list of (img [T,D], ev [T,D], class name) in list order; gt: 0/1 per raw frame,
    16 per embedding row (list/ucf_generate_gt.py:24).  Restates the reference loop:
    process_split chunking (data/tools.py:100-114) -> forward on [S,256,D] -> sigmoid ->
    first len_cur rows (ucf_test.py:112-114) -> concat -> np.repeat(.,16) -> AUC/AP
    (:151-152), Ano-AUC (:336-353) and class-wise AUC/AP (:164-178).
    Returns dict(scores, AUC, AP, ano_AUC, classwise={cls: (auc, ap)})."""
    fwd = fwd or forward
    scores = []
    by_cls: Dict[str, List[np.ndarray]] = {}
    gt_cls: Dict[str, List[np.ndarray]] = {}
    st = 0
    for img, ev, cls in videos:
        fi, n = process_split(np.nan_to_num(img, nan=0.0), maxlen)        # ucf_test.py:83-88
        fe, _ = process_split(np.nan_to_num(ev, nan=0.0), maxlen)
        if n < maxlen:                                                    # :79-81
            fi, fe = fi[None], fe[None]
        out = fwd(params, fi, fe, **fwd_kw)
        lg = np.asarray(out["logits"]).reshape(-1)[:n]                    # :112-114
        prob = sigmoid(lg.astype(np.float32)).astype(np.float32)
        scores.append(prob)
        by_cls.setdefault(cls, []).append(prob)
        gt_cls.setdefault(cls, []).append(gt[16 * st:16 * (st + n)])      # :122
        st += n
    allp = np.concatenate(scores)
    rep = np.repeat(allp.astype(np.float64), 16)
    res = {"scores": allp, "AUC": roc_auc_score(gt, rep), "AP": average_precision_score(gt, rep)}
    g_ab = [np.concatenate(gt_cls[k]) for k in gt_cls if k not in normal_keys]
    p_ab = [np.concatenate(by_cls[k]) for k in gt_cls if k not in normal_keys]
    if g_ab and len(np.unique(np.concatenate(g_ab))) > 1:
        res["ano_AUC"] = roc_auc_score(np.concatenate(g_ab), np.repeat(np.concatenate(p_ab).astype(np.float64), 16))
    else:
        res["ano_AUC"] = float("nan")
    cw = {}
    for k in by_cls:
        g = np.concatenate(gt_cls[k])
        if len(g) == 0 or g.sum() == 0:                                   # :167-168
            continue
        r = np.repeat(np.concatenate(by_cls[k]).astype(np.float64), 16)
        cw[k] = (roc_auc_score(g, r), average_precision_score(g, r))
    res["classwise"] = cw
    return res


# --------------------------------------------------------------------------
# D1-D4: the dead-code classes the north star names (model/layers.py, model/module.py)
# --------------------------------------------------------------------------


def similarity_adj(x: np.ndarray, weight0: np.ndarray, seq_len: Optional[Sequence[int]] = None) -> np.ndarray:
    """SimilarityAdj.forward, model/layers.py:130-158.  weight0 [Din, Dout] is used for both
    theta and phi (:132-133; weight1 is never read).  Cosine similarity with +1e-20 on the
    norm product (:137-140); F.threshold(.,0.7,0) then softmax(dim=1) per batch element, only on
    the top-left len x len block when seq_len is given (the rest stays 0)."""
    theta = x @ weight0
    sim = theta @ theta.transpose(0, 2, 1)
    nrm = np.sqrt((theta * theta).sum(axis=2, keepdims=True))
    sim = sim / (nrm @ nrm.transpose(0, 2, 1) + x.dtype.type(1e-20))
    out = np.zeros_like(sim)
    for i in range(sim.shape[0]):
        n = sim.shape[1] if seq_len is None else int(seq_len[i])
        t = sim[i, :n, :n]
        t = np.where(t > 0.7, t, 0).astype(x.dtype)
        out[i, :n, :n] = softmax(t, axis=1)
    return out


def distance_adj(batch_size: int, max_seqlen: int, dtype=np.float32) -> np.ndarray:
    """DistanceAdj.forward, model/layers.py:172-179: exp(-|i-j| / e); `sigma` is unused.
    (The reference hard-codes .to('cuda') so it cannot run on a CPU-only box; this follows
    the lines literally.)"""
    idx = np.arange(max_seqlen)
    dist = np.abs(idx[:, None] - idx[None, :]).astype(np.float32)
    adj = np.exp(-dist / np.exp(np.float32(1.0))).astype(dtype)
    return np.repeat(adj[None], batch_size, axis=0)


def graph_convolution(x: np.ndarray, adj: np.ndarray, weight: np.ndarray, bias: Optional[np.ndarray] = None,
                      residual: str = "identity", conv_w: Optional[np.ndarray] = None,
                      conv_b: Optional[np.ndarray] = None) -> np.ndarray:
    """GraphConvolution.forward, model/layers.py:91-106: adj @ (x @ W) (+bias) + residual.
    residual: 'identity' (Din==Dout), 'none' (residual=False -> +0) or 'conv'
    (Conv1d(Din->Dout, k=5, pad=2) along T, :84,98-102; conv_w [Dout, Din, 5])."""
    out = adj @ (x @ weight)
    if bias is not None:
        out = out + bias
    if residual == "identity":
        out = out + x
    elif residual == "conv":
        B, T, Din = x.shape
        xp = np.pad(x, ((0, 0), (2, 2), (0, 0)))
        res = np.zeros((B, T, conv_w.shape[0]), dtype=x.dtype)
        for k in range(5):
            res += xp[:, k:k + T] @ conv_w[:, :, k].T
        out = out + res + conv_b
    return out


def graph_convolution_distance_scan(x: np.ndarray, weight: np.ndarray) -> np.ndarray:
    """adj @ support for the DistanceAdj adjacency as a forward + backward first-order linear
    recurrence (SURVEY.md F3): y_t = s_t + r*(fwd_{t-1}) + r*(bwd_{t+1}), r = exp(-1/e)."""
    s = x @ weight
    r = x.dtype.type(np.exp(-1.0 / np.exp(np.float32(1.0))))
    f = np.zeros_like(s)
    b = np.zeros_like(s)
    T = s.shape[1]
    for t in range(1, T):
        f[:, t] = r * (f[:, t - 1] + s[:, t - 1])
    for t in range(T - 2, -1, -1):
        b[:, t] = r * (b[:, t + 1] + s[:, t + 1])
    return s + f + b


def quick_gelu(x: np.ndarray) -> np.ndarray:
    """model/module.py:15-17."""
    return x * sigmoid(x.dtype.type(1.702) * x)


def transformer(x: np.ndarray, blocks: List[Dict[str, np.ndarray]], heads: int,
                padding_mask: Optional[np.ndarray] = None, attn_mask: Optional[np.ndarray] = None) -> np.ndarray:
    """Transformer / ResidualAttentionBlock, model/module.py:20-54.  x is SEQ-FIRST [L, N, D]
    like the reference; each block: x += MHA(LN1(x)); x += c_proj(QuickGELU(c_fc(LN2(x)))).
    `blocks[i]` holds that block's state_dict entries without the `resblocks.i.` prefix."""
    xb = x.transpose(1, 0, 2)                                      # -> [N, L, D]
    for p in blocks:
        h = layer_norm(xb, p["ln_1.weight"], p["ln_1.bias"])
        xb = xb + multihead_self_attention(h, p["attn.in_proj_weight"], p["attn.in_proj_bias"],
                                           p["attn.out_proj.weight"], p["attn.out_proj.bias"], heads,
                                           key_padding_mask=padding_mask, attn_mask=attn_mask)
        h = layer_norm(xb, p["ln_2.weight"], p["ln_2.bias"])
        h = quick_gelu(linear(h, p["mlp.c_fc.weight"], p["mlp.c_fc.bias"]))
        xb = xb + linear(h, p["mlp.c_proj.weight"], p["mlp.c_proj.bias"])
    return xb.transpose(1, 0, 2)


# --------------------------------------------------------------------------
# synthetic event frames (row N4): extracting/ucf_gen_event.py
# --------------------------------------------------------------------------

def _r32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def gray_image(frames: np.ndarray) -> np.ndarray:
    """extracting/ucf_gen_event.py:22-33: torch.tensordot(frames.float(), [0.2989, 0.5870, 0.1140]) on the CPU.
    The contraction is an MKL sgemv with K = 3; its rounding is fl(fma(G, w1, fl(R w0)) + fl(B w2)) (found by
    comparing every fused / unfused association order with torch on 2e5 random pixels, pinned by the threshold-tie
    cases of tests/golden/event.npz).  float64 holds every float32 product and two-term sum exactly, so rounding a
    float64 result to float32 reproduces both the plain and the fused float32 operations."""
    w = np.array([0.2989, 0.5870, 0.1140], dtype=np.float32).astype(np.float64)
    f = np.asarray(frames).astype(np.float64)
    t = _r32(f[..., 0] * w[0])
    t = _r32(f[..., 1] * w[1] + t)                    # fma: one rounding
    u = _r32(f[..., 2] * w[2])
    return _r32(t + u).astype(np.float32)


def generate_event_image(frames: np.ndarray, threshold=25) -> np.ndarray:
    """extracting/ucf_gen_event.py:21-37.  frames uint8 [B, C, H, W, 3] -> [B, H, W] float32 event counts."""
    g = gray_image(frames)
    diffs = np.abs(g[:, 1:] - g[:, :-1])              # float32 subtraction (:34)
    return (diffs > np.float32(threshold)).astype(np.float32).sum(1)            # :36-37


def event_images(frames: np.ndarray, threshold=25, clamp=10) -> np.ndarray:
    """The caller's lines extracting/ucf_gen_event.py:91-95: clamp, divide by the batch maximum, stack 3 channels
    (an event-free batch divides 0 by 0 = NaN there too)."""
    event = np.clip(generate_event_image(frames, threshold), np.float32(0), np.float32(clamp))
    if event.size != 0:
        with np.errstate(invalid="ignore", divide="ignore"):
            event = (event / event.max()).astype(np.float32)
    return np.stack([event, event, event], 1)


# --------------------------------------------------------------------------
# Error metrics (SURVEY.md section 8c "metric definition")
# --------------------------------------------------------------------------


# --------------------------------------------------------------------------
# N5: temporal-localisation mAP (train/metrics.py:19-136; never called by the reference's live loops)
# --------------------------------------------------------------------------
LOC_CLASSLIST = ['Normal', 'Abuse', 'Arrest', 'Arson', 'Assault', 'Burglary', 'Explosion', 'Fighting', 'RoadAccidents',
                 'Robbery', 'Shooting', 'Shoplifting', 'Stealing', 'Vandalism']          # train/metrics.py:53


def loc_nms(dets: np.ndarray, thresh: float = 0.6) -> List[int]:
    """train/metrics.py:19-41: greedy 1-D NMS over [start, end] rows already sorted by score -> kept indices."""
    if len(dets) == 0:
        return []
    dets = np.asarray(dets, dtype=np.float64)
    x1, x2 = dets[:, 0], dets[:, 1]
    lengths = x2 - x1
    order = np.arange(len(dets))
    keep = []
    while order.size > 0:
        i = order[0]
        keep.append(int(i))
        xx1 = np.maximum(x1[i], x1[order[1:]])
        xx2 = np.minimum(x2[i], x2[order[1:]])
        inter = np.maximum(0.0, xx2 - xx1)
        ovr = inter / (lengths[i] + lengths[order[1:]] - inter)
        order = order[np.where(ovr <= thresh)[0] + 1]
    return keep


def loc_map(predictions, th: float, gtsegments, gtlabels, exclude_normal: bool = False):
    """train/metrics.py:44-126 (`getLocMAP`), statement by statement; predictions[i] is a float32 [T_i, 14] array."""
    if exclude_normal is True:                                               # :45-48
        predictions = predictions[:140]
    c_score, mod = [], []
    for p in predictions:                                                    # :58-65
        p = np.asarray(p, dtype=np.float32)
        pp = -np.sort(-p, axis=0)
        with np.errstate(invalid="ignore", divide="ignore"):
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                c_s = np.mean(pp[:int(p.shape[0] / 16), :], axis=0)
        c_score.append(c_s)
        mod.append(p * (c_s > 0.0))
    ap = []
    for c in range(14):                                                      # :68
        segment_predict = []
        for i in range(len(mod)):                                            # :71-88
            tmp = mod[i][:, c]
            if tmp.size == 0:
                continue
            threshold = np.max(tmp) - (np.max(tmp) - np.min(tmp)) * np.float64(0.6)
            vid_pred = np.concatenate([np.zeros(1), (tmp > threshold).astype('float32'), np.zeros(1)], axis=0)
            diff = vid_pred[1:] - vid_pred[:-1]
            s = np.nonzero(diff == 1)[0]
            e = np.nonzero(diff == -1)[0]
            cand = []
            for j in range(len(s)):
                if e[j] - s[j] >= 2:
                    cand.append([i, s[j], e[j], np.max(tmp[s[j]:e[j]]) + np.float32(0.7) * c_score[i][c]])
            if cand:
                cand = np.array(cand)
                cand = cand[np.argsort(-cand[:, -1], kind="stable")]
                segment_predict.extend(list(cand[loc_nms(cand[:, 1:-1], 0.6)]))
        segment_predict = np.array(segment_predict)
        if len(segment_predict) == 0:                                        # :92-93
            return 0
        segment_predict = segment_predict[np.argsort(-segment_predict[:, 3], kind="stable")]       # :96
        segment_gt = [[i, gtsegments[i][j][0], gtsegments[i][j][1]] for i in range(len(gtsegments))
                      for j in range(len(gtsegments[i])) if gtlabels[i][j] == LOC_CLASSLIST[c]]       # :99-100
        gtpos = len(segment_gt)
        tp, fp = [], []
        for i in range(len(segment_predict)):                                # :104-122
            flag, best_iou, best_j = 0.0, 0.0, -1
            for j in range(len(segment_gt)):
                if segment_predict[i][0] == segment_gt[j][0]:
                    gs, ge = int(segment_gt[j][1]), int(segment_gt[j][2])
                    ps, pe = int(segment_predict[i][1]), int(segment_predict[i][2])
                    lg, lp = max(ge - gs, 0), max(pe - ps, 0)
                    inter = max(min(pe, ge) - max(ps, gs), 0) if lg and lp else 0
                    iou = float(inter) / float(lg + lp - inter)
                    if iou >= th:
                        flag = 1.0
                        if iou > best_iou:
                            best_iou, best_j = iou, j
            if flag > 0:
                del segment_gt[best_j]
            tp.append(flag)
            fp.append(1.0 - flag)
        tp_c, fp_c = np.cumsum(tp), np.cumsum(fp)
        ap.append(0.0 if sum(tp) == 0 else float(np.sum((tp_c / (fp_c + tp_c)) * tp) / gtpos))    # :123-127
    return 100 * np.mean(ap)


def max_norm_err(x: np.ndarray, ref: np.ndarray) -> float:
    """max|x - ref| / max|ref| per tensor."""
    ref = np.asarray(ref, dtype=np.float64)
    return float(np.max(np.abs(np.asarray(x, dtype=np.float64) - ref)) / max(np.max(np.abs(ref)), 1e-300))


def score_rel_err(logits: np.ndarray, ref_logits: np.ndarray) -> float:
    """max |p - p_ref| / p_ref on sigmoid scores."""
    p = sigmoid(np.asarray(logits, dtype=np.float64))
    r = sigmoid(np.asarray(ref_logits, dtype=np.float64))
    return float(np.max(np.abs(p - r) / r))
