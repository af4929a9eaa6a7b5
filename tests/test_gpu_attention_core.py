"""The three tensor-core attention kernels (iefvad_attention_core) against float64 on their own 16-bit operands.  Needs
a B200.

Operands are drawn at random, rounded once to fp16 or bf16, and the reference is softmax(q k^T) v in float64 (on the
device) over exactly those rounded values.  The difference therefore measures the kernels' own arithmetic only.

Bound, per output element (row i, column d), with u = 2^-11 (fp16) or 2^-8 (bf16) and V_d = max_j |v_jd| over the keys
of the row's (batch, head) or ragged item:

    |got - ref| <= 2u (|ref| + V_d) + 2 e_s V_d  [+ n_sub 2^-23 V_d for fp16]

Derivation.  The kernels compute out = sum_j P16_j v_j / l with P16_j = round16(p_j), p_j = 2^(s_j log2e - m) in fp32
and l = sum_j p_j in fp32 (the unrounded p).
- P rounded to 16 bits: |P16_j - p_j| <= u p_j, so the numerator moves by at most u sum_j p_j |v_jd| <= u l V_d.
- Final 16-bit store: u |ref|.
- Score and exponent: the products of two 16-bit values are exact in fp32; the fp32 sum, the addition of a mask or of
  log(mult), the fused s log2e - m and ex2.approx each perturb p_j by a relative e_j.  sum_j p_j e_j (v_jd - out_d) / l
  is at most 2 max_j e_j V_d.  e_s = 2^-20 (1 + max_j (sum_d |q_d k_jd| + |mask_ij|)) bounds e_j: sixteen fp32
  roundings of the largest partial sum, plus the ex2.approx and __logf error (the 1).  The max runs over the keys whose
  float64 weight is at least 2^-100 of the row's largest; lighter keys give P = 0 in fp32 (ex2.approx flushes below
  2^-126), an error far below any bound here.  The term only matters for large scores or masks.
- fp32 accumulation of P.V and of l, and the fp32 division, add O(2^-17) relative at T = 16 384; the factor 2 on u
  covers them.
- fp16 P below 2^-14 is subnormal and rounds with an absolute error up to 2^-25 instead of u p_j.  The long kernel
  rounds P against its own half's maximum and then multiplies the packed fp16 value by a power of two, so a key can be
  rounded twice, and its unit 2^run can be up to twice the row maximum (l >= 1/2).  So each key whose float64 weight is
  below 2^-13 of the row's largest (n_sub of them) adds at most 4 * 2^-25 = 2^-23 V_d.  bf16 has fp32's exponent range
  and no such term.
Every fp16 output must also meet the bf16 bound divided by four: an fp16 case that quietly ran a bf16 step would not.

Inputs a correct kernel must never read, or may only multiply by an exact P = 0, are poisoned: NaN in the q / k pad
columns dh..dhp (the MMAs cover the first dh columns only) and in the vt columns T..Tpad (the TMA extent is T), and
large finite values in the rows between ragged items.  Every output element the kernel must not write holds a
sentinel that must survive.
"""
import functools
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

FMT = {"fp16": torch.float16, "bf16": torch.bfloat16}
U = {"fp16": 2.0 ** -11, "bf16": 2.0 ** -8}
SHORT_PAIRS = [(96, 96), (96, 128), (64, 64), (128, 128), (32, 64), (32, 32)]
WIDE_PAIRS = [(96, 128), (64, 64), (128, 128), (32, 64)]          # the long and flash kernels
SHORT_T = [1, 8, 31, 64, 65, 127, 128, 129, 255, 256]
LONG_T = [257, 319, 320, 383, 384, 385, 512, 513, 1000, 16384]
FLASH_T = [1, 129, 300]
# score distributions: batch element b of a dense case (ragged item b) draws DISTS[b % 9]
DISTS = ["uniform", "peaked", "last", "odd_half", "ramp", "equal", "subnormal", "neg_huge", "pos_huge"]
SENTINEL = -16384.0                     # exact in fp16 and bf16, far outside any convex combination of the values
POISON = 30000.0                        # finite in fp16 and bf16: rows between ragged items
KERNEL = {"short": "attn_short_kernel", "long": "attn_long_kernel", "flash": "attn_tc_kernel"}
HUGE_A = {32: 28, 64: 20, 96: 16, 128: 14}     # a^2 dh in [24 000, 26 000]
DEV = "cuda"


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from iefvad_b200 import ops as _ops
    return _ops


# ------------------------------------------------------------------------------------------------ operands
def make_head(dist, H, T, dh, seed):
    """fp32 (q, k, v) [H, T, dh] on the CPU with the score distribution `dist` (q already carries the 1/sqrt(dh))."""
    g = torch.Generator().manual_seed(seed)

    def r(*s):
        return torch.randn(*s, generator=g)

    v = r(H, T, dh)
    k = r(H, T, dh)
    j = torch.arange(T)
    if dist == "uniform":                                   # scores ~ N(0, 0.1^2)
        q = r(H, T, dh) * (0.1 / math.sqrt(dh))
    elif dist == "peaked":                                  # scores ~ N(0, 10^2): logits across about +-30
        q = r(H, T, dh) * (10 / math.sqrt(dh))
    elif dist in ("last", "odd_half", "ramp"):
        # score = 4 k_j0 + N(0, 1) with a +20 bump on the last 32 keys (the row max lies only in the last key block, and
        # for the short kernel in the second key half), on keys [64, 128) of every 128-key block (the second half of each
        # long-kernel block), or a ramp rising by 32 along the row (the running max moves in every block)
        q = r(H, T, dh) / math.sqrt(dh)
        q[..., 0] = 4.0
        k[..., 0] *= 0.5
        if dist == "last":
            k[:, max(T - 32, 0):, 0] += 5.0
        elif dist == "odd_half":
            k[:, (j // 64) % 2 == 1, 0] += 5.0
        else:
            k[..., 0] += 8.0 * j / T
    elif dist == "equal":                                   # every key of a row has the same score
        q = r(H, T, dh)
        k = r(H, 1, dh).expand(H, T, dh).clone()
    elif dist == "subnormal":
        # every 8th key at the max, the others 15-25 binades below it: fp16 P lands in the subnormal range
        q = r(H, T, dh) * 0.01
        q[..., 0] = 1.0
        k[..., 0] = -math.log(2.0) * (15 + 10 * torch.rand(H, T, generator=g))
        k[:, ::8, 0] = 0.0
    elif dist in ("neg_huge", "pos_huge"):
        # q_d = a + e, k_d = -+a + f with e, f in {-1/8, 0, 1/8} on 8 dims: every score in -+[24 000, 26 000], exact in
        # fp32 (products are multiples of 2^-6, sums below 2^15), a few units apart between keys
        a = float(HUGE_A[dh])
        q = torch.full((H, T, dh), a)
        k = torch.full((H, T, dh), -a if dist == "neg_huge" else a)
        q[..., :8] += torch.randint(-1, 2, (H, T, 8), generator=g) / 8
        k[..., :8] += torch.randint(-1, 2, (H, T, 8), generator=g) / 8
    else:
        raise ValueError(dist)
    return q, k, v


@functools.lru_cache(maxsize=4)
def dense_operands(B, H, T, dh):
    """fp32 [B, H, T, dh] q, k, v on the CPU; batch element b draws DISTS[b % 9]."""
    qs, ks, vs = zip(*(make_head(DISTS[b % len(DISTS)], H, T, dh, 17 * b + T) for b in range(B)))
    return torch.stack(qs), torch.stack(ks), torch.stack(vs)


def to16(x, fmt):
    return x.to(FMT[fmt]).to(DEV)


def pack_qk(x16, dhp):
    """[..., T, dh] -> [..., T, dhp] with NaN in the pad columns."""
    out = torch.full(x16.shape[:-1] + (dhp,), float("nan"), dtype=x16.dtype, device=x16.device)
    out[..., :x16.shape[-1]] = x16
    return out


def pack_vt(v16, Tpad):
    """[..., T, dh] -> [..., dh, Tpad] with NaN in the columns T..Tpad."""
    out = torch.full(v16.shape[:-2] + (v16.shape[-1], Tpad), float("nan"), dtype=v16.dtype, device=v16.device)
    out[..., :v16.shape[-2]] = v16.transpose(-1, -2)
    return out


def tpad_of(T):
    return (T + 7) // 8 * 8 + 8             # a NaN tail also where T % 8 == 0


# ------------------------------------------------------------------------------------------------ reference and bound
def attend(q, k, v, mask=None):
    """float64 softmax(q k^T + mask) v with the bound's e_s and n_sub per row.  q [..., R, dh], k / v [..., S, dh],
    mask additive [..., R, S] (may hold -inf).  A row whose keys are all -inf gives NaN, as nn.MultiheadAttention does."""
    s = q @ k.transpose(-1, -2)
    a = q.abs() @ k.abs().transpose(-1, -2)
    if mask is not None:
        s = s + mask
        a = a + torch.where(torch.isfinite(mask), mask.abs(), 0.0)
    w = torch.exp(s - s.amax(-1, keepdim=True))            # NaN for a fully masked row
    out = (w @ v) / w.sum(-1, keepdim=True)
    es = 2.0 ** -20 * (1 + torch.where(w >= 2.0 ** -100, a, 0.0).amax(-1))
    nsub = ((w > 0) & (w < 2.0 ** -13)).sum(-1).double()
    return out, es, nsub


def bound(ref, V, es, nsub, u, fp16):
    b = 2 * u * (ref.abs() + V) + 2 * es[..., None] * V
    if fp16:
        b = b + nsub[..., None] * 2.0 ** -23 * V
    return b


def ratio_to_bound(got, ref, V, es, nsub, fmt):
    """Worst |got - ref| / bound over the rows the reference does not leave NaN; a NaN pattern unlike the reference's
    counts as infinitely wrong."""
    nan_ref = torch.isnan(ref)
    if bool((torch.isnan(got) != nan_ref).any()):
        return math.inf
    r = torch.where(nan_ref, 0.0, (got - ref).abs() / bound(ref, V, es, nsub, U[fmt], fmt == "fp16"))
    return float(r.max()) if r.numel() else 0.0


def check(got, ref, V, es, nsub, fmt, label, groups):
    """got / ref [N, dh], V [N, dh], es / nsub [N], groups [N] (names for the failure message).  Asserts the NaN pattern
    and the bound, and for fp16 a quarter of the bf16 bound.  -> worst |got - ref| / bound."""
    nan_ref = torch.isnan(ref)
    bad = (torch.isnan(got) != nan_ref).any(-1)
    assert not bool(bad.any()), (f"{label}: {int(bad.sum())} rows whose NaN pattern differs from float64, in "
                                 f"{sorted(set(groups[bad.cpu().numpy()].tolist()))}; first got "
                                 f"{got[bad][0, :4].tolist()} where float64 has {ref[bad][0, :4].tolist()}")
    err = (got - ref).abs()
    ratio = torch.where(nan_ref, 0.0, err / bound(ref, V, es, nsub, U[fmt], fmt == "fp16")).amax(-1)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    print(f"attention-core ratio {label}: {worst:.3g}")
    if worst > 1:
        per = {gname: round(float(ratio[torch.as_tensor(groups == gname, device=ratio.device)].max()), 3)
               for gname in sorted(set(groups.tolist()))}
        raise AssertionError(f"{label}: error / bound = {worst:.3g}; worst per group {per}")
    if fmt == "fp16":
        q4 = float(torch.where(nan_ref, 0.0, err / (bound(ref, V, es, nsub, U["bf16"], False) / 4)).max())
        assert q4 <= 1, f"{label}: fp16 output misses a quarter of the bf16 bound ({q4:.3g})"
    return worst


# ------------------------------------------------------------------------------------------------ dense cases
def sample_rows(T):
    if T <= 2048:
        return torch.arange(T)
    g = torch.Generator().manual_seed(T)
    fixed = torch.tensor([0, 1, 127, 128, 255, 256, 257, 511, 512, T // 2, T - 129, T - 128, T - 2, T - 1])
    return torch.unique(torch.cat([fixed, torch.randperm(T, generator=g)[:242]]))


def key_pad_pattern(B, T):
    """[B, T] bool: b % 9 == 1 a fully padded 128-key prefix, 2 every key, 3 random 30 %, 4 the second half."""
    g = torch.Generator().manual_seed(5)
    kp = torch.zeros(B, T, dtype=torch.bool)
    for b in range(B):
        c = b % 9
        if c == 1:
            kp[b, :min(128, T - 1)] = True
        elif c == 2:
            kp[b] = True
        elif c == 3:
            kp[b] = torch.rand(T, generator=g) < 0.3
        elif c == 4:
            kp[b, (T + 1) // 2:] = True
    return kp


MASKS = {                     # name: (value above the diagonal or None for an all-zero mask, key padding)
    "zero": (None, False),
    "causal_1e4": (-1e4, False),
    "causal_1e4_pad": (-1e4, True),
    "causal_inf_pad": (float("-inf"), True),
    "pad": (None, True),
}


def run_dense(ops, fmt, dh, dhp, T, B=9, H=2, mask="none", use_row_out=False, drop_key=None, mask_shift=False):
    """One dense case through iefvad_attention_core.  mask: "none" (short / long kernel) or a MASKS key (flash kernel).
    -> (worst ratio, {wrong reference: ratio})."""
    q32, k32, v32 = dense_operands(B, H, T, dh)
    q16, k16, v16 = to16(q32, fmt), to16(k32, fmt), to16(v32, fmt)
    am = kp = None
    if mask != "none":
        fill, with_pad = MASKS[mask]
        am = torch.zeros(T, T, dtype=torch.float64, device=DEV)
        if fill is not None:
            am[torch.ones(T, T, dtype=torch.bool, device=DEV).triu(1)] = fill
        kp = key_pad_pattern(B, T).to(DEV) if with_pad else None
    ldo, rows_out = H * dh + 8, B * T + 8
    out = torch.full((rows_out, ldo), SENTINEL, dtype=FMT[fmt], device=DEV)
    if use_row_out:
        g = torch.Generator().manual_seed(T + dh)
        orow = torch.randperm(rows_out, generator=g)[:B * T].int()
        orow[torch.rand(B * T, generator=g) < 0.2] = -1
    else:
        orow = torch.arange(B * T, dtype=torch.int32)
    orow = orow.to(DEV)
    ops.attention_core(pack_qk(q16, dhp), pack_qk(k16, dhp), pack_vt(v16, tpad_of(T)),
                       attn_mask=am.float() if am is not None else None, key_padding_mask=kp,
                       row_out=orow if use_row_out else None, out=out)
    torch.cuda.synchronize()
    kernel = ("short" if T <= 256 else "long") if mask == "none" else "flash"
    label = f"{kernel} {fmt} ({dh},{dhp}) T={T} B={B} H={H} mask={mask}{' row_out' if use_row_out else ''}"
    orow = orow.long()
    written = torch.zeros(rows_out, ldo, dtype=torch.bool, device=DEV)
    written[orow[orow >= 0], :H * dh] = True
    assert bool((out[~written] == SENTINEL).all()), f"{label}: {int((out[~written] != SENTINEL).sum())} writes outside " \
                                                   f"the stored rows' head columns"
    rows = sample_rows(T).to(DEV)
    R = len(rows)
    got = out[orow.clamp(min=0)].double()[:, :H * dh].reshape(B, T, H, dh).permute(0, 2, 1, 3)[:, :, rows]
    sel = (orow >= 0).view(B, 1, T)[:, :, rows].expand(B, H, R).reshape(-1)
    qd, kd, vd = q16.double(), k16.double(), v16.double()
    V = vd.abs().amax(2, keepdim=True).expand(B, H, R, dh)
    groups = np.repeat(np.array([DISTS[b % 9] for b in range(B)]), H * R)[sel.cpu().numpy()]

    def flat(x):
        return x.reshape(B * H * R, -1)[sel]

    def reference(am_):
        full = am_[rows].expand(B, H, R, T) if am_ is not None else None
        if kp is not None:
            padm = torch.where(kp, float("-inf"), 0.0).double()[:, None, None, :]
            full = padm.expand(B, H, R, T) if full is None else full + padm
        ref, es, nsub = attend(qd[:, :, rows], kd, vd, full)
        return flat(ref), flat(es)[:, 0], flat(nsub)[:, 0]

    got, V = flat(got), flat(V)
    ref, es, nsub = reference(am)
    worst = check(got, ref, V, es, nsub, fmt, label, groups)
    wrong = {}
    if drop_key is not None:
        am_drop = am.clone() if am is not None else torch.zeros(T, T, dtype=torch.float64, device=DEV)
        am_drop[:, drop_key] = float("-inf")
        wrong["one key dropped"] = am_drop
    if mask_shift:
        wrong["mask shifted by one key"] = torch.roll(am, 1, dims=1)
    for name, am_ in wrong.items():
        r, e, n = reference(am_)
        wrong[name] = ratio_to_bound(got, r, V, e, n, fmt)
    return worst, wrong


# ------------------------------------------------------------------------------------------------ ragged items
def ragged_items(n=40, seed=3):
    """n items whose starts are multiples of 8 with gaps of poison rows between some, rows 1..256 (<= 128 and > 128
    mixed), mult 0, 1, 2 or 255, sorted longest first as Model::forward does.  -> (items [n, 4] int32, packed rows)."""
    g = np.random.default_rng(seed)
    specs = [(1, 0), (1, 255), (255, 1), (128, 0), (127, 1), (128, 2), (256, 0), (129, 255), (2, 2), (64, 1)]
    while len(specs) < n:
        mult = [0, 1, 2, 255][len(specs) % 4]
        specs.append((int(g.integers(1, 256 if mult else 257)), mult))
    items, cur = [], 0
    for i, (valid, mult) in enumerate(specs):
        rows = valid + (1 if mult else 0)
        items.append((cur, rows, valid, mult))
        cur = (cur + rows + 7) // 8 * 8 + (8 if i % 3 == 0 else 0)
    items.sort(key=lambda it: -it[1])
    return torch.tensor(items, dtype=torch.int32), cur + 8


def ragged_reference(q, k, v, items, mult_delta=0):
    """Per item: dense float64 attention of its rows over valid + mult keys, the last row repeated mult times (mult +
    mult_delta for a wrong reference).  q, k, v [H, M, dh] float64.  -> ref, V [H, M, dh], es, nsub [H, M]."""
    H, M, dh = q.shape
    ref = torch.full((H, M, dh), float("nan"), dtype=torch.float64, device=q.device)
    V = torch.zeros_like(ref)
    es = torch.zeros(H, M, dtype=torch.float64, device=q.device)
    nsub = torch.zeros_like(es)
    for start, rows, valid, mult in items.tolist():
        m = mult + mult_delta if mult else 0
        idx = torch.cat([torch.arange(start, start + valid), torch.full((m,), start + valid)]).to(q.device)
        o, e, n = attend(q[:, start:start + rows], k[:, idx], v[:, idx])
        ref[:, start:start + rows], es[:, start:start + rows], nsub[:, start:start + rows] = o, e, n
        V[:, start:start + rows] = v[:, idx].abs().amax(1, keepdim=True)
    return ref, V, es, nsub


def run_ragged(ops, fmt, dh, dhp, H=8, use_row_out=False, wrong_mult=False):
    """Ragged items on the short kernel.  -> (worst ratio, {wrong reference: ratio})."""
    items, M = ragged_items()
    q32 = torch.full((H, M, dh), POISON)
    k32, v32 = q32.clone(), q32.clone()
    row_group = np.full(M, "gap", dtype=object)
    for i, (start, rows, valid, mult) in enumerate(items.tolist()):
        q32[:, start:start + rows], k32[:, start:start + rows], v32[:, start:start + rows] = \
            make_head(DISTS[i % 9], H, rows, dh, 100 + i)
        row_group[start:start + rows] = f"{DISTS[i % 9]} mult {mult}"
    q16, k16, v16 = to16(q32, fmt), to16(k32, fmt), to16(v32, fmt)
    ldo, rows_out = H * dh + 8, M + 8
    out = torch.full((rows_out, ldo), SENTINEL, dtype=FMT[fmt], device=DEV)
    in_item = torch.as_tensor(row_group != "gap")
    if use_row_out:
        g = torch.Generator().manual_seed(dh)
        orow = torch.randperm(rows_out - 1, generator=g)[:M].int()
        orow[torch.rand(M, generator=g) < 0.2] = -1
        orow[~in_item] = rows_out - 1              # never read for rows outside the items: this row keeps its sentinel
    else:
        orow = torch.arange(M, dtype=torch.int32)
    orow = orow.to(DEV)
    ops.attention_core(pack_qk(q16[None], dhp), pack_qk(k16[None], dhp), pack_vt(v16[None], M + 8),
                       row_out=orow if use_row_out else None, items=items.to(DEV), out=out)
    torch.cuda.synchronize()
    label = f"short {fmt} ({dh},{dhp}) ragged items={items.shape[0]} H={H}{' row_out' if use_row_out else ''}"
    orow = orow.long()
    stored = in_item.to(DEV) & (orow >= 0)
    written = torch.zeros(rows_out, ldo, dtype=torch.bool, device=DEV)
    written[orow[stored], :H * dh] = True
    assert bool((out[~written] == SENTINEL).all()), f"{label}: writes outside the items' stored rows"
    got = out[orow.clamp(min=0)].double()[:, :H * dh].reshape(M, H, dh).permute(1, 0, 2)
    sel = stored.expand(H, M).reshape(-1)
    groups = np.tile(row_group, H)[sel.cpu().numpy()]

    def flat(x):
        return x.reshape(H * M, -1)[sel]

    qd, kd, vd = q16.double(), k16.double(), v16.double()
    ref, V, es, nsub = ragged_reference(qd, kd, vd, items)
    got, V = flat(got), flat(V)
    worst = check(got, flat(ref), V, flat(es)[:, 0], flat(nsub)[:, 0], fmt, label, groups)
    wrong = {}
    if wrong_mult:
        r, Vw, e, n = ragged_reference(qd, kd, vd, items, mult_delta=-1)
        wrong["multiplicity m - 1"] = ratio_to_bound(got, flat(r), flat(Vw), flat(e)[:, 0], flat(n)[:, 0], fmt)
    return worst, wrong


# ------------------------------------------------------------------------------------------------ tests
def _flash_pair(dh, dhp):
    """The flash kernel's q / k row length for a short-kernel pair: unpadded rows padded to a multiple of 64."""
    return dh, (dhp + 63) // 64 * 64


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
@pytest.mark.parametrize("dh,dhp", SHORT_PAIRS)
@pytest.mark.parametrize("T", SHORT_T)
def test_short_kernel_matches_float64(ops, fmt, dh, dhp, T):
    """T <= 256 without a mask: the short kernel at the tile, half and 32-key chunk edges; then the same operands
    through the flash kernel (all-zero mask)."""
    run_dense(ops, fmt, dh, dhp, T, use_row_out=T % 2 == 1)
    run_dense(ops, fmt, *_flash_pair(dh, dhp), T, mask="zero")


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
@pytest.mark.parametrize("dh,dhp", WIDE_PAIRS)
@pytest.mark.parametrize("T", LONG_T)
def test_long_kernel_matches_float64(ops, fmt, dh, dhp, T):
    """T > 256 without a mask: the long kernel at half-empty last blocks, 256-row item boundaries and config 5's
    T = 16 384 (sampled rows); then the same operands through the flash kernel (all-zero mask)."""
    H = 1 if T > 4096 else 2
    run_dense(ops, fmt, dh, dhp, T, H=H, use_row_out=T % 2 == 1)
    run_dense(ops, fmt, dh, dhp, T, H=H, mask="zero")


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
@pytest.mark.parametrize("dh,dhp", WIDE_PAIRS)
@pytest.mark.parametrize("T", FLASH_T)
@pytest.mark.parametrize("mask", list(MASKS))
def test_flash_kernel_masks_match_float64(ops, fmt, dh, dhp, T, mask):
    """Masked attention on the flash kernel: all-zero, causal -1e4 and causal -inf masks, key padding with a fully padded
    128-key prefix, a fully padded batch element (NaN rows, as float64 and nn.MultiheadAttention give) and random
    padding."""
    run_dense(ops, fmt, dh, dhp, T, mask=mask, use_row_out=T == 129)


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
@pytest.mark.parametrize("kernel,T,dh,dhp", [("short", 200, 64, 64), ("short", 100, 96, 96), ("long", 300, 96, 128),
                                             ("long", 700, 32, 64), ("flash", 150, 64, 64)])
def test_many_items_per_persistent_cta(ops, fmt, kernel, T, dh, dhp):
    """B*H (short) or B*H*ceil(T/256) (long) work items above 2 x 148, so that every persistent CTA runs several: ring
    and barrier parity across items, and K / V rows an earlier item leaves in shared memory."""
    B, H = (20, 8) if kernel == "long" else (40, 8)
    run_dense(ops, fmt, dh, dhp, T, B=B, H=H, mask="zero" if kernel == "flash" else "none", use_row_out=True)


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
@pytest.mark.parametrize("dh,dhp", SHORT_PAIRS)
@pytest.mark.parametrize("use_row_out", [False, True])
def test_ragged_items_match_float64(ops, fmt, dh, dhp, use_row_out):
    """The pad de-duplication's ragged items on the short kernel (40 items x 8 heads), the last row of an item counting
    `mult` times as a key, against dense float64 attention in which that row is repeated `mult` times."""
    run_ragged(ops, fmt, dh, dhp, use_row_out=use_row_out)


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_bound_rejects_wrong_references(ops, fmt):
    """Non-vacuity: the kernels' own outputs, within the bound of the right reference, exceed it several times over
    against a reference with one key dropped (each kernel), with multiplicity m - 1 (ragged items) and with the mask
    shifted by one key (flash).  The quarter-of-bf16 check on fp16 outputs runs inside every case."""
    for T, cases in ((129, {"short": {}, "flash": dict(mask="causal_1e4", mask_shift=True)}), (385, {"long": {}})):
        q32, k32, _ = dense_operands(9, 2, T, 64)
        j0 = int((q32[1, 0, 0] @ k32[1, 0].T).argmax())       # batch element 1 is "peaked": row 0's heaviest key
        for name, kw in cases.items():
            _, wrong = run_dense(ops, fmt, 64, 64, T, drop_key=j0, **kw)
            print(f"wrong references ({name} {fmt}):", {k: f"{v:.3g}" for k, v in wrong.items()})
            assert len(wrong) == 1 + ("mask_shift" in kw) and min(wrong.values()) > 4, (name, wrong)
    _, wrong = run_ragged(ops, fmt, 64, 64, wrong_mult=True)
    print(f"wrong references (ragged {fmt}):", {k: f"{v:.3g}" for k, v in wrong.items()})
    assert wrong["multiplicity m - 1"] > 4, wrong


def _launch(ops, fmt, kernel, dh, dhp, T, items=False):
    H = 2
    if items:
        it = torch.tensor([[0, 129, 128, 3], [136, 40, 40, 0]], dtype=torch.int32, device=DEV)
        q = torch.zeros(1, H, 176, dhp, dtype=FMT[fmt], device=DEV)
        return ops.attention_core(q, q.clone(), torch.zeros(1, H, dh, 176, dtype=FMT[fmt], device=DEV), items=it)
    q = torch.randn(1, H, T, dhp, device=DEV).to(FMT[fmt])
    vt = torch.randn(1, H, dh, tpad_of(T), device=DEV).to(FMT[fmt])
    am = torch.zeros(T, T, device=DEV) if kernel == "flash" else None
    return ops.attention_core(q, q.clone(), vt, attn_mask=am)


def test_dispatch_launches_the_kernel_each_case_names(ops):
    """torch.profiler: every case label above runs the kernel it names (T <= 256 or items: short, T > 256: long, any
    mask: flash) for each head-dim pair that kernel instantiates; other pairs fail before any launch."""
    from torch.profiler import ProfilerActivity, profile
    from iefvad_b200 import _lib
    plan = []
    for fmt in ("fp16", "bf16"):
        for dh, dhp in SHORT_PAIRS:
            plan += [(fmt, "short", dh, dhp, T, items) for T, items in ((1, False), (256, False), (0, True))]
        for dh, dhp in WIDE_PAIRS:
            plan += [(fmt, "long", dh, dhp, T, False) for T in (257, 1000)]
            plan += [(fmt, "flash", dh, dhp, T, False) for T in FLASH_T]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case in plan:
            _launch(ops, *case)
            torch.cuda.synchronize()
    events = sorted((e for e in prof.events() if "attn_" in e.name and "_kernel<" in e.name), key=lambda e: e.time_range.start)
    names = [e.name for e in events]
    assert len(names) == len(plan), (len(names), len(plan), names[:4])
    for case, name in zip(plan, names):
        _, kernel, dh, dhp, _, _ = case
        assert f"{KERNEL[kernel]}<{dh}, {dhp}>" in name, (case, name)
    n0 = _lib.lib.iefvad_launch_count()
    for kernel, dh, dhp, T in [("long", 96, 96, 300), ("long", 32, 32, 300), ("flash", 96, 96, 100),
                               ("flash", 32, 32, 100), ("short", 64, 128, 100), ("short", 48, 64, 100)]:
        with pytest.raises(_lib.IefvadError, match="unsupported head dim"):
            _launch(ops, "fp16", kernel, dh, dhp, T)
    assert _lib.lib.iefvad_launch_count() == n0
