"""Parity of the stand-alone CUDA operators (through the C ABI) against the CPU oracle.  Needs a B200."""
import numpy as np
import pytest
import torch

from oracle import iefvad_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from iefvad_b200 import ops as _ops
    return _ops


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# tolerance classes (max|x-ref| / max|ref|): fp32 kernels 1e-5; split-bf16 GEMM ~2^-16; plain bf16 GEMM ~2^-8
TOL = {"fp32": 1e-5, "split": 3e-5, "bf16": 1e-2, "fp16": 1.5e-3}    # fp16: 11-bit mantissa operands, 8x finer than bf16


@pytest.mark.parametrize("noise,nu", [("StudentT", 8), ("StudentT", 5), ("Gaussian", 8)])
def test_fuse_matches_oracle(ops, noise, nu):
    rng = np.random.default_rng(0)
    shape = (3, 37, 768)
    mi, me = rng.standard_normal(shape).astype(np.float32), rng.standard_normal(shape).astype(np.float32)
    li, le = (2 * rng.standard_normal(shape)).astype(np.float32), (2 * rng.standard_normal(shape)).astype(np.float32)
    li[0, 0, :8] = [-80, 80, 0, -0.0, 30, -30, 1e-8, 88]      # extremes: w -> 0 / inf-ish, epsilon matters
    wi, we, f = ops.fuse(_cuda(mi), _cuda(me), _cuda(li), _cuda(le), noise, nu)
    rwi, rwe, rf = O.fuse(mi, me, li, le, noise_model=noise, nu=nu)
    for got, ref in ((wi, rwi), (we, rwe), (f, rf)):
        got = got.cpu().numpy()
        finite = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), finite)
        # fused = w_i*mu_i + w_e*mu_e cancels, so its error is absolute (a few ulp of the O(1) products)
        np.testing.assert_allclose(got[finite], ref[finite], rtol=1e-5, atol=1e-6)


def test_fuse_rejects_unknown_noise_model_and_cpu_tensors(ops):
    x = torch.zeros(4, 768)
    with pytest.raises(ValueError, match="Unsupported noise_model"):
        ops.fuse(x.cuda(), x.cuda(), x.cuda(), x.cuda(), "Laplace")
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.fuse(x, x, x, x)


@pytest.mark.parametrize("D", [128, 512, 768, 1024])
def test_layernorm_single_and_double(ops, D):
    rng = np.random.default_rng(D)
    x = (3 * rng.standard_normal((5, 33, D)) + 1.5).astype(np.float32)
    w1, b1, w2, b2 = (rng.standard_normal(D).astype(np.float32) for _ in range(4))
    got = ops.layernorm(_cuda(x), _cuda(w1), _cuda(b1)).cpu().numpy()
    ref = O.layer_norm(x, w1, b1)
    assert O.max_norm_err(got, ref) < 1e-5
    got = ops.layernorm(_cuda(x), _cuda(w1), _cuda(b1), _cuda(w2), _cuda(b2)).cpu().numpy()
    ref = O.layer_norm(O.layer_norm(x, w1, b1), w2, b2)
    assert O.max_norm_err(got, ref) < 1e-5


@pytest.mark.parametrize("plan", ["fp32", "split", "bf16", "fp16"])
@pytest.mark.parametrize("rows,in_f,out_f,tile_n", [
    (256, 768, 768, 0), (1000, 768, 2304, 0), (130, 768, 1536, 64), (4096, 768, 768, 128),
    (4096, 768, 768, 256), (1, 768, 768, 0), (257, 128, 96, 0), (300, 3072, 768, 0), (20000, 768, 768, 0),
    (4096, 768, 768, 512), (1000, 768, 2304, 512), (130, 768, 1536, 512), (20000, 768, 768, 512), (257, 128, 256, 512)])
def test_linear_plain(ops, plan, rows, in_f, out_f, tile_n):
    if plan == "fp32" and tile_n:
        pytest.skip("tile_n only applies to the tcgen05 plans")
    rng = np.random.default_rng(rows + in_f)
    x = rng.standard_normal((rows, in_f)).astype(np.float32)
    w = (rng.standard_normal((out_f, in_f)) / np.sqrt(in_f)).astype(np.float32)
    b = rng.standard_normal(out_f).astype(np.float32)
    got = ops.linear(_cuda(x), _cuda(w), _cuda(b), plan=plan, tile_n=tile_n).cpu().numpy()
    ref = O.linear(x.astype(np.float64), w.astype(np.float64), b.astype(np.float64))
    assert got.shape == ref.shape
    assert O.max_norm_err(got, ref) < TOL[plan]


@pytest.mark.parametrize("plan", ["fp32", "split", "bf16", "fp16"])
@pytest.mark.parametrize("act", ["relu", "quickgelu", None])
@pytest.mark.parametrize("rows,tile_n", [(333, 0), (333, 512), (5000, 512), (5000, 256)])
def test_linear_epilogue_residual_alpha_act(ops, plan, act, rows, tile_n):
    if plan == "fp32" and tile_n:
        pytest.skip("tile_n only applies to the tcgen05 plans")
    rng = np.random.default_rng(5)
    D = 768
    x = rng.standard_normal((rows, D)).astype(np.float32)
    w = (rng.standard_normal((D, D)) / np.sqrt(D)).astype(np.float32)
    b = rng.standard_normal(D).astype(np.float32)
    r = rng.standard_normal((rows, D)).astype(np.float32)
    got = ops.linear(_cuda(x), _cuda(w), _cuda(b), resid=_cuda(r), alpha=-0.5, act=act, plan=plan,
                     tile_n=tile_n).cpu().numpy()
    y = O.linear(x.astype(np.float64), w.astype(np.float64), b.astype(np.float64))
    if act == "relu":
        y = np.maximum(y, 0)
    elif act == "quickgelu":
        y = O.quick_gelu(y)
    ref = r - 0.5 * y
    assert O.max_norm_err(got, ref) < TOL[plan]


def test_linear_split_is_much_tighter_than_bf16(ops):
    rng = np.random.default_rng(6)
    x = rng.standard_normal((512, 768)).astype(np.float32)
    w = (rng.standard_normal((768, 768)) / np.sqrt(768)).astype(np.float32)
    ref = x.astype(np.float64) @ w.astype(np.float64).T
    e_bf = O.max_norm_err(ops.linear(_cuda(x), _cuda(w), plan="bf16").cpu().numpy(), ref)
    e_sp = O.max_norm_err(ops.linear(_cuda(x), _cuda(w), plan="split").cpu().numpy(), ref)
    assert e_sp < 3e-5 and e_bf > 20 * e_sp


# the whole block: two chained 16-bit GEMMs plus attention, twice the linear class (as for bf16, 2e-2 against 1e-2)
MHA_TOL = {"fp32": 2e-5, "bf16": 2e-2, "fp16": 2 * TOL["fp16"]}


@pytest.mark.parametrize("plan", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("B,T,D,H", [(1, 256, 768, 8), (3, 40, 768, 8), (2, 129, 768, 8), (1, 1000, 768, 8),
                                     (2, 24, 128, 4), (1, 300, 512, 8), (2, 17, 128, 2), (1, 1, 768, 8)])
def test_mha_matches_oracle(ops, plan, B, T, D, H):
    rng = np.random.default_rng(B * 1000 + T)
    x = rng.standard_normal((B, T, D)).astype(np.float32)
    in_w = (rng.standard_normal((3 * D, D)) / np.sqrt(D)).astype(np.float32)
    in_b = (0.1 * rng.standard_normal(3 * D)).astype(np.float32)
    out_w = (rng.standard_normal((D, D)) / np.sqrt(D)).astype(np.float32)
    out_b = (0.1 * rng.standard_normal(D)).astype(np.float32)
    got = ops.mha(_cuda(x), _cuda(in_w), _cuda(in_b), _cuda(out_w), _cuda(out_b), H, plan=plan).cpu().numpy()
    ref = O.multihead_self_attention(x.astype(np.float64), in_w.astype(np.float64), in_b.astype(np.float64),
                                     out_w.astype(np.float64), out_b.astype(np.float64), H)
    err = O.max_norm_err(got, ref)
    print(f"mha {plan} B={B} T={T} D={D} H={H}: {err:.3g}")
    assert err < MHA_TOL[plan]


@pytest.mark.parametrize("plan", ["fp32", "bf16", "fp16"])
def test_mha_masks(ops, plan):
    rng = np.random.default_rng(77)
    B, T, D, H = 3, 150, 128, 4
    x = rng.standard_normal((B, T, D)).astype(np.float32)
    in_w = (rng.standard_normal((3 * D, D)) / np.sqrt(D)).astype(np.float32)
    in_b = (0.1 * rng.standard_normal(3 * D)).astype(np.float32)
    out_w = (rng.standard_normal((D, D)) / np.sqrt(D)).astype(np.float32)
    out_b = (0.1 * rng.standard_normal(D)).astype(np.float32)
    mask = np.zeros((T, T), dtype=np.float32)
    mask[np.triu(np.ones((T, T)), 9) > 0] = -1e4
    pad = np.zeros((B, T), dtype=bool)
    pad[1, 100:] = True
    pad[2, 5:] = True
    got = ops.mha(_cuda(x), _cuda(in_w), _cuda(in_b), _cuda(out_w), _cuda(out_b), H, attn_mask=_cuda(mask),
                  key_padding_mask=_cuda(pad), plan=plan).cpu().numpy()
    ref = O.multihead_self_attention(x.astype(np.float64), in_w.astype(np.float64), in_b.astype(np.float64),
                                     out_w.astype(np.float64), out_b.astype(np.float64), H,
                                     key_padding_mask=pad, attn_mask=mask)
    err = O.max_norm_err(got, ref)
    print(f"mha masks {plan}: {err:.3g}")
    assert err < MHA_TOL[plan]


def test_classifier(ops):
    rng = np.random.default_rng(8)
    x = rng.standard_normal((5, 77, 768)).astype(np.float32)
    w = rng.standard_normal((1, 768)).astype(np.float32)
    b = rng.standard_normal(1).astype(np.float32)
    logits, scores = ops.classifier(_cuda(x), _cuda(w), _cuda(b), with_scores=True)
    ref = O.linear(x.astype(np.float64), w.astype(np.float64), b.astype(np.float64))
    assert logits.shape == (5, 77, 1)
    assert O.max_norm_err(logits.cpu().numpy(), ref) < 1e-5
    assert O.max_norm_err(scores.cpu().numpy(), O.sigmoid(ref[..., 0])) < 1e-5


@pytest.mark.parametrize("rows,out_f,in_f", [(16384, 768, 768), (4096, 768, 2304), (1000, 256, 768), (333, 64, 96)])
def test_wgrad_split_k_matches_fp64(ops, rows, out_f, in_f):
    """iefvad_wgrad: dW = alpha * dY^T X (train/ucf_train.py:105's backward through every Linear) - operands transposed straight
    into the bf16 hi / lo form, K slices as extra row tiles where the output is small, slices summed in fixed order."""
    g = torch.Generator().manual_seed(rows + in_f)
    dy = torch.randn(rows, out_f, generator=g) * torch.logspace(-6, 0, out_f)     # gradients span many decades
    x = torch.randn(rows, in_f, generator=g)
    got = ops.wgrad(dy.cuda(), x.cuda(), alpha=-0.5)
    again = ops.wgrad(dy.cuda(), x.cuda(), alpha=-0.5)
    ref = -0.5 * dy.double().T @ x.double()
    assert torch.equal(got, again)                                               # no atomics: run-to-run identical
    err = (got.double().cpu() - ref).abs().max(dim=1).values / ref.abs().max(dim=1).values
    assert err.max().item() < 5e-5, err.max().item()                            # 3-term bf16 split, per output row (decade)


def test_linear_long_k_takes_the_split_k_path_and_matches(ops):
    g = torch.Generator().manual_seed(9)
    a = torch.randn(768, 16384, generator=g)
    b = torch.randn(768, 16384, generator=g)
    got = ops.linear(a.cuda(), b.cuda(), plan="split").double().cpu()
    ref = a.double() @ b.double().T
    assert (got - ref).abs().max().item() / ref.abs().max().item() < TOL["split"]
