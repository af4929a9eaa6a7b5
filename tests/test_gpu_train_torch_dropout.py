"""The "torch" dropout mode of the training attention (model.temporal.dropout_rng = "torch"): PyTorch's own CUDA dropout
mask, regenerated inside the kernels, and the generator stream of the reference's train() loop.

- iefvad_dropout_mask equals torch.native_dropout's mask bit for bit, and the generator offset after each call is torch's;
  an offset one step off, a launch width G +- 256 or swapped counter halves each give a different mask.
- The training attention in torch mode against float64 autograd with torch's own mask.
- The drop-in in train() mode against a stock-torch composition (real nn.MultiheadAttention modules, need_weights at its
  default, oracle/torch_port.py for the rest) under the same torch.cuda.manual_seed: outputs, loss, every gradient, the
  CUDA generator's offset afterwards, an untouched CPU generator, and two AdamW steps.
- The default "philox" mode is unchanged: its outputs and gradients hash to what the previous release produced.
Worst errors measured on an NVIDIA B200 (1000 W power limit) are quoted at each bound.  Needs a B200."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import torch_port
from oracle.torch_dropout import torch_dropout_keep
from test_gpu_train import reference_loss
from test_gpu_train_fp64 import attention_errors, attention_inputs, attention_ref, clas2_64, rel_err, small_batch, small_model

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    assert torch.cuda.is_available()
    import iefvad_b200
    from iefvad_b200 import ops, synth
    return iefvad_b200, ops, synth


def generator():
    torch.cuda.init()                     # default_generators is empty until CUDA is initialised
    return torch.cuda.default_generators[torch.cuda.current_device()]


def set_state(state):
    """Put the CUDA generator in one of three states -> (seed, offset)."""
    if state == "fresh":
        torch.cuda.manual_seed(1234)
    elif state == "seed_above_2^32":
        torch.cuda.manual_seed((1 << 40) + 77)
    else:                                                   # "advanced": unrelated draws moved the offset
        torch.cuda.manual_seed(5)
        torch.rand(1000, device="cuda")
        torch.rand(3, 7, device="cuda")
    g = generator()
    return g.initial_seed(), g.get_offset()


# ------------------------------------------------------------------------------------------------ the mask itself
MASK_CASES = [(B, H, T, p, s) for (B, H, T) in ((1, 8, 256), (2, 4, 48), (3, 8, 257), (128, 8, 256)) for p in (0.1, 0.5)
              for s in ("fresh", "seed_above_2^32", "advanced")]


@pytest.mark.parametrize("B, H, T, p, state", MASK_CASES, ids=[f"B{c[0]}-H{c[1]}-T{c[2]}-p{c[3]}-{c[4]}" for c in MASK_CASES])
def test_mask_equals_torch_native_dropout(pkg, B, H, T, p, state):
    _, ops, _ = pkg
    seed, off = set_state(state)
    G, advance = ops.torch_dropout_launch(B * H * T * T)
    mine = ops.dropout_mask(B, H, T, p, seed, "torch", off, G)
    assert generator().get_offset() == off                  # the library reads the state, it does not draw
    out, ref = torch.native_dropout(torch.ones(B * H, T, T, device="cuda"), p, True)
    assert generator().get_offset() == off + advance
    assert torch.equal(mine.bool(), ref)
    scale = float(np.float32(1.0 / np.float64(np.float32(1.0 - p))))
    assert float(out.max()) == scale                        # the scale the kernels apply to kept weights


def test_wrong_mappings_give_a_different_mask(pkg):
    _, ops, _ = pkg
    B, H, T, p = 128, 8, 256, 0.1                            # n / 4 > G: every thread runs several iterations
    seed, off = set_state("advanced")
    G, _ = ops.torch_dropout_launch(B * H * T * T)
    _, ref = torch.native_dropout(torch.ones(B * H, T, T, device="cuda"), p, True)
    assert torch.equal(ops.dropout_mask(B, H, T, p, seed, "torch", off, G).bool(), ref)
    for name, (o, g) in {"offset + 4": (off + 4, G), "offset - 4": (off - 4, G), "G + 256": (off, G + 256),
                         "G - 256": (off, G - 256)}.items():
        bad = ops.dropout_mask(B, H, T, p, seed, "torch", o, g).bool()
        frac = float((bad != ref).float().mean())
        print(f"{name}: {frac:.3f} of the mask differs")
        assert frac > 0.05, name
    B, H, T = 2, 4, 48
    seed, off = set_state("fresh")
    G, _ = ops.torch_dropout_launch(B * H * T * T)
    _, ref = torch.native_dropout(torch.ones(B * H, T, T, device="cuda"), p, True)
    ref = ref.cpu().numpy().reshape(B, H, T, T)
    assert np.array_equal(torch_dropout_keep(seed, off, B, H, T, p, G) > 0, ref)
    assert not np.array_equal(torch_dropout_keep(seed, off, B, H, T, p, G, swap_halves=True) > 0, ref)


# ------------------------------------------------------------------------------------------------ kernels vs float64
ATTN_CASES = [(dh, B, H, T) for dh in (32, 64, 96) for (B, H, T) in ((2, 2, 33), (2, 2, 129), (3, 4, 64))]


def torch_keep(B, H, T, p):
    """Generator state before the draw and torch's own multiplier [B, H, T, T] (float64)."""
    g = generator()
    seed, off = g.initial_seed(), g.get_offset()
    out, _ = torch.native_dropout(torch.ones(B * H, T, T, device="cuda"), p, True)
    return seed, off, out.double().cpu().reshape(B, H, T, T)


@pytest.mark.parametrize("dh, B, H, T", ATTN_CASES, ids=[f"dh{c[0]}-B{c[1]}-H{c[2]}-T{c[3]}" for c in ATTN_CASES])
def test_train_attention_matches_float64_with_torchs_mask(pkg, dh, B, H, T):
    """Bound 2e-5 as for the Philox mask (tests/test_gpu_train_fp64.py); odd T puts the two keys of one pair in
    different Philox groups."""
    _, ops, _ = pkg
    p = 0.1
    qkv, dout = attention_inputs(B, T, H, dh, 7 * dh + T)
    torch.cuda.manual_seed(dh + T)
    seed, off, keep = torch_keep(B, H, T, p)
    G, _ = ops.torch_dropout_launch(B * H * T * T)
    kw = dict(rng="torch", offset=off, threads=G)
    D = H * dh
    qkv_d, dout_d = qkv.cuda(), dout.cuda()
    out, lse = ops.attention_train_fwd(qkv_d, B, T, H, p, seed, **kw)
    dqkv = ops.attention_train_bwd(qkv_d, out, dout_d, lse, B, T, H, p, seed, **kw).cpu()
    got = (out.cpu(), lse.cpu(), dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:])
    errs = attention_errors(got, attention_ref(qkv, dout, B, T, H, keep), T)
    print(f"torch-mask attention dh {dh} B {B} H {H} T {T}:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) <= 2e-5, errs
    wrong = attention_errors(got, attention_ref(qkv, dout, B, T, H, keep.transpose(2, 3)), T)
    assert wrong["out"] > 1e-2, wrong                      # non-vacuity: a transposed mask is far outside the bound


# ------------------------------------------------------------------------------------------------ model vs stock torch
class StockComposition:
    """The reference's train() forward in stock torch: real nn.MultiheadAttention(batch_first=True) modules called with
    need_weights at its default (their dropout draws torch.native_dropout on the CUDA generator), oracle/torch_port.py
    for the rest, fp32.  Parameters are copies of the drop-in's, leaves of their own."""

    def __init__(self, m):
        t = m.temporal
        self.t = t
        self.P = {k: p.detach().clone().requires_grad_(True) for k, p in m.named_parameters()}
        self.by_weight = {}
        for mod in ("image", "event"):
            for i in range(t.num_layers):
                pre = f"temporal.{mod}_attn_layers.{i}."
                a = torch.nn.MultiheadAttention(t.embed_dim, t.num_heads, dropout=t.dropout, batch_first=True).cuda().train()
                a.in_proj_weight, a.in_proj_bias = self._param(pre + "in_proj_weight"), self._param(pre + "in_proj_bias")
                a.out_proj.weight, a.out_proj.bias = self._param(pre + "out_proj.weight"), self._param(pre + "out_proj.bias")
                self.by_weight[id(a.in_proj_weight)] = a
        self.outs = {}

    def _param(self, k):
        self.P[k] = torch.nn.Parameter(self.P[k].detach())
        return self.P[k]

    def __call__(self, img, ev, *_):
        def stock_mha(x, in_w, in_b, out_w, out_b, heads, keep=None):
            return self.by_weight[id(in_w)](x, x, x)[0]
        saved, torch_port.mha = torch_port.mha, stock_mha
        try:
            t = self.t
            self.outs = torch_port.forward(self.P, img, ev, heads=t.num_heads, lambda_ref=float(t.lambda_ref),
                                           noise_model=t.noise_model, nu=float(t.nu), epsilon=float(t.epsilon))
        finally:
            torch_port.mha = saved
        return self.outs


def step(model, CLAS2, img, ev, lengths, labels, nu, cuda_seed, params):
    """One loss.backward() under torch.cuda.manual_seed(cuda_seed) -> (loss, outputs, {name: grad}, offset after)."""
    for p in params.values():
        p.grad = None
    torch.cuda.manual_seed(cuda_seed)
    outs = {}

    def fn(i, e, *_):
        outs.update(model(i, e, None, None, None))
        return outs
    loss, _ = reference_loss(fn, CLAS2, img, ev, lengths, labels, nu)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in params.items()}
    return loss.detach(), {k: v.detach() for k, v in outs.items()}, grads, generator().get_offset()


def compare(got, ref, full_size):
    (l1, o1, g1, off1), (l2, o2, g2, off2) = got, ref
    assert off1 == off2, (off1, off2)                        # the same number of CUDA draws: later draws agree too
    assert abs(float(l1) - float(l2)) <= 2e-4 * abs(float(l2)), (float(l1), float(l2))
    oerr = {k: rel_err(o1[k], o2[k]) for k in o2}
    print("outputs:", {k: f"{v:.1e}" for k, v in oerr.items()})
    assert len(oerr) == 8 and max(oerr.values()) < 1e-3, oerr
    worst = 0.0
    for k, r in g2.items():
        g = g1[k].double().cpu().reshape(-1)
        r = r.double().cpu().reshape(-1)
        err = (g - r).abs() / max(float(r.abs().max()), 1e-20)
        if full_size:
            # as tests/test_gpu_train.py at full size: a ReLU pre-activation within rounding of zero may flip its gate
            assert float(torch.quantile(err.float(), 0.9)) < 1e-3 and float(err.max()) < 5e-2, (k, float(err.max()))
        else:
            assert float(err.max()) < 1e-3, (k, float(err.max()))
        worst = max(worst, float(err.max()))
    print(f"loss {float(l1):.6f} / {float(l2):.6f}, {len(g2)} gradients, worst {worst:.2e}")
    return len(g2)


def _torch_mode(m):
    m.train()
    m.temporal.dropout_rng = "torch"
    return m


def test_small_model_matches_stock_torch_in_train_mode(pkg):
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = _torch_mode(small_model(iefvad_b200, synth, 4, 2, 3, "StudentT", True))
    stock = StockComposition(m)
    img, ev, lengths, labels = small_batch()
    params = {**dict(m.named_parameters()), "img": img, "ev": ev}
    cpu_state = torch.get_rng_state()
    got = step(m, CLAS2, img, ev, lengths, labels, float(m.temporal.nu), 99, params)
    assert torch.equal(torch.get_rng_state(), cpu_state)     # torch mode leaves the CPU generator alone
    x = {n: t.detach().clone().requires_grad_(True) for n, t in (("img", img), ("ev", ev))}
    ref = step(stock, clas2_64, x["img"], x["ev"], lengths, labels, float(m.temporal.nu), 99, {**stock.P, **x})
    assert compare(got, ref, False) == len(stock.P) + 2
    # dropout really acts: another CUDA seed gives another loss
    other = step(m, CLAS2, img, ev, lengths, labels, float(m.temporal.nu), 100, params)
    assert float(other[0]) != float(got[0])


def test_full_size_matches_stock_torch_in_train_mode(pkg):
    """The 768-d model on 8 config-4 clips (T = 256, 8 heads): all 78 gradients."""
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = _torch_mode(synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda())
    stock = StockComposition(m)
    img, ev, lengths, labels = (t.cuda() for t in synth.make_c4_batch(8))
    got = step(m, CLAS2, img, ev, lengths, labels, float(m.temporal.nu), 7, dict(m.named_parameters()))
    ref = step(stock, clas2_64, img, ev, lengths, labels, float(m.temporal.nu), 7, stock.P)
    assert compare(got, ref, True) == 78


def test_two_adamw_steps_track_stock_torch(pkg):
    """train/ucf_train.py's loop body twice: the second step's masks come from the advanced generator."""
    iefvad_b200, _, synth = pkg
    from iefvad_b200.loss import CLAS2
    m = _torch_mode(small_model(iefvad_b200, synth, 4, 2, 3, "StudentT", True))
    stock = StockComposition(m)
    img, ev, lengths, labels = (t.detach() for t in small_batch())
    nu = float(m.temporal.nu)
    runs = []
    for model, loss_fn, params in ((m, CLAS2, dict(m.named_parameters())), (stock, clas2_64, stock.P)):
        opt = torch.optim.AdamW(list(params.values()), lr=2e-5)
        torch.cuda.manual_seed(2024)
        res = []
        for _ in range(2):
            outs = {}

            def fn(i, e, *_):
                outs.update(model(i, e, None, None, None))
                return outs
            opt.zero_grad()
            loss, _ = reference_loss(fn, loss_fn, img, ev, lengths, labels, nu)
            loss.backward()
            res.append((float(loss.detach()), {k: p.grad.detach().clone() for k, p in params.items()}))
            opt.step()
        runs.append((res, generator().get_offset()))
    (got, off_got), (ref, off_ref) = runs
    assert off_got == off_ref
    for (lg, gg), (lr_, gr) in zip(got, ref):
        assert abs(lg - lr_) <= 2e-4 * abs(lr_), (lg, lr_)
        for k in gr:
            assert rel_err(gg[k], gr[k]) < 1e-3, k
    assert got[0][0] != got[1][0]


# ------------------------------------------------------------------------------------------------ philox mode unchanged
# sha256 of the philox-mode results of the previous release (NVIDIA B200, 148 SMs); see philox_digests
PARENT_DIGESTS = {
    "attn_out": "a830bec436026a5fe45fe1723de564ad47bedcf6cd3187a7c3333203be630301",
    "attn_lse": "1f5ffe6fdd7148bb501763c1a406182b77a3eef4e2d7737f6befbf3c8713c618",
    "attn_dqkv": "bab2b77360bac2ec9aa85f250d2e1624998ac4a553377862c9bcc08ebfbe4002",
    "step_outputs": "9c55ec642f883ef84a792e95d09f82456d4d5fbbd7ee91ea5feffbdf5e518aa8",
    "step_grads": "f7f1bb0c2c7e609d6987ba759c5d3197958972b8e5f3d0171cabf5a28ca3d2f9",
}


def philox_digests(iefvad_b200, ops, synth):
    """sha256 of the bytes of the default (philox) mode's results: the attention operators at p = 0.1 and one train()
    step of the 128-d model (loss, 8 outputs, every parameter gradient, both input gradients)."""
    from iefvad_b200.loss import CLAS2
    res = {}
    B, T, H, dh = 2, 129, 2, 64
    qkv, dout = attention_inputs(B, T, H, dh, 5)
    qkv, dout = qkv.cuda(), dout.cuda()
    out, lse = ops.attention_train_fwd(qkv, B, T, H, 0.1, 0x7DEADBEEF)
    dqkv = ops.attention_train_bwd(qkv, out, dout, lse, B, T, H, 0.1, 0x7DEADBEEF)
    for n, t in (("attn_out", out), ("attn_lse", lse), ("attn_dqkv", dqkv)):
        res[n] = hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest()
    m = small_model(iefvad_b200, synth, 4, 2, 3, "StudentT", True)
    img, ev, lengths, labels = small_batch()
    params = {**dict(m.named_parameters()), "img": img, "ev": ev}
    torch.manual_seed(17)
    loss, outs, grads, _ = step(m, CLAS2, img, ev, lengths, labels, float(m.temporal.nu), 0, params)
    h = hashlib.sha256(loss.cpu().numpy().tobytes())
    for k in sorted(outs):
        h.update(outs[k].cpu().numpy().tobytes())
    res["step_outputs"] = h.hexdigest()
    h = hashlib.sha256()
    for k in sorted(grads):
        h.update(grads[k].cpu().numpy().tobytes())
    res["step_grads"] = h.hexdigest()
    return res


def test_philox_mode_is_unchanged(pkg):
    got = philox_digests(*pkg)
    print(got)
    assert got == PARENT_DIGESTS
