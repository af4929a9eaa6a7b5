"""Row N3 - the training objective in CUDA (csrc/train_loss.cu, iefvad_b200.loss.train_loss): CLAS2 + the cosine / norm
regulariser + the StudentT KL term of train/ucf_train.py:73-102 and their backward.

- The objective alone against float64 torch autograd of the loop's own ops on the same fp32 inputs, at the reference
  loop's full batch too, with torch's edge rows (zero row, equal norms, cos = +-1, large log-variances), each returned
  scalar's gradient on its own and the loss weights of both loops.
- Run-to-run identical bits, no host sync, a fixed number of library launches.
- The whole training step with `train_loss` in place of the caller's torch ops: against the reference goldens, against
  float64 oracle/torch_port.py with the exact dropout mask, and against the torch-composed objective.  Needs a B200."""
import numpy as np
import pytest
import torch

from conftest import load_golden, params_from_npz
from oracle import torch_port
from test_gpu_train import reference_loss
from test_gpu_train_fp64 import (O, assert_all_close, clas2_64, rel_err, small_batch, small_model)
from test_oracle_train_objective import GRADS, NAMES, objective_inputs, torch_objective, torch_reference

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    assert torch.cuda.is_available()
    import iefvad_b200
    from iefvad_b200 import _lib, synth
    from iefvad_b200.loss import train_loss
    return iefvad_b200, _lib, synth, train_loss


def native(train_loss, inputs, labels, lengths, nu, reg_weight=1.0, kl_weight=1.0, upstream=(1.0, 0.0, 0.0, 0.0)):
    """train_loss on CUDA copies of the fp32 inputs -> dict of the four scalars and the five input gradients."""
    xs = [torch.as_tensor(t).cuda().requires_grad_(True) for t in inputs]
    outs = dict(zip(("logits", "image_mu", "event_mu", "image_logvar", "event_logvar"), xs))
    res = train_loss(outs, torch.as_tensor(labels).cuda(), torch.as_tensor(lengths).cuda(), nu, reg_weight, kl_weight)
    picked = [o for g, o in zip(upstream, res) if g != 0]
    grads = torch.autograd.grad(picked, xs, [torch.full((), g, device="cuda") for g in upstream if g != 0])
    got = dict(zip(NAMES, (t.detach() for t in res)))
    got.update(zip(GRADS, grads))
    return got


def assert_objective_close(got, ref, what):
    for n in NAMES:
        g, r = float(got[n]), float(ref[n])
        assert abs(g - r) <= 1e-6 + 1e-5 * abs(r), (what, n, g, r)
    errs = {n: rel_err(got[n], ref[n]) for n in GRADS}
    assert max(errs.values()) <= 1e-5, (what, errs)
    return errs


SHAPES = [(3, 47, 128, True), (8, 256, 768, True), (128, 256, 768, False)]


@pytest.mark.parametrize("B, T, D, edge", SHAPES, ids=[f"{b}x{t}x{d}" for b, t, d, _ in SHAPES])
def test_objective_matches_float64_autograd(pkg, B, T, D, edge):
    _, _, _, train_loss = pkg
    inputs, labels, lengths = objective_inputs(B, T, D, seed=B + T + D, edge=edge)
    assert {1, 9, T} <= set(lengths.tolist())
    got = native(train_loss, inputs, labels, lengths, 5.0)
    ref = torch_reference(inputs, labels, lengths, 5.0, device="cuda")
    errs = assert_objective_close(got, ref, f"{B}x{T}x{D}")
    print(f"{B}x{T}x{D}: worst gradient error {max(errs.values()):.2e}")
    if edge:                                             # the zero row keeps torch's ~1e20 / (B T) normalize-clamp gradient
        z = float(got["d_mu_i"][0, 0].abs().max())
        assert z > 1e15 and abs(z - float(ref["d_mu_i"][0, 0].abs().max())) <= 1e-5 * z


def test_exp_overflow_gives_inf_like_torch_fp32(pkg):
    _, _, _, train_loss = pkg
    inputs, labels, lengths = objective_inputs(3, 47, 128, seed=1)
    inputs[3][1, 5, 7] = 100.0
    got = native(train_loss, inputs, labels, lengths, 5.0)
    ref32 = torch_reference(inputs, labels, lengths, 5.0, dtype=torch.float32, device="cuda")
    for n in ("total", "kl"):
        assert float(ref32[n]) == float("inf") and float(got[n]) == float("inf"), n
    assert float(got["regulariser"]) == pytest.approx(float(ref32["regulariser"]), rel=1e-5)


@pytest.mark.parametrize("weights", [(1.0, 1.0), (0.01, 0.01), (0.0, 1.0)])
@pytest.mark.parametrize("which", range(4), ids=NAMES)
def test_backward_from_each_scalar(pkg, weights, which):
    _, _, _, train_loss = pkg
    upstream = tuple(1.0 if i == which else 0.0 for i in range(4))
    inputs, labels, lengths = objective_inputs(3, 47, 128, seed=9, edge=True)
    got = native(train_loss, inputs, labels, lengths, 8.0, *weights, upstream=upstream)
    ref = torch_reference(inputs, labels, lengths, 8.0, *weights, upstream=upstream, device="cuda")
    assert_objective_close(got, ref, f"d {NAMES[which]}, weights {weights}")


def test_identical_bits_no_host_sync_and_fixed_launch_count(pkg):
    _, _lib, _, train_loss = pkg
    inputs, labels, lengths = objective_inputs(8, 256, 768, seed=4, edge=True)
    xs = [torch.as_tensor(t).cuda().requires_grad_(True) for t in inputs]
    outs = dict(zip(("logits", "image_mu", "event_mu", "image_logvar", "event_logvar"), xs))
    labels, lengths = torch.as_tensor(labels).cuda(), torch.as_tensor(lengths).cuda()
    runs = []
    for _ in range(2):
        for x in xs:
            x.grad = None
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            n0 = _lib.lib.iefvad_launch_count()
            res = train_loss(outs, labels, lengths, 8.0)
            n1 = _lib.lib.iefvad_launch_count()
            (res.total + res.regulariser).backward()
            n2 = _lib.lib.iefvad_launch_count()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert (n1 - n0, n2 - n1) == (4, 2)
        runs.append([t.detach().clone() for t in res] + [x.grad.clone() for x in xs])
    for a, b in zip(*runs):
        assert torch.equal(a, b)
    with torch.no_grad():                                # forward kernels only, no autograd node
        n0 = _lib.lib.iefvad_launch_count()
        res = train_loss(outs, labels, lengths, 8.0)
        assert _lib.lib.iefvad_launch_count() - n0 == 4 and res.total.grad_fn is None
    assert torch.equal(res.total, runs[0][0])


def test_rejects_bad_inputs(pkg):
    _, _, _, train_loss = pkg
    o = {k: torch.zeros(2, 16, 128, device="cuda") for k in ("image_mu", "event_mu", "image_logvar", "event_logvar")}
    o["logits"] = torch.zeros(2, 16, 1, device="cuda")
    labels, lengths = torch.zeros(2, 14, device="cuda"), torch.tensor([16, 3], device="cuda")
    for key, bad in (("image_mu", o["image_mu"].cpu()), ("event_logvar", torch.zeros(2, 16, 64, device="cuda")),
                     ("logits", torch.zeros(2, 16, device="cuda")), ("logits", torch.zeros(2, 15, 1, device="cuda"))):
        with pytest.raises(RuntimeError):
            train_loss({**o, key: bad}, labels, lengths, 8.0)
    with pytest.raises(RuntimeError):
        train_loss(o, labels, lengths.cpu(), 8.0)


# ------------------------------------------------------------------------------------------------ the whole training step
def native_loss(train_loss):
    """reference_loss's signature with train_loss in place of the caller's torch ops."""
    def loss_fn(model, _clas2, img, ev, lengths, labels, nu):
        res = train_loss(model(img, ev, None, None, lengths), labels, lengths, nu)
        return res.total, res.classification
    return loss_fn


def test_small_model_gradients_match_the_reference_goldens(pkg):
    iefvad_b200, _, synth, train_loss = pkg
    z = load_golden("train_small.npz")
    args = synth.default_args(noise_model="StudentT", nu=8, num_refinement_steps=3, visual_head=4)
    m = iefvad_b200.MMFMIL(14, 128, 256, 128, 8, 2, 8, 10, 10, "cuda", args)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params_from_npz(z).items()})
    m = m.cuda().eval()
    img, ev = torch.from_numpy(z["img"]).cuda(), torch.from_numpy(z["ev"]).cuda()
    lengths, labels = torch.from_numpy(z["lengths"]).cuda(), torch.from_numpy(z["labels"]).cuda()
    loss, lcls = native_loss(train_loss)(m, None, img, ev, lengths, labels, 8)
    assert abs(float(loss) - float(z["loss"])) < 2e-4 * abs(float(z["loss"]))
    assert abs(float(lcls) - float(z["loss_cls"])) < 2e-4
    loss.backward()
    for k, p in m.named_parameters():
        ref = z["grad:" + k]
        err = float(np.max(np.abs(p.grad.cpu().numpy() - ref)) / max(np.max(np.abs(ref)), 1e-12))
        assert err < 1e-3, (k, err)


def test_full_size_gradients_match_the_reference_goldens(pkg):
    iefvad_b200, _, synth, train_loss = pkg
    z = load_golden("train_full.npz")
    m = synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda().eval()
    img, ev, lengths, labels = synth.make_c4_batch(8)
    loss, _ = native_loss(train_loss)(m, None, img.cuda(), ev.cuda(), lengths.cuda(), labels.cuda(), 8)
    assert abs(float(loss) - float(z["loss"])) < 2e-4 * abs(float(z["loss"]))
    loss.backward()
    n = 0
    for k, p in m.named_parameters():
        g = p.grad.cpu().numpy().reshape(-1)
        norm_ref = float(z["norm:" + k])
        assert abs(np.linalg.norm(g.astype(np.float64)) - norm_ref) < 2e-3 * norm_ref + 1e-12, k
        scale = max(norm_ref / np.sqrt(g.size), float(np.max(np.abs(z["val:" + k])))) + 1e-20
        err = np.abs(g[z["idx:" + k]] - z["val:" + k]) / scale
        assert np.quantile(err, 0.9) < 1e-3 and err.max() < 5e-2, (k, float(np.quantile(err, 0.9)), float(err.max()))
        n += 1
    assert n == 78


STEP_SUBSET = [(4, 1, 3, "StudentT", False), (2, 2, 0, "Gaussian", True), (1, 2, 3, "StudentT", True)]


@pytest.mark.parametrize("H, L, R, noise, train", STEP_SUBSET,
                         ids=[f"H{c[0]}-L{c[1]}-R{c[2]}-{c[3]}-{'train' if c[4] else 'eval'}" for c in STEP_SUBSET])
def test_small_train_step_with_native_objective_matches_float64(pkg, H, L, R, noise, train):
    """ForwardFn + TrainLossFn against float64 autograd of oracle/torch_port.py and the loop's torch objective, the
    exact dropout mask in train mode (the same comparison as test_gpu_train_fp64, with the native objective)."""
    iefvad_b200, _, synth, train_loss = pkg
    m = small_model(iefvad_b200, synth, H, L, R, noise, train)
    img, ev, lengths, labels = small_batch()
    t = m.temporal
    B, T, _ = img.shape
    keep = None
    if m.training:
        torch.manual_seed(17)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        keep = {(mod, i): torch.from_numpy(O.attention_keep(seed + 1000 * mi + i, B, t.num_heads, T, float(t.dropout)))
                for mi, mod in enumerate(("image", "event")) for i in range(t.num_layers)}
        torch.manual_seed(17)
    outs = m(img, ev, None, None, None)
    res = train_loss(outs, labels, lengths, float(t.nu))
    res.total.backward()
    got = {"loss": res.total.detach(), **{k: v.detach() for k, v in outs.items()}}
    got.update({"grad:" + k: p.grad for k, p in m.named_parameters()})
    got.update({"grad:img": img.grad, "grad:ev": ev.grad})
    P = {k: p.detach().double().cpu().requires_grad_(True) for k, p in m.named_parameters()}
    x64 = {n: x.detach().double().cpu().requires_grad_(True) for n, x in (("img", img), ("ev", ev))}
    ref_outs = {}

    def ref_model(i, e, *_):
        ref_outs.update(torch_port.forward(P, i, e, heads=t.num_heads, lambda_ref=float(t.lambda_ref),
                                           noise_model=t.noise_model, nu=float(t.nu), epsilon=float(t.epsilon), keep=keep,
                                           dtype=torch.float64))
        return ref_outs
    ref_loss, _ = reference_loss(ref_model, clas2_64, x64["img"], x64["ev"], lengths.cpu(), labels.double().cpu(),
                                 float(t.nu))
    ref_loss.backward()
    ref = {"loss": ref_loss.detach(), **{k: v.detach() for k, v in ref_outs.items()}}
    ref.update({"grad:" + k: p.grad for k, p in P.items()})
    ref.update({"grad:img": x64["img"].grad, "grad:ev": x64["ev"].grad})
    assert_all_close(got, ref, 1e-3, f"native objective H{H} L{L} R{R} {noise} {'train' if train else 'eval'}")


def test_native_and_torch_composed_objectives_give_the_same_step(pkg):
    """The 768-d model in train() mode, same batch and dropout seed: loss, all 78 parameter gradients and both input
    gradients with train_loss against the caller's torch ops (CLAS2 unchanged).  The input gradients get the bound of the
    module's backward (1e-3, tests/test_gpu_train.py), not 1e-4: they pass every layer's split-bf16 GEMMs twice, and on a
    B200 a change of the objective's gradients at the 1e-7 level (torch's fp32 rounding; the native gradients of mu are
    float64-exact) moved them by 3e-4 - 7e-4, the native ones the closer to the step fed with float64 objective gradients."""
    iefvad_b200, _, synth, train_loss = pkg
    from iefvad_b200.loss import CLAS2
    m = synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda().train()
    img, ev, lengths, labels = (t.cuda() for t in synth.make_c4_batch(8))
    nu = m.temporal.nu

    def step(loss_fn):
        m.zero_grad()
        i, e = img.clone().requires_grad_(True), ev.clone().requires_grad_(True)
        torch.manual_seed(5)
        loss, _ = loss_fn(m, CLAS2, i, e, lengths, labels, nu)
        loss.backward()
        return float(loss), {k: p.grad.clone() for k, p in m.named_parameters()}, (i.grad, e.grad)

    l_t, g_t, in_t = step(reference_loss)
    l_n, g_n, in_n = step(native_loss(train_loss))
    assert abs(l_n - l_t) <= 1e-5 * abs(l_t), (l_n, l_t)
    assert len(g_n) == 78
    errs = {k: rel_err(g_n[k], g_t[k]) for k in g_t}
    worst = max(errs, key=errs.get)
    in_errs = {"img": rel_err(in_n[0], in_t[0]), "ev": rel_err(in_n[1], in_t[1])}
    print(f"native vs torch-composed objective: worst parameter {worst} {errs[worst]:.2e}, inputs {in_errs}")
    assert errs[worst] <= 1e-4, (worst, errs[worst])
    assert max(in_errs.values()) <= 1e-3, in_errs


def test_torch_objective_of_the_cpu_test_is_the_loops_formula():
    """The float64 reference used above is the same formula as tests/test_gpu_train.py's reference_loss."""
    inputs, labels, lengths = objective_inputs(2, 20, 128, seed=0)
    ts = [torch.as_tensor(t).double() for t in inputs]
    outs = dict(zip(("logits", "image_mu", "event_mu", "image_logvar", "event_logvar"), ts))
    a = reference_loss(lambda *_: outs, clas2_64, ts[1], ts[2], torch.as_tensor(lengths), torch.as_tensor(labels).double(), 8)
    b = torch_objective(ts[0], torch.as_tensor(labels).double(), torch.as_tensor(lengths), *ts[1:], 8)
    assert float(a[0]) == pytest.approx(float(b[0]), rel=1e-14) and float(a[1]) == float(b[1])
