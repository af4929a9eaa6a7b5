"""MIL top-k / CLAS2 / radix sort / AUC-AP kernels and the batched evaluator against the oracle, scikit-learn and
the reference's golden eval loop.  Needs a B200."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import iefvad_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from iefvad_b200 import ops as _ops
    return _ops


def test_clas2_matches_reference_golden(ops):
    z = load_golden("clas2.npz")
    loss, means = ops.clas2(torch.from_numpy(z["logits"]).cuda(), torch.from_numpy(z["labels"]).cuda(),
                            torch.from_numpy(z["lengths"]).cuda())
    assert abs(float(loss) - float(z["loss"])) < 1e-5 * max(1.0, abs(float(z["loss"])))     # fp32 class: 1e-5
    _, ref_means = O.clas2(z["logits"], z["labels"], z["lengths"], dtype=np.float64)
    np.testing.assert_allclose(means.cpu().numpy(), ref_means, rtol=1e-5, atol=1e-7)
    from iefvad_b200.loss import CLAS2
    assert float(CLAS2(torch.from_numpy(z["logits"]).cuda(), torch.from_numpy(z["labels"]), torch.from_numpy(z["lengths"]),
                       "cuda")) == float(loss)


@pytest.mark.parametrize("B,T", [(1, 256), (128, 256), (7, 100), (3, 1), (2, 4096), (1, 16384), (5, 33)])
def test_topk_indices_bit_exact_vs_stable_sort(ops, B, T):
    rng = np.random.default_rng(B * 100 + T)
    x = np.round(rng.standard_normal((B, T)), 1).astype(np.float32)        # heavy ties
    x[0, :min(T, 5)] = [0.0, -0.0, 0.0, 7.0, 7.0][:min(T, 5)]                # +-0 compare equal, ties by index
    lengths = rng.integers(1, T + 1, B)
    lengths[0] = T
    mean, idx = ops.mil_topk_mean(torch.from_numpy(x).cuda(), torch.from_numpy(lengths).cuda(), return_indices=True)
    mean, idx = mean.cpu().numpy(), idx.cpu().numpy()
    for i in range(B):
        n = int(lengths[i])
        k = int(n / 16 + 1)
        vals, ref_idx = O.mil_topk(x[i, :n], k)
        assert np.array_equal(idx[i, :k], ref_idx), i            # bit-exact ranking
        assert np.all(idx[i, k:] == -1)
        assert abs(mean[i] - vals.astype(np.float64).mean()) < 1e-6 * max(1, abs(vals.mean()))


@pytest.mark.parametrize("n", [1, 2, 255, 4096, 4097, 100_000, 1_000_003])
def test_sort_scores_is_stable_descending_argsort(ops, n):
    rng = np.random.default_rng(n)
    s = rng.standard_normal(n).astype(np.float32)
    if n > 10:
        s[rng.integers(0, n, n // 3)] = np.float32(0.25)          # big tie group
        s[:6] = [0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45]        # signed zeros, infinities, denormals
    order = ops.sort_scores(torch.from_numpy(s).cuda()).cpu().numpy()
    assert np.array_equal(order, np.argsort(-s, kind="stable"))


def _frames(pos):
    return (np.arange(16)[None, :] < pos[:, None]).astype(np.float64).reshape(-1)


def test_auc_ap_matches_sklearn_golden(ops):
    z = load_golden("sklearn_auc.npz")
    for i in range(int(z["n"])):
        s, pos = z[f"{i}:scores"], z[f"{i}:pos"].astype(np.int32)
        got = ops.auc_ap(torch.from_numpy(s).cuda(), torch.from_numpy(pos).cuda()).cpu().numpy()
        if np.isnan(z[f"{i}:auc"]):
            assert np.isnan(got[0])
        else:
            assert abs(got[0] - float(z[f"{i}:auc"])) < 1e-12
        assert abs(got[1] - float(z[f"{i}:ap"])) < 1e-12
        assert got[2] == pos.sum() and got[3] == 16 * len(pos) - pos.sum()


@pytest.mark.parametrize("n,ties", [(1, False), (17, True), (5000, True), (139_568 // 16, False), (300_000, True)])
def test_auc_ap_matches_live_sklearn_and_oracle(ops, n, ties):
    sk = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(n)
    s = rng.random(n).astype(np.float32)
    if ties:
        s = np.round(s, 2)
    pos = np.where(rng.random(n) < 0.3, rng.integers(1, 17, n), 0).astype(np.int32)
    got, order = ops.auc_ap(torch.from_numpy(s).cuda(), torch.from_numpy(pos).cuda(), return_order=True)
    got = got.cpu().numpy()
    auc, ap = O.auc_ap_segments(s, pos, 16)
    if np.isnan(auc):
        assert np.isnan(got[0])
    else:
        assert abs(got[0] - auc) < 1e-12
    assert abs(got[1] - ap) < 1e-12
    assert np.array_equal(order.cpu().numpy(), np.argsort(-s, kind="stable"))
    if n <= 20000 and 0 < pos.sum() < 16 * n:
        rep = np.repeat(s.astype(np.float64), 16)
        assert abs(got[0] - sk.roc_auc_score(_frames(pos), rep)) < 1e-12
        assert abs(got[1] - sk.average_precision_score(_frames(pos), rep)) < 1e-12


@pytest.mark.parametrize("n,nsub,ties", [(3000, 5, True), (77788, 16, False), (40000, 32, True)])
def test_auc_ap_multi_equals_per_subset_ranking(ops, n, nsub, ties):
    """Class-wise AUC / AP from ONE ranking pass == ranking every subset on its own (oracle / sklearn semantics),
    including subsets with one label value only (NaN AUC), empty subsets and ties across subset boundaries."""
    rng = np.random.default_rng(n + nsub)
    s = rng.random(n).astype(np.float32)
    if ties:
        s = np.round(s, 2)
    pos = np.where(rng.random(n) < 0.2, rng.integers(1, 17, n), 0).astype(np.int32)
    cls = rng.integers(0, nsub - 2, n) if nsub > 2 else np.zeros(n, dtype=np.int64)
    member = np.ones(n, dtype=np.uint32)                      # bit 0: everything
    member |= np.where(cls % 2 == 1, 2, 0).astype(np.uint32)  # bit 1: an "abnormal"-style union of classes
    for c in range(nsub - 2):
        member |= np.where(cls == c, np.uint32(4) << np.uint32(c), 0).astype(np.uint32)
    if nsub > 3:
        pos[cls == 0] = 0                                     # a class without positives -> AUC NaN, AP 0
    if nsub == 32:
        member &= ~np.uint32(1 << 31)                         # the last subset is empty
    got = ops.auc_ap_multi(torch.from_numpy(s).cuda(), torch.from_numpy(pos).cuda(),
                           torch.from_numpy(member.view(np.int32)).cuda(), nsub).cpu().numpy()
    for k in range(nsub):
        sel = ((member >> np.uint32(k)) & 1).astype(bool)
        if not sel.any():
            assert np.isnan(got[k, 0]) and got[k, 2] == 0 and got[k, 3] == 0
            continue
        auc, ap = O.auc_ap_segments(s[sel], pos[sel], 16)
        assert got[k, 2] == pos[sel].sum() and got[k, 3] == 16 * sel.sum() - pos[sel].sum()
        if np.isnan(auc):
            assert np.isnan(got[k, 0])
        else:
            assert abs(got[k, 0] - auc) < 1e-12, (k, got[k, 0], auc)
        if pos[sel].sum() > 0:
            assert abs(got[k, 1] - ap) < 1e-12, (k, got[k, 1], ap)


def test_auc_stress_2_pow_24(ops):
    """SURVEY 8d stress point: N = 2^24 scores, 5 % positives, 10 % forced ties; checked through size-independent
    properties (sortedness of the rank permutation, permutation validity, invariance to input order)."""
    n = 1 << 24
    g = torch.Generator(device="cuda").manual_seed(0)
    s = torch.rand(n, device="cuda", generator=g)
    tie = torch.rand(n, device="cuda", generator=g) < 0.10
    s = torch.where(tie, torch.round(s * 64) / 64, s)
    pos = (torch.rand(n, device="cuda", generator=g) < 0.05).to(torch.int32) * 16
    out, order = ops.auc_ap(s, pos, return_order=True)
    o = order.long()
    sorted_s = s[o]
    assert bool((sorted_s[:-1] >= sorted_s[1:]).all())
    same = sorted_s[:-1] == sorted_s[1:]
    assert bool((o[:-1][same] < o[1:][same]).all())                        # ties keep ascending index
    assert int(torch.bincount(o, minlength=n).max()) == 1                  # a permutation
    perm = torch.randperm(n, device="cuda", generator=g)
    out2 = ops.auc_ap(s[perm], pos[perm])
    assert torch.equal(out[[0, 2, 3]], out2[[0, 2, 3]])                    # exact-integer AUC: order independent
    assert abs(float(out[1]) - float(out2[1])) < 1e-12
    assert abs(float(out[0]) - 0.5) < 5e-3                                 # random scores


def test_evaluator_matches_reference_eval_loop(ops):
    """The reference's own train/ucf_test.py:test() on 30 synthetic videos (golden) vs the batched GPU evaluator."""
    import iefvad_b200
    from iefvad_b200 import synth
    from iefvad_b200.evaluate import Evaluator
    z = load_golden("eval_loop.npz")
    T, classes = z["lengths"], [str(c) for c in z["classes"]]
    gt = synth.make_gt(T, classes)
    model = synth.build_model(iefvad_b200.MMFMIL, seed=0).cuda().eval()
    ev = Evaluator(model, T, classes, gt)
    fi, fe = [], []
    for v in range(len(T)):
        a, b = synth.make_video(100 + v, int(T[v]))
        fi.append(a)
        fe.append(b)
    ev.set_device_features(ev.chunk_features(fi), ev.chunk_features(fe))
    for plan, tol in (("fp32", 1e-5), ("B", 1e-3), ("HH", 1e-3)):
        model.temporal.precision = plan
        with torch.no_grad():
            res = ev.step()
        scores = res["scores"].cpu().numpy()
        assert np.max(np.abs(scores - z["scores"]) / z["scores"]) < tol, plan
        # AUC / AP given OUR scores must equal the oracle's sklearn restatement on the same scores
        rep = np.repeat(scores.astype(np.float64), 16)
        assert abs(res["AUC"] - O.roc_auc_score(gt, rep)) < 1e-12
        assert abs(res["AP"] - O.average_precision_score(gt, rep)) < 1e-12
        assert abs(res["AUC"] - float(z["AUC"])) < 2e-3 and abs(res["AP"] - float(z["AP"])) < 2e-3
    # pinned-host path gives the same bits
    ev.set_host_features(ev.chunk_features(fi), ev.chunk_features(fe))
    with torch.no_grad():
        res2 = ev.step(host_inputs=True)
    assert torch.equal(res2["scores"], res["scores"])
    # ragged pinned-host path (raw [T_v, D] features, process_split on the device): the same bits again
    ev.set_host_ragged(fi, fe)
    with torch.no_grad():
        res3 = ev.step(host_inputs=True)
    assert torch.equal(res3["scores"], res["scores"]) and res3["AUC"] == res["AUC"] and res3["AP"] == res["AP"]
    # ... the full-rows path (every stage on every pad row) agrees to the rounding of one softmax term: the
    # valid-rows mode computes the identical zero-pad rows of a chunk once (pad de-duplication) ...
    ev.valid_rows_only = False
    ev.set_device_features(ev.chunk_features(fi), ev.chunk_features(fe))
    with torch.no_grad():
        res4 = ev.step()
    assert ((res4["scores"] - res["scores"]).abs() / res4["scores"]).max().item() < 3e-4
    # ... and bit for bit once de-duplication is switched off
    from iefvad_b200 import _lib
    ev.valid_rows_only = True
    model.temporal.pad_dedup = False
    with torch.no_grad():
        res5 = ev.step()
    model.temporal.pad_dedup = True
    assert torch.equal(res4["scores"], res5["scores"])
    # class-wise and Ano-AUC against the oracle on our scores
    st = 0
    by, gby = {}, {}
    for v, c in enumerate(classes):
        by.setdefault(c, []).append(scores[st:st + T[v]])
        gby.setdefault(c, []).append(gt[16 * st:16 * (st + T[v])])
        st += int(T[v])
    for c, (auc, ap) in res["classwise"].items():
        rep = np.repeat(np.concatenate(by[c]).astype(np.float64), 16)
        assert abs(auc - O.roc_auc_score(np.concatenate(gby[c]), rep)) < 1e-12
        assert abs(ap - O.average_precision_score(np.concatenate(gby[c]), rep)) < 1e-12
    assert "Normal" not in res["classwise"]
    ab = [c for c in by if c != "Normal"]
    rep = np.repeat(np.concatenate([np.concatenate(by[c]) for c in ab]).astype(np.float64), 16)
    # Ano-AUC concatenates class by class (train/ucf_test.py:339-345); AUC is order independent
    assert abs(res["ano_AUC"] - O.roc_auc_score(np.concatenate([np.concatenate(gby[c]) for c in ab]), rep)) < 1e-12


def test_localisation_map_matches_reference_and_oracle():
    """Row N5: getDetectionMAP on the GPU (csrc/locmap.cu) against the reference's own output (train/metrics.py run as-is,
    tests/golden/locmap.npz) and against the oracle on further cases incl. the `return 0` quirk."""
    from iefvad_b200 import metrics, synth
    z = load_golden("locmap.npz")
    preds, segs, labels = synth.make_locmap_case()
    dmap, ious = metrics.getDetectionMAP([torch.from_numpy(p).cuda() for p in preds], segs, labels)
    assert ious == [0.1, 0.2, 0.3, 0.4, 0.5]
    assert np.max(np.abs(np.array(dmap) - z["dmap"])) < 1e-6, (dmap, z["dmap"])
    assert abs(metrics.getLocMAP(preds[:9], 0.3, segs[:9], labels[:9], False) - float(z["short"])) < 1e-6
    dead = [p.copy() for p in preds]
    for p in dead:
        p[:, 5] = -1.0
    assert metrics.getLocMAP(dead, 0.3, segs, labels, False) == 0
    p2, s2, l2 = synth.make_locmap_case(n_videos=120, seed=77)
    for th in (0.1, 0.5):
        assert abs(metrics.getLocMAP(p2, th, s2, l2, False) - O.loc_map(p2, th, s2, l2)) < 1e-6
