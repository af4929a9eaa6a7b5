"""The "torch" dropout mode of the training attention without a GPU: its numpy restatement (oracle/torch_dropout.py)
against Philox known-answer vectors and a loop-by-loop replay of curand's state machine, the launch arithmetic, the
argument checks of the new C entry points (made before the device is touched) and the ValueError of an unknown
`dropout_rng`."""
import ctypes

import numpy as np
import pytest

from oracle import iefvad_oracle as O
from oracle.torch_dropout import torch_dropout_keep, torch_dropout_launch, torch_dropout_words

M32 = 0xFFFFFFFF


def test_philox_known_answers():
    """Random123's kat_vectors for philox4x32_10 (the block function curand's Philox4_32_10 runs)."""
    kat = [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((M32,) * 4, (M32, M32), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for ctr, key, want in kat:
        assert tuple(int(w) for w in O.philox4x32_10(ctr, key)) == want


def _curand_replay(seed, offset, n, G):
    """torch's fused_dropout_kernel_vec with VEC = 4, loop by loop: thread t runs curand_init(seed, t, offset) (counter
    (0, 0, t lo, t hi) advanced by offset / 4) and one curand_uniform4 per iteration over linearIndex = 4 t, 4 t + 4 G, ..."""
    words = np.zeros(n, dtype=np.uint64)
    for t in range(G):
        ctr = offset // 4
        for lin in range(4 * t, n, 4 * G):
            r = O.philox4x32_10((ctr & M32, ctr >> 32, t & M32, t >> 32), (seed & M32, seed >> 32))
            words[lin:lin + 4] = [int(w) for w in r][:n - lin]
            ctr += 1
    return words


@pytest.mark.parametrize("seed, offset, n, G", [(1234, 0, 4 * 97, 8), ((1 << 40) + 77, 8, 2 * 8 * 5 * 5, 16),
                                                (5, 2 ** 33 + 12, 256, 64), (2 ** 63 + 3, 4, 64, 256)])
def test_counter_mapping_replays_curands_state_machine(seed, offset, n, G):
    got = torch_dropout_words(seed, offset, n, G)
    assert np.array_equal(got, _curand_replay(seed, offset, n, G))
    # the negative control of the GPU tests really moves the words
    if n // 4 > 1:
        assert not np.array_equal(torch_dropout_words(seed, offset, n, G, swap_halves=True), got)


def test_keep_decision_and_scale():
    """float32(word) * 2^-32 + 2^-33 < float32(1 - p): the boundary word of p = 0.5 and the kept fraction / scale."""
    keep = torch_dropout_keep(7, 0, 2, 4, 64, 0.1, 1024)
    kept = keep[keep > 0]
    assert keep.shape == (2, 4, 64, 64)
    assert np.all(kept == np.float64(np.float32(1 / np.float64(np.float32(0.9)))))
    assert abs(kept.size / keep.size - 0.9) < 0.01
    # u(w) = float32(w) 2^-32 + 2^-33 < 0.5 exactly for w < 2^31 (float32(2^31 - 1) rounds up to 2^31)
    w = np.array([2 ** 31 - 129, 2 ** 31 - 64, 2 ** 31 - 1, 2 ** 31], dtype=np.uint64)
    u = w.astype(np.float64).astype(np.float32) * np.float32(2.0 ** -32) + np.float32(2.0 ** -33)
    assert list(u < np.float32(0.5)) == [True, False, False, False]


def test_launch_arithmetic():
    """grid = min(SMs * 8, ceil(n / 256)) blocks of 256 on a 148-SM, 2048-thread-per-SM device (NVIDIA B200)."""
    assert torch_dropout_launch(128 * 8 * 256 * 256, 148) == (303104, 224)
    assert torch_dropout_launch(1 * 8 * 256 * 256, 148) == (303104, 4)
    assert torch_dropout_launch(2 * 4 * 48 * 48, 148) == (18432, 4)
    assert torch_dropout_launch(3 * 8 * 257 * 257, 148) == (303104, 8)
    with pytest.raises(ValueError):
        torch_dropout_keep(0, 0, 1, 1, 3, 0.1, 256)            # 9 elements: torch's VEC would be 1


def test_new_entry_points_reject_bad_arguments_without_a_gpu():
    from iefvad_b200 import _lib
    L = _lib.lib
    p = 1 << 20                                     # never read: every case fails its checks first

    def call(fn, drop, B=2, H=4, T=48, dh=32):
        d = None if drop is None else ctypes.byref(drop)
        if fn == "fwd":
            return L.iefvad_attention_train_fwd_dropout(p, B, T, H, dh, d, p, p, None)
        if fn == "bwd":
            return L.iefvad_attention_train_bwd_dropout(p, p, p, p, B, T, H, dh, d, p, None)
        if fn == "philox fwd":
            return L.iefvad_attention_train_fwd(p, B, T, H, dh, 0.1, 3, p, p, None)
        if fn == "philox bwd":
            return L.iefvad_attention_train_bwd(p, p, p, p, B, T, H, dh, 0.1, 3, p, None)
        return L.iefvad_dropout_mask(d, B, H, T, p, None)

    torch_ok = dict(kind=1, p=0.1, seed=3, offset=8, threads=18432)
    bad = [
        (dict(kind=2), {}, "kind"), (dict(kind=-1), {}, "kind"),
        (dict(p=0.0), {}, "probability"), (dict(p=1.0), {}, "probability"), (dict(p=-0.5), {}, "probability"),
        (dict(threads=0), {}, "threads"), (dict(threads=-256), {}, "threads"), (dict(threads=1 << 31), {}, "threads"),
        (dict(offset=6), {}, "offset"),
        ({}, dict(B=1, H=1, T=3), "multiple of 4"), ({}, dict(B=3, H=1, T=257), "multiple of 4"),
        (dict(kind=0, p=1.0), {}, "probability"),
        (None, {}, "descriptor"),
        ({}, dict(T=-1), "bad B / T"), ({}, dict(H=0), "bad B / T"),
    ]
    for fn in ("fwd", "bwd", "mask"):
        for change, sizes, word in bad:
            drop = None if change is None else _lib.Dropout(**{**torch_ok, **change})
            rc = call(fn, drop, **sizes)
            assert rc != 0 and word in _lib.last_error(), (fn, change, sizes, rc, _lib.last_error())
    # sizes and head sizes the kernels are not built for, on both attention pairs (the philox pair takes no descriptor)
    sized = [(dict(T=-1), "bad B / T"), (dict(H=0), "bad B / T"), (dict(dh=48), "head dim"), (dict(dh=0), "head dim")]
    for fn in ("fwd", "bwd", "philox fwd", "philox bwd"):
        for sizes, word in sized:
            rc = call(fn, _lib.Dropout(**torch_ok), **sizes)
            assert rc != 0 and word in _lib.last_error(), (fn, sizes, rc, _lib.last_error())
    # null tensors
    d = _lib.Dropout(**torch_ok)
    assert L.iefvad_attention_train_fwd_dropout(None, 2, 48, 4, 32, ctypes.byref(d), p, p, None) != 0
    assert "null" in _lib.last_error()
    assert L.iefvad_dropout_mask(ctypes.byref(d), 2, 4, 48, None, None) != 0 and "null" in _lib.last_error()


def test_unknown_dropout_rng_raises_value_error():
    import torch
    import iefvad_b200
    from iefvad_b200 import ops, synth
    args = synth.default_args(visual_head=4)
    m = iefvad_b200.MMFMIL(14, 128, 256, 128, 4, 2, 8, 10, 10, "cpu", args)
    assert m.temporal.dropout_rng == "philox"                      # the default is unchanged
    m.temporal.dropout_rng = "curand"
    x = torch.zeros(1, 4, 128)
    with pytest.raises(ValueError, match="dropout_rng"):
        m(x, x)
    m.train()
    with pytest.raises(ValueError, match="dropout_rng"):
        m(x, x)
    with pytest.raises(ValueError, match="rng"):
        ops.dropout_mask(1, 4, 4, 0.1, 0, rng="numpy")
