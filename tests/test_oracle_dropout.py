"""The attention-dropout mask of the training step as the oracle states it (oracle/iefvad_oracle.py: philox4x32_10,
attention_keep): Philox4x32-10 against Random123's known-answer vectors, and the dropped fraction against the binomial
law.  CPU only; tests/test_gpu_train_fp64.py compares the CUDA kernels with this mask."""
import math

import numpy as np
import pytest

from oracle import iefvad_oracle as O


@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox4x32_10_known_answers(ctr, key, want):
    assert tuple(int(w) for w in O.philox4x32_10(ctr, key)) == want


def test_attention_keep_follows_the_documented_counter_and_word():
    seed = (0x1234567 << 32) | 0x89ABCDEF
    B, H, T, p = 2, 3, 9, 0.5
    keep = O.attention_keep(seed, B, H, T, p)
    thresh = int(np.float64(np.float32(p)) * 2 ** 32)
    for b, h, q, k in ((0, 0, 0, 0), (1, 2, 8, 7), (1, 0, 3, 5), (0, 2, 6, 2)):
        words = O.philox4x32_10((k >> 2, q, b * H + h, 0), (seed & 0xFFFFFFFF, seed >> 32))
        assert keep[b, h, q, k] == (2.0 if int(words[k & 3]) >= thresh else 0.0)
    assert np.array_equal(O.attention_keep(seed, B, H, T, 0.0), np.ones((B, H, T, T)))


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_attention_keep_drops_a_binomial_fraction(p):
    B, H, T = 2, 3, 300
    keep = O.attention_keep(2 ** 62 - 12345, B, H, T, p)
    scale = float(np.float32(1) / (np.float32(1) - np.float32(p)))
    assert set(np.unique(keep).tolist()) == {0.0, scale}
    n = keep.size
    dropped = float((keep == 0).mean())
    assert abs(dropped - p) < 5 * math.sqrt(p * (1 - p) / n), dropped
