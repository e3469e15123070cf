"""The Philox4x32-10 oracle (tests/philox_oracle.py) against the Random123 known-answer vectors and a plain-Python
transcription of the kernel's round function; no GPU needed."""
import numpy as np
import pytest
import torch

import philox_oracle as ph

# Random123 kat_vectors, philox4x32_10: (counter, key, result)
KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
     (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def _philox_scalar(ctr, key):
    """csrc/common.cuh philox4x32_10, line by line in Python integers."""
    c, k = list(ctr), list(key)
    for _ in range(10):
        p0, p1 = ph.M0 * c[0], ph.M1 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k[0], p1 & 0xFFFFFFFF, (p0 >> 32) ^ c[3] ^ k[1], p0 & 0xFFFFFFFF]
        k = [(k[0] + ph.W0) & 0xFFFFFFFF, (k[1] + ph.W1) & 0xFFFFFFFF]
    return tuple(c)


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_known_answer_vectors(ctr, key, want):
    assert _philox_scalar(ctr, key) == want
    got = ph.philox4x32_10(ctr, key)
    assert tuple(int(v) for v in got) == want


def test_vectorised_oracle_equals_scalar_transcription():
    """Counter layout (i_lo, i_hi, off_lo, off_hi), key (seed_lo, seed_hi), with the high words of all three in use."""
    seed, offset = (1 << 32) + 7, (1 << 33) + 5
    idx = [0, 1, 2, 1023, (1 << 32) - 1, 1 << 32, (5 << 32) + 9]
    words = ph.philox4x32_10((np.array([i & 0xFFFFFFFF for i in idx]), np.array([i >> 32 for i in idx]),
                              offset & 0xFFFFFFFF, offset >> 32), (seed & 0xFFFFFFFF, seed >> 32))
    for n, i in enumerate(idx):
        want = _philox_scalar((i & 0xFFFFFFFF, i >> 32, offset & 0xFFFFFFFF, offset >> 32), (seed & 0xFFFFFFFF, seed >> 32))
        assert tuple(int(w[n]) for w in words) == want
    flat = ph.philox_words(1030, seed, offset)
    assert tuple(int(v) for v in flat[1023]) == _philox_scalar((1023, 0, offset & 0xFFFFFFFF, offset >> 32),
                                                               (seed & 0xFFFFFFFF, seed >> 32))
    # every 32-bit half of seed and offset changes the stream
    for s, o in ((seed & 0xFFFFFFFF, offset), (seed, offset & 0xFFFFFFFF), (seed + (1 << 32), offset), (seed, offset + (1 << 32))):
        assert not np.array_equal(ph.philox_words(8, s, o), ph.philox_words(8, seed, offset))


def test_dropout_oracle_keep_rule():
    """Threshold = uint32(float32(p) * 2^32), word >= threshold keeps; kept values are scaled by 1/(1-p); p = 0 keeps everything."""
    assert ph.keep_threshold(0.0) == 0
    assert ph.keep_threshold(0.5) == 1 << 31
    assert ph.keep_threshold(0.2) == int(float(np.float32(0.2)) * 2 ** 32)
    x = torch.ones(4096 * 4, dtype=torch.bfloat16)
    seed, off, p = 99, 3, 0.25
    y = ph.dropout_bf16(x, p, seed, off)
    words = ph.philox_words(4096, seed, off).reshape(-1)
    thr = ph.keep_threshold(p)
    assert np.array_equal((y != 0).numpy(), words >= thr)
    assert abs((y == 0).float().mean().item() - p) < 0.02
    assert torch.all(y[y != 0] == torch.tensor(1.0 / 0.75).to(torch.bfloat16))
    assert torch.equal(ph.dropout_bf16(x, 0.0, seed, off), x)


def test_normal_oracle_is_standard_normal():
    z = ph.normals(400002, 7, 1)
    assert z.shape == (400002,)
    assert abs(z.mean()) < 1e-2 and abs(z.std() - 1.0) < 1e-2
    assert abs((z ** 4).mean() - 3.0) < 0.05
