"""The host reference of the in-kernel noise (tests/philox_ref.py): Philox4x32-10 known-answer vectors and the project's counter
layout.  No GPU needed; tests/test_gpu_philox.py compares the kernels with this reference."""
import numpy as np
import pytest

import philox_ref as P


# Known-answer vectors of Philox4x32-10 (the Random123 distribution's kat_vectors)
@pytest.mark.parametrize("ctr,key,expected", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox4x32_10_known_answers(ctr, key, expected):
    got = P.philox4x32_10(*ctr, *key)
    assert tuple(int(v) for v in got) == expected
    # vectorised: the same counter repeated in an array gives the same answer in every lane
    arr = P.philox4x32_10(*(np.full(5, c, dtype=np.uint32) for c in ctr), *key)
    assert all((a == e).all() for a, e in zip(arr, expected))


def test_step_words_are_unique_per_step_and_draw():
    words = [P.step_word(s, d) for s in range(-1, 1000) for d in range(8)]
    assert len(set(words)) == len(words)
    assert P.step_word(-1) == 0                    # x_T
    assert P.step_word(0, 7) == 15 and P.step_word(999, 0) == 8000


def test_stream_word_folds_the_high_half():
    assert P.stream_word(0) == 0 and P.stream_word(3) == 3
    assert P.stream_word(2 ** 32 + 5) == (5 ^ 0x9E3779B9)
    assert len({P.stream_word(s) for s in (0, 1, 3, 2 ** 32, 2 ** 32 + 5, 2 ** 33)}) == 6


def test_key_uses_both_seed_words_and_quad_index_is_64_bit():
    q = np.array([0, 1, 2 ** 32, 2 ** 32 + 1], dtype=np.uint64)
    a = P.raw_quads(0x1_0000_0007, 0, 8, q)
    b = P.raw_quads(0x7, 0, 8, q)
    assert not (a == b).all(axis=1).any()          # the high seed word changes every quad
    assert len({tuple(r) for r in a}) == 4         # quads 0 and 2^32 differ (the high counter word is used)
    # randn lays quad i out as elements 4i .. 4i + 3
    z = P.randn(5, 1, 3, 64)
    np.testing.assert_array_equal(z.reshape(-1, 4)[9], P.normal4(5, 1, P.step_word(3), [9])[0])


def test_uniforms_and_box_muller_edges():
    r = np.array([[0xFFFFFFFF, 0, 0, 0xFFFFFFFF], [0xFFFFFF80, 1 << 31, 0xFFFFFF7F, 0], [0xFFFFFE80, 0, 0xFFFFFE81, 0]],
                 dtype=np.uint32)
    u = P.uniforms(r)
    assert u.dtype == np.float32
    assert u[0, 0] == 1.0 and u[0, 3] == 1.0 and u[0, 1] == 0.0    # (float)0xFFFFFFFF rounds to 2^32
    # round to nearest even: 2^32 - 128 -> 2^32, 2^32 - 384 -> 2^32 - 512
    assert u[1, 0] == 1.0 and u[1, 2] == np.float32(1 - 2 ** -24) and u[1, 1] == 0.5
    assert u[2, 0] == np.float32(1 - 2 ** -23) and u[2, 2] == np.float32(1 - 2 ** -24)
    z = P.box_muller(u)
    assert np.isfinite(z).all() and (z[0, :2] == 0).all()        # radius 0 at u = 1
    assert abs(z[0, 2] - np.sqrt(-2 * np.log(2.0 ** -32))) < 1e-9  # r.z = 0: the largest radius, angle 0
    x = P.randn(1234, 0, -1, 1 << 16)
    assert abs(x.mean()) < 0.02 and abs(x.var() - 1) < 0.02
