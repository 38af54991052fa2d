"""Acceleration primitives on the device (hs_b200_accel_find) against the
reference's shuftiExec / truffleExec / vermicelliExec / vermicelliDoubleExec
(oracle/_ref), plus the reference's own KATs (unit/internal/shufti.cpp:165-182,
truffle.cpp, vermicelli.cpp)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VERM, VERM_NC, DVERM, DVERM_NC, SHUFTI, TRUFFLE = 1, 2, 3, 4, 13, 15


def shufti_masks(chars):
    """lo/hi nibble masks with lo[c & 15] & hi[c >> 4] != 0 <=> c in chars
    (the construction of src/nfa/shufticompile.cpp:54-105: one bit per
    distinct low-nibble set)."""
    by_hi = {}
    for c in chars:
        by_hi.setdefault(c >> 4, set()).add(c & 15)
    sets = []
    lo, hi = [0] * 16, [0] * 16
    for h, s in sorted(by_hi.items()):
        fs = frozenset(s)
        if fs not in sets:
            sets.append(fs)
        hi[h] |= 1 << sets.index(fs)
    if len(sets) > 8:
        return None
    for b, fs in enumerate(sets):
        for n in fs:
            lo[n] |= 1 << b
    return bytes(lo), bytes(hi)


def truffle_masks(chars):
    """src/nfa/trufflecompile.cpp:59+: mask1 covers bytes < 0x80, mask2 the rest;
    entry[low nibble] has bit (high nibble & 7)."""
    m1, m2 = [0] * 16, [0] * 16
    for c in chars:
        (m1 if c < 0x80 else m2)[c & 15] |= 1 << ((c >> 4) & 7)
    return bytes(m1), bytes(m2)


def find(hs, typ, params, data):
    L = hs.lib()
    L.hs_b200_accel_find.argtypes = [C.c_uint, C.c_char_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_ulonglong)]
    pos = C.c_ulonglong()
    rc = L.hs_b200_accel_find(typ, params, bytes(data), len(data), C.byref(pos))
    assert rc == 0
    return pos.value


def ref_find(ref, typ, params, data):
    return ref.accel_find(typ, params, data)


def test_shufti_exec_match1_kat(hs, ref):
    lo, hi = shufti_masks([ord("a")])
    t1 = b"b" * 33 + b"a" + b"b" * 14 + b"a" + b"b" * 12
    for i in range(32):
        assert find(hs, SHUFTI, lo + hi, t1[i:]) == 33 - i
        assert ref_find(ref, SHUFTI, lo + hi, t1[i:]) == 33 - i
    assert find(hs, SHUFTI, lo + hi, b"b" * 100) == 100


@pytest.mark.parametrize("seed", range(6))
def test_random_classes_and_buffers(hs, ref, seed):
    rng = np.random.default_rng(seed)
    for _ in range(12):
        n = int(rng.integers(1, 5000))
        alpha = rng.integers(0, 256, size=int(rng.integers(2, 40)), dtype=np.uint8)
        data = alpha[rng.integers(0, alpha.size, size=n)]
        k = int(rng.integers(1, 6))
        chars = [int(c) for c in rng.integers(0, 256, size=k)]
        if rng.random() < 0.5:
            data = data[~np.isin(data, chars)]
            if data.size == 0:
                continue
            if rng.random() < 0.7:
                data[int(rng.integers(0, data.size))] = chars[0]
        data = data.tobytes()
        sm = shufti_masks(chars)
        if sm:
            assert find(hs, SHUFTI, sm[0] + sm[1], data) == ref_find(ref, SHUFTI, sm[0] + sm[1], data)
        tm = truffle_masks(chars)
        assert find(hs, TRUFFLE, tm[0] + tm[1], data) == ref_find(ref, TRUFFLE, tm[0] + tm[1], data)
        c = bytes([chars[0]])
        assert find(hs, VERM, c + b"\0", data) == ref_find(ref, VERM, c + b"\0", data)


def test_vermicelli_nocase_and_double(hs, ref):
    rng = np.random.default_rng(9)
    for _ in range(40):
        n = int(rng.integers(16, 3000))  # the reference asserts >= VERM_BOUNDARY for some paths
        data = rng.choice(np.frombuffer(b"abxyABXY..", dtype=np.uint8), size=n).tobytes()
        for c in (b"A", b"X", b"Q"):
            assert find(hs, VERM_NC, c + b"\0", data) == ref_find(ref, VERM_NC, c + b"\0", data)
        for pair in (b"ab", b"xy", b"b.", b"zz"):
            assert find(hs, DVERM, pair, data) == ref_find(ref, DVERM, pair, data)
        for pair in (b"AB", b"XY"):
            assert find(hs, DVERM_NC, pair, data) == ref_find(ref, DVERM_NC, pair, data)
    # partial match at the end (src/nfa/vermicelli.h:238-245)
    d = b"." * 40 + b"a"
    assert find(hs, DVERM, b"ab", d) == 40 == ref_find(ref, DVERM, b"ab", d)


def test_large_buffer_first_hit(hs, ref):
    data = np.full(8 << 20, ord("b"), dtype=np.uint8)
    lo, hi = shufti_masks([ord("a"), ord("z")])
    assert find(hs, SHUFTI, lo + hi, data.tobytes()) == data.size
    data[5_000_001] = ord("z")
    data[7_000_000] = ord("a")
    assert find(hs, SHUFTI, lo + hi, data.tobytes()) == 5_000_001
