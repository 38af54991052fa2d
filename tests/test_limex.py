"""LimEx NFA, 32-state model (SURVEY.md section 8a rows a20 LimEx, a21 struct NFA / mq):
engines emitted by the host builder in the reference's byte layout run on the UNMODIFIED
reference engine -- the way Rose runs an outfix in block mode: a queue {START@0, TOP@0,
END@len} through nfaExecLimEx32_Q, then nfaExecLimEx32_testEOD (oracle/ref/ref_limex.c) --
which pins the emitter and the Python restatement of the runtime (oracle/limex.py); on the
GPU box the device kernel must fire the same (report, block, offset) multiset."""
import numpy as np
import pytest

from hyperscan_b200 import synth
import oracle.brute as brute
import oracle.limex as model


def _triples(recs):
    return sorted((int(r["id"]), int(r["block"]), int(r["to"])) for r in recs)


LIT_SETS = [([b"abc", b"bcd", b"xyz", b"ab"], [0, 0, 1, 0]), ([b"a"], [0]), ([b"aaaa", b"aa"], [0, 0]),
            ([b"abcdefghijklmnopqrstuvwxyzABCDE"], [1]), ([b"ab", b"cd", b"ef", b"gh", b"ab", b"b", b"hgfedcba"], [0, 1] * 3 + [0])]
LENS = [0, 1, 2, 3, 4, 15, 16, 17, 31, 32, 33, 100, 127, 128, 129, 1000, 1024, 1025, 3000]


def _lit_case(i):
    lits, cl = LIT_SETS[i]
    ids = [100 + (k % 3) for k in range(len(lits))]                  # shared report ids
    data, off, ln = synth.ragged_corpus(LENS, lits, seed=40 + i, plant_per_kb=40, alphabet=b"abcdefghxyzXYZAB")
    return lits, cl, ids, data, off, ln


@pytest.mark.parametrize("i", range(len(LIT_SETS)))
def test_literal_nfas_run_on_the_reference(hs, ref, i):
    lits, cl, ids, data, off, ln = _lit_case(i)
    eng = hs.limex32_from_literals(lits, cl, ids)
    assert eng[8] == (0 if sum(map(len, lits)) < 32 else 1)            # NFA.type = LIMEX_NFA_32 / _64
    walk = model.walk_blocks(eng, data, off, ln)
    got = _triples(ref.nfa_exec_blocks(eng, data, off, ln, like=walk))
    want = brute.scan_blocks(lits, cl, ids, data, off, ln)
    # one callback per accepting STATE: two literals with one report id ending together fire it twice
    assert sorted(set(got)) == sorted({(int(r["id"]), int(r["block"]), int(r["to"])) for r in want})
    assert got == sorted(walk)
    assert len(got) > 20


def _random_nfa(seed, wide=False):
    """reach, init, succ, reports, eod reports, squash: anything goes -- the reference runs any
    well-formed LimEx structure, so the emitter's choice of shifts / exceptions is exercised too"""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(33, 65)) if wide else int(rng.integers(2, 33))
    full = (1 << n) - 1
    classes = rng.integers(0, 5, size=256)
    rand = lambda: (int(rng.integers(0, 1 << 32)) | (int(rng.integers(0, 1 << 32)) << 32)) & full
    masks = [rand() for _ in range(5)]
    masks[0] |= 1                                                     # keep the automaton alive on class 0
    reach = np.array([masks[c] for c in classes], dtype=np.uint64)
    succ = np.zeros(n, dtype=np.uint64)
    for s in range(n):
        m = 0
        if rng.random() < 0.8 and s + 1 < n:
            m |= 1 << (s + 1)
        for _ in range(int(rng.integers(0, 4))):
            m |= 1 << int(rng.integers(0, n))
        if rng.random() < 0.3:
            m |= 1 << s
        succ[s] = np.uint64(m)
    succ[0] |= np.uint64(1)
    reports = [sorted(set(rng.integers(0, 6, size=int(rng.integers(1, 3))).tolist())) if rng.random() < 0.25 else []
               for _ in range(n)]
    eod = [[int(rng.integers(50, 54))] if rng.random() < 0.2 else [] for _ in range(n)]
    kind = np.array([int(rng.choice([0, 0, 0, 1, 3])) for _ in range(n)], dtype=np.uint8)
    sqm = np.array([rand() for _ in range(n)], dtype=np.uint64)
    init = 1 | (rand() & 0x7)
    return reach, init, succ, reports, eod, sqm, kind


def _emit(hs, spec):
    reach, init, succ, reports, eod, sqm, kind = spec
    if len(succ) <= 32 and int(np.max(reach)) < (1 << 32):
        return hs.limex32_from_spec(reach.astype(np.uint32), init, init, succ.astype(np.uint32), reports, eod,
                                    sqm.astype(np.uint32), kind)
    return hs.limex_from_spec64(reach, init, init, succ, reports, eod, sqm, kind)


def _random_corpus(seed):
    rng = np.random.default_rng(seed)
    data, off, ln = synth.ragged_corpus(LENS[:16], None, seed=seed, plant_per_kb=0)
    return rng.integers(0, 256, size=data.size, dtype=np.uint8), off, ln


@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("seed", range(12))
def test_random_nfas_reference_equals_restatement(hs, ref, seed, wide):
    eng = _emit(hs, _random_nfa(seed, wide))
    assert eng[8] == (1 if wide else 0)
    data, off, ln = _random_corpus(100 + seed)
    walk = model.walk_blocks(eng, data, off, ln)
    got = _triples(ref.nfa_exec_blocks(eng, data, off, ln, like=walk))
    assert got == sorted(walk)


def _random_wide_nfa(seed, n):
    """the same over n > 64 states, state sets as Python ints; sparse enough that the automaton neither dies at
    once nor saturates: every state has a neighbour edge (a limited shift unless it crosses a 64-bit lane) and a
    few far ones (exceptions)"""
    rng = np.random.default_rng(seed)
    full = (1 << n) - 1

    def rand(density):
        return sum(1 << i for i in np.flatnonzero(rng.random(n) < density).tolist())
    classes = rng.integers(0, 6, size=256)
    masks = [rand(0.5) | 1 for _ in range(6)]
    reach = [masks[c] for c in classes]
    succ = []
    for s in range(n):
        m = 0
        for d in (1, 2, 5):
            if rng.random() < (0.8 if d == 1 else 0.25) and s + d < n:
                m |= 1 << (s + d)
        for _ in range(int(rng.integers(0, 3))):
            m |= 1 << int(rng.integers(0, n))
        if rng.random() < 0.2:
            m |= 1 << s
        succ.append(m)
    succ[0] |= 1
    reports = [sorted(set(rng.integers(0, 6, size=int(rng.integers(1, 3))).tolist())) if rng.random() < 0.1 else []
               for _ in range(n)]
    eod = [[int(rng.integers(50, 54))] if rng.random() < 0.1 else [] for _ in range(n)]
    kind = [int(rng.choice([0, 0, 0, 0, 1, 3])) for _ in range(n)]
    sqm = [rand(0.9) for _ in range(n)]
    init = 1 | (rand(0.02) & full)
    return reach, init, succ, reports, eod, sqm, kind


WIDE_SIZES = [(65, 2), (100, 2), (128, 2), (129, 3), (200, 3), (256, 3), (257, 5), (300, 5), (384, 5), (450, 5), (512, 5)]


@pytest.mark.parametrize("n,kind", WIDE_SIZES)
def test_random_wide_nfas_reference_equals_restatement(hs, ref, n, kind):
    for seed in range(3):
        reach, init, succ, reports, eod, sqm, sk = _random_wide_nfa(1000 * n + seed, n)
        eng = hs.limex_from_spec_wide(reach, init, init, succ, reports, eod, sqm, sk)
        assert eng[8] == kind                                         # LIMEX_NFA_128 / _256 / _512
        data, off, ln = _random_corpus(300 + seed)
        walk = model.walk_blocks(eng, data, off, ln)
        got = _triples(ref.nfa_exec_blocks(eng, data, off, ln, like=walk))
        assert got == sorted(walk)
        assert len(got) > 50


def test_builder_limits(hs):
    with pytest.raises(hs.HsError):
        hs.limex32_from_literals([b"a" * 512], [0], [1])             # 513 states
    assert hs.limex32_from_literals([b"a" * 31], [0], [1])[8] == 0
    assert hs.limex32_from_literals([b"a" * 32], [0], [1])[8] == 1   # 33 states: the 64-state model
    assert hs.limex32_from_literals([b"a" * 64], [0], [1])[8] == 2   # 65: LIMEX_NFA_128
    assert hs.limex32_from_literals([b"ab" * 100], [0], [1])[8] == 3
    assert hs.limex32_from_literals([b"abc" * 100], [0], [1])[8] == 5


# ---- device --------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(LIT_SETS)))
def test_device_limex_equals_reference_literals(hs, ref, i):
    lits, cl, ids, data, off, ln = _lit_case(i)
    eng = hs.limex32_from_literals(lits, cl, ids)
    corpus = hs.Corpus.upload(data, off, ln)
    got, ms = hs.nfa_scan_corpus(eng, corpus)
    assert _triples(got) == _triples(ref.nfa_exec_blocks(eng, data, off, ln, like=got))
    corpus.free()


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("seed", range(24))
def test_device_limex_equals_reference_random(hs, ref, seed, wide):
    eng = _emit(hs, _random_nfa(seed, wide))
    data, off, ln = _random_corpus(200 + seed)
    corpus = hs.Corpus.upload(data, off, ln)
    got, ms = hs.nfa_scan_corpus(eng, corpus, cap=64)                 # forces the grow-and-retry path
    want = ref.nfa_exec_blocks(eng, data, off, ln, like=got)
    assert _triples(got) == _triples(want)
    corpus.free()


@pytest.mark.gpu
@pytest.mark.parametrize("n,kind", WIDE_SIZES)
def test_device_wide_limex_equals_reference_random(hs, ref, n, kind):
    for seed in range(3):
        reach, init, succ, reports, eod, sqm, sk = _random_wide_nfa(1000 * n + seed, n)
        eng = hs.limex_from_spec_wide(reach, init, init, succ, reports, eod, sqm, sk)
        assert eng[8] == kind
        data, off, ln = _random_corpus(300 + seed)
        corpus = hs.Corpus.upload(data, off, ln)
        got, ms = hs.nfa_scan_corpus(eng, corpus, cap=64)
        assert _triples(got) == _triples(ref.nfa_exec_blocks(eng, data, off, ln, like=got))
        corpus.free()


@pytest.mark.gpu
@pytest.mark.parametrize("reps,kind", [(10, 2), (30, 3), (70, 5)])
def test_device_wide_limex_literals(hs, ref, reps, kind):
    lits = [b"needle" * reps, b"hay", b"stack" * 3, b"ne"]
    eng = hs.limex32_from_literals(lits, [0, 1, 0, 0], [1, 2, 3, 4])
    assert eng[8] == kind
    data, off, ln, _ = synth.block_corpus(512, 1024, lits, plant_per_kb=2.0, seed=12)
    corpus = hs.Corpus.upload(data, off, ln)
    got, ms = hs.nfa_scan_corpus(eng, corpus)
    want = ref.nfa_exec_blocks(eng, data, off, ln, like=got)
    assert _triples(got) == _triples(want) and len(want) > 300
    corpus.free()


@pytest.mark.gpu
def test_device_limex_uniform_blocks(hs, ref):
    lits = [b"needle", b"hay", b"stack", b"ne"]
    eng = hs.limex32_from_literals(lits, [0, 1, 0, 0], [1, 2, 3, 4])
    data, off, ln, _ = synth.block_corpus(2048, 1024, lits, plant_per_kb=2.0, seed=12)
    corpus = hs.Corpus.upload(data, off, ln)
    got, ms = hs.nfa_scan_corpus(eng, corpus)
    want = ref.nfa_exec_blocks(eng, data, off, ln, like=got)
    assert _triples(got) == _triples(want) and len(want) > 1000
    corpus.free()


@pytest.mark.gpu
def test_device_refuses_bounded_repeats(hs):
    import struct
    eng = bytearray(hs.limex32_from_literals([b"ab"], [0], [1]))
    struct.pack_into("<I", eng, 64 + 300, 1)                          # LimExNFA32.repeatCount
    data, off, ln = synth.ragged_corpus([64], None, seed=1, plant_per_kb=0)
    corpus = hs.Corpus.upload(data, off, ln)
    with pytest.raises(hs.HsError) as e:
        hs.nfa_scan_corpus(bytes(eng), corpus)
    assert e.value.code == hs.HS_ARCH_ERROR
    corpus.free()
