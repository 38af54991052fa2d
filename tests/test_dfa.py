"""DFA engines (SURVEY.md section 8a rows a18 McClellan, a19 Sheng, a21 struct NFA):
engines emitted by the host builder in the reference's byte layout run on the
UNMODIFIED reference engines (nfaExecMcClellan8_B / nfaExecMcClellan16_B /
nfaExecSheng_B through oracle/_ref) -- which pins the emitters -- and, on the GPU
box, on the device kernels, which must fire the same (report, block, end) set.
The definition-level oracle is a plain Python walk of the automaton."""
import numpy as np
import pytest

from hyperscan_b200 import synth
import oracle.brute as brute

KINDS = {"auto": 0, "mcclellan8": 1, "mcclellan16": 2, "sheng": 3}


def _lit_case(seed, nlits, alphabet, lo, hi, caseless_frac=0.2):
    lits, flags, ids = synth.literal_set(nlits, min_len=lo, max_len=hi, seed=seed, caseless_frac=caseless_frac,
                                         alphabet=alphabet)
    ids = [100 + (i % max(1, nlits // 2)) for i in ids]            # shared reports
    lens = [0, 1, 2, 3, 15, 16, 17, 31, 32, 33, 100, 1000, 1024, 1025, 5000]
    data, off, ln = synth.ragged_corpus(lens, lits, seed=seed + 1, plant_per_kb=20, alphabet=alphabet + b"XY")
    return lits, flags, ids, data, off, ln


def _definition(lits, flags, ids, data, off, ln):
    """every (report, block, to) with the literal ending at `to`, one per distinct triple"""
    recs = brute.scan_blocks(lits, flags, ids, data, off, ln)
    return sorted({(int(r["id"]), int(r["block"]), int(r["to"])) for r in recs})


def _triples(recs):
    return sorted((int(r["id"]), int(r["block"]), int(r["to"])) for r in recs)


CASES = [("sheng", 2, b"ab", 2, 3), ("sheng", 4, b"abc", 1, 3), ("mcclellan8", 12, b"abcd", 2, 5),
         ("mcclellan8", 30, b"abcdefgh", 2, 4), ("mcclellan16", 12, b"abcd", 2, 5),
         ("mcclellan16", 200, b"abcdefgh", 3, 8), ("auto", 60, b"abcdefghijklmnopqrstuvwxyz", 3, 7)]


@pytest.mark.parametrize("kind,nlits,alphabet,lo,hi", CASES)
@pytest.mark.parametrize("sherman", [0, 1])
def test_emitted_engines_run_on_the_reference(hs, ref, kind, nlits, alphabet, lo, hi, sherman):
    lits, flags, ids, data, off, ln = _lit_case(nlits, nlits, alphabet, lo, hi, 0.0 if kind == "sheng" else 0.2)
    eng = hs.dfa_from_literals(lits, [f & 1 for f in flags], ids, kind=KINDS[kind], sherman=sherman)
    assert eng[8] in (6, 7, 17)                                   # NFA.type
    want = _definition(lits, flags, ids, data, off, ln)
    got = ref.nfa_exec_blocks(eng, data, off, ln, like=want)
    # the reference fires one callback per report of the accept state's list: a set per (block, to)
    assert _triples(got) == want


def _random_table(seed, nstates, nreports=5, dead_frac=0.1):
    rng = np.random.default_rng(seed)
    nxt = rng.integers(1, nstates, size=(nstates, 256)).astype(np.uint16)
    # make the table compressible: a few byte classes, rows similar to state 1's
    classes = rng.integers(0, 6, size=256)
    base = rng.integers(1, nstates, size=6)
    for s in range(nstates):
        row = base.copy()
        for k in rng.choice(6, size=int(rng.integers(0, 4)), replace=False):
            row[k] = rng.integers(0 if rng.random() < dead_frac else 1, nstates)
        nxt[s] = row[classes]
    nxt[0] = 0                                                      # dead state
    reports = [[] for _ in range(nstates)]
    eod = [[] for _ in range(nstates)]
    for s in range(1, nstates):
        if rng.random() < 0.3:
            reports[s] = sorted(set(rng.integers(0, nreports, size=int(rng.integers(1, 3))).tolist()))
        if rng.random() < 0.2:
            eod[s] = [int(rng.integers(50, 55))]
    return nxt, reports, eod


def _walk(nxt, reports, eod, start, data, off, ln):
    out = []
    for b, (o, n) in enumerate(zip(off, ln)):
        s = start
        for i in range(int(n)):
            if s == 0:
                break
            s = int(nxt[s][int(data[int(o) + i])])
            for r in reports[s]:
                out.append((r, b, i + 1))
        for r in eod[s]:
            out.append((r, b, int(n)))
    return sorted(out)


TABLES = [("sheng", 9), ("sheng", 16), ("mcclellan8", 40), ("mcclellan8", 256), ("mcclellan16", 40),
          ("mcclellan16", 700)]


@pytest.mark.parametrize("kind,nstates", TABLES)
@pytest.mark.parametrize("sherman", [0, 1])
def test_random_tables_reference_equals_definition(hs, ref, kind, nstates, sherman):
    nxt, reports, eod = _random_table(nstates + sherman, nstates)
    eng = hs.dfa_from_table(nxt, 1, 1, reports, eod, kind=KINDS[kind], sherman=sherman)
    rng = np.random.default_rng(nstates)
    lens = [0, 1, 5, 16, 17, 200, 1024]
    data, off, ln = synth.ragged_corpus(lens, None, seed=nstates, plant_per_kb=0)
    data = rng.integers(0, 256, size=data.size, dtype=np.uint8)
    want = _walk(nxt, reports, eod, 1, data, off, ln)
    got = ref.nfa_exec_blocks(eng, data, off, ln, like=want)
    assert _triples(got) == want


def test_builder_refuses_what_does_not_fit(hs):
    lits, flags, ids = synth.literal_set(200, min_len=3, max_len=8, seed=3, alphabet=b"abcdefgh")
    with pytest.raises(hs.HsError):
        hs.dfa_from_literals(lits, None, ids, kind=KINDS["sheng"])
    with pytest.raises(hs.HsError):
        hs.dfa_from_literals(lits, None, ids, kind=KINDS["mcclellan8"])
    assert hs.dfa_from_literals(lits, None, ids, kind=KINDS["mcclellan16"])[8] == 7


# ---- device --------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kind,nlits,alphabet,lo,hi", CASES)
@pytest.mark.parametrize("sherman", [0, 1])
def test_device_engines_equal_reference_literals(hs, ref, kind, nlits, alphabet, lo, hi, sherman):
    lits, flags, ids, data, off, ln = _lit_case(nlits + 7, nlits, alphabet, lo, hi, 0.0 if kind == "sheng" else 0.2)
    eng = hs.dfa_from_literals(lits, [f & 1 for f in flags], ids, kind=KINDS[kind], sherman=sherman)
    corpus = hs.Corpus.upload(data, off, ln)
    got, ms = hs.nfa_scan_corpus(eng, corpus)
    want = ref.nfa_exec_blocks(eng, data, off, ln, like=got)
    assert _triples(got) == _triples(want)
    assert len(want) > 20
    corpus.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,nstates", TABLES)
@pytest.mark.parametrize("sherman", [0, 1])
def test_device_engines_equal_reference_random_tables(hs, ref, kind, nstates, sherman):
    rng = np.random.default_rng(nstates + 1)
    lens = [0, 1, 5, 15, 16, 17, 33, 200, 1024, 3000] * 7
    data, off, ln = synth.ragged_corpus(lens, None, seed=nstates, plant_per_kb=0)
    data = rng.integers(0, 256, size=data.size, dtype=np.uint8)
    corpus = hs.Corpus.upload(data, off, ln)
    busy = 0
    for k in range(6):                                           # some random automata die at once: take several
        nxt, reports, eod = _random_table(3 * nstates + sherman + 1000 * k, nstates)
        eng = hs.dfa_from_table(nxt, 1, 1, reports, eod, kind=KINDS[kind], sherman=sherman)
        got, ms = hs.nfa_scan_corpus(eng, corpus, cap=64)        # forces the grow-and-retry path
        want = ref.nfa_exec_blocks(eng, data, off, ln, like=got)
        assert _triples(got) == _triples(want)
        busy += len(want) > 100
    assert busy >= 2
    corpus.free()


@pytest.mark.gpu
def test_device_dfa_uniform_blocks_and_big_table(hs, ref):
    """hsbench-shaped corpus (uniform 1 KiB blocks) against a 16-bit DFA whose table
    does not fit shared memory (read through L1/L2)."""
    lits, flags, ids = synth.literal_set(2000, min_len=4, max_len=8, seed=9, caseless_frac=0.0)
    eng = hs.dfa_from_literals(lits, [f & 1 for f in flags], ids, kind=KINDS["mcclellan16"])
    data, off, ln, _ = synth.block_corpus(512, 1024, lits, plant_per_kb=1.0, seed=10)
    corpus = hs.Corpus.upload(data, off, ln)
    got, ms = hs.nfa_scan_corpus(eng, corpus)
    want = ref.nfa_exec_blocks(eng, data, off, ln, like=got)
    assert _triples(got) == _triples(want) and len(want) > 300
    corpus.free()


@pytest.mark.gpu
def test_device_refuses_other_engines(hs):
    import ctypes as C
    eng = bytearray(hs.dfa_from_literals([b"ab"], None, [1], kind=KINDS["mcclellan16"]))
    data, off, ln = synth.ragged_corpus([64], None, seed=1, plant_per_kb=0)
    corpus = hs.Corpus.upload(data, off, ln)
    eng[8] = 4                                                   # LIMEX_NFA_384: not built
    with pytest.raises(hs.HsError) as e:
        hs.nfa_scan_corpus(bytes(eng), corpus)
    assert e.value.code == hs.HS_ARCH_ERROR
    corpus.free()
