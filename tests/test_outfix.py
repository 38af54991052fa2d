"""Single-outfix databases (ROSE_RUNTIME_SINGLE_OUTFIX): hs_scan -> soleOutfixBlockExec
(src/runtime.c:245-280) runs ONE engine over the whole block through nfaQueueExec with the
queue {START@0, TOP@0, END@len}, its reports are report programs run by roseReportAdaptor ->
roseRunProgram (src/rose/match.c:611-633), EOD accepts through nfaCheckFinalState.  The
build option "outfix_engine" makes the literal compiler emit such a database around a
McClellan-8 / -16, Sheng or LimEx-32 engine over the whole literals.

CPU half: the UNMODIFIED reference hs_scan scanning those databases returns exactly the
definition's matches (which pins the emitted RoseEngine / NfaInfo / programs and, through
the real runtime, the engines once more).  GPU half: hs_scan / hs_b200_scan_blocks of this
runtime on the same database against the reference hs_scan."""
import numpy as np
import pytest

from hyperscan_b200 import synth
import oracle.brute as brute

F_CASELESS, F_SINGLE = 1, 8
KINDS = {"dfa_auto": 1, "mcclellan8": 2, "mcclellan16": 3, "sheng": 4, "limex32": 5}
SETS = {
    "mixed": ([b"abc", b"bcd", b"xyz", b"ab", b"abcdefghij"], [0, 0, F_CASELESS, F_SINGLE, 0], [10, 11, 12, 13, 10]),
    "tiny": ([b"ab", b"b"], [0, F_CASELESS], [1, 2]),
    "shared": ([b"hay", b"stack", b"needle", b"ne"], [F_SINGLE, F_SINGLE, 0, 0], [7, 7, 8, 8]),
}
LENS = [0, 1, 2, 3, 10, 69, 70, 71, 100, 1000, 1024, 1025, 4000]


def _compile(hs, kind, lits, flags, ids):
    hs.set_build_option("outfix_engine", KINDS[kind])
    try:
        return hs.compile_lit_multi(lits, flags, ids)
    finally:
        hs.set_build_option("outfix_engine", 0)


def _fits(kind, name):
    return not (kind == "sheng" and name != "tiny")            # 16 states


CASES = [(k, n) for k in KINDS for n in SETS if _fits(k, n)]


@pytest.mark.parametrize("kind,name", CASES)
def test_reference_hs_scan_runs_our_outfix_databases(hs, ref, kind, name):
    lits, flags, ids = SETS[name]
    db = _compile(hs, kind, lits, flags, ids)
    assert db.info().runtime_impl == 2                             # ROSE_RUNTIME_SINGLE_OUTFIX
    data, off, ln = synth.ragged_corpus(LENS, lits, seed=5, plant_per_kb=40, alphabet=b"abcdxyzXYZefghijnestackhy")
    want = np.sort(brute.scan_blocks(lits, flags, ids, data, off, ln), order=["block", "to", "id"])
    got = ref.scan_sorted(db.ptr, data, off, ln, like=want)
    assert np.array_equal(got, want) and got.size > 30


def test_outfix_database_limits(hs):
    with pytest.raises(hs.HsError):
        _compile(hs, "sheng", *SETS["mixed"])                      # more than 16 states
    with pytest.raises(hs.HsError):
        _compile(hs, "limex32", [b"a" * 520], [0], [1])            # more than 512 positions
    hs.set_build_option("outfix_engine", 3)
    try:
        with pytest.raises(hs.HsError):                            # block mode only
            hs.compile_lit_multi([b"ab"], [0], [1], mode=hs.HS_MODE_STREAM)
    finally:
        hs.set_build_option("outfix_engine", 0)


# ---- device --------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kind,name", CASES)
def test_device_scans_outfix_databases(hs, ref, kind, name):
    lits, flags, ids = SETS[name]
    db = _compile(hs, kind, lits, flags, ids)
    data, off, ln = synth.ragged_corpus(LENS, lits, seed=6, plant_per_kb=40, alphabet=b"abcdxyzXYZefghijnestackhy")
    scratch = hs.Scratch(db)
    got = np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"])
    want = ref.scan_sorted(db.ptr, data, off, ln, like=got)
    assert np.array_equal(got, want) and want.size > 30
    # the stock hs_scan, one block at a time, callbacks in order
    for b in (3, 5, 8, 12):
        buf = data[int(off[b]):int(off[b]) + int(ln[b])].tobytes()
        rc, out = hs.scan(db, buf, scratch)
        assert rc == hs.HS_SUCCESS
        exp = [(int(r["id"]), int(r["to"])) for r in want[want["block"] == b]]
        assert sorted(out) == sorted(exp)
    # resident corpus path
    corpus = hs.Corpus.upload(data, off, ln)
    hs.scan_corpus_async(db, corpus, scratch)
    rc, n, _ = hs.scan_corpus_finish(scratch)
    assert rc == hs.HS_SUCCESS
    got2 = np.sort(hs.fetch_matches(db, scratch), order=["block", "to", "id"])
    assert np.array_equal(got2, want)
    corpus.free()
    scratch.free()


@pytest.mark.gpu
def test_device_outfix_many_uniform_blocks_and_ring_growth(hs, ref):
    lits, flags, ids = SETS["shared"]
    db = _compile(hs, "mcclellan8", lits, flags, ids)
    data, off, ln, _ = synth.block_corpus(4096, 1024, lits, plant_per_kb=3.0, seed=8)
    hs.set_runtime_option("initial_ring", 64)
    try:
        scratch = hs.Scratch(db)
        got = np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"])
    finally:
        hs.set_runtime_option("initial_ring", 1 << 20)
    want = ref.scan_sorted(db.ptr, data, off, ln, like=got)
    assert np.array_equal(got, want) and want.size > 3000
    scratch.free()


@pytest.mark.gpu
def test_device_outfix_termination(hs, ref):
    lits, flags, ids = SETS["mixed"]
    db = _compile(hs, "limex32", lits, flags, ids)
    scratch = hs.Scratch(db)
    rc, out = hs.scan(db, b"..abc..abc..xyz", scratch, stop_after=2)
    assert rc == hs.HS_SCAN_TERMINATED and len(out) == 2
    scratch.free()
