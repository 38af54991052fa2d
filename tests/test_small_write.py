"""Small-write engine (src/smallwrite/, used by hs_scan for buffers shorter than 70
bytes: src/runtime.c:401-413): literal databases carry a DFA over the whole literals
(Sheng or McClellan in the reference's layout, host/dfa_build.cpp) whose reports are
report-program offsets.  The UNMODIFIED reference hs_scan takes that path for short
buffers and must deliver what the definition demands; the device ignores the switch
(same results by construction) and is checked against the reference as everywhere."""
import json
import os
import struct

import numpy as np
import pytest

from hyperscan_b200 import synth
import oracle.brute as brute

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "ref_layout.json")) as f:
    LAYOUT = json.load(f)


def _small_write(db):
    """(smallWriteOffset, largestBuffer, NFA.type) read from the serialized bytecode"""
    bc = db.serialize()[32:]
    off = struct.unpack_from("<I", bc, LAYOUT["RoseEngine.smallWriteOffset"])[0]
    if not off:
        return 0, 0, None
    largest, start, size = struct.unpack_from("<III", bc, off)
    return off, largest, bc[off + 64 + 8]


CASES = [(1, b"abcdef", 3, 6, 0.0), (3, b"ab", 1, 3, 0.0), (12, b"abcd", 2, 6, 0.3), (40, b"abcdefgh", 2, 12, 0.2),
         (300, b"abcdefgh", 3, 9, 0.1)]


@pytest.mark.parametrize("nl,alphabet,lo,hi,cf", CASES)
def test_reference_small_write_path_on_our_engines(hs, ref, nl, alphabet, lo, hi, cf):
    lits, flags, ids = synth.literal_set(nl, min_len=lo, max_len=hi, seed=nl + 3, caseless_frac=cf,
                                         alphabet=alphabet, singlematch_frac=0.1)
    ids = [i // 2 for i in ids]                                   # shared report ids -> dedupe keys
    fm = {}
    for k in range(nl):
        fm.setdefault(ids[k], flags[k] & 8)
        flags[k] = (flags[k] & ~8) | fm[ids[k]]
    db = hs.compile_lit_multi(lits, flags, ids)
    off, largest, typ = _small_write(db)
    assert off and largest == 70 and typ in (6, 7, 17)
    lens = list(range(0, 70)) * 3 + [70, 71, 100, 5000]           # < 70: small-write DFA; >= 70: rose
    data, o, l = synth.ragged_corpus(lens, lits, seed=nl, plant_per_kb=300, alphabet=alphabet + b"AB")
    want = brute.scan_blocks(lits, flags, ids, data, o, l)
    got = ref.scan_sorted(db.ptr, data, o, l, like=want)
    assert np.array_equal(got, want)
    assert want.size > 50


def test_no_small_write_when_the_automaton_would_be_large(hs):
    lits, flags, ids = synth.literal_set(5000)                      # > 12 000 literal bytes
    assert _small_write(hs.compile_lit_multi(lits, flags, ids))[0] == 0
    stream = hs.compile_lit_multi([b"abc"], mode=hs.HS_MODE_STREAM)  # block mode only (src/runtime.c:401)
    assert _small_write(stream)[0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("nl,alphabet,lo,hi,cf", CASES)
def test_device_equals_reference_on_short_buffers(hs, ref, nl, alphabet, lo, hi, cf):
    lits, flags, ids = synth.literal_set(nl, min_len=lo, max_len=hi, seed=nl + 3, caseless_frac=cf, alphabet=alphabet)
    db = hs.compile_lit_multi(lits, flags, ids)
    lens = list(range(0, 70)) * 3 + [70, 71, 100, 5000]
    data, o, l = synth.ragged_corpus(lens, lits, seed=nl, plant_per_kb=300, alphabet=alphabet + b"AB")
    scratch = hs.Scratch(db)
    got = np.sort(hs.scan_blocks(db, data, o, l, scratch), order=["block", "to", "id"])
    assert np.array_equal(got, ref.scan_sorted(db.ptr, data, o, l, like=got))
    # and the engine itself on the device: the DFA's reports are report-program offsets
    bc = db.serialize()[32:]
    off = _small_write(db)[0]
    size = struct.unpack_from("<III", bc, off)[2]
    eng = bytes(bc[off + 64:off + size])
    corpus = hs.Corpus.upload(data, o, l)
    recs, ms = hs.nfa_scan_corpus(eng, corpus)
    want = ref.nfa_exec_blocks(eng, data, o, l, like=recs)
    assert np.array_equal(np.sort(recs, order=["block", "to", "id"]), want) and want.size > 50
    corpus.free()
    scratch.free()
