"""Expression sets larger than one automaton: hs_compile_multi / hs_compile_ext_multi split a set whose character
positions exceed the 512-state model into several engines (McClellan-8 / -16 groups first, then LimEx), each an
outfix of a FULL_ROSE database that holds nothing else (hyperscan_b200/csrc/host/rose_build.cpp partitionEngines,
finishEnginesRose).  Sets that fit one automaton compile exactly as before.

CPU half: the bytes of sets that fit are pinned; the UNMODIFIED reference hs_scan on the split databases reports
what the definition (test_regex._ends) gives, and what the recorded hscollider vectors hold.
GPU half: the device runs every engine of one model in one launch; its answers on every block entry point equal the
reference's."""
import base64
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_golden import COLLIDER_REGEX, _collider_blocks
from test_regex import PATTERNS, SINGLE, TAILS, _data, _ends, _ends_ext

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "ref_layout.json")) as f:
    LAYOUT = json.load(f)
with open(os.path.join(ROOT, "tests", "golden", "regex_set_digests.json")) as f:
    DIGESTS = json.load(f)

# recorded expressions the NFA route takes one at a time: no single-match flag, no extended parameters
POOL = [c for c in COLLIDER_REGEX if "H" not in c["flag_letters"] and not c.get("ext")]


def today_sets():
    """seeded sets that fit one automaton (the parent of this change compiled them): (expressions, flags, ids,
    regex_dfa)"""
    out = []
    for seed in range(16):
        rng = np.random.default_rng(100 + seed)
        n = int(rng.integers(2, 8))
        picks = [POOL[int(i)] for i in rng.choice(len(POOL), size=n, replace=False)]
        pats = [PATTERNS[int(i)] for i in rng.choice(len(PATTERNS), size=4, replace=False)]
        exprs = [base64.b64decode(c["pattern"]) for c in picks] + [p for p, _ in pats]
        flags = [c["hs_flags"] for c in picks] + [f for _, f in pats]
        out.append((exprs, flags, [k % 5 for k in range(len(exprs))], seed % 3 != 2))
    return out


def _compile(hs, exprs, flags, ids, dfa=True, ext=None):
    hs.set_build_option("regex_dfa", 1 if dfa else 0)
    try:
        if ext is None:
            return hs.compile_multi(exprs, flags, ids)
        return hs.compile_ext_multi(exprs, flags, ids, ext)
    finally:
        hs.set_build_option("regex_dfa", 1)


def _digest(db):
    import hashlib
    return hashlib.sha256(db.serialize()).hexdigest()


def split_set(seed, n, dfa=True, shared=False, single=False, ext=False):
    """a seeded set of n expressions (the PATTERNS of test_regex, all of them, and recorded ones) that does not fit
    one automaton.  ids: PATTERNS[k] -> k (or k // 3 when shared), recorded -> 1000 + index.  single: every third
    PATTERNS id is HS_FLAG_SINGLEMATCH.  ext: extended parameters on some PATTERNS."""
    rng = np.random.default_rng(seed)
    big = [c for c in POOL if len(base64.b64decode(c["pattern"])) > 40]
    nb = min(len(big), 12, n - len(PATTERNS))
    picks = [big[int(i)] for i in rng.choice(len(big), size=nb, replace=False)]
    picks += [POOL[int(i)] for i in rng.choice(len(POOL), size=n - len(PATTERNS) - nb, replace=False)]
    exprs, flags, ids, exts = [], [], [], []
    for k, (p, f) in enumerate(PATTERNS):
        i = k // 3 if shared else k
        exprs.append(p)
        flags.append(f | (SINGLE if single and i % 3 == 0 else 0))
        ids.append(i)
        unbounded = ext and (b"+" in p or b"*" in p) and b"\\z" not in p  # (parameters its matches can satisfy)
        exts.append({"min_offset": 3} if unbounded and k % 4 == 1 else {"max_offset": 30} if unbounded and k % 4 == 2
                    else {"min_length": 4} if unbounded and k % 4 == 3 else None)
    order = rng.permutation(len(picks) + len(PATTERNS))
    for c in picks:
        exprs.append(base64.b64decode(c["pattern"]))
        flags.append(c["hs_flags"])
        ids.append(1000 + len(ids))
        exts.append(None)
    exprs, flags, ids, exts = ([x[int(i)] for i in order] for x in (exprs, flags, ids, exts))
    return exprs, flags, ids, (exts if ext else None), dfa


SPLIT = [  # (seed, n, dfa, shared ids, singlematch, extended parameters)
    (1, 50, True, False, False, False), (2, 60, True, True, False, False), (3, 100, True, False, True, False),
    (4, 200, True, True, True, False), (5, 60, False, False, False, False), (6, 80, True, False, False, True),
    (7, 120, False, True, True, False),
]


def _blocks(seed, count=10):
    """buffers for the definition: random ones, ones with the end-anchor tails, one shorter than any match, and an
    empty one"""
    datas = [_data(seed * 100 + k) + TAILS[k % len(TAILS)] for k in range(count)] + [b"a", b""]
    off, buf = [], bytearray()
    for d in datas:
        while len(buf) % 16:
            buf.append(0)
        off.append(len(buf))
        buf += d
    return datas, np.frombuffer(bytes(buf) + b"\0" * 16, dtype=np.uint8), np.array(off, np.uint64), \
        np.array([len(d) for d in datas], np.uint32)


def _want(exprs, flags, ids, exts, datas):
    """(block, id) -> the definition's match ends, for the ids of PATTERNS; single-match ids: the first"""
    want = {}
    for b, d in enumerate(datas):
        for k, (p, f, i) in enumerate(zip(exprs, flags, ids)):
            if i >= 1000:
                continue
            e = exts[k] if exts else None
            ends = _ends_ext(p, f, d, e.get("min_offset", 0), e.get("max_offset"), e.get("min_length", 0)) if e \
                else _ends(p, f, d)
            want[(b, i)] = sorted(set(want.get((b, i), [])) | set(ends))
    for (b, i), v in want.items():
        if v and any(f & SINGLE for f, j in zip(flags, ids) if j == i):
            want[(b, i)] = v[:1]
    return want


def _check_definition(recs, want):
    for (b, i), v in want.items():
        got = [int(r["to"]) for r in recs if r["block"] == b and r["id"] == i]
        assert got == v, (b, i, got, v)


def test_sets_that_fit_one_automaton_keep_their_bytes(hs):
    sets = today_sets()
    assert len(sets) == len(DIGESTS["today"])
    for (exprs, flags, ids, dfa), want in zip(sets, DIGESTS["today"]):
        db = _compile(hs, exprs, flags, ids, dfa)
        assert db.info().runtime_impl == 2        # one engine, as before
        assert _digest(db) == want


@pytest.mark.parametrize("si", range(len(SPLIT)))
def test_reference_on_split_sets_equals_definition(hs, ref, si):
    exprs, flags, ids, exts, dfa = split_set(*SPLIT[si])
    db = _compile(hs, exprs, flags, ids, dfa, exts)
    engines = db.engines()
    assert db.info().runtime_impl == 0 and len(engines) > 1
    assert dfa or all(m.startswith("LimEx") for m, _ in engines)
    datas, data, off, ln = _blocks(si)
    recs = ref.scan_sorted(db.ptr, data, off, ln)
    _check_definition(recs, _want(exprs, flags, ids, exts, datas))


def test_split_sets_mix_every_engine_model(hs):
    models = set()
    for row in SPLIT:
        exprs, flags, ids, exts, dfa = split_set(*row)
        models |= {m for m, _ in _compile(hs, exprs, flags, ids, dfa, exts).engines()}
    assert {"McClellan-8", "McClellan-16"} <= models and any(m.startswith("LimEx") for m in models)


def test_one_id_raised_by_two_engines_at_one_offset_is_reported_once(hs, ref):
    """the same expression twice under one id, in a set that splits: two engines raise the id at the same end, and
    the set-wide dedupe key delivers it once"""
    exprs, flags, ids, _, _ = split_set(9, 60)
    exprs, flags, ids = [rb"qz+y"] + exprs + [rb"qz+y"], [0] + flags + [0], [77] + ids + [77]
    db = _compile(hs, exprs, flags, ids)
    assert len(db.engines()) > 1
    data = np.frombuffer(b"aqzzy qzy" + b"\0" * 16, np.uint8)
    recs = ref.scan_sorted(db.ptr, data, np.array([0], np.uint64), np.array([9], np.uint32))
    assert [int(r["to"]) for r in recs if r["id"] == 77] == [5, 9]


@pytest.mark.skipif(os.environ.get("HS_REF_RECORD") == "1", reason="18 M reference records: too many to record")
def test_all_recorded_expressions_in_one_database(hs, ref):
    """all 1 128 recorded regex patterns of hscollider in ONE database, id = case id: on every recorded corpus the
    reference reports, under the corpus' own id, exactly the recorded ends (single-match: one of them)"""
    import oracle.ref as r
    if not r.live():
        pytest.skip("the reference's answer (18 M records) is checked where oracle/_ref is built")
    db, blocks, data, off, ln = all_recorded(hs)
    _check_recorded(r.scan_sorted(db.ptr, data, off, ln), blocks)


def all_recorded(hs):
    cases = COLLIDER_REGEX
    db = hs.compile_ext_multi([base64.b64decode(c["pattern"]) for c in cases], [c["hs_flags"] for c in cases],
                              [c["id"] for c in cases], [c.get("ext") for c in cases])
    blocks, datas = [], []
    for c in cases:
        _, _, _, ends = _collider_blocks(c)
        for k, want in zip(c["corpora"], ends):
            datas.append(base64.b64decode(k["data"]))
            blocks.append((c, want))
    off, buf = [], bytearray()
    for d in datas:
        while len(buf) % 16:
            buf.append(0)
        off.append(len(buf))
        buf += d
    return db, blocks, np.frombuffer(bytes(buf) + b"\0" * 16, np.uint8), np.array(off, np.uint64), \
        np.array([len(d) for d in datas], np.uint32)


def _check_recorded(recs, blocks):
    ids = recs["id"].astype(np.int64)
    blk = recs["block"].astype(np.int64)
    for b, (c, want) in enumerate(blocks):
        lo, hi = np.searchsorted(blk, b), np.searchsorted(blk, b, side="right")
        tos = [int(t) for t, i in zip(recs["to"][lo:hi], ids[lo:hi]) if i == c["id"]]
        if "H" in c["flag_letters"]:
            assert (len(tos) == 1 and tos[0] in want) if want else not tos, (c["id"], b, tos, want)
        else:
            assert tos == want, (c["id"], b, tos, want)


def test_split_compile_is_deterministic(hs):
    exprs, flags, ids, _, _ = split_set(4, 200, shared=True, single=True)
    a = _digest(_compile(hs, exprs, flags, ids))
    assert a == _digest(_compile(hs, exprs, flags, ids))
    code = ("import sys, hashlib; sys.path[:0] = [%r, %r]\n"
            "from hyperscan_b200 import capi\nimport test_regex_sets as t\n"
            "capi.LIB_PATH = %r\n"
            "e, f, i, _, _ = t.split_set(4, 200, shared=True, single=True)\n"
            "print(hashlib.sha256(capi.compile_multi(e, f, i).serialize()).hexdigest())"
            % (ROOT, os.path.join(ROOT, "tests"), hs.LIB_PATH))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=ROOT)
    assert out.stdout.strip() == a


def test_engine_listing_reads_the_layout(hs):
    assert (hs._ROSE_QUEUE_COUNT, hs._ROSE_NFA_INFO, hs._NFA_INFO_SIZE, hs._NFA_TYPE, hs._NFA_POSITIONS) == \
        (LAYOUT["RoseEngine.queueCount"], LAYOUT["RoseEngine.nfaInfoOffset"], LAYOUT["sizeof(NfaInfo)"],
         LAYOUT["NFA.type"], LAYOUT["NFA.nPositions"])
    assert [m for m, _ in _compile(hs, [rb"ab+c"], [0], [1]).engines()] == ["McClellan-8"]
    assert [m for m, _ in _compile(hs, [rb"ab+c"], [0], [1], dfa=False).engines()] == ["LimEx-32"]


def test_too_large_expression_and_other_modes_stay_refused(hs):
    exprs, flags, ids, _, _ = split_set(1, 40)
    with pytest.raises(hs.HsError, match="too large"):
        hs.compile_multi(exprs + [rb"[a-z]{600}x+"], flags + [0], ids + [5])
    with pytest.raises(hs.HsError, match="block mode only"):
        hs.compile_multi(exprs, flags, ids, mode=hs.HS_MODE_STREAM)


# ---- GPU half ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("si", range(len(SPLIT)))
def test_device_on_split_sets_equals_reference(hs, ref, si):
    exprs, flags, ids, exts, dfa = split_set(*SPLIT[si])
    db = _compile(hs, exprs, flags, ids, dfa, exts)
    datas, data, off, ln = _blocks(50 + si)  # (other inputs than the CPU half's: the store keeps both answers)
    scratch = hs.Scratch(db)
    got = np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"])
    want = ref.scan_sorted(db.ptr, data, off, ln, like=got)
    assert np.array_equal(got, want)
    _check_definition(got, _want(exprs, flags, ids, exts, datas))
    # hs_scan, one buffer at a time: callbacks in non-decreasing `to`
    for b, d in enumerate(datas):
        out = []
        rc, _ = hs.scan(db, d, scratch, on_event=lambda i, frm, to, fl: out.append((to, i)) or 0)
        assert rc == 0
        assert [t for t, _ in out] == sorted(t for t, _ in out)
        assert sorted((i, t) for t, i in out) == sorted((int(r["id"]), int(r["to"])) for r in want[want["block"] == b])
    # the resident corpus
    corpus = hs.Corpus.upload(data, off, ln)
    res = np.sort(hs.scan_corpus(db, corpus, scratch), order=["block", "to", "id"])
    assert np.array_equal(res, want)


@pytest.mark.gpu
def test_device_ring_growth_and_termination_on_split_sets(hs, ref):
    exprs, flags, ids, _, dfa = split_set(*SPLIT[3])
    db = _compile(hs, exprs, flags, ids, dfa)
    datas, data, off, ln = _blocks(11, count=40)
    hs.set_runtime_option("initial_ring", 64)
    try:
        scratch = hs.Scratch(db)
        got = np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"])
    finally:
        hs.set_runtime_option("initial_ring", 0)
    assert got.size > 64 * 8
    assert np.array_equal(got, ref.scan_sorted(db.ptr, data, off, ln, like=got))
    # termination: the callback stops the scan after its third match (which three at a tied offset is not
    # part of the API; their offsets are)
    d = datas[0] + datas[1]
    full = []
    hs.scan(db, d, scratch, on_event=lambda i, frm, to, fl: full.append(to) or 0)
    seen = []
    rc, _ = hs.scan(db, d, scratch, on_event=lambda i, frm, to, fl: seen.append(to) or (1 if len(seen) == 3 else 0))
    assert rc == hs.HS_SCAN_TERMINATED and seen == full[:3]


@pytest.mark.gpu
def test_device_runs_every_engine_model_of_a_split_set(hs, ref):
    """one database whose engines are McClellan-8, McClellan-16 and LimEx of several sizes: every instantiation of
    the engine-table launch runs, each over several engines"""
    exprs, flags, ids, _, _ = split_set(4, 200, shared=True, single=True)
    e2, f2, i2, _, _ = split_set(7, 120, dfa=False)
    db = _compile(hs, exprs, flags, ids)
    models = [m for m, _ in db.engines()]
    assert {"McClellan-8", "McClellan-16"} <= set(models) and any(m.startswith("LimEx") for m in models)
    datas, data, off, ln = _blocks(13, count=30)
    for d in (db, _compile(hs, e2, f2, i2, False)):
        scratch = hs.Scratch(d)
        got = np.sort(hs.scan_blocks(d, data, off, ln, scratch), order=["block", "to", "id"])
        assert np.array_equal(got, ref.scan_sorted(d.ptr, data, off, ln, like=got))


@pytest.mark.gpu
@pytest.mark.parametrize("field,value", [("fmatcherOffset", 64), ("leftfixBeginQueue", 1), ("eodProgramOffset", 64),
                                         ("activeLeftCount", 1)])
def test_device_refuses_more_than_outfixes(hs, field, value):
    """a split database patched to carry anything besides outfixes is refused when the scratch is allocated"""
    import ctypes as C
    exprs, flags, ids, _, _ = split_set(*SPLIT[0][:2])
    db = _compile(hs, exprs, flags, ids)
    p = db.ptr.value
    length, bc = C.c_uint32.from_address(p + 8).value, C.c_uint32.from_address(p + 36).value
    C.c_uint32.from_address(p + bc + LAYOUT["RoseEngine." + field]).value = value
    C.c_uint32.from_address(p + 24).value = _crc32c(C.string_at(p + bc, length))
    with pytest.raises(hs.HsError) as e:
        hs.Scratch(db)
    assert e.value.code == hs.HS_ARCH_ERROR


def _crc32c(b):
    """CRC32C, initial value 0, no final xor (the database header's checksum)"""
    crc = 0
    for x in b:
        crc ^= x
        for _ in range(8):
            crc = (crc >> 1) ^ (0x82F63B78 & -(crc & 1))
    return crc


@pytest.mark.gpu
def test_device_all_recorded_expressions_in_one_database(hs, real_gpu):
    """the 1 128-pattern database on the device, against the recorded hscollider ends directly"""
    db, blocks, data, off, ln = all_recorded(hs)
    scratch = hs.Scratch(db)
    _check_recorded(np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"]), blocks)
