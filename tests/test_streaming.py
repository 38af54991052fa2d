"""Streaming mode for literal databases (SURVEY.md section 8f rank 2, the
pure-literal part): our compiler's HS_MODE_STREAM databases drive the UNMODIFIED
reference stream runtime (hs_open_stream / hs_scan_stream / hs_close_stream) to
the matches the definition demands over any cut of the data into writes; the
C restatement reproduces the reference's callbacks, order and termination; on
the GPU box the device stream API does the same."""
import ctypes as C

import numpy as np
import pytest

from hyperscan_b200 import synth
import oracle.brute as brute
import oracle.port as port


def make(hs, nl, seed, lo=2):
    lits, flags, ids = synth.literal_set(nl, min_len=1 if nl < 10 else lo, max_len=8, seed=seed,
                                         caseless_frac=0.2, alphabet=b"abcdef", singlematch_frac=0.15)
    ids = [i // 2 for i in ids]
    fm = {}
    for k in range(nl):
        fm.setdefault(ids[k], flags[k] & 8)
        flags[k] = (flags[k] & ~8) | fm[ids[k]]
    db = hs.compile_lit_multi(lits, flags, ids, mode=hs.HS_MODE_STREAM)
    data, off, ln = synth.ragged_corpus([7000], lits, seed=seed + 1, plant_per_kb=15, alphabet=b"abcdefAB")
    return lits, flags, ids, db, data, off, ln


def cuts_of(n, seed, k=40):
    rng = np.random.default_rng(seed)
    cuts = sorted(set(rng.integers(0, n, size=k).tolist() + [0, n, 1, 2, 3, n - 1]))
    return np.diff(np.array(cuts)).astype(np.uint32)


@pytest.mark.parametrize("nl", [1, 6, 40, 300, 1500])
def test_streaming_databases_on_reference_runtime(hs, ref, nl):
    lits, flags, ids, db, data, off, ln = make(hs, nl, nl)
    want = sorted((int(r["id"]), int(r["to"])) for r in brute.scan_blocks(lits, flags, ids, data, off, ln))
    for seed in (1, 2):
        wl = cuts_of(data.size, seed)
        a, ea = ref.stream_collect(db.ptr, data, wl)
        assert ea == 0 and sorted((int(r["id"]), int(r["to"])) for r in a) == want
        b, eb = port.stream_collect(db.ptr, data, wl)
        assert eb == 0 and np.array_equal(a, b)          # same callbacks in the same order
        a, ea = ref.stream_collect(db.ptr, data, wl, stop_after=4)
        b, eb = port.stream_collect(db.ptr, data, wl, stop_after=4)
        assert ea == eb == hs.HS_SCAN_TERMINATED and np.array_equal(a, b)
    # byte-at-a-time writes
    small = data[:300]
    a, _ = ref.stream_collect(db.ptr, small, np.ones(300, dtype=np.uint32))
    b, _ = port.stream_collect(db.ptr, small, np.ones(300, dtype=np.uint32))
    assert np.array_equal(a, b)


def test_stream_compile_rules(hs, ref):
    import ctypes
    db = hs.compile_lit_multi([b"abcdefgh", b"xy"], mode=hs.HS_MODE_STREAM)
    sz = ctypes.c_size_t()
    assert hs.lib().hs_stream_size(db.ptr, ctypes.byref(sz)) == 0
    assert sz.value == 16 + 1 + 1 + 7            # struct hs_stream + status + groups + history (src/runtime.c:1058)
    assert ref.stream_size(db.ptr) == (0, sz.value)
    info = ctypes.c_void_p()
    assert hs.lib().hs_database_info(db.ptr, ctypes.byref(info)) == 0
    assert b"Mode: STREAM" in ctypes.string_at(info)
    with pytest.raises(hs.HsError) as e:          # long literals need the long-literal table
        hs.compile_lit_multi([b"abcdefghi"], mode=hs.HS_MODE_STREAM)
    assert "long literal" in e.value.message
    with pytest.raises(hs.HsError):               # one (and only one) of BLOCK / STREAM / VECTORED
        hs.compile_lit_multi([b"abc"], mode=hs.HS_MODE_VECTORED | hs.HS_MODE_STREAM)


@pytest.mark.gpu
@pytest.mark.parametrize("nl", [1, 6, 40, 300, 1500])
def test_device_stream_api_equals_reference(hs, ref, nl):
    lits, flags, ids, db, data, off, ln = make(hs, nl, nl + 50)
    scratch = hs.Scratch(db)
    for seed in (3, 4):
        wl = cuts_of(data.size, seed, k=25)
        want, err = ref.stream_collect(db.ptr, data, wl)
        st = hs.Stream(db)
        got, pos = [], 0
        for i, n in enumerate(wl):
            rc, out = st.scan(data[pos:pos + int(n)], scratch)
            assert rc == hs.HS_SUCCESS
            got += [(i, idv, to) for (idv, to) in out]
            pos += int(n)
        assert st.close(scratch) == hs.HS_SUCCESS
        # per write the API promises non-decreasing `to`; compare as sets per write
        exp = sorted((int(r["block"]), int(r["id"]), int(r["to"])) for r in want)
        assert sorted(got) == exp
        tos = [t for (_, _, t) in got]
        assert tos == sorted(tos)


@pytest.mark.gpu
def test_device_stream_termination_copy_reset(hs, ref):
    lits, flags, ids, db, data, off, ln = make(hs, 40, 99)
    scratch = hs.Scratch(db)
    st = hs.Stream(db)
    rc, out = st.scan(data[:3000], scratch, stop_after=3)
    assert rc == hs.HS_SCAN_TERMINATED and len(out) == 3
    rc, out = st.scan(data[3000:4000], scratch)           # broken stream stays broken
    assert rc == hs.HS_SCAN_TERMINATED and out == []
    st.reset(scratch)
    rc, a = st.scan(data[:2000], scratch)
    assert rc == 0
    twin = st.copy()                                       # same state, independent afterwards
    rc, b1 = st.scan(data[2000:5000], scratch)
    rc, b2 = twin.scan(data[2000:5000], scratch)
    assert b1 == b2 and len(b1) > 0
    want, _ = ref.stream_collect(db.ptr, data[:5000], np.array([2000, 3000], dtype=np.uint32))
    assert sorted(a + b1) == sorted((int(r["id"]), int(r["to"])) for r in want)
    L = hs.lib()
    assert L.hs_scan_stream(None, b"x", 1, 0, scratch.ptr, hs.MATCH_CB(), None) == hs.HS_INVALID
    blk = hs.compile_lit_multi([b"abc"])                  # block database: wrong mode for streams
    p = C.c_void_p()
    assert L.hs_open_stream(blk.ptr, 0, C.byref(p)) == hs.HS_DB_MODE_ERROR
    rc, _ = hs.scan(db, b"abc", scratch)                  # and a stream database is refused by hs_scan
    assert rc == hs.HS_DB_MODE_ERROR
    st.close(scratch)
    twin.close(scratch)


@pytest.mark.gpu
@pytest.mark.parametrize("nl,wlen,fat", [(40, 64, 0), (300, 1024, 0), (1, 33, 0), (80, 200, 1)])
def test_stream_set_equals_per_stream_reference(hs, ref, nl, wlen, fat):
    """hs_b200_streams_scan (state in HBM) == one reference stream per stream.
    fat: compiled for an AVX2 platform -> 16-bucket Teddy (FK_BYTE64 first stage)."""
    lits, flags, ids = synth.literal_set(nl, min_len=2, max_len=8, seed=nl + 7, caseless_frac=0.2,
                                         alphabet=b"abcdef")
    plat = None
    if fat:
        if ref.best_isa() == "corei7":
            pytest.skip("the reference build on this host has no fat Teddy")
        plat = C.byref(hs.PlatformInfo(0, hs.HS_CPU_FEATURES_AVX2, 0, 0))
    db = hs.compile_lit_multi(lits, flags, ids, mode=hs.HS_MODE_STREAM, platform=plat)
    if fat:
        assert 3 <= db.info().engine_id <= 10
    scratch = hs.Scratch(db)
    nstreams = 257
    sset = hs.StreamSet(db, nstreams)
    rng = np.random.default_rng(nl)
    rounds = []
    for rnd in range(4):
        if rnd == 2:   # a ragged round (some streams get nothing)
            ln = rng.integers(0, wlen + 1, size=nstreams).astype(np.uint32)
        else:
            ln = np.full(nstreams, wlen, dtype=np.uint32)
        data, off, _ = synth.ragged_corpus([int(x) for x in ln], lits, seed=100 * nl + rnd, plant_per_kb=30,
                                           align=1, alphabet=b"abcdefAB")
        rounds.append((data, off, ln))
    got = []
    for rnd, (data, off, ln) in enumerate(rounds):
        recs = sset.scan(data, off, ln, scratch)
        got.append(recs)
    sset.close()
    # reference: every stream on its own, writes = its slice of every round
    for s in rng.choice(nstreams, size=40, replace=False).tolist() + [0, nstreams - 1]:
        pieces = [d[int(o[s]):int(o[s]) + int(l[s])] for (d, o, l) in rounds]
        cat = np.concatenate(pieces) if sum(p.size for p in pieces) else np.zeros(0, np.uint8)
        wl = np.array([p.size for p in pieces], dtype=np.uint32)
        want, err = ref.stream_collect(db.ptr, cat, wl)
        assert err == 0
        exp = sorted((int(r["block"]), int(r["id"]), int(r["to"])) for r in want)
        mine = []
        for rnd, recs in enumerate(got):
            sel = recs[recs["block"] == s]
            mine += [(rnd, int(r["id"]), int(r["to"])) for r in sel]
        assert sorted(mine) == exp, (s, sorted(mine)[:5], exp[:5])


@pytest.mark.gpu
def test_stream_set_rejects_what_it_cannot_do(hs):
    blk = hs.compile_lit_multi([b"abc"])
    with pytest.raises(hs.HsError) as e:
        hs.StreamSet(blk, 4)
    assert e.value.code == hs.HS_DB_MODE_ERROR
    single = hs.compile_lit_multi([b"abc"], flags=[8], mode=hs.HS_MODE_STREAM)
    with pytest.raises(hs.HsError) as e:
        hs.StreamSet(single, 4)
    assert e.value.code == hs.HS_ARCH_ERROR


@pytest.mark.gpu
def test_stream_compress_expand_round_trip(hs, ref):
    """hs_compress_stream / hs_expand_stream / hs_reset_and_expand_stream
    (src/runtime.c:1177-1282): a stream expanded from the bytes continues exactly
    as the compressed one; the whole run equals the reference's uninterrupted stream."""
    lits, flags, ids, db, data, off, ln = make(hs, 40, 123)
    scratch = hs.Scratch(db)
    st = hs.Stream(db)
    rc, a = st.scan(data[:2500], scratch)
    assert rc == 0
    blob = st.compress()
    assert len(blob) >= 32 and st.compress() == blob                  # deterministic
    L = hs.lib()
    used = C.c_size_t()
    small = C.create_string_buffer(8)
    assert L.hs_compress_stream(st.ptr, small, 8, C.byref(used)) == hs.HS_INSUFFICIENT_SPACE
    assert used.value == len(blob)
    assert L.hs_compress_stream(st.ptr, None, 8, C.byref(used)) == hs.HS_INVALID
    twin = hs.Stream.expand(db, blob)
    rc, b1 = st.scan(data[2500:6000], scratch)
    rc, b2 = twin.scan(data[2500:6000], scratch)
    assert b1 == b2 and len(b1) > 0
    want, _ = ref.stream_collect(db.ptr, data[:6000], np.array([2500, 3500], dtype=np.uint32))
    assert sorted(a + b1) == sorted((int(r["id"]), int(r["to"])) for r in want)
    # reset_and_expand rewinds an existing stream to the compressed point
    assert twin.reset_and_expand(blob, scratch) == 0
    rc, b3 = twin.scan(data[2500:6000], scratch)
    assert b3 == b1
    # a damaged buffer is refused and leaves the stream untouched
    bad = bytearray(blob)
    bad[0] ^= 0xff
    assert twin.reset_and_expand(bytes(bad), scratch) == hs.HS_INVALID
    assert twin.reset_and_expand(blob[:-1], scratch) == hs.HS_INVALID
    p = C.c_void_p()
    assert L.hs_expand_stream(db.ptr, C.byref(p), bytes(bad), len(bad)) == hs.HS_INVALID
    other = hs.compile_lit_multi([b"zz"], mode=hs.HS_MODE_STREAM)       # another database's stream bytes
    assert L.hs_expand_stream(other.ptr, C.byref(p), blob, len(blob)) == hs.HS_INVALID
    blk = hs.compile_lit_multi([b"zz"])
    assert L.hs_expand_stream(blk.ptr, C.byref(p), blob, len(blob)) == hs.HS_DB_MODE_ERROR
    rc, b4 = twin.scan(data[6000:7000], scratch)
    rc, b5 = st.scan(data[6000:7000], scratch)
    assert b4 == b5
    st.close(scratch)
    twin.close(scratch)
