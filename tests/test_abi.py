"""The C-ABI library loads on a CPU-only box and exports every symbol
include/hs_b200.h declares; argument checks and error codes follow the
reference (unit/hyperscan/arg_checks.cpp, serialize.cpp)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle.port as port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "hs_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set(re.findall(r"\b(hs_[a-z0-9_]+)\s*\(", src))
    return sorted(n for n in names if not n.endswith("_t"))


def test_exports_every_declared_symbol(hs):
    L = hs.lib()
    names = declared_functions()
    assert len(names) >= 40
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_version_and_error_codes(hs):
    assert hs.lib().hs_version().startswith(b"5.4.2")
    assert (hs.HS_SUCCESS, hs.HS_INVALID, hs.HS_SCAN_TERMINATED, hs.HS_UNKNOWN_ERROR) == (0, -1, -3, -13)


def test_compile_arg_checks(hs):
    L = hs.lib()
    db = C.c_void_p()
    err = C.POINTER(hs.CompileError)()
    # NULL expression (unit/hyperscan/arg_checks.cpp CompileNullExpression...)
    assert L.hs_compile(None, 0, hs.HS_MODE_BLOCK, None, C.byref(db), C.byref(err)) == hs.HS_COMPILER_ERROR
    assert err and b"NULL" in err.contents.message
    L.hs_free_compile_error(err)
    # no mode / two modes / bad mode
    for mode in (0, hs.HS_MODE_BLOCK | hs.HS_MODE_STREAM, 1 << 10):
        err = C.POINTER(hs.CompileError)()
        assert L.hs_compile(b"foo", 0, mode, None, C.byref(db), C.byref(err)) == hs.HS_COMPILER_ERROR
        assert err.contents.expression == -1
        L.hs_free_compile_error(err)
    # NULL db
    err = C.POINTER(hs.CompileError)()
    assert L.hs_compile(b"foo", 0, hs.HS_MODE_BLOCK, None, None, C.byref(err)) == hs.HS_COMPILER_ERROR
    L.hs_free_compile_error(err)
    # NULL error pointer
    assert L.hs_compile(b"foo", 0, hs.HS_MODE_BLOCK, None, C.byref(db), None) == hs.HS_COMPILER_ERROR
    # unsupported construct reports the expression index
    with pytest.raises(hs.HsError) as e:
        hs.compile_multi([b"abc", rb"a.*(?=b)b"])        # look-around is beyond both the literal and the NFA route
    assert e.value.expression == 1
    with pytest.raises(hs.HsError):
        hs.compile_lit_multi([b""])
    with pytest.raises(hs.HsError):
        hs.compile_multi([b"abc"], flags=[1 << 20])


def test_regex_literal_escapes(hs, ref):
    db = hs.compile_multi([rb"a\.b\x41\n", b"xyz"], flags=[0, hs.HS_FLAG_CASELESS], ids=[3, 4])
    data = b"..a.bA\n..XyZ"
    got = ref.scan_sorted(db.ptr, data, [0], [len(data)])
    assert [(int(r["id"]), int(r["to"])) for r in got] == [(3, 7), (4, 12)]


def test_serialize_roundtrip_and_errors(hs, ref):
    L = hs.lib()
    db = hs.compile_lit_multi([b"hatstand", b"teakettle", b"badgerbrush"], ids=[1, 2, 3])
    blob = db.serialize()
    size = C.c_size_t()
    assert L.hs_serialized_database_size(blob, len(blob), C.byref(size)) == 0
    dsz = C.c_size_t()
    assert L.hs_database_size(db.ptr, C.byref(dsz)) == 0 and dsz.value == size.value
    info = C.c_void_p()
    assert L.hs_serialized_database_info(blob, len(blob), C.byref(info)) == 0
    assert b"Version: 5.4.2" in C.string_at(info) and b"Mode: BLOCK" in C.string_at(info)
    db2 = hs.Database.deserialize(blob)
    assert db2.serialize() == blob
    data = b"...hatstand...teakettle"
    a = ref.scan_sorted(db.ptr, data, [0], [len(data)])
    b = ref.scan_sorted(db2.ptr, data, [0], [len(data)])
    assert a.size == 2 and (a == b).all()
    # deserialize_at at 16 alignments (unit/hyperscan/serialize.cpp)
    for al in (8, 16, 24, 40, 56):
        raw = C.create_string_buffer(size.value + 128)
        base = (C.addressof(raw) + 63) // 64 * 64 + al
        assert L.hs_deserialize_database_at(blob, len(blob), C.c_void_p(base)) == 0
        r = ref.scan_sorted(base, data, [0], [len(data)])
        assert (r == a).all()
    assert L.hs_deserialize_database_at(blob, len(blob), C.c_void_p(base + 1)) == hs.HS_BAD_ALIGN
    out = C.c_void_p()
    # corrupt bytecode -> CRC failure; truncated; bad magic; bad version
    bad = bytearray(blob)
    bad[200] ^= 0xFF
    assert L.hs_deserialize_database(bytes(bad), len(bad), C.byref(out)) == hs.HS_INVALID
    assert L.hs_deserialize_database(blob, len(blob) - 1, C.byref(out)) == hs.HS_INVALID
    bad = bytearray(blob)
    bad[0] = 0
    assert L.hs_deserialize_database(bytes(bad), len(bad), C.byref(out)) == hs.HS_INVALID
    bad = bytearray(blob)
    bad[5] ^= 1
    assert L.hs_deserialize_database(bytes(bad), len(bad), C.byref(out)) == hs.HS_DB_VERSION_ERROR
    assert L.hs_deserialize_database(None, 10, C.byref(out)) == hs.HS_INVALID
    ss = C.c_size_t()
    assert L.hs_stream_size(db.ptr, C.byref(ss)) == hs.HS_DB_MODE_ERROR


def test_reference_accepts_our_database_container(hs, ref):
    """The reference's own hs_deserialize/hs_database_info read our container."""
    db = hs.compile_lit_multi([b"needle"])
    rc, info, r = ref.read_container(db.serialize(), b"xxneedlexx")
    assert rc == 0
    assert "5.4.2" in info and "BLOCK" in info
    assert [(int(x["id"]), int(x["to"])) for x in r] == [(0, 8)]


def test_no_gpu_fails_loudly(hs):
    """Without a CUDA device the scan path refuses to run (no CPU fallback)."""
    if hs.lib().hs_valid_platform() == 0:
        pytest.skip("a CUDA device is present")
    db = hs.compile_lit_multi([b"abc"])
    with pytest.raises(hs.HsError) as e:
        hs.Scratch(db)
    assert e.value.code == hs.HS_ARCH_ERROR


def test_allocator_hooks(hs):
    L = hs.lib()
    calls = {"a": 0, "f": 0}
    libc = C.CDLL(None)
    libc.malloc.restype = C.c_void_p
    libc.malloc.argtypes = [C.c_size_t]
    libc.free.argtypes = [C.c_void_p]
    AT = C.CFUNCTYPE(C.c_void_p, C.c_size_t)
    FT = C.CFUNCTYPE(None, C.c_void_p)

    def a(n):
        calls["a"] += 1
        return libc.malloc(n)

    def f(p):
        calls["f"] += 1
        libc.free(p)

    ac, fc = AT(a), FT(f)
    L.hs_set_database_allocator.argtypes = [AT, FT]
    assert L.hs_set_database_allocator(ac, fc) == 0
    try:
        db = hs.compile_lit_multi([b"abc"])
        del db
        assert calls["a"] == 1 and calls["f"] == 1
        # misaligned allocator -> HS_COMPILER_ERROR, like the reference's HS_BAD_ALLOC path
        bad = AT(lambda n: libc.malloc(n + 8) + 4)
        nofree = FT(lambda p: None)  # keep alive while installed
        L.hs_set_database_allocator(bad, nofree)
        with pytest.raises(hs.HsError):
            hs.compile_lit_multi([b"abc"])
    finally:
        L.hs_set_database_allocator(AT(), FT())


def test_expression_info(hs):
    # unit/hyperscan/expr_info.cpp: widths of plain literals
    class Info(C.Structure):
        _fields_ = [("min_width", C.c_uint), ("max_width", C.c_uint), ("unordered_matches", C.c_char),
                    ("matches_at_eod", C.c_char), ("matches_only_at_eod", C.c_char)]
    L = hs.lib()
    L.hs_expression_info.argtypes = [C.c_char_p, C.c_uint, C.POINTER(C.POINTER(Info)),
                                     C.POINTER(C.POINTER(hs.CompileError))]
    info = C.POINTER(Info)()
    err = C.POINTER(hs.CompileError)()
    assert L.hs_expression_info(rb"foo\.bar", 0, C.byref(info), C.byref(err)) == 0
    assert (info.contents.min_width, info.contents.max_width) == (7, 7)
    assert info.contents.unordered_matches == b"\0" and info.contents.matches_at_eod == b"\0"
    C.CDLL(None).free(info)
    assert L.hs_expression_info(b"foo.*bar", 0, C.byref(info), C.byref(err)) == 0      # NFA route: widths known
    assert (info.contents.min_width, info.contents.max_width) == (6, 0xffffffff)
    C.CDLL(None).free(info)
    assert L.hs_expression_info(rb"foo.*(?!x)bar", 0, C.byref(info), C.byref(err)) == hs.HS_COMPILER_ERROR
    assert err and err.contents.message
    L.hs_free_compile_error(err)
    assert L.hs_expression_info(None, 0, C.byref(info), C.byref(err)) == hs.HS_COMPILER_ERROR
    L.hs_free_compile_error(err)


FINITE = [
    (rb"(foo){2,3}bar", 0), (rb"x?(foo){2,3}bar", 0), (rb"[fg]oo|ba[rz]", 0), (rb"abc|bc|c", 0),
    (rb"a{3}", 0), (rb"a{3}", 1), (rb"(ab|ba){2}", 0), (rb"[a-c]{2}d", 1), (rb"(?:ab)?cd", 0),
    (rb"[]a]b", 0), (rb"[a\-c]b", 0), (rb"[A-C-E]", 0), (rb"a[\x62\x63]", 0), (rb"((a|b)(c|d)){2}", 0),
    (rb"ab{0,2}c", 0), (rb"(a|ab)(c|bcd)", 0),
]


@pytest.mark.parametrize("pat,caseless", [(p, c) for (p, c) in FINITE], ids=[p.decode() for (p, _) in FINITE])
def test_finite_language_expressions(hs, ref, pat, caseless):
    """hs_compile accepts expressions that denote a finite set of literals (groups,
    alternation, classes, bounded repeats): every end offset where Python's re
    (PCRE-compatible for these constructs) finds a match ending -- and no other --
    is reported once by the reference runtime scanning our database."""
    import re
    rng = np.random.default_rng(len(pat))
    data = bytes(rng.choice(np.frombuffer(b"abcdfoorzABC-]", dtype=np.uint8), size=700).tolist())
    data += b"foofoobar xfoofoofoobar abccd ab]b a-b bab"
    rx = re.compile(b"(?:" + pat + rb")\Z", re.I if caseless else 0)
    want = [e for e in range(1, len(data) + 1) if rx.search(data[:e])]
    db = hs.compile_multi([pat], flags=[hs.HS_FLAG_CASELESS if caseless else 0], ids=[9])
    got = ref.scan_sorted(db.ptr, data, [0], [len(data)])
    assert [int(r["to"]) for r in got] == want and all(int(r["id"]) == 9 for r in got)
    b = port.scan_sorted(db.ptr, np.frombuffer(data, dtype=np.uint8), np.array([0], dtype=np.uint64),
                         np.array([len(data)], dtype=np.uint32))
    assert np.array_equal(b, got)


def test_finite_language_limits_and_errors(hs):
    # (expressions with unbounded repeats, ".", "^", negated classes or class escapes are no longer errors:
    # they compile through the NFA route, tests/test_regex.py)
    for bad, why in [(rb"a*", "empty buffer"), (rb"a$b", "Embedded end anchors"), (rb"(?<=a)b", "Look-around"), (rb"a|", "empty buffer"),
                     (rb"(ab", "parenthesis"), (rb"ab)", "parentheses"), (rb"(a)\1", "Escape sequence"),
                     (rb"a??", "empty buffer"), (rb"[[:nope:]]", "POSIX"), (rb"a{3,2}", "min > max"),
                     (rb"*a", "nothing to repeat"), (rb"[ab", "Unterminated"), (rb"[a-z]{1001}x+", "too large")]:
        with pytest.raises(hs.HsError) as e:
            hs.compile_multi([b"ok", bad])
        assert why in e.value.message, (bad, e.value.message)
        assert e.value.expression == 1
    # widths reported by hs_expression_info follow the language
    class Info(C.Structure):
        _fields_ = [("min_width", C.c_uint), ("max_width", C.c_uint), ("unordered_matches", C.c_char),
                    ("matches_at_eod", C.c_char), ("matches_only_at_eod", C.c_char)]
    L = hs.lib()
    L.hs_expression_info.argtypes = [C.c_char_p, C.c_uint, C.POINTER(C.POINTER(Info)),
                                     C.POINTER(C.POINTER(hs.CompileError))]
    info = C.POINTER(Info)()
    err = C.POINTER(hs.CompileError)()
    assert L.hs_expression_info(rb"x?(foo){2,3}bar", 0, C.byref(info), C.byref(err)) == 0
    assert (info.contents.min_width, info.contents.max_width) == (9, 13)
    C.CDLL(None).free(info)
    assert L.hs_expression_info(rb"ab+c?|x{2,4}y", 0, C.byref(info), C.byref(err)) == 0
    assert (info.contents.min_width, info.contents.max_width) == (2, 0xffffffff)
    C.CDLL(None).free(info)
