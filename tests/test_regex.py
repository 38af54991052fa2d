"""Expressions that are not a finite set of literals: hs_compile* builds their position
(Glushkov) automaton as ONE LimEx-32 NFA and wraps it in a single-outfix database
(hyperscan_b200/csrc/host/regex_nfa.cpp, rose_build.cpp buildRegexRose).

CPU half: the UNMODIFIED reference hs_scan scanning those databases reports exactly the
match ends the definition gives -- every end offset e such that some data[s:e] is in the
expression's language (Hyperscan reports all match ends, doc/dev-reference/compilation.rst
"Semantics"), computed with Python's re.fullmatch -- which pins the compiler; the recorded
vectors of the reference's own regression suite are in test_zz_recorded_vectors_gpu.py.
GPU half: this runtime's hs_scan / scan_blocks on the same database against the reference."""
import base64
import json
import os
import re

import numpy as np
import pytest

from hyperscan_b200 import synth

CASELESS, DOTALL, MULTILINE, SINGLE = 1, 2, 4, 8
PATTERNS = [
    (rb"ab+c", 0), (rb"a[bc]*d", 0), (rb"x.y", 0), (rb"x.y", DOTALL), (rb"\d+\.\d\d", 0), (rb"^abc", 0),
    (rb"(ab|cd)+e", 0), (rb"[^a-z]{2,3}q", 0), (rb"fo{1,}d?", CASELESS), (rb"a(bc)?d|x+y", 0),
    (rb"^a.*b", DOTALL), (rb"\w+@\w+", 0), (rb"[a-c]{3}", 0), (rb"q\s*=\s*\d", 0), (rb"(?:ab){2,}c", 0),
    (rb"a+?b", 0), (rb"^x|y\x41z", 0), (rb"[\d\-x]+y", 0), (rb"a.{2,4}b", 0), (rb"\Sq\S", CASELESS),
    (rb"\bab", 0), (rb"\w+\b", 0), (rb"\Bq\B", 0), (rb"a\b.\bb", 0), (rb"^\b\d", 0), (rb"x\B|\by", 0),
    # anchors inside groups, where the reference takes them (nothing consumed before / after on any way there)
    (rb"(^a|b)c", 0), (rb"(a|^)b+c", 0), (rb"(^|x)ab+", 0), (rb"(^)?ab+", 0), (rb"fo+($)?", CASELESS), (rb"ab+(\z|c)", 0),
    (rb"\bab+$", 0), (rb"(^a|b)c", MULTILINE), (rb"b+($|x)", MULTILINE), (rb"[a-c]+(\Z|\d)", 0), (rb"(\Aa|^b|c)d+", MULTILINE),
]
ALPHA = b"abcdxyqAB.12e\nfoFOD =@-_z"
TAILS = [b"", b" abb", b"1abb\n", b"bcd\n", b"\nfoo", b"xbb\n\n"]   # for the end anchors
SEED_TEXT = b"abc abbcd acbd x\ny 3.14 ababe 12q fOOd ad xxy a\nb u_1@v2 cab q = 7 ababababc aab yAz 1-x2y a123b .q, "


def _ends(pat, flags, data):
    """every end offset e such that the expression matches some data[s:e] in context (\\b / \\B see the bytes
    around the match): a fixed-width look-behind pins the match end to e"""
    fl = (re.I if flags & CASELESS else 0) | (re.S if flags & DOTALL else 0) | (re.M if flags & MULTILINE else 0)
    out = []
    pat = pat.replace(b"\\Z", b"(?=\n?\0)").replace(b"\\z", b"\\Z").replace(b"\0", b"\\Z")   # PCRE \Z, \z in Python's spelling
    for e in range(1, len(data) + 1):
        rx = re.compile(b"(?:" + pat + b")(?<=(?s:\\A.{%d}))" % e, fl)
        if any(rx.match(data, s) for s in range(e)):
            out.append(e)
    return out


def _ends_ext(pat, flags, data, min_offset=0, max_offset=None, min_length=0):
    """_ends under hs_expr_ext: the match end within [min_offset, max_offset], the match at least min_length long"""
    fl = (re.I if flags & CASELESS else 0) | (re.S if flags & DOTALL else 0) | (re.M if flags & MULTILINE else 0)
    out = []
    for e in range(max(1, min_offset), len(data) + 1):
        if max_offset is not None and e > max_offset:
            break
        rx = re.compile(b"(?:" + pat + b")(?<=(?s:\\A.{%d}))" % e, fl)
        if any(rx.match(data, s) for s in range(e - max(min_length, 1) + 1)):
            out.append(e)
    return out


def _data(seed, n=48):
    rng = np.random.default_rng(seed)
    a = np.frombuffer(ALPHA, dtype=np.uint8)
    return a[rng.integers(0, a.size, size=n)].tobytes()


def _ref_ends(ref, db, data):
    a = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(0, np.uint8)
    r = ref.scan_sorted(db.ptr, a, np.array([0], np.uint64), np.array([len(data)], np.uint32))
    return [(int(x["id"]), int(x["to"])) for x in r]


@pytest.mark.parametrize("dfa", [1, 0])
@pytest.mark.parametrize("pi", range(len(PATTERNS)))
def test_reference_hs_scan_on_compiled_expressions_equals_definition(hs, ref, pi, dfa):
    pat, fl = PATTERNS[pi]
    hs.set_build_option("regex_dfa", dfa)            # the engine of the outfix: McClellan if small (default), or LimEx
    try:
        db = hs.compile_multi([pat], [fl], [7])
    finally:
        hs.set_build_option("regex_dfa", 1)
    assert db.info().runtime_impl == (1 if pat == rb"[a-c]{3}" else 2)   # single outfix, unless the language is finite
    if db.info().runtime_impl == 2:
        assert db.info().engine_id in ((6, 7) if dfa else (0, 1, 2, 3, 5))
    hits = 0
    for seed in range(10):
        data = (SEED_TEXT if seed == 0 else b"") + _data(100 * pi + seed) + TAILS[seed % len(TAILS)]
        want = [(7, e) for e in _ends(pat, fl, data)]
        assert _ref_ends(ref, db, data) == want, (pat, data)
        hits += len(want)
    assert hits > 0


def test_several_expressions_share_one_nfa_and_report_rules_hold(hs, ref):
    pats = [rb"ab+", rb"b+c", rb"[xy]z", rb"a.c"]
    flags = [0, 0, SINGLE, 0]
    ids = [1, 1, 2, 3]
    db = hs.compile_multi(pats, flags, ids)
    for seed in range(8):
        data = _data(900 + seed, 80) + b"abbbc xz yz"
        want = set()
        for p, f, i in zip(pats, flags, ids):
            e = _ends(p, f, data)
            want |= {(i, x) for x in (e[:1] if f & SINGLE else e)}   # SINGLEMATCH: the first match only
        assert sorted(_ref_ends(ref, db, data), key=lambda t: (t[1], t[0])) == sorted(want, key=lambda t: (t[1], t[0]))


@pytest.mark.parametrize("pat,fl,ext", [
    (rb"ab+c", 0, {"min_offset": 20}), (rb"ab+c", 0, {"max_offset": 30}), (rb"a.*d", DOTALL, {"min_offset": 10, "max_offset": 60}),
    (rb"a.*d", DOTALL, {"min_length": 6}), (rb"a[bc]*d", 0, {"min_length": 4, "min_offset": 8}), (rb"x.y|ab+", 0, {"min_length": 3}),
    (rb"\w+@\w+", 0, {"min_length": 7, "max_offset": 90}), (rb"b+(cd)?$", 0, {"min_offset": 5}), (rb"\bab+", 0, {"min_length": 3}),
    (rb"^a.*b", DOTALL, {"min_length": 10}), (rb"[a-c]{2,}", 0, {"min_length": 4})])
def test_extended_parameters_equal_definition(hs, ref, pat, fl, ext):
    """hs_compile_ext_multi: min_offset / max_offset (CHECK_BOUNDS in the report programs) and min_length (levels in
    the automaton), checked like the plain expressions -- the unmodified reference hs_scan on the database against
    the definition; the reference's own vectors for them (tools/hscollider extparams.txt) are in the golden file"""
    hits = 0
    for dfa in (1, 0):
        hs.set_build_option("regex_dfa", dfa)
        try:
            db = hs.compile_ext_multi([pat], [fl], [7], [ext])
        finally:
            hs.set_build_option("regex_dfa", 1)
        assert db.info().runtime_impl == 2
        for seed in range(8):
            data = (SEED_TEXT if seed == 0 else b"") + _data(300 + seed) + TAILS[seed % len(TAILS)]
            want = [(7, e) for e in _ends_ext(pat, fl, data, **ext)]
            assert _ref_ends(ref, db, data) == want, (pat, ext, data)
            hits += len(want)
    assert hits > 0


def test_an_expression_that_cannot_match_is_refused(hs):
    """as the reference does after it has resolved the assertions ("Pattern can never match."): the expression's own
    automaton, determinised and minimised, is the dead state alone"""
    for pat in (rb"^\Bfoo", rb"can't_match\b\B", rb"mkdzo(x|u)(\b)kd"):
        with pytest.raises(hs.HsError) as e:
            hs.compile_multi([rb"fo+d", pat], [0, 0], [1, 2])
        assert "Pattern can never match." in str(e.value) and e.value.expression == 1


def test_extended_parameter_errors(hs):
    for ext, msg in [({"min_offset": 9, "max_offset": 3}, "min_offset must be less"), ({"min_length": 9, "max_offset": 3}, "min_length must be less"),
                     ({"edit_distance": 1}, "Approximate"), ({"hamming_distance": 1}, "Approximate")]:
        with pytest.raises(hs.HsError) as e:
            hs.compile_ext_multi([rb"ab+c"], [0], [1], [ext])
        assert msg in str(e.value)
    with pytest.raises(hs.HsError):
        hs.compile_ext_multi([rb"a.{600}b"], [0], [1], [{"min_length": 600}])      # beyond the 512-state model
    for pat, ext, msg in [(rb"^fo+d?", {"min_offset": 3}, None), (rb"^food", {"min_offset": 5}, "anchored and cannot satisfy min_offset=5"),
                          (rb"fo+bar", {"min_length": 3}, None), (rb"foobar", {"min_length": 20}, "min_length=20 but can only produce matches of length 6"),
                          (rb"foobar", {"max_offset": 3}, "max_offset=3 but requires 6 bytes")]:
        if msg is None:
            hs.compile_ext_multi([pat], [0], [1], [ext])
            continue
        with pytest.raises(hs.HsError) as e:
            hs.compile_ext_multi([pat], [0], [1], [ext])
        assert msg in str(e.value)


@pytest.mark.parametrize("a,b,fl", [
    (rb"foo(?i)bar+", rb"foo(?i:bar+)", 0), (rb"(?i)fo+(?-i)d", rb"[fF][oO]+d", 0), (rb"\Qa.b\E+c", rb"a\.b+c", 0),
    (rb"\x{41}+b", rb"A+b", 0), (rb"[\060-\071]+x", rb"[0-9]+x", 0), (rb"\cAb+", rb"\x01b+", 0), (rb"\h+a", rb"[\t \xa0]+a", 0),
    (rb"[\Qa]\E]+y", rb"[a\]]+y", 0), (rb"a(?s).b+", rb"a(?s:.)b+", 0), (rb"\V+\v", rb"[^\n\x0b\f\r\x85]+[\n\x0b\f\r\x85]", 0),
    (rb"(?m)^ab+", rb"^ab+", MULTILINE), (rb"x\N+y", rb"x[^\n]+y", DOTALL), (rb"\0+a", rb"\x00+a", 0)])
def test_other_spellings_of_the_same_expression(hs, ref, a, b, fl):
    """option groups, \\Q..\\E, \\x{..}, octal, \\c, \\h \\v \\N against the plain spelling of the same language (the reference's
    own vectors for these, tools/hscollider test cases 11xxx / 19xxx / 24xxx, are in tests/golden/hscollider_regex.json)"""
    da, dbb = hs.compile_multi([a], [fl], [7]), hs.compile_multi([b], [fl], [7])
    alpha = b"abfoFOBARbar.dD\n\t \xa0\x00\x01A019]xy\x0b\x85"
    hits = 0
    for seed in range(12):
        rng = np.random.default_rng(seed)
        data = np.frombuffer(alpha, dtype=np.uint8)[rng.integers(0, len(alpha), size=200)].tobytes()
        data += b" fooBARr foobaR FoOd food a.bbc a.b.bc AAb 0129x \x01bb \t \xa0a a]ay a\nbb a\nb q\n\x0b\n abb\nabb x12y xy \x00\x00a "
        got = _ref_ends(ref, da, data)
        assert got == _ref_ends(ref, dbb, data), (a, b, data)
        hits += len(got)
    assert hits > 0


@pytest.mark.parametrize("pat,msg", [
    (rb"a*", "empty"), (rb"a$b", "Embedded end"), (rb"(a$|b)c", "Embedded end"), (rb"a^b", "Embedded start"), (rb"(^a)+b", "Embedded start"), (rb"\b+ab", "quantifier"), (rb"(?=a)b", "Look-around"), (rb"a++b", "Possessive"),
    (rb"(a|b)\1", "Escape"), (rb"[a-z]{600}x+", "too large"), (rb"(abcdefghijklmnopqrstuvwxyz0123456){2}+", "Possessive"), (rb"(abcdefghijklmnopqrstuvwxyz0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ_+){9}", "too large"), (rb"(a{40}){40}b+", "too large")])
def test_what_the_nfa_route_refuses(hs, pat, msg):
    with pytest.raises(hs.HsError) as e:
        hs.compile_multi([pat], [0], [1])
    assert msg.lower() in str(e.value).lower()


def test_nfa_route_is_block_mode_only_and_literal_sets_are_untouched(hs):
    with pytest.raises(hs.HsError):
        hs.compile_multi([rb"ab+c"], [0], [1], mode=hs.HS_MODE_STREAM)
    assert hs.compile_multi([rb"ab(c|d)e"], [0], [1]).info().runtime_impl == 1    # finite: pure literal as before


# ---- device --------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("pi", range(len(PATTERNS)))
def test_device_scans_compiled_expressions(hs, ref, pi):
    pat, fl = PATTERNS[pi]
    db = hs.compile_multi([pat], [fl], [7])
    scratch = hs.Scratch(db)
    lens = [0, 1, 2, 3, 17, 64, 100, 1000, 1024, 1025]
    rng = np.random.default_rng(pi)
    a = np.frombuffer(ALPHA, dtype=np.uint8)
    data, off, ln = synth.ragged_corpus(lens, None, seed=pi, plant_per_kb=0)
    data = a[rng.integers(0, a.size, size=data.size)].astype(np.uint8)
    got = np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"])
    want = ref.scan_sorted(db.ptr, data, off, ln, like=got)
    assert np.array_equal(got, want)
    b = 8
    buf = data[int(off[b]):int(off[b]) + int(ln[b])].tobytes()
    rc, out = hs.scan(db, buf, scratch)
    assert rc == hs.HS_SUCCESS and sorted(out) == sorted((int(r["id"]), int(r["to"])) for r in want[want["block"] == b])
    scratch.free()


@pytest.mark.gpu
def test_device_expression_set_with_report_rules(hs, ref):
    pats = [rb"ab+", rb"b+c", rb"[xy]z", rb"a.c", rb"\d{2,}"]
    db = hs.compile_multi(pats, [0, 0, SINGLE, 0, CASELESS], [1, 1, 2, 3, 4])
    data, off, ln, _ = synth.block_corpus(512, 512, [b"abbbc", b"xz", b"a1c22"], plant_per_kb=8.0, seed=3)
    scratch = hs.Scratch(db)
    got = np.sort(hs.scan_blocks(db, data, off, ln, scratch), order=["block", "to", "id"])
    want = ref.scan_sorted(db.ptr, data, off, ln, like=got)
    assert np.array_equal(got, want) and want.size > 500
    scratch.free()


with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bad_patterns.json")) as _f:
    BAD = json.load(_f)["cases"]
@pytest.mark.parametrize("case", BAD, ids=[str(i) for i in range(len(BAD))])
def test_what_the_reference_refuses_is_refused(hs, case):
    """unit/hyperscan/bad_patterns.txt: none of the reference's bad patterns compiles here either (the wording of the
    error is the reference's own where this compiler detects the same thing; otherwise it names what is missing)"""
    ext = case["ext"]
    if ext and any(not isinstance(v, int) for v in ext.values()):
        ext = None            # a malformed parameter in the file: the expression parser's error, not hs_compile's
    with pytest.raises(hs.HsError):
        hs.compile_ext_multi([base64.b64decode(case["pattern"])], [case["hs_flags"]], [1], [ext])


def _large_offset_cases():
    """unit/hyperscan/extparam.cpp:40-122 (LargeMinOffset, LargeExactOffset): (ext, corpus, expected ends)"""
    pad = lambda n: b"hatstand" + b"_" * n + b"teakettle"
    return [({"min_offset": 100000}, pad(80000), []), ({"min_offset": 100000}, pad(100000 - 17), [100000]),
            ({"min_offset": 200000, "max_offset": 200000}, pad(199982), []),
            ({"min_offset": 200000, "max_offset": 200000}, pad(199983), [200000]),
            ({"min_offset": 200000, "max_offset": 200000}, pad(199984), [])]


def test_large_offset_bounds_reference_runtime(hs, ref):
    for ext, corpus, want in _large_offset_cases():
        db = hs.compile_ext_multi([rb"hatstand.*teakettle"], [0], [0], [ext])
        assert [e for _, e in _ref_ends(ref, db, corpus)] == want
    with pytest.raises(hs.HsError):        # extparam.cpp:125 LargeMinLength: the length counter is in the automaton here
        hs.compile_ext_multi([rb"hatstand.*teakettle"], [0], [0], [{"min_length": 100000}])


@pytest.mark.gpu
def test_large_offset_bounds_device(hs):
    for ext, corpus, want in _large_offset_cases():
        db = hs.compile_ext_multi([rb"hatstand.*teakettle"], [0], [0], [ext])
        scratch = hs.Scratch(db)
        tos = []
        hs.scan(db, corpus, scratch, on_event=lambda i, frm, to, fl: tos.append(to) or 0)
        assert tos == want
