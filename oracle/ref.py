"""ctypes binding of the unmodified reference runtime built into oracle/_ref/
(see oracle/ref/Makefile, oracle/ref/ref_driver.c).  TEST INFRASTRUCTURE ONLY.

The reference runtime can only be built where its sources are.  Everywhere else
the answers it gave are replayed from tests/golden/ref_results/ (written by
tests/golden/gen_ref_results.py): every call below is keyed by a digest of its
inputs -- the database bytes included -- so a replayed answer is the one the
reference gave for exactly these inputs, and inputs it never saw fail loudly.
Where the runtime is built, its answers are also checked against the recorded
ones.  HS_REF_RECORD=1 adds the answers of a live run to the store."""
import atexit
import ctypes as C
import fcntl
import hashlib
import json
import lzma
import os
import struct

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(_HERE, "_ref")
STORE_DIR = os.path.join(os.path.dirname(_HERE), "tests", "golden", "ref_results")
REC_DTYPE = np.dtype([("id", "<u4"), ("block", "<u4"), ("to", "<u8")])
RECORD = os.environ.get("HS_REF_RECORD") == "1"

_libs = {}


def cpu_flags():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return set(line.split(":", 1)[1].split())
    except OSError:
        pass
    return set()


def host_isa():
    """Highest ISA level of the reference's fat runtime this host can run
    (reference: src/dispatcher.c:50-90)."""
    fl = cpu_flags()
    if {"avx512vbmi", "avx512bw", "avx512f"} <= fl:
        return "avx512vbmi"
    if {"avx512bw", "avx512f"} <= fl:
        return "avx512"
    if "avx2" in fl:
        return "avx2"
    return "corei7"


def live():
    """The reference runtime itself is built here (oracle/_ref)."""
    return os.path.exists(os.path.join(REF_DIR, "libhsref_%s.so" % host_isa()))


def best_isa():
    """The ISA level whose answers calls get: this host's where the runtime is
    built, else the one the recorded answers were taken with."""
    if live():
        return host_isa()
    return _store().isa or host_isa()


def available():
    """Answers can be had: from the runtime, or recorded."""
    return live() or bool(_store().entries)


class _Store:
    """Recorded answers, one lzma file per test module: a JSON header (ISA, keys,
    record counts, scalar values, digests) and the record columns (id, block, to).
    A large answer is kept as a digest when something else can offer it: the C
    restatement (oracle/port.py) reproducing it exactly ("port"), or the test's
    own result ("like", over the records sorted by (block, to, id))."""

    def __init__(self):
        self.entries, self.isa, self.new = {}, None, {}
        if not os.path.isdir(STORE_DIR):
            return
        for name in sorted(os.listdir(STORE_DIR)):
            if name.endswith(".xz"):
                isa, entries = self._read(os.path.join(STORE_DIR, name))
                self.isa = self.isa or isa
                self.entries.update(entries)

    @staticmethod
    def _read(path):
        with open(path, "rb") as f:
            raw = lzma.decompress(f.read())
        hlen = struct.unpack_from("<I", raw)[0]
        head = json.loads(raw[4:4 + hlen])
        counts = np.array(head["counts"], dtype=np.int64)
        total = int(counts.sum())
        cols = np.frombuffer(raw, dtype="<u4", count=4 * total, offset=4 + hlen)
        recs = np.zeros(total, dtype=REC_DTYPE)
        recs["id"] = cols[:total]
        recs["block"] = np.cumsum(cols[total:2 * total].astype(np.int32), dtype=np.int64)
        recs["to"] = cols[2 * total:3 * total].astype(np.uint64) | (cols[3 * total:].astype(np.uint64) << 32)
        ends = np.cumsum(counts)
        entries = {}
        for k, v, d, e, n in zip(head["keys"], head["values"], head["digests"], ends, counts):
            entries[bytes.fromhex(k)] = (recs[e - n:e], v, d)
        return head["isa"], entries

    @staticmethod
    def _write(path, isa, entries):
        keys = sorted(entries)
        recs = np.concatenate([entries[k][0] for k in keys]) if keys else np.zeros(0, REC_DTYPE)
        block = recs["block"].astype(np.int64)
        head = json.dumps({"isa": isa, "keys": [k.hex() for k in keys],
                           "counts": [int(entries[k][0].size) for k in keys],
                           "values": [entries[k][1] for k in keys],
                           "digests": [entries[k][2] for k in keys]}, separators=(",", ":")).encode()
        cols = np.concatenate([recs["id"], np.diff(block, prepend=0).astype(np.uint32),
                               (recs["to"] & 0xFFFFFFFF).astype(np.uint32), (recs["to"] >> 32).astype(np.uint32)])
        with open(path, "wb") as f:
            f.write(lzma.compress(struct.pack("<I", len(head)) + head + cols.astype("<u4").tobytes(),
                                  preset=9 | lzma.PRESET_EXTREME))

    def flush(self):
        """Merge the answers recorded by this process into the store files."""
        if not self.new:
            return
        os.makedirs(STORE_DIR, exist_ok=True)
        fd = os.open(STORE_DIR, os.O_RDONLY)
        try:
            fcntl.flock(fd, fcntl.LOCK_EX)      # recording processes (spawned test workers) merge one at a time
            for shard, new in self.new.items():
                path = os.path.join(STORE_DIR, shard + ".xz")
                old = self._read(path)[1] if os.path.exists(path) else {}
                old.update(new)
                self._write(path, host_isa(), old)
        finally:
            os.close(fd)
        self.new = {}


_the_store = None


def _store():
    global _the_store
    if _the_store is None:
        _the_store = _Store()
        if RECORD:
            atexit.register(_the_store.flush)
    return _the_store


def _bytes(p):
    if isinstance(p, bytes):
        return p
    if isinstance(p, np.ndarray):
        return np.ascontiguousarray(p).tobytes()
    return repr(p).encode()


def _db_bytes(db_ptr):
    """Platform word and bytecode of an hs_database_t (struct hs_database,
    hyperscan_b200/csrc/ref_layout.h DbHeader)."""
    p = db_ptr.value if isinstance(db_ptr, C.c_void_p) else int(db_ptr)
    length = C.c_uint32.from_address(p + 8).value
    bytecode = C.c_uint32.from_address(p + 36).value
    return C.string_at(p + 16, 8) + C.string_at(p + bytecode, length)


DIGEST_ABOVE = 64           # answers with more records are recorded as a digest where something can offer them


def _canon(recs):
    """records (a structured array with id / block / to, or (id, block, to)
    triples) as REC_DTYPE sorted by (block, to, id)"""
    if isinstance(recs, np.ndarray):
        r = np.zeros(recs.size, dtype=REC_DTYPE)
        for f in ("id", "block", "to"):
            r[f] = recs[f]
    else:
        r = np.array([tuple(int(x) for x in t) for t in recs], dtype=REC_DTYPE)
    return np.sort(r, order=["block", "to", "id"])


def _digest(how, recs):
    return "%s:%d:%s" % (how, recs.size, hashlib.blake2b(recs.tobytes(), digest_size=16).hexdigest())


def _same(entry, recs, value):
    old, old_value, dg = entry
    if old_value != value:
        return False
    if dg is None:
        return np.array_equal(old, recs)
    how = dg.split(":")[0]
    return dg == _digest(how, _canon(recs) if how == "like" else recs)


def _answer(kind, isa, parts, compute, restate=None, like=None):
    """(records, value) of one reference call: from the runtime where it is built
    (checked against the recorded answer, if any), else the recorded answer.
    restate: the C restatement of the same call.  like: the caller's own answer
    (records or (id, block, to) triples), offered where only a digest of the
    reference's is recorded; it is returned, sorted by (block, to, id), when it
    has that digest, and a different one fails the calling test."""
    h = hashlib.blake2b(digest_size=10)
    for p in (kind, isa) + tuple(parts):
        b = _bytes(p)
        h.update(struct.pack("<Q", len(b)) + b)
    key = h.digest()
    store = _store()
    if live():
        recs, value = compute()
        recs = np.ascontiguousarray(recs, dtype=REC_DTYPE)
        old = store.entries.get(key)
        if old is not None and not _same(old, recs, value):
            raise AssertionError("the reference runtime's %s answer differs from the one recorded in %s"
                                 % (kind, STORE_DIR))
        if RECORD:
            entry = (recs, value, None)
            if recs.size > DIGEST_ABOVE and like is not None:
                entry = (recs[:0], value, _digest("like", _canon(recs)))
            elif recs.size > DIGEST_ABOVE and restate is not None:
                r2, v2 = restate()
                if v2 == value and np.array_equal(np.asarray(r2, dtype=REC_DTYPE), recs):
                    entry = (recs[:0], value, _digest("port", recs))
            test = os.environ.get("PYTEST_CURRENT_TEST", "")
            shard = os.path.splitext(os.path.basename(test.split("::")[0]))[0] if test else "other"
            store.new.setdefault(shard, {})[key] = entry
        return recs, value
    if key not in store.entries:
        raise RuntimeError("no recorded reference answer for this %s call: the reference runtime never saw these "
                           "inputs (record them with tests/golden/gen_ref_results.py where oracle/_ref is built)"
                           % kind)
    recs, value, dg = store.entries[key]
    if dg is None:
        return recs.copy(), value
    if dg.startswith("port:"):
        recs = np.ascontiguousarray(restate()[0], dtype=REC_DTYPE)
        if _digest("port", recs) != dg:
            raise AssertionError("the C restatement no longer reproduces the reference's recorded %s answer" % kind)
        return recs, value
    if like is None:
        raise RuntimeError("only a digest of the reference's %s answer is recorded: the caller must offer its own"
                           % kind)
    recs = _canon(like)
    if _digest("like", recs) != dg:
        raise AssertionError("%d records differ from the reference's %s answer recorded for these inputs (%s)"
                             % (recs.size, kind, dg.split(":")[1]))
    return recs, value


def lib(isa=None):
    isa = isa or best_isa()
    if isa not in _libs:
        path = os.path.join(REF_DIR, "libhsref_%s.so" % isa)
        if not os.path.exists(path):
            raise RuntimeError("reference runtime not built: %s (run `make -C oracle/ref REF=<reference "
                               "source tree>`)" % path)
        L = C.CDLL(path)
        vp = C.c_void_p
        L.ref_scan_collect.restype = C.c_long
        L.ref_scan_collect.argtypes = [vp, vp, vp, vp, C.c_size_t, vp, C.c_size_t, C.c_size_t,
                                       C.POINTER(C.c_int)]
        L.ref_stream_collect.restype = C.c_long
        L.ref_vector_collect.restype = C.c_long
        L.ref_vector_collect.argtypes = [vp, vp, vp, C.c_size_t, vp, C.c_size_t, C.c_size_t, C.POINTER(C.c_int)]
        L.ref_stream_collect.argtypes = [vp, vp, vp, C.c_size_t, vp, C.c_size_t, C.c_size_t, C.POINTER(C.c_int)]
        L.ref_scan_blocks_mt.restype = C.c_double
        L.ref_scan_blocks_mt.argtypes = [vp, vp, vp, vp, C.c_size_t, C.c_uint, C.c_uint,
                                         C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
        L.ref_hwlm_exec.restype = C.c_long
        L.ref_hwlm_exec.argtypes = [vp, vp, C.c_size_t, C.c_size_t, C.c_ulonglong, vp, C.c_size_t,
                                    C.c_size_t]
        for f in (L.ref_shufti, L.ref_truffle):
            f.restype = C.c_long
            f.argtypes = [vp, vp, vp, C.c_size_t]
        L.ref_vermicelli.restype = C.c_long
        L.ref_vermicelli.argtypes = [C.c_ubyte, C.c_int, vp, C.c_size_t]
        L.ref_dvermicelli.restype = C.c_long
        L.ref_dvermicelli.argtypes = [C.c_ubyte, C.c_ubyte, C.c_int, vp, C.c_size_t]
        _libs[isa] = L
    return _libs[isa]


def _u8(data):
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    return np.frombuffer(bytes(data), dtype=np.uint8)


def scan_collect(db_ptr, data, offsets, lengths, stop_after=0, isa=None, cap=None, like=None):
    """Reference hs_scan() over blocks; records in delivery order.
    Returns (records, last_error).  like: see _answer."""
    a = _u8(data)
    keep = a if a.size else np.zeros(1, dtype=np.uint8)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.uint32)
    isa = isa or best_isa()

    def compute(cap=cap or (1 << 20)):
        while True:
            out = np.zeros(cap, dtype=REC_DTYPE)
            err = C.c_int()
            n = lib(isa).ref_scan_collect(db_ptr, keep.ctypes.data, off.ctypes.data, ln.ctypes.data, off.size,
                                          out.ctypes.data, cap, stop_after, C.byref(err))
            if n < 0:
                raise RuntimeError("reference hs_alloc_scratch failed: %d" % n)
            if n <= cap:
                return out[:n], err.value
            cap = int(n) + 16
    def restate():
        from . import port
        return port.scan_collect(db_ptr, data, off, ln, stop_after)
    return _answer("hs_scan", isa, (_db_bytes(db_ptr), a, off, ln, stop_after), compute, restate, like)


def stream_collect(db_ptr, data, write_lengths, stop_after=0, isa=None, like=None):
    """Reference streaming scan of `data` cut into consecutive writes; records
    (id, write index, to = stream offset) in delivery order + last error."""
    a = _u8(data)
    keep = a if a.size else np.zeros(1, dtype=np.uint8)
    wl = np.ascontiguousarray(write_lengths, dtype=np.uint32)
    assert int(wl.sum()) == a.size
    isa = isa or best_isa()

    def compute(cap=1 << 18):
        while True:
            out = np.zeros(cap, dtype=REC_DTYPE)
            err = C.c_int()
            n = lib(isa).ref_stream_collect(db_ptr, keep.ctypes.data, wl.ctypes.data, wl.size, out.ctypes.data,
                                            cap, stop_after, C.byref(err))
            if n < 0:
                raise RuntimeError("reference stream open failed: %d" % n)
            if n <= cap:
                return out[:n], err.value
            cap = int(n) + 16
    def restate():
        from . import port
        return port.stream_collect(db_ptr, data, wl, stop_after)
    return _answer("stream", isa, (_db_bytes(db_ptr), a, wl, stop_after), compute, restate, like)


def vector_collect(db_ptr, data, buf_lengths, stop_after=0, isa=None, like=None):
    """Reference hs_scan_vector over `data` cut into consecutive buffers; records
    (id, 0, to counted from the first buffer) in delivery order + the call's
    return code."""
    a = _u8(data)
    keep = a if a.size else np.zeros(1, dtype=np.uint8)
    bl = np.ascontiguousarray(buf_lengths, dtype=np.uint32)
    assert int(bl.sum()) == a.size
    isa = isa or best_isa()

    def compute(cap=1 << 18):
        while True:
            out = np.zeros(cap, dtype=REC_DTYPE)
            err = C.c_int()
            n = lib(isa).ref_vector_collect(db_ptr, keep.ctypes.data, bl.ctypes.data, bl.size, out.ctypes.data,
                                            cap, stop_after, C.byref(err))
            if n < 0:
                raise RuntimeError("reference scratch allocation failed: %d" % n)
            if n <= cap:
                return out[:n], err.value
            cap = int(n) + 16
    def restate():
        from . import port
        return port.vector_collect(db_ptr, data, bl, stop_after)
    return _answer("vector", isa, (_db_bytes(db_ptr), a, bl, stop_after), compute, restate, like)


def scan_sorted(db_ptr, data, offsets, lengths, isa=None, like=None):
    """Match multiset sorted by (block, to, id): what 'bit-exact' is defined on
    (SURVEY.md F8)."""
    r, err = scan_collect(db_ptr, data, offsets, lengths, isa=isa, like=like)
    if err:
        raise RuntimeError("reference hs_scan error %d" % err)
    return np.sort(r, order=["block", "to", "id"])


def physical_core_cpus():
    """CPUs of the affinity mask, one hardware thread per physical core first (then
    the SMT siblings), for pinning the bench threads 1:1 the way hsbench does."""
    cpus = sorted(os.sched_getaffinity(0))
    first, rest, seen = [], [], set()
    for c in cpus:
        try:
            with open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c) as f:
                sib = f.read().strip()
        except OSError:
            sib = str(c)
        if sib in seen:
            rest.append(c)
        else:
            seen.add(sib)
            first.append(c)
    return first + rest


def pin_bench_threads(cpus):
    """Pin bench thread i to cpus[i % len(cpus)]; an empty list unpins."""
    arr = (C.c_int * max(1, len(cpus)))(*cpus)
    lib().ref_set_bench_cpus(arr, len(cpus))


def bench_blocks(db_ptr, data, offsets, lengths, threads, repeats, isa=None):
    """hsbench-style timing loop (tools/hsbench/main.cpp:503-527).  Returns
    (seconds, matches, bytes)."""
    a = _u8(data)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.uint32)
    m = C.c_ulonglong()
    b = C.c_ulonglong()
    t = lib(isa).ref_scan_blocks_mt(db_ptr, a.ctypes.data, off.ctypes.data, ln.ctypes.data, off.size,
                                    threads, repeats, C.byref(m), C.byref(b))
    if t < 0:
        raise RuntimeError("reference bench failed")
    return t, int(m.value), int(b.value)


def hwlm_exec(hwlm_bytes, data, start=0, groups=0xFFFFFFFFFFFFFFFF, stop_after=0, isa=None):
    """Reference hwlmExec() on a raw HWLM table (64-byte aligned copy)."""
    raw = np.zeros(len(hwlm_bytes) + 64, dtype=np.uint8)
    o = (-raw.ctypes.data) % 64
    raw[o:o + len(hwlm_bytes)] = np.frombuffer(hwlm_bytes, dtype=np.uint8)
    a = _u8(data)
    # the reference engines may read a few bytes around the buffer: pad it
    buf = np.zeros(a.size + 128, dtype=np.uint8)
    buf[64:64 + a.size] = a
    isa = isa or best_isa()

    def compute(cap=1 << 16):
        out = np.zeros(cap, dtype=REC_DTYPE)
        n = lib(isa).ref_hwlm_exec(raw.ctypes.data + o, buf.ctypes.data + 64, a.size, start, groups,
                                   out.ctypes.data, cap, stop_after)
        return out[:min(n, cap)], 0
    def restate():
        from . import port
        got = port.hwlm_exec(hwlm_bytes, data, start=start, groups=groups, stop_after=stop_after)
        return np.array([(i, 0, to) for to, i in got], dtype=REC_DTYPE), 0
    out, _ = _answer("hwlmExec", isa, (bytes(hwlm_bytes), a, start, groups, stop_after), compute, restate)
    return [(int(r["to"]), int(r["id"])) for r in out]


def nfa_exec_blocks(nfa_bytes, data, offsets, lengths, isa=None, cap=1 << 20, like=None):
    """Reference nfaExecMcClellan8_B / 16_B / nfaExecSheng_B over every block (offset 0):
    the callbacks as records sorted by (block, to, id)."""
    a = _u8(data)
    keep = a if a.size else np.zeros(1, dtype=np.uint8)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.uint32)
    raw = np.zeros(len(nfa_bytes) + 64, dtype=np.uint8)     # struct NFA is cache-line aligned
    shift = (-raw.ctypes.data) % 64
    raw[shift:shift + len(nfa_bytes)] = np.frombuffer(nfa_bytes, dtype=np.uint8)
    isa = isa or best_isa()

    def compute(cap=cap):
        L = lib(isa)
        L.ref_nfa_exec_blocks.restype = C.c_long
        L.ref_nfa_exec_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                          C.c_size_t]
        while True:
            out = np.zeros(cap, dtype=REC_DTYPE)
            n = L.ref_nfa_exec_blocks(raw.ctypes.data + shift, keep.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                      off.size, out.ctypes.data, cap)
            if n < 0:
                raise RuntimeError("reference: engine type not handled")
            if n <= cap:
                return np.sort(out[:n], order=["block", "to", "id"]), 0
            cap = int(n) + 16
    return _answer("nfaExec", isa, (bytes(nfa_bytes), a, off, ln), compute, like=like)[0]


ACCEL_VERM, ACCEL_VERM_NOCASE, ACCEL_DVERM, ACCEL_DVERM_NOCASE, ACCEL_SHUFTI, ACCEL_TRUFFLE = 1, 2, 3, 4, 13, 15


def accel_find(typ, params, data, isa=None):
    """Reference shuftiExec / truffleExec / vermicelliExec / vermicelliDoubleExec
    (`typ` as hs_b200_accel_find takes it) over `data`: the offset of the first
    byte found, len(data) for none."""
    a = bytes(data)
    isa = isa or best_isa()

    def compute():
        R = lib(isa)
        buf = np.zeros(len(a) + 192, dtype=np.uint8)
        buf[64:64 + len(a)] = np.frombuffer(a, dtype=np.uint8)
        p = buf.ctypes.data + 64
        if typ == ACCEL_SHUFTI:
            pos = R.ref_shufti(params[:16], params[16:], p, len(a))
        elif typ == ACCEL_TRUFFLE:
            pos = R.ref_truffle(params[:16], params[16:], p, len(a))
        elif typ in (ACCEL_VERM, ACCEL_VERM_NOCASE):
            pos = R.ref_vermicelli(params[0], typ == ACCEL_VERM_NOCASE, p, len(a))
        else:
            pos = R.ref_dvermicelli(params[0], params[1], typ == ACCEL_DVERM_NOCASE, p, len(a))
        return np.zeros(0, REC_DTYPE), int(pos)
    return _answer("accel", isa, (typ, bytes(params), a), compute)[1]


def stream_size(db_ptr, isa=None):
    """The reference's hs_stream_size() for a streaming database."""
    isa = isa or best_isa()

    def compute():
        R = lib(isa)
        R.hs_stream_size.argtypes = [C.c_void_p, C.POINTER(C.c_size_t)]
        sz = C.c_size_t()
        rc = R.hs_stream_size(db_ptr, C.byref(sz))
        return np.zeros(0, REC_DTYPE), [int(rc), int(sz.value)]
    return tuple(_answer("hs_stream_size", isa, (_db_bytes(db_ptr),), compute)[1])


def read_container(blob, data, isa=None):
    """The reference's hs_deserialize_database() and hs_database_info() on a
    serialized database, and its hs_scan() of `data` as one block on the result:
    (deserialize rc, info text, matches sorted by (block, to, id))."""
    blob = bytes(blob)
    a = _u8(data)
    isa = isa or best_isa()

    def compute():
        R = lib(isa)
        out = C.c_void_p()
        R.hs_deserialize_database.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]
        rc = R.hs_deserialize_database(blob, len(blob), C.byref(out))
        if rc != 0:
            return np.zeros(0, REC_DTYPE), [int(rc), ""]
        info = C.c_char_p()
        R.hs_database_info.argtypes = [C.c_void_p, C.POINTER(C.c_char_p)]
        if R.hs_database_info(out, C.byref(info)) != 0:
            raise RuntimeError("reference hs_database_info failed")
        return scan_sorted(out.value, a, [0], [a.size], isa=isa), [0, info.value.decode()]
    recs, (rc, info) = _answer("hs_deserialize", isa, (blob, a), compute)
    return rc, info, recs
