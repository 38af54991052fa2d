"""ctypes binding of libhs_b200.so (include/hs_b200.h) for the Python harness
(tests/, bench.py, __graft_entry__.py).

The product is the C-ABI library; this module only marshals arguments.  It
fails loudly when the library has not been built -- there is no Python or CPU
fallback for the scan path.
"""
import ctypes as C
import os
import struct

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libhs_b200.so")

HS_SUCCESS = 0
HS_INVALID = -1
HS_NOMEM = -2
HS_SCAN_TERMINATED = -3
HS_COMPILER_ERROR = -4
HS_DB_VERSION_ERROR = -5
HS_DB_PLATFORM_ERROR = -6
HS_DB_MODE_ERROR = -7
HS_BAD_ALIGN = -8
HS_BAD_ALLOC = -9
HS_SCRATCH_IN_USE = -10
HS_ARCH_ERROR = -11
HS_INSUFFICIENT_SPACE = -12
HS_UNKNOWN_ERROR = -13

HS_FLAG_CASELESS = 1
HS_FLAG_DOTALL = 2
HS_FLAG_MULTILINE = 4
HS_FLAG_SINGLEMATCH = 8
HS_FLAG_ALLOWEMPTY = 16
HS_FLAG_UTF8 = 32
HS_FLAG_SOM_LEFTMOST = 256
HS_MODE_BLOCK = 1
HS_MODE_STREAM = 2
HS_MODE_VECTORED = 4
HS_CPU_FEATURES_AVX2 = 1 << 2

MATCH_DTYPE = np.dtype([("id", "<u4"), ("block", "<u4"), ("to", "<u8")])


class CompileError(C.Structure):
    _fields_ = [("message", C.c_char_p), ("expression", C.c_int)]


class PlatformInfo(C.Structure):
    _fields_ = [("tune", C.c_uint), ("cpu_features", C.c_ulonglong),
                ("reserved1", C.c_ulonglong), ("reserved2", C.c_ulonglong)]


class DbInfo(C.Structure):
    _fields_ = [("runtime_impl", C.c_uint), ("hwlm_type", C.c_uint), ("engine_id", C.c_uint),
                ("fdr_domain", C.c_uint), ("fdr_stride", C.c_uint), ("num_literals", C.c_uint),
                ("bytecode_len", C.c_uint), ("min_width", C.c_uint)]


MATCH_CB = C.CFUNCTYPE(C.c_int, C.c_uint, C.c_ulonglong, C.c_ulonglong, C.c_uint, C.c_void_p)
BLOCK_CB = C.CFUNCTYPE(C.c_int, C.c_uint, C.c_uint, C.c_ulonglong, C.c_ulonglong, C.c_uint, C.c_void_p)

_lib = None


class HsError(RuntimeError):
    def __init__(self, code, what=""):
        super().__init__("hs error %d %s" % (code, what))
        self.code = code


def lib():
    """Load libhs_b200.so (built by hyperscan_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libhs_b200.so is not built (%s): run `python -m hyperscan_b200.build`; "
                "there is no fallback scan path" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, cp, u32p, u64p = C.c_void_p, C.c_char_p, C.POINTER(C.c_uint), C.POINTER(C.c_ulonglong)
        L.hs_compile_lit_multi.argtypes = [C.POINTER(cp), u32p, u32p, C.POINTER(C.c_size_t), C.c_uint,
                                           C.c_uint, C.POINTER(PlatformInfo), C.POINTER(vp),
                                           C.POINTER(C.POINTER(CompileError))]
        L.hs_compile_multi.argtypes = [C.POINTER(cp), u32p, u32p, C.c_uint, C.c_uint,
                                       C.POINTER(PlatformInfo), C.POINTER(vp),
                                       C.POINTER(C.POINTER(CompileError))]
        L.hs_compile.argtypes = [cp, C.c_uint, C.c_uint, C.POINTER(PlatformInfo), C.POINTER(vp),
                                 C.POINTER(C.POINTER(CompileError))]
        L.hs_compile_lit.argtypes = [cp, C.c_uint, C.c_size_t, C.c_uint, C.POINTER(PlatformInfo),
                                     C.POINTER(vp), C.POINTER(C.POINTER(CompileError))]
        L.hs_free_compile_error.argtypes = [C.POINTER(CompileError)]
        L.hs_free_database.argtypes = [vp]
        L.hs_serialize_database.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
        L.hs_deserialize_database.argtypes = [cp, C.c_size_t, C.POINTER(vp)]
        L.hs_deserialize_database_at.argtypes = [cp, C.c_size_t, vp]
        L.hs_database_size.argtypes = [vp, C.POINTER(C.c_size_t)]
        L.hs_serialized_database_size.argtypes = [cp, C.c_size_t, C.POINTER(C.c_size_t)]
        L.hs_stream_size.argtypes = [vp, C.POINTER(C.c_size_t)]
        L.hs_database_info.argtypes = [vp, C.POINTER(vp)]
        L.hs_serialized_database_info.argtypes = [cp, C.c_size_t, C.POINTER(vp)]
        L.hs_version.restype = cp
        L.hs_alloc_scratch.argtypes = [vp, C.POINTER(vp)]
        L.hs_clone_scratch.argtypes = [vp, C.POINTER(vp)]
        L.hs_scratch_size.argtypes = [vp, C.POINTER(C.c_size_t)]
        L.hs_free_scratch.argtypes = [vp]
        L.hs_scan.argtypes = [vp, vp, C.c_uint, C.c_uint, vp, MATCH_CB, vp]
        L.hs_b200_streams_open.argtypes = [vp, C.c_size_t, C.c_int, C.POINTER(vp)]
        L.hs_b200_streams_scan.argtypes = [vp, vp, vp, vp, vp, BLOCK_CB, vp, u64p]
        L.hs_b200_streams_scan_collect.argtypes = [vp, vp, vp, vp, vp, vp, C.c_size_t, u64p]
        L.hs_b200_streams_close.argtypes = [vp]
        L.hs_b200_streams_state_bytes.argtypes = [vp]
        L.hs_b200_streams_state_bytes.restype = C.c_size_t
        L.hs_open_stream.argtypes = [vp, C.c_uint, C.POINTER(vp)]
        L.hs_scan_stream.argtypes = [vp, vp, C.c_uint, C.c_uint, vp, MATCH_CB, vp]
        L.hs_scan_vector.argtypes = [vp, vp, vp, C.c_uint, C.c_uint, vp, MATCH_CB, vp]
        L.hs_compress_stream.argtypes = [vp, cp, C.c_size_t, C.POINTER(C.c_size_t)]
        L.hs_expand_stream.argtypes = [vp, C.POINTER(vp), cp, C.c_size_t]
        L.hs_reset_and_expand_stream.argtypes = [vp, cp, C.c_size_t, vp, MATCH_CB, vp]
        L.hs_close_stream.argtypes = [vp, vp, MATCH_CB, vp]
        L.hs_reset_stream.argtypes = [vp, C.c_uint, vp, MATCH_CB, vp]
        L.hs_copy_stream.argtypes = [C.POINTER(vp), vp]
        L.hs_reset_and_copy_stream.argtypes = [vp, vp, vp, MATCH_CB, vp]
        L.hs_b200_scan_blocks.argtypes = [vp, vp, vp, vp, C.c_size_t, vp, BLOCK_CB, vp, u64p]
        L.hs_b200_scan_blocks_collect.argtypes = [vp, vp, vp, vp, C.c_size_t, vp, vp, C.c_size_t, u64p]
        L.hs_b200_corpus_upload.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, C.POINTER(vp)]
        L.hs_b200_corpus_wrap.argtypes = [vp, C.c_size_t, vp, vp, C.c_size_t, C.c_int, C.POINTER(vp)]
        L.hs_b200_corpus_free.argtypes = [vp]
        L.hs_b200_corpus_bytes.argtypes = [vp]
        L.hs_b200_corpus_bytes.restype = C.c_size_t
        L.hs_b200_scan_corpus_async.argtypes = [vp, vp, vp, vp]
        L.hs_b200_scan_corpus_finish.argtypes = [vp, u64p, C.POINTER(vp)]
        L.hs_b200_copy_records.argtypes = [vp, vp, C.c_size_t]
        L.hs_b200_export_records_async.argtypes = [vp, vp, C.c_size_t, vp, vp]
        L.hs_b200_peer_buffer_alloc.argtypes = [C.c_size_t, C.POINTER(vp), C.c_char_p]
        L.hs_b200_peer_buffer_open.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.hs_b200_peer_buffer_close.argtypes = [vp, C.c_int]
        L.hs_b200_peer_buffer_read.argtypes = [vp, vp, C.c_size_t]
        L.hs_b200_set_peer_exchange.argtypes = [vp, C.c_uint, C.c_uint, C.POINTER(vp), C.c_size_t, C.c_uint]
        L.hs_b200_postprocess_matches.argtypes = [vp, vp, C.c_size_t, u64p]
        L.hs_b200_fetch_matches.argtypes = [vp, vp, vp, C.c_size_t, u64p]
        L.hs_b200_db_info.argtypes = [vp, C.POINTER(DbInfo)]
        L.hs_b200_set_build_option.argtypes = [cp, C.c_int]
        L.hs_b200_set_runtime_option.argtypes = [cp, C.c_int]
        L.hs_b200_last_counters.argtypes = [vp, C.POINTER(C.c_uint * 8)]
        L.hs_b200_launch_count.restype = C.c_ulonglong
        L.hs_b200_last_kernel_ms.argtypes = [vp]
        L.hs_b200_last_kernel_ms.restype = C.c_float
        _lib = L
    return _lib


def _check(rc, what=""):
    if rc != HS_SUCCESS:
        raise HsError(rc, what)


class Database:
    """Owner of an hs_database_t* produced by this library's compiler."""

    def __init__(self, ptr):
        self.ptr = C.c_void_p(ptr) if not isinstance(ptr, C.c_void_p) else ptr

    def __del__(self):
        try:
            if self.ptr:
                lib().hs_free_database(self.ptr)
                self.ptr = None
        except Exception:
            pass

    def info(self):
        d = DbInfo()
        _check(lib().hs_b200_db_info(self.ptr, C.byref(d)))
        return d

    def serialize(self):
        out = C.c_void_p()
        n = C.c_size_t()
        _check(lib().hs_serialize_database(self.ptr, C.byref(out), C.byref(n)))
        b = C.string_at(out, n.value)
        C.CDLL(None).free(out)
        return b

    @staticmethod
    def deserialize(b):
        out = C.c_void_p()
        _check(lib().hs_deserialize_database(b, len(b), C.byref(out)))
        return Database(out)

    def engines(self):
        """The engines of an outfix database, one per queue in queue order: [(model, states)], model one of
        ENGINE_MODELS' values, states the engine's NFA.nPositions.  [] for a database without engines."""
        bc = self.serialize()[32:]  # the bytecode follows the 32-byte serialization header
        n, info_at = struct.unpack_from("<I", bc, _ROSE_QUEUE_COUNT)[0], struct.unpack_from("<I", bc, _ROSE_NFA_INFO)[0]
        if not info_at:
            return []
        out = []
        for q in range(n):
            nfa = struct.unpack_from("<I", bc, info_at + q * _NFA_INFO_SIZE)[0]
            out.append((ENGINE_MODELS.get(bc[nfa + _NFA_TYPE], "type %d" % bc[nfa + _NFA_TYPE]),
                        struct.unpack_from("<I", bc, nfa + _NFA_POSITIONS)[0]))
        return out


# NFA.type (src/nfa/nfa_internal.h:53-78) of the engines this library builds
ENGINE_MODELS = {0: "LimEx-32", 1: "LimEx-64", 2: "LimEx-128", 3: "LimEx-256", 5: "LimEx-512", 6: "McClellan-8",
                 7: "McClellan-16", 17: "Sheng"}
# byte offsets of RoseEngine.queueCount, RoseEngine.nfaInfoOffset, sizeof(NfaInfo), NFA.type, NFA.nPositions
_ROSE_QUEUE_COUNT, _ROSE_NFA_INFO, _NFA_INFO_SIZE, _NFA_TYPE, _NFA_POSITIONS = 156, 236, 20, 8, 20


def _raise_compile(rc, err):
    msg, idx = "?", -1
    if err:
        msg = (err.contents.message or b"").decode("latin1")
        idx = err.contents.expression
        lib().hs_free_compile_error(err)
    e = HsError(rc, "compile: %s (expression %d)" % (msg, idx))
    e.message = msg
    e.expression = idx
    raise e


def compile_lit_multi(lits, flags=None, ids=None, mode=HS_MODE_BLOCK, platform=None):
    """hs_compile_lit_multi (src/hs_compile.h:501-560): raw byte literals."""
    n = len(lits)
    lits = [bytes(x) for x in lits]
    flags = list(flags) if flags is not None else [0] * n
    ids = list(ids) if ids is not None else list(range(n))
    bufs = [C.create_string_buffer(x, len(x) + 1) for x in lits]
    arr = (C.c_char_p * n)(*[C.cast(b, C.c_char_p) for b in bufs])
    fl = (C.c_uint * n)(*flags)
    idv = (C.c_uint * n)(*ids)
    lens = (C.c_size_t * n)(*[len(x) for x in lits])
    db = C.c_void_p()
    err = C.POINTER(CompileError)()
    rc = lib().hs_compile_lit_multi(arr, fl, idv, lens, n, mode, platform, C.byref(db), C.byref(err))
    if rc != HS_SUCCESS:
        _raise_compile(rc, err)
    return Database(db)


def compile_multi(exprs, flags=None, ids=None, mode=HS_MODE_BLOCK, platform=None):
    """hs_compile_multi (src/hs_compile.h:360-420): NUL-terminated regex strings."""
    n = len(exprs)
    exprs = [x if isinstance(x, bytes) else x.encode("latin1") for x in exprs]
    flags = list(flags) if flags is not None else [0] * n
    ids = list(ids) if ids is not None else list(range(n))
    arr = (C.c_char_p * n)(*exprs)
    fl = (C.c_uint * n)(*flags)
    idv = (C.c_uint * n)(*ids)
    db = C.c_void_p()
    err = C.POINTER(CompileError)()
    rc = lib().hs_compile_multi(arr, fl, idv, n, mode, platform, C.byref(db), C.byref(err))
    if rc != HS_SUCCESS:
        _raise_compile(rc, err)
    return Database(db)


class ExprExt(C.Structure):
    _fields_ = [("flags", C.c_ulonglong), ("min_offset", C.c_ulonglong), ("max_offset", C.c_ulonglong),
                ("min_length", C.c_ulonglong), ("edit_distance", C.c_uint), ("hamming_distance", C.c_uint)]


def compile_ext_multi(exprs, flags=None, ids=None, ext=None, mode=HS_MODE_BLOCK, platform=None):
    """hs_compile_ext_multi (src/hs_compile.h:422-520); ext: one dict per expression (or None) with any of
    min_offset, max_offset, min_length, edit_distance, hamming_distance."""
    n = len(exprs)
    exprs = [x if isinstance(x, bytes) else x.encode("latin1") for x in exprs]
    flags = list(flags) if flags is not None else [0] * n
    ids = list(ids) if ids is not None else list(range(n))
    bits = {"min_offset": 1, "max_offset": 2, "min_length": 4, "edit_distance": 8, "hamming_distance": 16}
    structs, ptrs = [], (C.POINTER(ExprExt) * n)()
    for i, e in enumerate(ext or [None] * n):
        if e:
            x = ExprExt()
            for k, v in e.items():
                x.flags |= bits[k]
                setattr(x, k, int(v))
            structs.append(x)
            ptrs[i] = C.pointer(x)
    arr = (C.c_char_p * n)(*exprs)
    fl = (C.c_uint * n)(*flags)
    idv = (C.c_uint * n)(*ids)
    db = C.c_void_p()
    err = C.POINTER(CompileError)()
    rc = lib().hs_compile_ext_multi(arr, fl, idv, ptrs, n, mode, platform, C.byref(db), C.byref(err))
    if rc != HS_SUCCESS:
        _raise_compile(rc, err)
    return Database(db)


def set_build_option(key, value):
    _check(lib().hs_b200_set_build_option(key.encode(), int(value)), key)


def set_runtime_option(key, value):
    _check(lib().hs_b200_set_runtime_option(key.encode(), int(value)), key)


def _as_u8(data):
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    else:
        a = np.frombuffer(bytes(data), dtype=np.uint8)
    return a


def _blocks(offsets, lengths):
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.uint32)
    assert off.shape == ln.shape
    return off, ln


class Scratch:
    def __init__(self, db):
        self.ptr = C.c_void_p()
        _check(lib().hs_alloc_scratch(db.ptr, C.byref(self.ptr)), "hs_alloc_scratch")

    def add(self, db):
        _check(lib().hs_alloc_scratch(db.ptr, C.byref(self.ptr)), "hs_alloc_scratch")

    def free(self):
        if self.ptr:
            lib().hs_free_scratch(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def size(self):
        n = C.c_size_t()
        _check(lib().hs_scratch_size(self.ptr, C.byref(n)))
        return n.value

    def counters(self):
        """[records, error, candidates, confirmed, prefilter_pass, ...] of the last scan."""
        out = (C.c_uint * 8)()
        _check(lib().hs_b200_last_counters(self.ptr, C.byref(out)))
        return list(out)

    def last_kernel_ms(self):
        return float(lib().hs_b200_last_kernel_ms(self.ptr))


def scan(db, data, scratch, on_event=None, stop_after=0):
    """hs_scan(): returns (rc, [(id, to), ...]) in delivery order."""
    a = _as_u8(data)
    out = []

    def cb(i, frm, to, flags, ctx):
        out.append((int(i), int(to)))
        if on_event is not None:
            return int(on_event(i, frm, to, flags))
        if stop_after and len(out) >= stop_after:
            return 1
        return 0

    keep = np.zeros(1, dtype=np.uint8) if a.size == 0 else a
    rc = lib().hs_scan(db.ptr, keep.ctypes.data, a.size, 0, scratch.ptr, MATCH_CB(cb), None)
    return rc, out


def scan_blocks(db, data, offsets, lengths, scratch, collect=True):
    """hs_b200_scan_blocks() on HOST buffers: returns a MATCH_DTYPE array in
    (block, to, id) order (or just the count when collect=False)."""
    a = _as_u8(data)
    off, ln = _blocks(offsets, lengths)
    n = C.c_ulonglong()
    if not collect:
        rc = lib().hs_b200_scan_blocks(db.ptr, a.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                       off.size, scratch.ptr, BLOCK_CB(), None, C.byref(n))
        _check(rc, "hs_b200_scan_blocks")
        return int(n.value)
    recs = []

    def cb(block, i, frm, to, flags, ctx):
        recs.append((i, block, to))
        return 0

    rc = lib().hs_b200_scan_blocks(db.ptr, a.ctypes.data, off.ctypes.data, ln.ctypes.data, off.size,
                                   scratch.ptr, BLOCK_CB(cb), None, C.byref(n))
    _check(rc, "hs_b200_scan_blocks")
    return np.array(recs, dtype=MATCH_DTYPE) if recs else np.zeros(0, dtype=MATCH_DTYPE)


def scan_blocks_collect(db, data, offsets, lengths, scratch, out):
    """hs_b200_scan_blocks_collect() on HOST buffers: the delivered matches, ordered
    by (block, to, id), land in the caller's MATCH_DTYPE array `out`; returns the
    count (grows nothing: HsError HS_INSUFFICIENT_SPACE if `out` is too small)."""
    a = _as_u8(data)
    off, ln = _blocks(offsets, lengths)
    n = C.c_ulonglong()
    rc = lib().hs_b200_scan_blocks_collect(db.ptr, a.ctypes.data, off.ctypes.data, ln.ctypes.data, off.size,
                                           scratch.ptr, out.ctypes.data, out.size, C.byref(n))
    _check(rc, "hs_b200_scan_blocks_collect")
    return int(n.value)


class Corpus:
    """Device-resident corpus (hs_b200_corpus_upload / hs_b200_corpus_wrap)."""

    def __init__(self, ptr, keep=None):
        self.ptr = ptr
        self._keep = keep

    @staticmethod
    def upload(data, offsets, lengths, device=0):
        a = _as_u8(data)
        off, ln = _blocks(offsets, lengths)
        out = C.c_void_p()
        _check(lib().hs_b200_corpus_upload(a.ctypes.data, off.ctypes.data, ln.ctypes.data, off.size,
                                           device, C.byref(out)), "corpus_upload")
        return Corpus(out)

    @staticmethod
    def wrap(dev_ptr, nbytes, offsets, lengths, device=0, keep=None):
        off, ln = _blocks(offsets, lengths)
        out = C.c_void_p()
        _check(lib().hs_b200_corpus_wrap(C.c_void_p(dev_ptr), nbytes, off.ctypes.data, ln.ctypes.data,
                                         off.size, device, C.byref(out)), "corpus_wrap")
        return Corpus(out, keep)

    def payload_bytes(self):
        return int(lib().hs_b200_corpus_bytes(self.ptr))

    def free(self):
        if self.ptr:
            lib().hs_b200_corpus_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def scan_corpus_async(db, corpus, scratch, stream=None):
    _check(lib().hs_b200_scan_corpus_async(db.ptr, corpus.ptr, scratch.ptr, C.c_void_p(stream or 0)),
           "scan_corpus_async")


def scan_corpus_finish(scratch):
    """Returns (rc, nrecords, device pointer of the raw record array)."""
    n = C.c_ulonglong()
    p = C.c_void_p()
    rc = lib().hs_b200_scan_corpus_finish(scratch.ptr, C.byref(n), C.byref(p))
    return rc, int(n.value), p.value


def fetch_matches(db, scratch):
    n = C.c_ulonglong()
    _check(lib().hs_b200_fetch_matches(db.ptr, scratch.ptr, None, 0, C.byref(n)), "fetch count")
    out = np.zeros(int(n.value), dtype=MATCH_DTYPE)
    if n.value:
        _check(lib().hs_b200_fetch_matches(db.ptr, scratch.ptr, out.ctypes.data, out.size, C.byref(n)),
               "fetch")
    return out


def scan_corpus(db, corpus, scratch, fetch=True):
    """Scan a device-resident corpus; re-runs once if the record ring had to grow."""
    for _ in range(3):
        scan_corpus_async(db, corpus, scratch)
        rc, n, _ = scan_corpus_finish(scratch)
        if rc == HS_INSUFFICIENT_SPACE:
            continue
        _check(rc, "scan_corpus_finish")
        return fetch_matches(db, scratch) if fetch else n
    raise HsError(HS_INSUFFICIENT_SPACE, "record ring")


def postprocess_matches(db, recs):
    """Host-side report rules over raw records (no GPU needed)."""
    recs = np.array(recs, dtype=MATCH_DTYPE, copy=True)
    n = C.c_ulonglong()
    _check(lib().hs_b200_postprocess_matches(db.ptr, recs.ctypes.data, recs.size, C.byref(n)))
    return recs[: int(n.value)]


def launch_count():
    return int(lib().hs_b200_launch_count())


class Stream:
    """hs_open_stream / hs_scan_stream / hs_close_stream."""

    def __init__(self, db, ptr=None):
        self.db = db
        self.ptr = ptr or C.c_void_p()
        if ptr is None:
            _check(lib().hs_open_stream(db.ptr, 0, C.byref(self.ptr)), "hs_open_stream")

    def scan(self, data, scratch, stop_after=0):
        """Returns (rc, [(id, to), ...]) for one write."""
        a = _as_u8(data)
        out = []

        def cb(i, frm, to, flags, ctx):
            out.append((int(i), int(to)))
            return 1 if (stop_after and len(out) >= stop_after) else 0

        keep = np.zeros(1, dtype=np.uint8) if a.size == 0 else a
        rc = lib().hs_scan_stream(self.ptr, keep.ctypes.data, a.size, 0, scratch.ptr, MATCH_CB(cb), None)
        return rc, out

    def copy(self):
        p = C.c_void_p()
        _check(lib().hs_copy_stream(C.byref(p), self.ptr), "hs_copy_stream")
        return Stream(self.db, p)

    def compress(self):
        """hs_compress_stream: size query with a NULL buffer, then the bytes."""
        used = C.c_size_t()
        rc = lib().hs_compress_stream(self.ptr, None, 0, C.byref(used))
        if rc != HS_INSUFFICIENT_SPACE:
            raise HsError(rc, "hs_compress_stream size query")
        buf = C.create_string_buffer(used.value)
        _check(lib().hs_compress_stream(self.ptr, buf, used.value, C.byref(used)), "hs_compress_stream")
        return buf.raw[:used.value]

    @staticmethod
    def expand(db, blob):
        p = C.c_void_p()
        _check(lib().hs_expand_stream(db.ptr, C.byref(p), blob, len(blob)), "hs_expand_stream")
        return Stream(db, p)

    def reset_and_expand(self, blob, scratch):
        return lib().hs_reset_and_expand_stream(self.ptr, blob, len(blob), scratch.ptr, MATCH_CB(), None)

    def reset(self, scratch):
        _check(lib().hs_reset_stream(self.ptr, 0, scratch.ptr, MATCH_CB(), None))

    def close(self, scratch):
        if self.ptr:
            rc = lib().hs_close_stream(self.ptr, scratch.ptr, MATCH_CB(), None)
            self.ptr = C.c_void_p()
            return rc
        return HS_SUCCESS


def scan_vector(db, buffers, scratch, stop_after=0):
    """hs_scan_vector(): `buffers` = list of bytes-like; returns (rc, [(id, to), ...])
    in delivery order, `to` counted from the start of the first buffer."""
    arrs = [_as_u8(b) for b in buffers]
    pad = np.zeros(1, dtype=np.uint8)
    ptrs = (C.c_void_p * max(1, len(arrs)))(*[(a if a.size else pad).ctypes.data for a in arrs])
    lens = (C.c_uint * max(1, len(arrs)))(*[a.size for a in arrs])
    out = []

    def cb(i, frm, to, flags, ctx):
        out.append((int(i), int(to)))
        return 1 if (stop_after and len(out) >= stop_after) else 0

    rc = lib().hs_scan_vector(db.ptr, ptrs, lens, len(arrs), 0, scratch.ptr, MATCH_CB(cb), None)
    return rc, out


class StreamSet:
    """hs_b200_streams_open / scan / close: many streams, state resident in HBM."""

    def __init__(self, db, nstreams, device=0, out_cap=1 << 22):
        self.db = db
        self.n = nstreams
        self._out = np.zeros(out_cap, dtype=MATCH_DTYPE)
        self.ptr = C.c_void_p()
        _check(lib().hs_b200_streams_open(db.ptr, nstreams, device, C.byref(self.ptr)), "streams_open")

    def scan(self, data, offsets, lengths, scratch, collect=True):
        a = _as_u8(data)
        off, ln = _blocks(offsets, lengths)
        assert off.size == self.n
        n = C.c_ulonglong()
        keep = a if a.size else np.zeros(1, dtype=np.uint8)
        if not collect:
            rc = lib().hs_b200_streams_scan(self.ptr, keep.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                            scratch.ptr, BLOCK_CB(), None, C.byref(n))
            _check(rc, "streams_scan")
            return int(n.value)
        rc = lib().hs_b200_streams_scan_collect(self.ptr, keep.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                                scratch.ptr, self._out.ctypes.data, self._out.size, C.byref(n))
        if rc == HS_INSUFFICIENT_SPACE:
            raise HsError(rc, "streams_scan_collect: %d matches exceed the harness buffer" % n.value)
        _check(rc, "streams_scan_collect")
        return self._out[: int(n.value)].copy()

    def close(self):
        if self.ptr:
            lib().hs_b200_streams_close(self.ptr)
            self.ptr = C.c_void_p()


def test_program_base():
    lib().hs_b200_test_program_base.restype = C.c_uint
    return lib().hs_b200_test_program_base()


def compile_programs(lits, nocase, prog_off, area, ekey_count=0, inv_dkey=()):
    """hs_b200_test_compile_programs: pure-literal block database whose literal
    programs are the raw instruction bytes in `area` (test hook)."""
    n = len(lits)
    lits = [bytes(x) for x in lits]
    bufs = [C.create_string_buffer(x, len(x) + 1) for x in lits]
    arr = (C.c_char_p * n)(*[C.cast(b, C.c_char_p) for b in bufs])
    lens = (C.c_size_t * n)(*[len(x) for x in lits])
    nc = (C.c_uint * n)(*[int(bool(x)) for x in nocase])
    po = (C.c_uint * n)(*prog_off)
    inv = (C.c_uint * max(1, len(inv_dkey)))(*inv_dkey)
    db = C.c_void_p()
    L = lib()
    L.hs_b200_test_compile_programs.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_size_t),
                                                C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.c_uint,
                                                C.c_char_p, C.c_size_t, C.c_uint, C.POINTER(C.c_uint),
                                                C.c_uint, C.POINTER(C.c_void_p)]
    area = bytes(area)
    _check(L.hs_b200_test_compile_programs(arr, lens, nc, po, n, area, len(area), ekey_count, inv,
                                           len(inv_dkey), C.byref(db)), "test_compile_programs")
    return Database(db)


def dfa_from_literals(lits, caseless=None, reports=None, anchored=False, kind=0, sherman=False):
    """hs_b200_dfa_from_literals: Aho-Corasick DFA of a literal set as a reference-format
    engine (struct NFA + McClellan 8/16 or Sheng).  Returns the bytes."""
    n = len(lits)
    lits = [bytes(x) for x in lits]
    bufs = [C.create_string_buffer(x, len(x) + 1) for x in lits]
    arr = (C.c_char_p * n)(*[C.cast(b, C.c_char_p) for b in bufs])
    lens = (C.c_size_t * n)(*[len(x) for x in lits])
    cl = (C.c_uint * n)(*[int(bool(x)) for x in (caseless or [0] * n)])
    rp = (C.c_uint * n)(*(reports if reports is not None else list(range(n))))
    L = lib()
    L.hs_b200_dfa_from_literals.restype = C.c_long
    L.hs_b200_dfa_from_literals.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), C.POINTER(C.c_uint),
                                            C.POINTER(C.c_uint), C.c_uint, C.c_int, C.c_int, C.c_int,
                                            C.c_void_p, C.c_size_t]
    cap = 64 << 20
    out = C.create_string_buffer(cap)
    sz = L.hs_b200_dfa_from_literals(arr, lens, cl, rp, n, int(anchored), kind, int(sherman), out, cap)
    if sz < 0:
        raise HsError(HS_COMPILER_ERROR, "dfa_from_literals")
    return out.raw[:sz]


def dfa_from_table(next_table, start_anchored, start_floating, reports, reports_eod, kind=0, sherman=False):
    """hs_b200_dfa_from_table: next_table uint16 [nstates, 256]; reports / reports_eod: one list
    of report ids per state.  Returns the engine bytes."""
    nt = np.ascontiguousarray(next_table, dtype=np.uint16)
    n = nt.shape[0]

    def flat(lists):
        off = np.zeros(n + 1, dtype=np.uint32)
        off[1:] = np.cumsum([len(x) for x in lists])
        vals = np.array([v for x in lists for v in x] + [0], dtype=np.uint32)
        return off, vals

    ro, rv = flat(reports)
    eo, ev = flat(reports_eod)
    L = lib()
    L.hs_b200_dfa_from_table.restype = C.c_long
    L.hs_b200_dfa_from_table.argtypes = [C.c_uint, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t]
    cap = 64 << 20
    out = C.create_string_buffer(cap)
    sz = L.hs_b200_dfa_from_table(n, nt.ctypes.data, start_anchored, start_floating, ro.ctypes.data, rv.ctypes.data,
                                  eo.ctypes.data, ev.ctypes.data, kind, int(sherman), out, cap)
    if sz < 0:
        raise HsError(HS_COMPILER_ERROR, "dfa_from_table")
    return out.raw[:sz]


def limex32_from_literals(lits, caseless, reports):
    """hs_b200_limex32_from_literals: the engine bytes (struct NFA + LimExNFA32 ...)."""
    n = len(lits)
    arr = (C.c_char_p * n)(*[bytes(x) for x in lits])
    lens = (C.c_size_t * n)(*[len(x) for x in lits])
    cl = (C.c_uint * n)(*[int(bool(x)) for x in (caseless or [0] * n)])
    rp = (C.c_uint * n)(*[int(x) for x in reports])
    L = lib()
    L.hs_b200_limex32_from_literals.restype = C.c_long
    L.hs_b200_limex32_from_literals.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p,
                                                C.c_size_t]
    cap = 1 << 20
    out = C.create_string_buffer(cap)
    sz = L.hs_b200_limex32_from_literals(arr, lens, cl, rp, n, out, cap)
    if sz < 0:
        raise HsError(HS_COMPILER_ERROR, "limex32_from_literals")
    return out.raw[:sz]


def limex32_from_spec(reach, init, init_ds, succ, reports, reports_eod, squash_mask=None, squash_kind=None):
    """hs_b200_limex32_from_spec: reach uint32[256], succ uint32[nstates], reports / reports_eod one
    list of report ids per state, squash_kind uint8[nstates] (0 / 1 / 3) with squash_mask."""
    sc = np.ascontiguousarray(succ, dtype=np.uint32)
    n = sc.size
    rc = np.ascontiguousarray(reach, dtype=np.uint32)

    def flat(lists):
        off = np.zeros(n + 1, dtype=np.uint32)
        off[1:] = np.cumsum([len(x) for x in lists])
        vals = np.array([v for x in lists for v in x] + [0], dtype=np.uint32)
        return off, vals

    ro, rv = flat(reports)
    eo, ev = flat(reports_eod)
    sm = np.ascontiguousarray(squash_mask if squash_mask is not None else np.full(n, 0xffffffff), dtype=np.uint32)
    sk = np.ascontiguousarray(squash_kind if squash_kind is not None else np.zeros(n), dtype=np.uint8)
    L = lib()
    L.hs_b200_limex32_from_spec.restype = C.c_long
    L.hs_b200_limex32_from_spec.argtypes = [C.c_uint, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_size_t]
    cap = 1 << 20
    out = C.create_string_buffer(cap)
    sz = L.hs_b200_limex32_from_spec(n, rc.ctypes.data, int(init), int(init_ds), sc.ctypes.data, sm.ctypes.data,
                                     sk.ctypes.data, ro.ctypes.data, rv.ctypes.data, eo.ctypes.data, ev.ctypes.data,
                                     out, cap)
    if sz < 0:
        raise HsError(HS_COMPILER_ERROR, "limex32_from_spec")
    return out.raw[:sz]


def limex_from_spec64(reach, init, init_ds, succ, reports, reports_eod, squash_mask=None, squash_kind=None):
    """hs_b200_limex_from_spec64: as limex32_from_spec over uint64 state sets (up to 64 states)."""
    sc = np.ascontiguousarray(succ, dtype=np.uint64)
    n = sc.size
    rc = np.ascontiguousarray(reach, dtype=np.uint64)

    def flat(lists):
        off = np.zeros(n + 1, dtype=np.uint32)
        off[1:] = np.cumsum([len(x) for x in lists])
        vals = np.array([v for x in lists for v in x] + [0], dtype=np.uint32)
        return off, vals

    ro, rv = flat(reports)
    eo, ev = flat(reports_eod)
    sm = np.ascontiguousarray(squash_mask if squash_mask is not None else np.full(n, 0xffffffffffffffff, dtype=np.uint64),
                              dtype=np.uint64)
    sk = np.ascontiguousarray(squash_kind if squash_kind is not None else np.zeros(n), dtype=np.uint8)
    L = lib()
    L.hs_b200_limex_from_spec64.restype = C.c_long
    L.hs_b200_limex_from_spec64.argtypes = [C.c_uint, C.c_void_p, C.c_ulonglong, C.c_ulonglong, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_size_t]
    cap = 1 << 20
    out = C.create_string_buffer(cap)
    sz = L.hs_b200_limex_from_spec64(n, rc.ctypes.data, int(init), int(init_ds), sc.ctypes.data, sm.ctypes.data,
                                     sk.ctypes.data, ro.ctypes.data, rv.ctypes.data, eo.ctypes.data, ev.ctypes.data,
                                     out, cap)
    if sz < 0:
        raise HsError(HS_COMPILER_ERROR, "limex_from_spec64")
    return out.raw[:sz]


def limex_from_spec_wide(reach, init, init_ds, succ, reports, reports_eod, squash_mask=None, squash_kind=None):
    """hs_b200_limex_from_spec_wide: state sets are Python ints (bit i = state i), up to 512 states; the model
    emitted is the smallest of 32 / 64 / 128 / 256 / 512 that holds len(succ) states."""
    n = len(succ)
    words = max(1, (n + 63) // 64)
    m64 = (1 << 64) - 1

    def sets(vals):
        return np.array([(int(v) >> (64 * j)) & m64 for v in vals for j in range(words)], dtype=np.uint64)

    def flat(lists):
        off = np.zeros(n + 1, dtype=np.uint32)
        off[1:] = np.cumsum([len(x) for x in lists])
        vals = np.array([v for x in lists for v in x] + [0], dtype=np.uint32)
        return off, vals

    ro, rv = flat(reports)
    eo, ev = flat(reports_eod)
    rc, sc = sets(reach), sets(succ)
    i0, i1 = sets([init]), sets([init_ds])
    sm = sets(squash_mask if squash_mask is not None else [(1 << (64 * words)) - 1] * n)
    sk = np.ascontiguousarray(squash_kind if squash_kind is not None else np.zeros(n), dtype=np.uint8)
    L = lib()
    L.hs_b200_limex_from_spec_wide.restype = C.c_long
    L.hs_b200_limex_from_spec_wide.argtypes = [C.c_uint, C.c_uint] + [C.c_void_p] * 11 + [C.c_size_t]
    cap = 4 << 20
    out = C.create_string_buffer(cap)
    sz = L.hs_b200_limex_from_spec_wide(n, words, rc.ctypes.data, i0.ctypes.data, i1.ctypes.data, sc.ctypes.data,
                                        sm.ctypes.data, sk.ctypes.data, ro.ctypes.data, rv.ctypes.data, eo.ctypes.data,
                                        ev.ctypes.data, out, cap)
    if sz < 0:
        raise HsError(HS_COMPILER_ERROR, "limex_from_spec_wide")
    return out.raw[:sz]


def nfa_scan_corpus(nfa_bytes, corpus, cap=1 << 20):
    """hs_b200_nfa_scan_corpus: the engine over every block of a resident corpus.
    Returns (records MATCH_DTYPE ordered by (block, to, id), kernel ms)."""
    L = lib()
    L.hs_b200_nfa_scan_corpus.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.POINTER(C.c_ulonglong), C.POINTER(C.c_float)]
    n = C.c_ulonglong()
    ms = C.c_float()
    for _ in range(3):
        out = np.zeros(cap, dtype=MATCH_DTYPE)
        rc = L.hs_b200_nfa_scan_corpus(nfa_bytes, len(nfa_bytes), corpus.ptr, out.ctypes.data, cap, C.byref(n),
                                       C.byref(ms))
        if rc == HS_INSUFFICIENT_SPACE:
            cap = int(n.value) + 16
            continue
        _check(rc, "nfa_scan_corpus")
        return out[: int(n.value)], float(ms.value)
    raise HsError(HS_INSUFFICIENT_SPACE, "nfa_scan_corpus")
