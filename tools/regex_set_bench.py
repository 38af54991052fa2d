"""Expression sets split into several engines, on the device: every engine of one model in one launch, against
the same engines run one at a time.

  python tools/regex_set_bench.py [--sizes 50,200,1000] [--mib 512] [--repeats 5] [--out DIR]

Workload: seeded sets of recorded hscollider regex patterns (tests/golden/hscollider_regex.json), over a resident
corpus of --mib MiB (larger than the 126 MB L2) of seeded printable text in 1 KiB blocks.  Patterns that match
more than once per KiB of a sample are left out of the sets: their records, not the scan, would be measured.
Reports per set: the engines by model, compile time, kernel time by CUDA events (warmed up, best and median of
--repeats) and Gbit/s of
  - the new launch over the corpus (hs_b200_scan_corpus),
  - (a) the same engines one at a time through hs_b200_nfa_scan_corpus, times summed,
  - (b) hs_scan-sized work: one 1 MiB buffer, the new launch against per-engine launches,
  - (c) the unmodified reference hs_scan on all cores (where oracle/_ref is built; over a 16 MiB slice),
and the record counts of both device paths (the per-engine path's are raw engine reports, before the report programs
resolve them).  One JSON line per set, with the card's name and power limit."""
import argparse
import base64
import json
import os
import struct
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hyperscan_b200 import capi  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def corpus(mib, seed=7):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz ABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789 .,;:-_/=\n", np.uint8)
    data = alpha[rng.integers(0, alpha.size, size=mib << 20, dtype=np.uint8)]
    n = (mib << 20) // 1024
    return data, np.arange(n, dtype=np.uint64) * 1024, np.full(n, 1024, np.uint32)


def engines_bytes(db):
    """the serialized engines of a database, queue order (RoseEngine.nfaInfoOffset -> NfaInfo -> struct NFA)"""
    bc = db.serialize()[32:]
    n = struct.unpack_from("<I", bc, capi._ROSE_QUEUE_COUNT)[0]
    at = struct.unpack_from("<I", bc, capi._ROSE_NFA_INFO)[0]
    out = []
    for q in range(n):
        off = struct.unpack_from("<I", bc, at + q * capi._NFA_INFO_SIZE)[0]
        length = struct.unpack_from("<I", bc, off + 4)[0]
        out.append(bc[off:off + length])
    return out


def timed(fn, repeats):
    fn()
    ms = [fn() for _ in range(repeats)]
    return min(ms), float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="50,200,1000")
    ap.add_argument("--mib", type=int, default=512)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    with open(os.path.join(ROOT, "tests", "golden", "hscollider_regex.json")) as f:
        cases = json.load(f)
    cases = cases["cases"] if isinstance(cases, dict) else cases
    name = card()
    data, off, ln = corpus(a.mib)
    big = capi.Corpus.upload(data, off, ln)
    one = capi.Corpus.upload(data[: 1 << 20], np.array([0], np.uint64), np.array([1 << 20], np.uint32))
    sample = capi.Corpus.upload(data[: 1 << 20], off[:1024], ln[:1024])
    # the pool: every recorded pattern that compiles alone and matches at most once per KiB of the sample
    pool = [c for c in cases if not c.get("ext")]
    every = capi.compile_multi([base64.b64decode(c["pattern"]) for c in pool], [c["hs_flags"] for c in pool],
                               list(range(len(pool))))
    s = capi.Scratch(every)
    counts = np.bincount(capi.scan_corpus(every, sample, s)["id"].astype(np.int64), minlength=len(pool))
    s.free()
    pool = [c for c, k in zip(pool, counts) if k <= 1024]
    results = []
    for size in [int(x) for x in a.sizes.split(",")]:
        rng = np.random.default_rng(size)
        pick = [pool[int(i)] for i in sorted(rng.choice(len(pool), size=min(size, len(pool)), replace=False))]
        t0 = time.perf_counter()
        db = capi.compile_multi([base64.b64decode(c["pattern"]) for c in pick], [c["hs_flags"] for c in pick],
                                [c["id"] for c in pick])
        compile_s = time.perf_counter() - t0
        models = {}
        for m, _ in db.engines():
            models[m] = models.get(m, 0) + 1
        scratch = capi.Scratch(db)

        def launch(c):
            def run():
                capi.scan_corpus(db, c, scratch, fetch=False)
                return scratch.last_kernel_ms()
            return run
        new_best, new_med = timed(launch(big), a.repeats)
        one_best, one_med = timed(launch(one), a.repeats)
        got = np.sort(capi.scan_corpus(db, big, scratch), order=["block", "to", "id"])
        engs = engines_bytes(db)
        per, per_one, raw = [], [], 0
        for e in engs:
            r, _ = capi.nfa_scan_corpus(e, big)
            raw += r.size
            per.append(timed(lambda: capi.nfa_scan_corpus(e, big, cap=r.size + 16)[1], a.repeats))
            per_one.append(timed(lambda: capi.nfa_scan_corpus(e, one, cap=1 << 16)[1], a.repeats))
        ref = None
        import oracle.ref as oref
        if oref.live():
            sl = 16 << 10
            secs, _, nbytes = oref.bench_blocks(db.ptr, data[: sl * 1024], off[:sl], ln[:sl],
                                                len(os.sched_getaffinity(0)), 1)
            ref = {"gbit_s": round(nbytes * 8 / secs / 1e9, 3), "threads": len(os.sched_getaffinity(0)),
                   "mib": 16}
        gbit = lambda ms, nbytes: round(nbytes * 8 / (ms * 1e-3) / 1e9, 2)  # noqa: E731
        per_sum = sum(b for b, _ in per)
        per_one_sum = sum(b for b, _ in per_one)
        res = {"set": size, "engines": models, "compile_s": round(compile_s, 2), "records": int(got.size),
               "corpus_mib": a.mib, "block_bytes": 1024,
               "new_launch_ms": round(new_best, 3), "new_launch_median_ms": round(new_med, 3),
               "new_launch_gbit_s": gbit(new_best, a.mib << 20),
               "a_per_engine_sum_ms": round(per_sum, 3), "a_per_engine_gbit_s": gbit(per_sum, a.mib << 20),
               "b_1mib_new_ms": round(one_best, 4), "b_1mib_per_engine_sum_ms": round(per_one_sum, 4),
               "c_reference_cpu": ref or "not measured (oracle/_ref not built)",
               "per_engine_raw_records": raw, "card": name}
        print(json.dumps(res), flush=True)
        results.append(res)
        scratch.free()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "regex_set_bench.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
