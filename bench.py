#!/usr/bin/env python
"""hsbench-style block-mode throughput of the B200 scan runtime.

  python bench.py --gpus N --steps K --warmup W            (ours)
  python bench.py --impl reference --gpus N --steps K ...  (reference CPU arm)

Workload = BASELINE.json configs[1]: 1 000 short literals, 1 GiB synthetic corpus
as 2^20 blocks x 1 KiB, block mode, one B200 (per rank; blocks shard by rank).
One "step" = one hsbench repeat GROUP: --passes-per-step (default 40) passes of the
literal scan path over the whole resident corpus (hsbench's inner loop: every block
through hs_scan once per repeat, -n repeats, tools/hsbench/main.cpp:503-527); the
default --steps 10 therefore times 400 passes (~146 ms per GPU), so that a barrier
is < 0.5 % of the region and nvidia-smi gets its samples.  The region is timed with
CUDA events on the launching stream, max over ranks (the wall clock with the closing
barrier is printed beside it).  Metric: Gbit/s = 8 * corpus bytes * passes / seconds /
1e9 (main.cpp:721-725), whole job.

Prints ONE JSON line (rank 0):
  value      corpus resident in HBM, device-timed region, max over ranks
  e2e        hs_b200_scan_blocks_collect() on HOST (pinned) buffers: H2D of the
             corpus, scan, D2H of the records, host ordering -- the delivered
             match list in (block, to, id) order lands in a host array
  roofline   dominant kernel (class-pair first stage + confirm) by CUDA events
             recorded by the library around it on its stream
  secondary  (N = 1) the other literal configurations of BASELINE.json, each with
             kernel-event roofline and a bit-exact check against the reference
             runtime: config 1 through the stock hs_scan, Teddy 48, fat Teddy 96,
             config-5 shape (50 000 literals), config-4 shape (stream set), the DFA
             engines (McClellan 8 / 16, Sheng) against the reference engines
             (N > 1) the config-5 shape sharded at 8 GiB per GPU
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "hsbench block-mode scan throughput (Gbit/s scanned), match set bit-exact vs CPU ref"
KERNEL_SRC = os.path.join(ROOT, "hyperscan_b200", "csrc", "device", "scan_kernels.cu")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--passes-per-step", type=int, default=40)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--lits", type=int, default=1000)
    ap.add_argument("--blocks", type=int, default=1 << 20)
    ap.add_argument("--block-len", type=int, default=1024)
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 5)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--cpu-sample-mb", type=int, default=1024)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--verify-blocks", type=int, default=4096)
    ap.add_argument("--secondary-mb", type=int, default=512)
    ap.add_argument("--shard-gib", type=int, default=8, help="N>1 secondary: config-5 shape, GiB per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the matches of the last timed pass (rank 0) to DIR/match_{block,to,id}.npy")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: p2p = records stored into every rank's buffer by the confirm kernel itself over "
                         "NVLink peer memory; nccl = one all-gather per pass")
    return ap.parse_args()


def workload(args, rank):
    """Seeded literal set (same on every rank) and this rank's shard of blocks."""
    from hyperscan_b200 import synth
    lits, flags, ids = synth.literal_set(args.lits, min_len=4, max_len=8, caseless_frac=0.1, seed=2)
    data, off, ln, planted = synth.block_corpus(args.blocks, args.block_len, lits, plant_per_kb=0.01,
                                                seed=7 + 1000 * rank)
    return lits, flags, ids, data, off, ln, planted


def config_of(args, n, info=None):
    c = {"workload": "hsbench configs[1]: %d short literals (len 4-8, [a-z], 10%% caseless), "
                     "%d blocks x %d B per GPU, block mode" % (args.lits, args.blocks, args.block_len),
         "corpus_bytes_per_gpu": args.blocks * args.block_len,
         "passes_per_step": args.passes_per_step,
         "l2": "inputs larger than L2 (corpus >> 126 MB), no flush needed",
         "sharding": "blocks sharded by rank, database replicated" if n > 1 else "single GPU"}
    if args.blocks * args.block_len <= 256 << 20:
        c["l2"] = "WARNING: corpus not much larger than L2"
    if info is not None:
        c["engine"] = engine_name(info)
    return c


def engine_name(info):
    if info.hwlm_type == 12 and info.engine_id == 0:
        return "FDR domain %d stride %d" % (info.fdr_domain, info.fdr_stride)
    return "Teddy id %d" % info.engine_id if info.hwlm_type == 12 else "noodle"


def usable_cores():
    """Host cores this container may actually use: the cgroup CPU quota when
    there is one (the GPU boxes expose 128 logical CPUs but cap the container at
    16 to 96 CPUs' worth of time; more runnable threads than that only get
    throttled), else the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def close(self):
        if self.proc:
            self.proc.terminate()
            self.proc = None

    def window(self, t0, t1):
        """median SM clock / throttle reasons of the samples taken in [t0, t1] (wall clock)"""
        if not self.proc:
            return None
        time.sleep(0.15)
        sm, mx, reasons = [], 0, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"],
                               f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": mx or None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def pinned_threads():
    """hsbench pins its scan threads 1:1 to cores (tools/hsbench/main.cpp:211-222):
    one thread per usable core, each pinned to its own physical core."""
    import oracle.ref as ref
    threads = usable_cores()
    cpus = ref.physical_core_cpus()
    if len(cpus) >= threads:
        ref.pin_bench_threads(cpus[:threads])
        return threads, "pinned 1:1 to cpus %s" % (",".join(map(str, cpus[:threads])))
    ref.pin_bench_threads([])
    return threads, "unpinned (affinity mask smaller than the thread count)"


def cpu_reference_run(db, data, off, ln, sample_mb, seconds):
    """Time the reference's own CPU hs_scan (oracle/_ref, unmodified sources)
    on a bounded sample of the workload, hsbench style."""
    import oracle.ref as ref
    threads, pin = pinned_threads()
    nblk = max(1, min(len(off), (sample_mb << 20) // max(1, int(ln[0]))))
    o, l = off[:nblk], ln[:nblk]
    sample_bytes = int(l.sum())
    ref.bench_blocks(db.ptr, data, o, l, threads, 1)            # warm (threads, page cache)
    t3, _, _ = ref.bench_blocks(db.ptr, data, o, l, threads, 3)
    reps = max(1, min(2000, int(seconds / max(t3 / 3, 1e-4))))
    t, m, b = ref.bench_blocks(db.ptr, data, o, l, threads, reps)
    # hsbench runs every thread over the whole corpus; ref_driver splits the
    # blocks across threads, so `b` is the bytes all threads scanned
    return {"value": b * 8 / t / 1e9, "unit": "Gbit/s", "cores": threads, "kind": "reference",
            "isa": ref.best_isa(), "threads": pin,
            "sample": "first %d blocks (%.0f MiB) of the same corpus x %d repeats, %d threads, "
                      "unmodified reference hs_scan (oracle/_ref, -O3 %s)" %
                      (nblk, sample_bytes / 2**20, reps, threads, ref.best_isa()),
            "seconds": t, "matches_per_pass": m // reps}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    from hyperscan_b200 import capi
    lits, flags, ids, data, off, ln, _ = workload(args, 0)
    db = capi.compile_lit_multi(lits, flags, ids)
    K, W = args.steps, args.warmup
    import oracle.ref as ref
    threads, pin = pinned_threads()
    nblk = max(1, min(len(off), (args.cpu_sample_mb << 20) // args.block_len))
    o, l = off[:nblk], ln[:nblk]
    for _ in range(W):
        ref.bench_blocks(db.ptr, data, o, l, threads, 1)
    t, m, b = ref.bench_blocks(db.ptr, data, o, l, threads, K)
    val = b * 8 / t / 1e9
    cb = {"value": val, "unit": "Gbit/s", "cores": threads, "kind": "reference", "threads": pin,
          "sample": "each step = first %d blocks (%.0f MiB) of the corpus, one pass, %d threads, unmodified "
                    "reference hs_scan (oracle/_ref %s)" % (nblk, int(l.sum()) / 2**20, threads, ref.best_isa())}
    cfg = config_of(args, args.gpus, db.info())
    cfg["passes_per_step"] = 1
    print(json.dumps({"metric": METRIC, "value": val, "unit": "Gbit/s", "n_gpus": args.gpus, "steps": K,
                      "warmup": W, "ms_per_step": t / K * 1e3, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "impl": "reference", "config": cfg, "cpu_baseline": cb,
                      "e2e": {"value": val, "unit": "Gbit/s", "h2d_bytes_per_step": 0,
                              "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


class Passes:
    """Back-to-back passes over one resident shard, all stream-ordered on ONE
    stream: scan kernel (+ confirm kernel) -> (N>1) the records land in every rank's
    exchange buffer, stored by the confirm kernel over NVLink peer mappings, or one
    NCCL all-gather per pass -> next pass.  The host only enqueues (two scratches
    = two record rings, so it runs up to two passes ahead) and retires a pass's
    counters two passes later."""

    def __init__(self, capi, hdist, torch, dist, db, corpus, dev, world, rank, exchange, block_base):
        self.capi, self.hdist, self.torch, self.dist = capi, hdist, torch, dist
        self.db, self.corpus, self.dev, self.world, self.rank = db, corpus, dev, world, rank
        self.rings = (capi.Scratch(db), capi.Scratch(db))
        self.stream = torch.cuda.Stream(device=dev)
        self.peerx = None
        self.cap = 0
        self.bufs = None
        self.phase = {}
        # one unpipelined pass per record ring: a ring (or its candidate list) that is too small
        # for this workload grows here, not in the timed region
        n0 = 0
        for sc in self.rings:
            for attempt in range(4):
                capi.scan_corpus_async(db, corpus, sc)
                rc, n0, _ = capi.scan_corpus_finish(sc)
                if rc != capi.HS_INSUFFICIENT_SPACE:
                    break
            capi._check(rc, "first pass")
        if world > 1:
            # capacity of the exchange buffers: from that pass, with headroom, same on all ranks
            n_all = torch.tensor([n0], dtype=torch.int64, device=dev)
            dist.all_reduce(n_all, op=dist.ReduceOp.MAX)
            self.cap = (int(n_all.item()) * 3 // 2 + 4095) // 4096 * 4096
            self.bufs = [torch.zeros((self.cap + 1, 2), dtype=torch.int64, device=dev) for _ in range(2)]
            if exchange == "p2p":
                try:
                    self.peerx = hdist.PeerExchange(self.cap)
                    for s in self.rings:
                        self.peerx.attach(s, block_base)
                except Exception as e:   # no peer access on this box: fall back to the collective
                    print("[bench rank %d] peer exchange unavailable (%s): using NCCL all-gather" % (rank, e),
                          file=sys.stderr, flush=True)
                    self.peerx = None
                ok = torch.tensor([1 if self.peerx is not None else 0], dtype=torch.int64, device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if int(ok.item()) == 0 and self.peerx is not None:
                    for s in self.rings:
                        self.peerx.detach(s)
                    self.peerx = None

    def run(self, k):
        capi, torch, dist = self.capi, self.torch, self.dist
        st = self.stream.cuda_stream
        kms, outs, n = [], [], 0

        def retire(sc):
            rc, cnt, _ = capi.scan_corpus_finish(sc)
            if rc != capi.HS_SUCCESS:   # incl. a record ring that had to grow
                raise RuntimeError("scan failed %d (rerun)" % rc)
            kms.append(sc.last_kernel_ms())
            return cnt

        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.stream):
            e0.record(self.stream)
            for i in range(k):
                sc = self.rings[i % 2]
                if i >= 2:
                    n = retire(sc)          # pass i-2 used this scratch
                capi.scan_corpus_async(self.db, self.corpus, sc, st)
                if self.world > 1 and self.peerx is None:
                    buf = self.bufs[i % 2]
                    capi._check(capi.lib().hs_b200_export_records_async(
                        sc.ptr, buf[1:].data_ptr(), self.cap, buf[0:1].data_ptr(), st))
                    out = torch.empty((self.world,) + tuple(buf.shape), dtype=torch.int64, device=self.dev)
                    dist.all_gather_into_tensor(out.view(-1), buf.view(-1))
                    outs = [out]
            e1.record(self.stream)
            for i in range(max(0, k - 2), k):
                n = retire(self.rings[i % 2])
        self.stream.synchronize()
        self.device_ms = e0.elapsed_time(e1)   # first launch .. last kernel (+ exchange) on the launching stream
        res = None
        for out in outs:
            res = self.hdist.fused_result(out, self.cap)
            if res is None:
                raise RuntimeError("record exchange overflowed its buffer (cap %d)" % self.cap)
        return n, res, kms

    def last_scratch(self, k):
        return self.rings[(k - 1) % 2]

    def close(self):
        if self.peerx is not None:
            for s in self.rings:
                self.peerx.detach(s)
            self.peerx.close()
        for s in self.rings:
            s.free()


def replant(base, nblocks, block_len, lits, per_kb, seed):
    """A copy of the first nblocks blocks of `base` with literals of another set planted."""
    rng = np.random.default_rng(seed)
    data = base[: nblocks * block_len].copy()
    nplant = int(nblocks * block_len / 1024.0 * per_kb)
    for w, b, p in zip(rng.integers(0, len(lits), size=nplant), rng.integers(0, nblocks, size=nplant),
                       rng.random(size=nplant)):
        lit = lits[int(w)]
        s = int(b) * block_len + int(p * (block_len - len(lit) + 1))
        data[s:s + len(lit)] = np.frombuffer(lit, dtype=np.uint8)
    return data


def reference_sorted(db, data, off, ln):
    """The reference runtime's matches sorted by (block, to, id); None where
    oracle/_ref is not built (the bit-exact fields are then null)."""
    import oracle.ref as ref
    return ref.scan_sorted(db.ptr, data, off, ln) if ref.live() else None


def same_matches(got, want):
    return None if want is None else bool(np.array_equal(np.sort(got, order=["block", "to", "id"]), want))


DUMP_BYTES = 64 << 20


def dump_outputs(path, matches):
    """The match arrays a caller of the timed path receives, in (block, to, id)
    order, as float64 columns; above DUMP_BYTES a fixed seeded sample of rows."""
    m = np.sort(matches, order=["block", "to", "id"])
    rows = DUMP_BYTES // (3 * 8)
    if m.size > rows:
        m = m[np.sort(np.random.default_rng(0).choice(m.size, size=rows, replace=False))]
    os.makedirs(path, exist_ok=True)
    for f in ("block", "to", "id"):
        np.save(os.path.join(path, "match_%s.npy" % f), m[f].astype(np.float64))


def secondary_block(capi, ref, name, lits, flags, ids, base, nblocks, block_len, peak, platform=None, passes=7):
    """Kernel-event roofline + bit-exact check of one more literal configuration."""
    db = capi.compile_lit_multi(lits, flags, ids, platform=platform)
    data = replant(base, nblocks, block_len, lits, 0.01, 99)
    off = np.arange(nblocks, dtype=np.uint64) * np.uint64(block_len)
    ln = np.full(nblocks, block_len, dtype=np.uint32)
    corpus = capi.Corpus.upload(data, off, ln)
    sc = capi.Scratch(db)
    ms = []
    n = 0
    for i in range(3 + passes):
        capi.scan_corpus_async(db, corpus, sc)
        rc, n, _ = capi.scan_corpus_finish(sc)
        if rc == capi.HS_INSUFFICIENT_SPACE:
            continue
        capi._check(rc, name)
        if i >= 3:
            ms.append(sc.last_kernel_ms())
    got = capi.fetch_matches(db, sc)
    vb = min(4096, nblocks)
    exact = same_matches(got[got["block"] < vb], reference_sorted(db, data, off[:vb], ln[:vb]))
    c = sc.counters()
    kms = float(np.median(ms))
    nbytes = nblocks * block_len
    ach = (nbytes + 16 * int(n)) / (kms * 1e-3) / 1e9
    out = {"engine": engine_name(db.info()), "literals": len(lits), "corpus_bytes": nbytes, "kernel_ms": kms,
           "value_gbit_s_resident": nbytes * 8 / (kms * 1e-3) / 1e9, "roofline_gbs": ach,
           "roofline_frac": ach / peak, "records": int(n), "candidates_per_kb": c[2] / (nbytes / 1024.0),
           "verified_blocks": vb, "bit_exact_vs_reference": exact}
    corpus.free()
    sc.free()
    return out, db, data


def secondary_single_gpu(args, capi, torch, base, peak):
    """The other literal configurations BASELINE.json names, one GPU."""
    import ctypes as C
    import oracle.ref as ref
    from hyperscan_b200 import synth
    sec = {}
    bl = args.block_len
    nb = min(args.blocks, (args.secondary_mb << 20) // bl)

    # configs[0]: simplegrep -- 1 literal, 1 MiB buffer, through the STOCK hs_scan (per-call latency)
    lits, flags, ids = synth.literal_set(1, min_len=6, max_len=6, seed=1)
    out, db, data = secondary_block(capi, ref, "noodle", lits, flags, ids, base, nb, bl, peak)
    one = data[: 1 << 20].tobytes()
    sc = capi.Scratch(db)
    lat = []
    for i in range(60):
        t0 = time.perf_counter()
        rc, m = capi.scan(db, one, sc)
        lat.append(time.perf_counter() - t0)
    want = reference_sorted(db, np.frombuffer(one, dtype=np.uint8), np.array([0], np.uint64),
                            np.array([len(one)], np.uint32))
    out.update({"hs_scan_1mib_call_ms_median": float(np.median(lat[10:]) * 1e3),
                "hs_scan_1mib_gbit_s": len(one) * 8 / float(np.median(lat[10:])) / 1e9,
                "hs_scan_bit_exact": None if want is None else
                sorted(m) == sorted((int(r["id"]), int(r["to"])) for r in want),
                "api": "stock hs_scan(): pack -> H2D -> kernels -> D2H -> ordered callbacks, one call per buffer"})
    sc.free()
    sec["config1_noodle_1lit"] = out

    lits, flags, ids = synth.literal_set(48, min_len=4, max_len=8, seed=48)
    sec["teddy_48lits"], _, _ = secondary_block(capi, ref, "teddy48", lits, flags, ids, base, nb, bl, peak)

    if ref.best_isa() != "corei7":
        lits, flags, ids = synth.literal_set(96, min_len=4, max_len=8, seed=96)
        plat = C.byref(capi.PlatformInfo(0, capi.HS_CPU_FEATURES_AVX2, 0, 0))
        sec["fat_teddy_96lits"], _, _ = secondary_block(capi, ref, "fat96", lits, flags, ids, base, nb, bl, peak,
                                                        platform=plat)

    lits, flags, ids = synth.literal_set(50000, min_len=4, max_len=16, caseless_frac=0.1, seed=5)
    sec["config5_shape_50k_lits"], _, _ = secondary_block(capi, ref, "50k", lits, flags, ids, base, nb, bl, peak)

    # configs[3] shape: stream set, state resident in HBM, writes from pinned host memory
    lits, flags, ids = synth.literal_set(5000, min_len=4, max_len=8, caseless_frac=0.1, seed=4)
    db = capi.compile_lit_multi(lits, flags, ids, mode=capi.HS_MODE_STREAM)
    ns = min(nb, 1 << 18)
    sset = capi.StreamSet(db, ns)
    sc = capi.Scratch(db)
    data = replant(base, ns, bl, lits, 0.01, 98)
    pinned = torch.empty(data.size, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = data
    off = np.arange(ns, dtype=np.uint64) * np.uint64(bl)
    ln = np.full(ns, bl, dtype=np.uint32)
    rounds, got = 4, []
    sset.scan(pinned.numpy(), off, ln, sc, collect=False)          # warm (allocations)
    t0 = time.perf_counter()
    kms = []
    for r in range(rounds):
        got.append(sset.scan(pinned.numpy(), off, ln, sc))
        kms.append(sc.last_kernel_ms())
    dt = time.perf_counter() - t0
    ok = True if ref.live() else None
    for s in (0, ns // 2, ns - 1) if ref.live() else ():          # 5 writes of the same 1 KiB per stream
        cat = np.tile(data[s * bl:(s + 1) * bl], rounds + 1)
        want, err = ref.stream_collect(db.ptr, cat, np.full(rounds + 1, bl, dtype=np.uint32))
        exp = sorted((int(r["block"]) - 1, int(r["id"]), int(r["to"])) for r in want if int(r["block"]) >= 1)
        mine = sorted((r_, int(x["id"]), int(x["to"])) for r_, recs in enumerate(got) for x in recs[recs["block"] == s])
        ok = ok and err == 0 and mine == exp
    sec["config4_shape_stream_set"] = {
        "engine": engine_name(db.info()), "literals": 5000, "streams": ns, "write_bytes": bl, "rounds": rounds,
        "state_bytes_in_hbm": ns * 16, "e2e_gbit_s": ns * bl * 8 * rounds / dt / 1e9, "ms_per_round": dt / rounds * 1e3,
        "scan_kernel_ms": float(np.median(kms)), "sampled_streams_bit_exact_vs_reference_stream_runtime": ok,
        "api": "hs_b200_streams_scan_collect(pinned host writes) -> ordered records on host"}
    sset.close()
    sc.free()

    # DFA / NFA engines (SURVEY section 8a a18-a20): literal-set automata in the reference layout, one block per thread
    kinds = {"mcclellan16_2000lits": (2, 2000, 4, 8), "mcclellan8_30lits": (1, 30, 2, 4), "sheng_4lits": (3, 4, 1, 3),
             "limex32_6lits": (-1, 6, 4, 5)}
    ndfa = nb
    off = np.arange(ndfa, dtype=np.uint64) * np.uint64(bl)
    ln = np.full(ndfa, bl, dtype=np.uint32)
    for name, (kind, nl, lo, hi) in kinds.items():
        alpha = b"abcdefghijklmnopqrstuvwxyz" if nl > 100 else (b"abcdefgh" if nl > 4 else b"abc")
        lits, flags, ids = synth.literal_set(nl, min_len=lo, max_len=hi, seed=nl, caseless_frac=0.0, alphabet=alpha)
        if kind < 0:      # LimEx-32 position automaton of the literals (<= 31 literal bytes)
            eng = capi.limex32_from_literals(lits, None, ids)
        else:
            eng = capi.dfa_from_literals(lits, None, ids, kind=kind)
        data = replant(base, ndfa, bl, lits, 0.01, 97)
        corpus = capi.Corpus.upload(data, off, ln)
        ms = []
        for i in range(6):
            got, kms = capi.nfa_scan_corpus(eng, corpus)
            if i >= 2:
                ms.append(kms)
        vb = min(2048, ndfa)
        def triples(r):
            t = np.stack([r["block"].astype(np.int64), r["to"].astype(np.int64), r["id"].astype(np.int64)], axis=1)
            return t[np.lexsort((t[:, 2], t[:, 1], t[:, 0]))]
        exact = bool(np.array_equal(triples(got[got["block"] < vb]),
                                    triples(ref.nfa_exec_blocks(eng, data, off[:vb], ln[:vb])))) if ref.live() else None
        kms = float(np.median(ms))
        ach = (ndfa * bl + 16 * got.size) / (kms * 1e-3) / 1e9
        sec["dfa_" + name] = {"engine_bytes": len(eng), "blocks": ndfa, "block_len": bl, "kernel_ms": kms,
                              "roofline_gbs": ach, "roofline_frac": ach / peak, "records": int(got.size),
                              "verified_blocks": vb, "bit_exact_vs_reference_engine": exact,
                              "api": "hs_b200_nfa_scan_corpus (nfaExecMcClellan16_B / 8_B / Sheng_B / LimEx32_Q + testEOD "
                                     "semantics)"}
        corpus.free()

    # a regular-expression database: hs_compile -> position automaton -> McClellan DFA when its determinisation
    # stays small (here), else LimEx -> single-outfix database, scanned through the ordinary entry points
    # (DESIGN.md section 10b)
    pats = [rb"ab+c", rb"[0-9]{2,}\.[0-9]", rb"^GET\s", rb"(foo|bar)x*z", rb"q.{2,4}w$"]
    db = capi.compile_multi(pats, [0, 0, 0, capi.HS_FLAG_CASELESS, 0], list(range(1, len(pats) + 1)))
    data = replant(base, ndfa, bl, [b"abbbc", b"123.4", b"GET /", b"fooxxz", b"q123w"], 0.05, 96)
    corpus = capi.Corpus.upload(data, off, ln)
    sc = capi.Scratch(db)
    ms = []
    for i in range(6):
        capi.scan_corpus_async(db, corpus, sc)
        rc, n, _ = capi.scan_corpus_finish(sc)
        if rc == capi.HS_INSUFFICIENT_SPACE:
            continue
        capi._check(rc, "regex")
        if i >= 2:
            ms.append(sc.last_kernel_ms())
    got = capi.fetch_matches(db, sc)
    vb = min(2048, ndfa)
    exact = same_matches(got[got["block"] < vb], reference_sorted(db, data, off[:vb], ln[:vb]))
    kms = float(np.median(ms))
    ach = (ndfa * bl + 16 * int(got.size)) / (kms * 1e-3) / 1e9
    info = db.info()
    engine = {0: "LimEx-32", 1: "LimEx-64", 2: "LimEx-128", 3: "LimEx-256", 5: "LimEx-512", 6: "McClellan-8",
              7: "McClellan-16"}.get(int(info.engine_id), str(int(info.engine_id)))
    sec["regex_5_expressions"] = {
        "expressions": [p.decode() for p in pats], "engine": engine, "engine_states": int(info.num_literals),
        "blocks": ndfa, "block_len": bl, "kernel_ms": kms,
        "roofline_gbs": ach, "roofline_frac": ach / peak, "matches": int(got.size), "verified_blocks": vb,
        "bit_exact_vs_reference_hs_scan": exact,
        "api": "hs_compile_multi -> single-outfix database -> hs_b200_scan_corpus_* / fetch_matches"}
    corpus.free()
    sc.free()
    return sec


def traffic_record():
    """dram bytes per launch from the committed ncu capture, valid only for the kernel
    source it was taken from (profiles/traffic.json carries the source hash)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        with open(KERNEL_SRC, "rb") as f:
            sha = hashlib.sha256(f.read()).hexdigest()[:16]
        if t.get("kernel_source_sha16") != sha:
            return None, "profiles/traffic.json was captured from another build of scan_kernels.cu (%s != %s)" % (
                t.get("kernel_source_sha16"), sha)
        return t.get("dram_bytes_per_launch"), "ncu dram__bytes_read.sum + dram__bytes_write.sum of %s over %s" % (
            t.get("kernel"), t.get("command"))
    except (OSError, ValueError) as e:
        return None, "no capture: %s" % e


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    # libraries (NCCL) print banners on fd 1: keep it for the ONE JSON line
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from hyperscan_b200 import capi, dist as hdist, synth
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the scan path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    lits, flags, ids, data, off, ln, planted = workload(args, rank)
    db = capi.compile_lit_multi(lits, flags, ids)
    info = db.info()
    corpus = capi.Corpus.upload(data, off, ln, device=local)
    corpus_bytes = int(ln.sum())
    K, W, P = args.steps, args.warmup, max(1, args.passes_per_step)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    passes = Passes(capi, hdist, torch, dist, db, corpus, dev, world, rank, args.exchange, rank * args.blocks)
    # the sampler forks nvidia-smi (~100 ms): start it BEFORE the warm-up so that
    # rank 0 enters the timed region together with the other ranks
    sampler = ClockSampler(local) if rank == 0 else None
    passes.run(W * P)
    barrier()
    launches0 = capi.launch_count()
    t0w = time.time()
    t0 = time.perf_counter()
    n, last, kernel_ms = passes.run(K * P)
    t_run = time.perf_counter() - t0
    barrier()
    dt = time.perf_counter() - t0
    t1w = time.time()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, capi.fetch_matches(db, passes.last_scratch(K * P)))
    wall = dt
    dt = passes.device_ms * 1e-3          # CUDA events on the launching stream; the wall clock is printed beside it
    print("[bench rank %d] %d passes: device %.3f ms (events), host run %.3f ms, with barrier %.3f ms, kernel sum %.3f ms"
          % (rank, K * P, dt * 1e3, t_run * 1e3, wall * 1e3, sum(kernel_ms)), file=sys.stderr, flush=True)
    launches = capi.launch_count() - launches0
    clocks = sampler.window(t0w, t1w) if sampler else None
    more = 1 if (sampler and clocks is not None and clocks["samples"] < 3) else 0
    if world > 1:
        mt = torch.tensor([more], dtype=torch.int64, device=dev)
        dist.all_reduce(mt, op=dist.ReduceOp.MAX)
        more = int(mt.item())
    if more:
        # nvidia-smi came up too late for so short a region: every rank keeps the same passes
        # running for about 0.6 s and rank 0 samples those
        t0c = time.time()
        passes.run(max(P, int(0.6 / max(dt / (K * P), 1e-6))))
        if sampler:
            clocks = sampler.window(t0c, time.time())
            clocks["note"] = "sampled over ~0.6 s of the same passes right after the timed region"
    if sampler:
        sampler.close()
    if world > 1:
        tt = torch.tensor([dt, wall], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt, wall = float(tt[0].item()), float(tt[1].item())
        tb = torch.tensor([corpus_bytes, launches], dtype=torch.int64, device=dev)
        dist.all_reduce(tb, op=dist.ReduceOp.SUM)
        total_bytes, launches = int(tb[0].item()), int(tb[1].item())
    else:
        total_bytes = corpus_bytes
    value = total_bytes * 8 * K * P / dt / 1e9

    # ---- parity spot-check on this run's data (not timed) ----------------------
    verify = {}
    matches = capi.fetch_matches(db, passes.last_scratch(K * P))
    verify["matches_per_pass_rank0"] = int(matches.size)
    if rank == 0 and args.verify_blocks and not args.no_cpu:
        vb = min(args.verify_blocks, len(off))
        verify["verified_blocks"] = vb
        verify["bit_exact_vs_reference"] = same_matches(matches[matches["block"] < vb],
                                                        reference_sorted(db, data, off[:vb], ln[:vb]))
    if world > 1:
        verify["exchange"] = "p2p: the confirm kernel stores records into every rank's buffer over NVLink" \
            if passes.peerx is not None else "nccl all_gather_into_tensor per pass"
        barrier()   # every rank's last pass (and its peer stores) has completed
        if rank == 0:
            if passes.peerx is not None:
                counts, merged = passes.peerx.read()
            else:
                counts, gathered = last
                merged = hdist.merge_gathered(counts, gathered, [r * args.blocks for r in range(world)])
            final = capi.postprocess_matches(db, merged)
            verify["gathered_records"] = int(sum(counts))
            verify["merged_matches_all_ranks"] = int(final.size)
            mine = final[final["block"] < args.blocks]
            verify["rank0_slice_equals_local_fetch"] = bool(np.array_equal(
                mine, np.sort(matches, order=["block", "to", "id"])))
            verify["ranks_with_records"] = int(sum(1 for c in counts if c > 0))
        barrier()

    # ---- e2e: host (pinned) buffers through the C ABI ----------------------------
    e2e = None
    scratch = passes.rings[0]
    if not args.no_e2e:
        pinned = torch.empty(data.size, dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = data
        hview = pinned.numpy()
        Ke = args.e2e_steps or min(K, 5)
        recs = np.zeros(max(1 << 16, 4 * int(matches.size)), dtype=capi.MATCH_DTYPE)
        for _ in range(min(W, 3)):
            capi.scan_blocks_collect(db, hview, off, ln, scratch, recs)
        barrier()
        t0 = time.perf_counter()
        nm = 0
        for _ in range(Ke):
            nm = capi.scan_blocks_collect(db, hview, off, ln, scratch, recs)
        barrier()
        de = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([de], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            de = float(tt.item())
        ordered = bool(np.all(np.diff(recs[:nm]["block"].astype(np.int64)) >= 0))
        e2e = {"value": total_bytes * 8 * Ke / de / 1e9, "unit": "Gbit/s",
               "h2d_bytes_per_step": int(data.size),   # uniform blocks: no block table travels
               "d2h_bytes_per_step": int(32 + nm * 16),
               "steps": Ke, "passes_per_step": 1, "ms_per_step": de / Ke * 1e3,
               "matches_delivered_per_step": int(nm), "delivered_in_block_order": ordered,
               "api": "hs_b200_scan_blocks_collect(host pinned buffer): H2D, scan + confirm kernels, D2H of the "
                      "records, report rules and (block, to, id) ordering on the host -> match array on host",
               "bound": "one PCIe Gen5 x16 link per GPU: the H2D copy of the corpus is ~95 % of the call "
                        "(tools/h2d_ceiling.py); the scan itself needs < 3 % of that time"}
        # the same call path with the corpus ALREADY in device memory (a framework that produces its
        # input on the GPU): wrap the device buffer, scan, fetch the ordered matches to the host
        dcorp = torch.from_numpy(data).to(dev)
        wrapped = capi.Corpus.wrap(dcorp.data_ptr(), data.size, off, ln, device=local, keep=dcorp)
        for _ in range(2):
            capi.scan_corpus(db, wrapped, scratch)
        barrier()
        t0 = time.perf_counter()
        for _ in range(Ke * 4):
            got = capi.scan_corpus(db, wrapped, scratch)
        barrier()
        dr = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dr], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dr = float(tt.item())
        e2e["device_resident_input"] = {
            "value": total_bytes * 8 * Ke * 4 / dr / 1e9, "unit": "Gbit/s", "steps": Ke * 4,
            "ms_per_step": dr / (Ke * 4) * 1e3, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(32 + got.size * 16),
            "api": "hs_b200_corpus_wrap(device pointer) once; per step hs_b200_scan_corpus_async + _finish + "
                   "hs_b200_fetch_matches -> ordered match array on host"}
        wrapped.free()
        del dcorp

    # ---- secondary configurations -------------------------------------------------
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    secondary = None
    if not args.no_secondary:
        try:
            secondary = secondary_single_gpu(args, capi, torch, data, peak) if world == 1 else {}
        except Exception as e:   # never lose the headline line to a secondary failure
            secondary = {"error": "%s: %s" % (type(e).__name__, e)}
        sharded = secondary_sharded(args, capi, hdist, torch, dist, dev, world, rank, local, data, peak, barrier)
        if rank == 0:
            secondary.update(sharded)
    passes.close()

    if rank == 0:
        peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        kms = float(np.mean(kernel_ms))
        alg_bytes = corpus_bytes + 16 * int(n)
        achieved = alg_bytes / (kms * 1e-3) / 1e9
        traffic, traffic_src = traffic_record()
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel": "scanKernelPair (class-pair first stage, prefilter) + confirmKernel, CUDA events on "
                          "the launching stream around both",
                "kernel_ms": kms, "algorithmic_bytes_per_launch": alg_bytes}
        cpu = None
        if not args.no_cpu:
            try:
                cpu = cpu_reference_run(db, data, off, ln, args.cpu_sample_mb, args.cpu_seconds)
            except Exception as e:  # oracle/_ref missing on this box
                cpu = {"value": None, "unit": "Gbit/s", "cores": 0, "kind": "reference",
                       "sample": "unavailable: %s" % e}
        out = {"metric": METRIC, "value": value, "unit": "Gbit/s", "n_gpus": world, "steps": K, "warmup": W,
               "ms_per_step": dt / K * 1e3, "wall_ms_per_step_with_barrier": wall / K * 1e3,
               "timing": "CUDA events on the launching stream around the K x P passes, max over ranks",
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "u8", "data": "synthetic", "config": config_of(args, world, info), "e2e": e2e,
               "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
               "verify": verify, "secondary": secondary}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def secondary_sharded(args, capi, hdist, torch, dist, dev, world, rank, local, base, peak, barrier):
    """BASELINE configs[4] shape: 50 000 literals, --shard-gib GiB of blocks per GPU
    (64 GiB over 8 GPUs), records exchanged every pass.  The shard is the rank's
    1 GiB corpus (with this literal set planted) tiled in device memory."""
    from hyperscan_b200 import synth
    lits, flags, ids = synth.literal_set(50000, min_len=4, max_len=16, caseless_frac=0.1, seed=5)
    db = capi.compile_lit_multi(lits, flags, ids)
    bl = args.block_len
    nb1 = args.blocks
    one = replant(base, nb1, bl, lits, 0.01, 97 + rank)
    reps = max(1, (args.shard_gib << 30) // one.size)
    d1 = torch.from_numpy(one).to(dev)
    big = d1.repeat(reps)
    del d1
    nb = nb1 * reps
    off = np.arange(nb, dtype=np.uint64) * np.uint64(bl)
    ln = np.full(nb, bl, dtype=np.uint32)
    corpus = capi.Corpus.wrap(big.data_ptr(), big.numel(), off, ln, device=local, keep=big)
    passes = Passes(capi, hdist, torch, dist, db, corpus, dev, world, rank, args.exchange, rank * nb)
    passes.run(3)
    barrier()
    t0 = time.perf_counter()
    T = 20
    n, last, kms = passes.run(T)
    barrier()
    wall = time.perf_counter() - t0
    dt = passes.device_ms * 1e-3      # CUDA events on the launching stream, max over ranks below
    cnt = torch.tensor([n], dtype=torch.int64, device=dev)
    if world > 1:
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    out = None
    if rank == 0:
        got = capi.fetch_matches(db, passes.last_scratch(T))
        vb = 2048
        exact = same_matches(got[got["block"] < vb], reference_sorted(db, one, off[:vb], ln[:vb]))
        kmean = float(np.mean(kms))
        out = {"config5_shape_sharded": {
            "engine": engine_name(db.info()), "literals": 50000, "bytes_per_gpu": int(big.numel()),
            "total_bytes": int(big.numel()) * world, "passes": T, "ms_per_pass": dt / T * 1e3,
            "wall_ms_per_pass_with_barrier_rank0": wall / T * 1e3,
            "value_gbit_s": int(big.numel()) * world * 8 * T / dt / 1e9, "records_per_pass_all_ranks": int(cnt.item()),
            "rank0_kernel_ms": kmean, "rank0_roofline_frac": (big.numel() + 16 * int(n)) / (kmean * 1e-3) / 1e9 / peak,
            "exchange": ("p2p peer stores" if passes.peerx is not None else "nccl all-gather per pass")
            if world > 1 else "none (one GPU)",
            "rank0_verified_blocks": vb, "rank0_bit_exact_vs_reference": exact,
            "note": "weak scaling: every --gpus N run prints this shape; the ratio of value_gbit_s at N=8 and "
                    "N=1 is the scaling of BASELINE configs[4]"}}
    passes.close()
    corpus.free()
    return out


if __name__ == "__main__":
    main()
