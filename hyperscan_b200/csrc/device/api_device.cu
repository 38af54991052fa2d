/*
 * api_device.cu -- device half of the C ABI: scratch, corpus handles and the
 * scan entry points (include/hs_b200.h).  The thin host shim around the
 * sm_100a kernels in scan_kernels.cu:
 *
 *   hs_alloc_scratch / hs_clone_scratch / hs_scratch_size / hs_free_scratch
 *        src/scratch.c:244-460 -- here a scratch owns a CUDA stream, the
 *        match-record ring in HBM and the device images of the databases it
 *        was allocated for.
 *   hs_scan   src/runtime.c:316-475 -- argument checks and early-outs follow
 *        the reference; the body is "copy block to HBM, launch, read records
 *        back, replay callbacks in offset order".
 *   hs_b200_* the batched / device-resident forms of the same (hsbench scans
 *        a set of blocks: tools/hsbench/main.cpp:503-527).
 *
 * There is no CPU scan path in this library: without a usable CUDA device
 * hs_alloc_scratch fails with HS_ARCH_ERROR.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../host/api_internal.h"
#include "../host/db_walk.h"
#include "../host/pair_table.h"
#include "kernels.h"

using namespace hsb;

namespace {

const u32 SCRATCH_MAGIC = 0x544F4259; /* src/scratch.h:48 */
const size_t FRONT_PAD = 256;         /* readable bytes before corpus position 0 */

std::atomic<unsigned long long> g_launches{0};

/* runtime tunables (hs_b200_set_runtime_option / HSB200_* environment) */
struct RuntimeOpts {
    int warps = 0;           /* per CTA; 0 = what measured best for the kernel (28 in direct mode: 896
                              * threads x 72 registers; 32 with TMA staging) */
    int tileBytes = 1024;
    int stages = 2;
    int wideFdr = 0;         /* 1: use all 8 FDR slots (u64 entries) when they fit */
    int stride = 1;          /* first-stage sampling stride (0 = as compiled into the FDR table) */
    int prefilter = 1;       /* shared-memory bitmap in front of the hash confirm */
    int rebuild = 1;         /* rebuild the FDR first-stage table over slots 1..4 from the literals */
    int domain = 0;          /* rebuilt table: hash domain bits (0 = as compiled) */
    int direct = 1;          /* 1: corpus straight into registers; 0: TMA-staged tiles */
    int pfDist = 8;          /* direct mode: L2 prefetch distance in 512-byte steps */
    int replicas = 1;        /* rebuilt table: copies per entry (0 = fill up to 128 KB, max 16);
                              * measured: no gain, and a small footprint lets NCCL CTAs co-reside */
    int queue = 2;           /* candidates go through the per-warp shared-memory queue: 0 never, 1 always,
                              * 2 for the per-byte tables (Teddy, noodle: measured +15 %) but not for the
                              * FDR hash table, whose kernel is shared-memory bound either way */
    int wide = 1;            /* 1: wide-step kernel (32-byte lanes, always queued) for FK_BYTE32 / FK_HASH32.
                              * Measured with split=1 and 28 warps: Teddy-48 4.14 TB/s against 3.08 for the
                              * 16-byte queued kernel, noodle 4.43 against 3.19 (profiles/r02_*) */
    int split = 1;           /* 1 (with wide): scan kernel stops at the prefilter, confirmKernel finishes the
                              * candidates from a list in HBM (second half of the record ring) */
    int firstStage = 3;      /* FDR databases: 3 = class-pair tables (FK_PAIR32: two conflict-free lookups per
                              * byte), 1 = two-byte hash table (FK_HASH32, ~3.3-way bank conflicts), 2 = per-byte
                              * table (FK_BYTE32, conflict-free, many more candidates), 0 = choose between 1
                              * and 2 by the modelled candidate rate of the per-byte table */
    int bigSet = 0;          /* FK_PAIR32: sets that would overfill the 32 KiB bitmap trade classes of the
                              * second byte for a large contiguous bitmap */
    int gram = 1;            /* FDR sets: 1 = class 4-gram first stage (FK_GRAM4) for sets that would fill the
                              * pair kernel's 32 KiB bitmap beyond 10 % (all literals >= 4 bytes), 2 = whenever
                              * possible, 0 = never */
    int heavy = 1;           /* FK_PAIR32 candidate path: 0 = per-lane entries, 2 = per-word entries (sets that
                              * pass many candidates), 1 = by the modelled first-stage rate */
    int bigSetClasses = 4;   /* ... classes left to the second byte (pair table = 4 KiB each) */
    int dfaIlp = 1;          /* DFA kernels: blocks walked by one lane at a time; 2 = two interleaved state chains
                              * per lane, measured SLOWER (half the warps per block count: profiles/r02_dfa.log) */
    int fatPair = 1;         /* fat Teddy (16 buckets): 1 = class-pair first stage with the buckets folded onto
                              * 8 bits (3.0 TB/s), 0 = 64-bit per-byte entries (FK_BYTE64, 1.75 TB/s) */
    int chunkMB = 128;       /* host->device pipeline granularity */
    int initialRing = 1 << 20;
};
RuntimeOpts g_opts;
bool g_optsInit = false;

void initOpts() {
    if (g_optsInit) {
        return;
    }
    g_optsInit = true;
    struct { const char *env; int *v; } e[] = {
        {"HSB200_WARPS", &g_opts.warps},       {"HSB200_TILE", &g_opts.tileBytes},
        {"HSB200_STAGES", &g_opts.stages},     {"HSB200_WIDE_FDR", &g_opts.wideFdr},
        {"HSB200_CHUNK_MB", &g_opts.chunkMB},  {"HSB200_RING", &g_opts.initialRing},
        {"HSB200_STRIDE", &g_opts.stride},     {"HSB200_PREFILTER", &g_opts.prefilter},
        {"HSB200_REBUILD", &g_opts.rebuild},   {"HSB200_DOMAIN", &g_opts.domain},
        {"HSB200_DIRECT", &g_opts.direct},     {"HSB200_REPLICAS", &g_opts.replicas},
        {"HSB200_PF_DIST", &g_opts.pfDist},    {"HSB200_QUEUE", &g_opts.queue},
        {"HSB200_FIRST_STAGE", &g_opts.firstStage}, {"HSB200_WIDE", &g_opts.wide},
        {"HSB200_SPLIT", &g_opts.split},       {"HSB200_BIG_SET", &g_opts.bigSet},
        {"HSB200_BIG_SET_CLASSES", &g_opts.bigSetClasses}, {"HSB200_HEAVY", &g_opts.heavy},
        {"HSB200_GRAM", &g_opts.gram},         {"HSB200_FAT_PAIR", &g_opts.fatPair},
        {"HSB200_DFA_ILP", &g_opts.dfaIlp}};
    for (auto &x : e) {
        const char *s = getenv(x.env);
        if (s && *s) {
            *x.v = atoi(s);
        }
    }
}

/* ---- device image of one database --------------------------------------- */

struct DevImage {
    const hs_database_t *db = nullptr;   /* identity of the database the image was built from (a key: never
                                          * dereferenced -- the application may have freed it) */
    std::vector<u8> dbCopy;
    u32 dbCopyShift = 0;              /* its bytes (header + bytecode, bytecode offset preserved), so that
                                          * hs_clone_scratch can rebuild the image without the original */
    u32 crc = 0, length = 0;
    u8 *d_bc = nullptr;
    u8 *d_table = nullptr;
    u32 tableBytes = 0;
    u8 *d_bitmap = nullptr;
    u32 bitmapBytes = 0, bitmapShift = 0, keyBytes = 0;
    u32 pairBytes = 0, bitmapHoles = 0, bitmapBits = 0; /* FK_PAIR32 layout (kernels.h) */
    u32 bucketFold = 0;
    /* FK_OUTFIX: the engines (one per queue), grouped by model, and one launch per model: `engines` of each
     * launch points into d_engines */
    DfaEngine *d_engines = nullptr;
    std::vector<DfaParams> engineLaunches;
    /* FK_OUTFIX: report program offset -> its (onmatch, offset_adjust) list, filled as programs are met */
    mutable std::unordered_map<u32, std::vector<ProgReport>> progReports;
    double pairRate = 0;     /* FK_PAIR32: modelled first-stage candidates per byte (printable ASCII) */
    u8 *d_bitmap2 = nullptr; /* second level (HBM / L2) for large literal sets */
    u32 bitmap2Shift = 0;
    int kind = FK_BYTE32;
    int stride = 1;
    int slotBase = 0;
    u32 repShift = 0;
    u32 indexMask = 0;
    u32 confOff = 0, engineOff = 0;
    u32 confirmKind = CK_FDR;
    u64 groups = 0;
    u32 minWidth = 0;
    bool hasDedupe = false;              /* RoseEngine.dkeyCount != 0 */
    mutable std::unordered_set<u32> exhaustible; /* report ids under HS_FLAG_SINGLEMATCH (FK_OUTFIX: found with the programs) */
    size_t deviceBytes = 0;
};

/* A scratch (and a corpus / stream set) is bound to the CUDA device that was current
 * when it was created: its streams, events, record ring and database images live
 * there.  The reference lets any thread use any scratch, and a fresh thread's current
 * device is 0, so every entry point that touches one switches to its device for the
 * duration of the call and restores the caller's. */
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
            switched = cudaSetDevice(dev) == cudaSuccess;
        }
    }
    ~DeviceGuard() {
        if (switched) {
            cudaSetDevice(prev);
        }
    }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};

#define CUDA_TRY(expr)                                                                     \
    do {                                                                                   \
        cudaError_t e__ = (expr);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            return e__ == cudaErrorMemoryAllocation ? HS_NOMEM : HS_UNKNOWN_ERROR;         \
        }                                                                                  \
    } while (0)

/* Second-stage prefilter: a bitmap over a hash of each literal's last
 * keyBytes bytes (don't-care bits of LitInfo.msk -- caseless letters --
 * enumerated).  A clear bit proves no literal ends at a candidate position, so
 * the hash confirm in HBM/L2 is only reached by ~1% of the first stage's false
 * positives.  Returns an empty vector when the set cannot be keyed usefully. */
std::vector<u8> buildBitmap(const std::vector<LitTail> &tails, u32 *keyBytes, u32 *shift,
                            std::vector<u8> *level2 = nullptr, u32 *shift2 = nullptr) {
    std::vector<u8> bm;
    if (tails.empty()) {
        return bm;
    }
    u32 m = 4;
    for (const LitTail &t : tails) {
        m = std::min(m, t.size);
    }
    if (m < 2) {
        return bm; /* single-byte literals: the first stage is already exact */
    }
    std::vector<u32> keys;
    for (const LitTail &t : tails) {
        const u32 v = (u32)(t.v >> 32) >> (8 * (4 - m));
        const u32 care = (u32)(t.msk >> 32) >> (8 * (4 - m));
        const u32 full = m == 4 ? 0xffffffffu : (1u << (8 * m)) - 1;
        const u32 dc = ~care & full;
        if (__builtin_popcount(dc) > 10) {
            return std::vector<u8>(); /* too loose to enumerate */
        }
        u32 sub = 0;
        do {
            keys.push_back((v & care) | sub);
            sub = (sub - dc) & dc;
        } while (sub);
    }
    u32 lg = 13; /* 8 Kbit .. 512 Kbit (64 KB), ~256 bits per key when possible */
    while (lg < 19 && (1ull << lg) < (u64)keys.size() * 256) {
        lg++;
    }
    bm.assign((size_t)1 << (lg - 3), 0);
    for (u32 k : keys) {
        const u32 h = (k * 0x9E3779B1u) >> (32 - lg);
        bm[h >> 3] |= (u8)(1u << (h & 7));
    }
    *keyBytes = m;
    *shift = 32 - lg;
    if (level2 && shift2 && keys.size() * 32 > ((size_t)1 << lg)) {
        /* the shared-memory bitmap is more than ~3 % full: add a level with
         * ~1024 bits per key (<= 64 MB), probed only by its survivors */
        u32 lg2 = lg + 1;
        while (lg2 < 29 && (1ull << lg2) < (u64)keys.size() * 1024) {
            lg2++;
        }
        level2->assign((size_t)1 << (lg2 - 3), 0);
        for (u32 k : keys) {
            const u32 h = (k * 0x85EBCA6Bu) >> (32 - lg2);
            (*level2)[h >> 3] |= (u8)(1u << (h & 7));
        }
        *shift2 = 32 - lg2;
    }
    return bm;
}

/* Keys of the prefilter bitmaps: every literal's last m <= 4 bytes with the
 * don't-care bits of LitInfo.msk enumerated.  false = cannot be keyed usefully. */
bool tailKeys(const std::vector<LitTail> &tails, u32 *keyBytes, std::vector<u32> *keys) {
    if (tails.empty()) {
        return false;
    }
    u32 m = 4;
    for (const LitTail &t : tails) {
        m = std::min(m, t.size);
    }
    if (m < 2) {
        return false;
    }
    for (const LitTail &t : tails) {
        const u32 v = (u32)(t.v >> 32) >> (8 * (4 - m));
        const u32 care = (u32)(t.msk >> 32) >> (8 * (4 - m));
        const u32 full = m == 4 ? 0xffffffffu : (1u << (8 * m)) - 1;
        const u32 dc = ~care & full;
        if (__builtin_popcount(dc) > 10) {
            return false;
        }
        u32 sub = 0;
        do {
            keys->push_back((v & care) | sub);
            sub = (sub - dc) & dc;
        } while (sub);
    }
    *keyBytes = m;
    return true;
}

/* FK_PAIR32 bitmaps: first level of `bits` bits (index = mulhi(key * K, bits)) in
 * shared memory, second level (~1024 bits per key, <= 64 MB) in HBM / L2 when the
 * first is more than ~3 % full. */
void buildPairBitmaps(const std::vector<u32> &keys, u32 bits, std::vector<u8> *level1,
                      std::vector<u8> *level2, u32 *shift2) {
    level1->assign((size_t)(bits + 31) / 32 * 4, 0);
    for (u32 k : keys) {
        const u32 h = (u32)(((u64)(k * 0x9E3779B1u) * bits) >> 32);
        (*level1)[h >> 3] |= (u8)(1u << (h & 7));
    }
    *shift2 = 0;
    if (keys.size() * 32 > bits) {
        u32 lg2 = 20;
        while (lg2 < 29 && (1ull << lg2) < (u64)keys.size() * 1024) {
            lg2++;
        }
        level2->assign((size_t)1 << (lg2 - 3), 0);
        for (u32 k : keys) {
            const u32 h = (k * 0x85EBCA6Bu) >> (32 - lg2);
            (*level2)[h >> 3] |= (u8)(1u << (h & 7));
        }
        *shift2 = 32 - lg2;
    }
}

/* FK_GRAM4 tables: a byte -> class map (<= 32 classes) and the 1 Mbit bitmap of the class
 * 4-grams that some literal's last four bytes can produce (caseless letters through
 * LitInfo.msk).  Bytes no tail uses share class 0; if more than 31 byte values are in
 * use, the two cases of a letter share a class first (a case-sensitive literal then also
 * admits the other case at the first stage -- the exact 4-byte bitmap in L2 and the
 * confirm sort that out), then the rarest byte values are folded together. */
bool buildGramTables(const std::vector<LitTail> &tails, std::vector<u8> *classWords, std::vector<u8> *bitmap) {
    u32 count[256] = {0};
    for (const LitTail &t : tails) {
        if (t.size < 4) {
            return false; /* needs four known bytes per literal */
        }
        for (u32 p = 0; p < 4; p++) {
            const u8 c = (u8)(t.v >> (8 * (7 - p))), m = (u8)(t.msk >> (8 * (7 - p)));
            for (u32 b = 0; b < 256; b++) {
                if ((b & m) == c) {
                    count[b]++;
                }
            }
        }
    }
    u32 cls[256];
    std::vector<std::vector<u32>> groups; /* groups[i] = byte values of class i + 1 */
    for (u32 b = 0; b < 256; b++) {
        if (count[b]) {
            groups.push_back({b});
        }
    }
    auto weight = [&](const std::vector<u32> &g) {
        u64 w = 0;
        for (u32 b : g) {
            w += count[b];
        }
        return w;
    };
    if (groups.size() > 31) { /* fold the cases of letters */
        std::vector<std::vector<u32>> folded;
        std::vector<bool> done(256, false);
        for (const auto &g : groups) {
            const u32 b = g[0];
            if (done[b]) {
                continue;
            }
            done[b] = true;
            std::vector<u32> ng = {b};
            const bool alpha = (b >= 'a' && b <= 'z') || (b >= 'A' && b <= 'Z');
            if (alpha && count[b ^ 0x20]) {
                ng.push_back(b ^ 0x20);
                done[b ^ 0x20] = true;
            }
            folded.push_back(ng);
        }
        groups.swap(folded);
    }
    while (groups.size() > 31) { /* fold the two rarest groups */
        size_t a = 0, b = 1;
        if (weight(groups[b]) < weight(groups[a])) {
            std::swap(a, b);
        }
        for (size_t i = 2; i < groups.size(); i++) {
            if (weight(groups[i]) < weight(groups[a])) {
                b = a;
                a = i;
            } else if (weight(groups[i]) < weight(groups[b])) {
                b = i;
            }
        }
        groups[std::min(a, b)].insert(groups[std::min(a, b)].end(), groups[std::max(a, b)].begin(),
                                      groups[std::max(a, b)].end());
        groups.erase(groups.begin() + (long)std::max(a, b));
    }
    for (u32 b = 0; b < 256; b++) {
        cls[b] = 0;
    }
    for (size_t i = 0; i < groups.size(); i++) {
        for (u32 b : groups[i]) {
            cls[b] = (u32)i + 1;
        }
    }
    classWords->resize(256 * 4);
    for (u32 b = 0; b < 256; b++) {
        const u32 e = cls[b] * 4;
        memcpy(classWords->data() + 4 * b, &e, 4);
    }
    /* word index c[e-3] + 33 c[e-2] + 1025 c[e-1] (kernels.h FK_GRAM4): sized like the kernel's window */
    bitmap->assign((size_t)scanSmemBytes(FK_GRAM4, 0, 0, 0, 0, 0, 0) - 65536, 0);
    for (const LitTail &t : tails) {
        /* classes each of the last four bytes can take: [0] = byte e-3 ... [3] = byte e */
        u32 opts[4] = {0, 0, 0, 0}; /* bitmask over classes */
        for (u32 p = 0; p < 4; p++) {
            const u8 c = (u8)(t.v >> (8 * (7 - p))), m = (u8)(t.msk >> (8 * (7 - p)));
            for (u32 b = 0; b < 256; b++) {
                if ((b & m) == c) {
                    opts[3 - p] |= 1u << cls[b];
                }
            }
        }
        for (u32 c3 = 0; c3 < 32; c3++) {
            if (!((opts[0] >> c3) & 1)) continue;
            for (u32 c2 = 0; c2 < 32; c2++) {
                if (!((opts[1] >> c2) & 1)) continue;
                for (u32 c1 = 0; c1 < 32; c1++) {
                    if (!((opts[2] >> c1) & 1)) continue;
                    const u32 word = c3 + 33 * c2 + 1025 * c1;
                    u32 w;
                    memcpy(&w, bitmap->data() + 4 * (size_t)word, 4);
                    w |= opts[3];
                    memcpy(bitmap->data() + 4 * (size_t)word, &w, 4);
                }
            }
        }
    }
    return true;
}

/* First-stage table rebuilt from the literal tails (LitInfo v/msk) and their
 * bucket assignment: u32 entry = 4 slots x 8 buckets indexed by the FDR hash
 * (two bytes & domain mask, src/fdr/fdr.c:157-170); slot i stands for suffix
 * distance i + slotBase.  With slotBase 1 the sample at x tests the pairs
 * (char 1, char 0) .. (char 4, char 3): every character of a 4-byte tail is in a
 * full two-byte sample, which the reference's slot 0 (second byte unknown)
 * cannot give, and literals of 5+ bytes gain a sample.  Same construction as
 * setupTab (src/fdr/fdr_compile.cpp:527-632): bit SET = impossible. */
std::vector<u8> rebuildHashTable(const std::vector<LitTail> &tails, u32 domain, u32 slotBase) {
    const u32 entries = 1u << domain, dmask = entries - 1;
    std::vector<u32> tab(entries, 0xffffffffu);
    u32 dead = 0;
    const u32 hiBits = domain - 8;
    for (const LitTail &t : tails) {
        for (u32 i = 0; i < 4; i++) {
            const u32 p = i + slotBase;
            const u32 bit = 1u << (8 * i + t.bucket);
            if (p >= t.size) {
                dead |= bit; /* shorter literal: this slot cannot constrain the bucket */
                continue;
            }
            const u8 c0 = (u8)(t.v >> (8 * (7 - p))), m0 = (u8)(t.msk >> (8 * (7 - p)));
            u8 c1 = 0, m1 = 0; /* p == 0: the following byte is unknown */
            if (p > 0) {
                c1 = (u8)(t.v >> (8 * (8 - p)));
                m1 = (u8)(t.msk >> (8 * (8 - p)));
            }
            const u8 hm = (u8)((1u << hiBits) - 1);
            bool seen1[256] = {false};
            for (u32 b1 = 0; b1 < 256; b1++) {
                if ((b1 & m1) != c1 || seen1[b1 & hm]) {
                    continue;
                }
                seen1[b1 & hm] = true;
                for (u32 b0 = 0; b0 < 256; b0++) {
                    if ((b0 & m0) == c0) {
                        tab[(b0 | (b1 << 8)) & dmask] &= ~bit;
                    }
                }
            }
        }
    }
    std::vector<u8> out((size_t)entries * 4);
    for (u32 i = 0; i < entries; i++) {
        const u32 e = tab[i] & ~dead;
        memcpy(&out[(size_t)i * 4], &e, 4);
    }
    return out;
}

/* Per-byte first-stage table for an FDR literal set: entry b, slot i, bucket k
 * is CLEAR iff some literal of bucket k can have byte b at suffix distance i
 * (caseless letters through LitInfo.msk).  The Teddy construction
 * (src/fdr/teddy_compile.cpp:440-509) applied to the FDR buckets: a weaker
 * filter than the two-byte hash, but its 256-row table is replicated per lane,
 * so the lookups are bank-conflict free.  *rate = modelled candidates per byte
 * on uniformly random printable ASCII. */
std::vector<u8> buildByteTable(const std::vector<LitTail> &tails, double *rate) {
    u32 tab[256];
    for (u32 b = 0; b < 256; b++) {
        tab[b] = 0xffffffffu;
    }
    u32 dead = 0;
    for (const LitTail &t : tails) {
        for (u32 i = 0; i < 4; i++) {
            const u32 bit = 1u << (8 * i + t.bucket);
            if (i >= t.size) {
                dead |= bit;
                continue;
            }
            const u8 c = (u8)(t.v >> (8 * (7 - i))), m = (u8)(t.msk >> (8 * (7 - i)));
            for (u32 b = 0; b < 256; b++) {
                if ((b & m) == c) {
                    tab[b] &= ~bit;
                }
            }
        }
    }
    std::vector<u8> out(256 * 4);
    double total = 0;
    for (u32 k = 0; k < 8; k++) {
        double pr = 1;
        for (u32 i = 0; i < 4; i++) {
            u32 n = 0;
            for (u32 b = 0x20; b < 0x7f; b++) {
                n += !(((tab[b] & ~dead) >> (8 * i + k)) & 1);
            }
            pr *= n / 95.0;
        }
        total += pr;
    }
    *rate = total;
    for (u32 b = 0; b < 256; b++) {
        const u32 e = tab[b] & ~dead;
        memcpy(&out[b * 4], &e, 4);
    }
    return out;
}

/* What launchDfa needs to know about a serialized engine (struct NFA + McClellan 8 / 16,
 * Sheng or LimEx-32 ... -512), checked against its length.  HS_ARCH_ERROR: an engine or a feature
 * (wide states, bounded repeats) the DFA / NFA kernels do not implement. */
hs_error_t engineParams(const void *nfa, size_t nfa_len, DfaParams *out) {
    if (!nfa || nfa_len < sizeof(NFA) + 64) {
        return HS_INVALID;
    }
    NFA hdr;
    memcpy(&hdr, nfa, sizeof(hdr));
    if (hdr.length > nfa_len) {
        return HS_INVALID;
    }
    DfaParams &p = *out;
    memset(&p, 0, sizeof(p));
    p.kind = hdr.type;
    p.ilp = g_opts.dfaIlp == 2 ? 2u : 1u;
    if (hdr.type == NFA_MCCLELLAN_8 || hdr.type == NFA_MCCLELLAN_16) {
        if (nfa_len < sizeof(NFA) + sizeof(McClellan)) {
            return HS_INVALID;
        }
        McClellan m;
        memcpy(&m, (const u8 *)nfa + sizeof(NFA), sizeof(m));
        if (m.has_wide) {
            return HS_ARCH_ERROR; /* wide states (mcclellan.c:168-225) are not built here */
        }
        const u32 rows = hdr.type == NFA_MCCLELLAN_16 ? m.sherman_limit : m.state_count;
        p.tableBytes = (rows << m.alphaShift) * (hdr.type == NFA_MCCLELLAN_16 ? 2u : 1u);
        p.states = m.state_count;
        if (hdr.type == NFA_MCCLELLAN_8 && (m.state_count == 0 || m.state_count > 256)) {
            return HS_INVALID;
        }
        if (sizeof(NFA) + sizeof(McClellan) + p.tableBytes > nfa_len) {
            return HS_INVALID;
        }
    } else if (hdr.type == NFA_SHENG) {
        if (nfa_len < sizeof(NFA) + sizeof(Sheng)) {
            return HS_INVALID;
        }
    } else if (hdr.type == NFA_LIMEX_32 || hdr.type == NFA_LIMEX_64 || hdr.type == NFA_LIMEX_128 ||
               hdr.type == NFA_LIMEX_256 || hdr.type == NFA_LIMEX_512) {
        /* (the 384-state model is not built: the emitter here never produces it) */
        size_t structSize, excSize, stateBytes, shiftCountAt;
        switch (hdr.type) {
#define HSB_LIMEX_MODEL(T, L, E, B)                                                     \
        case T:                                                                         \
            structSize = sizeof(L), excSize = sizeof(E), stateBytes = B, shiftCountAt = offsetof(L, shiftCount); \
            break;
            HSB_LIMEX_MODEL(NFA_LIMEX_32, LimExNFA32, NFAException32, 4)
            HSB_LIMEX_MODEL(NFA_LIMEX_64, LimExNFA64, NFAException64, 8)
            HSB_LIMEX_MODEL(NFA_LIMEX_128, LimExNFA128, NFAException128, 16)
            HSB_LIMEX_MODEL(NFA_LIMEX_256, LimExNFA256, NFAException256, 32)
        default:
            HSB_LIMEX_MODEL(NFA_LIMEX_512, LimExNFA512, NFAException512, 64)
#undef HSB_LIMEX_MODEL
        }
        if (nfa_len < sizeof(NFA) + structSize) {
            return HS_INVALID;
        }
        /* the count / offset fields precede the state-sized ones and sit at the same offsets in every model */
        LimExNFA32 lx;
        memcpy(&lx, (const u8 *)nfa + sizeof(NFA), offsetof(LimExNFA32, init));
        u32 shiftCount;
        memcpy(&shiftCount, (const u8 *)nfa + sizeof(NFA) + shiftCountAt, 4);
        if (lx.repeatCount) {
            return HS_ARCH_ERROR; /* bounded repeats (repeat control blocks, tug / pos triggers) are not built */
        }
        if (stateBytes > 8 && ((uintptr_t)nfa & 7)) {
            return HS_INVALID; /* the wide state sets are read as 64-bit words */
        }
        const size_t body = nfa_len - sizeof(NFA);
        if (shiftCount > 8 || lx.exceptionCount > 8 * stateBytes ||
            structSize + stateBytes * lx.reachSize > body ||
            (size_t)lx.exceptionOffset + (size_t)lx.exceptionCount * excSize > body ||
            (size_t)lx.acceptOffset + (size_t)lx.acceptCount * sizeof(NFAAccept) > body ||
            (size_t)lx.acceptEodOffset + (size_t)lx.acceptEodCount * sizeof(NFAAccept) > body) {
            return HS_INVALID;
        }
        p.states = hdr.nPositions;
        for (u32 i = 0; i < lx.exceptionCount; i++) {
            /* hasSquash sits right after the two state-sized masks and the two u32 of every model's exception */
            const u8 kind = *((const u8 *)nfa + sizeof(NFA) + lx.exceptionOffset + i * excSize + 2 * stateBytes + 8);
            p.squashes |= kind == LIMEX_SQUASH_CYCLIC || kind == LIMEX_SQUASH_REPORT;
        }
    } else {
        return HS_ARCH_ERROR; /* LimEx-384, McSheng, Gough, Castle, ...: not built */
    }
    return HS_SUCCESS;
}

void freeImage(DevImage *im) {
    if (!im) {
        return;
    }
    cudaFree(im->d_bc);
    cudaFree(im->d_engines);
    cudaFree(im->d_table);
    cudaFree(im->d_bitmap);
    cudaFree(im->d_bitmap2);
    delete im;
}

/* Derive the device image: a copy of the bytecode plus the first-stage table
 * in the form the shift-OR kernel consumes (DESIGN.md section 3). */
hs_error_t buildImage(const hs_database_t *db, DevImage **out) {
    initOpts();
    const DbHeader *h = (const DbHeader *)db;
    const RoseEngine *r = dbRose(db);
    const u8 *bc = (const u8 *)r;
    const bool soleOutfix = r->runtimeImpl == RUNTIME_SINGLE_OUTFIX && r->mode == MODE_BLOCK && r->queueCount == 1 &&
                            r->outfixBeginQueue == 0 && r->outfixEndQueue == 1 && r->nfaInfoOffset &&
                            !r->amatcherOffset && !r->ematcherOffset && !r->fmatcherOffset && !r->hasSom;
    if (!soleOutfix && !outfixesOnly(r, h->length) && (r->runtimeImpl != RUNTIME_PURE_LITERAL || !r->fmatcherOffset)) {
        /* other FULL_ROSE databases need the full rose interpreter and the catch-up machinery
         * (SURVEY.md section 8f rank 1): not in this build */
        return HS_ARCH_ERROR;
    }
    DevImage *im = new (std::nothrow) DevImage();
    if (!im) {
        return HS_NOMEM;
    }
    im->db = db;
    {
        /* same address modulo 64 as the original, so that every offset-derived alignment holds */
        const size_t total = sizeof(DbHeader) + h->length;
        im->dbCopy.resize(total + 128);
        const size_t want = (uintptr_t)db & 63, have = (uintptr_t)im->dbCopy.data() & 63;
        im->dbCopyShift = (u32)((want + 64 - have) & 63);
        memcpy(im->dbCopy.data() + im->dbCopyShift, db, std::min(total, (size_t)h->bytecode + h->length));
    }
    im->crc = h->crc32;
    im->length = h->length;
    im->groups = r->initialGroups & r->floating_group_mask;
    im->minWidth = r->minWidth;
    im->hasDedupe = r->dkeyCount != 0;
    if (r->runtimeImpl != RUNTIME_PURE_LITERAL) {
        /* hs_scan -> soleOutfixBlockExec (src/runtime.c:245-280), or roseBlockExec over outfixes only: every engine
         * runs over the whole block, its reports are report programs (roseReportAdaptor / roseNfaAdaptor, src/rose/
         * match.c:611-633).  The engines run on the DFA / NFA kernels (dfa_kernels.cu) straight from the bytecode
         * copy, one launch per engine model; the programs are resolved on the host when the records are ordered
         * (postprocess). */
        struct Eng {
            DfaParams p;
            u32 offset;
        };
        std::vector<Eng> engs;
        for (u32 q = 0; q < r->queueCount; q++) {
            const u64 at = (u64)r->nfaInfoOffset + (u64)q * sizeof(NfaInfo);
            if (at + sizeof(NfaInfo) > h->length) {
                delete im;
                return HS_INVALID;
            }
            NfaInfo ni;
            memcpy(&ni, bc + at, sizeof(ni));
            if (ni.nfaOffset % 64 || (size_t)ni.nfaOffset + sizeof(NFA) > h->length) {
                delete im;
                return HS_INVALID;
            }
            NFA nh;
            memcpy(&nh, bc + ni.nfaOffset, sizeof(nh));
            if ((size_t)ni.nfaOffset + nh.length > h->length) {
                delete im;
                return HS_INVALID;
            }
            Eng e;
            const hs_error_t er = engineParams(bc + ni.nfaOffset, nh.length, &e.p);
            if (er != HS_SUCCESS) {
                delete im;
                return er;
            }
            e.offset = ni.nfaOffset;
            engs.push_back(e);
        }
        std::stable_sort(engs.begin(), engs.end(), [](const Eng &a, const Eng &b) { return a.p.kind < b.p.kind; });
        im->kind = FK_OUTFIX;
        im->groups = 0;
        cudaError_t e = cudaMalloc(&im->d_bc, HSB_ROUNDUP(h->length, 16));
        if (e == cudaSuccess) {
            e = cudaMemcpy(im->d_bc, bc, h->length, cudaMemcpyHostToDevice);
        }
        std::vector<DfaEngine> table(engs.size());
        for (size_t i = 0; i < engs.size(); i++) {
            const DfaParams &ep = engs[i].p;
            table[i] = {im->d_bc + engs[i].offset, ep.tableBytes, ep.states, ep.squashes, 0};
        }
        if (e == cudaSuccess) {
            e = cudaMalloc(&im->d_engines, table.size() * sizeof(DfaEngine));
        }
        if (e == cudaSuccess) {
            e = cudaMemcpy(im->d_engines, table.data(), table.size() * sizeof(DfaEngine), cudaMemcpyHostToDevice);
        }
        if (e != cudaSuccess) {
            freeImage(im);
            return e == cudaErrorMemoryAllocation ? HS_NOMEM : HS_UNKNOWN_ERROR;
        }
        for (size_t i = 0; i < engs.size(); i++) {
            const DfaParams &ep = engs[i].p;
            if (im->engineLaunches.empty() || im->engineLaunches.back().kind != ep.kind) {
                im->engineLaunches.push_back(ep);
                im->engineLaunches.back().engines = im->d_engines + i;
                im->engineLaunches.back().nengines = 0;
            }
            DfaParams &l = im->engineLaunches.back();
            l.nengines++;
            l.tableBytes = std::max(l.tableBytes, ep.tableBytes);
            l.states = std::max(l.states, ep.states);
            l.squashes |= ep.squashes;
        }
        im->deviceBytes = HSB_ROUNDUP(h->length, 16) + table.size() * sizeof(DfaEngine);
        *out = im;
        return HS_SUCCESS;
    }
    const HWLM *hw = (const HWLM *)(bc + r->fmatcherOffset);
    const u32 engOff = r->fmatcherOffset + HWLM_ENGINE_OFFSET;
    std::vector<u8> table, pairBitmap, pairBitmap2;
    std::vector<LitTail> tails;
    bool programsOk = true;
    /* FK_PAIR32 / FK_GRAM4 tables from the literals' tails (FDR sets, and fat Teddy with its 16
     * buckets folded onto 8 first-stage bits) */
    auto pairStage = [&](bool allowGram) {
        int dev = 0, maxSmem = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&maxSmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
                u32 minSize = 8;
                for (const LitTail &t : tails) {
                    minSize = std::min(minSize, t.size);
                }
                im->kind = FK_PAIR32;
                im->stride = 1;
                im->slotBase = minSize >= 2 ? 1 : 0;
                /* shared memory: 64 KiB class rows + pair table + (large sets) bitmap +
                 * queues.  Small sets: 32 x 32 classes (128 KiB pair table), the 32 KiB
                 * bitmap in the class rows' upper halves.  Sets whose keys would fill that
                 * bitmap beyond ~10 %: the pair filter is saturated anyway, so the second
                 * byte gets few classes and the freed space a large contiguous bitmap. */
                std::vector<u32> keys;
                u32 kb = 0;
                const bool keyed = g_opts.prefilter && tailKeys(tails, &kb, &keys);
                const bool large = keyed && keys.size() * 10 > 262144; /* would fill the 32 KiB bitmap > 10 % */
                std::vector<u8> gramBitmap;
                /* measured crossover (DESIGN.md section 3.7): 5 000 literals (12.5 k keys) scan
                 * 10 % faster through the 4-gram kernel, 1 000 literals 38 % slower */
                const bool gramWorth = keys.size() >= 10000;
                if (allowGram && (g_opts.gram == 2 || (g_opts.gram == 1 && gramWorth)) && keyed && kb == 4 &&
                    buildGramTables(tails, &table, &gramBitmap)) {
                    /* the pair evidence saturates for such sets: exact class 4-gram membership
                     * instead (FK_GRAM4), exact raw 4-byte keys in L2 behind it */
                    im->kind = FK_GRAM4;
                    im->keyBytes = 4;
                    pairBitmap.swap(gramBitmap);
                    /* second level in L2: one BYTE per slot = the buckets of the literals whose
                     * raw 4-byte key hashes there (~64 slots per key, <= 64 MB), so that a
                     * survivor reaches confirm with its real buckets, not all eight */
                    u32 lg2 = 16;
                    while (lg2 < 26 && (1ull << lg2) < (u64)keys.size() * 64) {
                        lg2++;
                    }
                    pairBitmap2.assign((size_t)1 << lg2, 0);
                    for (const LitTail &t : tails) {
                        const u32 v = (u32)(t.v >> 32), care = (u32)(t.msk >> 32), dc = ~care;
                        u32 sub = 0;
                        do {
                            const u32 k = (v & care) | sub;
                            pairBitmap2[(k * 0x85EBCA6Bu) >> (32 - lg2)] |= (u8)(1u << (t.bucket & 7));
                            sub = (sub - dc) & dc;
                        } while (sub);
                    }
                    im->bitmap2Shift = 32 - lg2;
                    return;
                }
                {
                const bool big = large && g_opts.bigSet != 0;
                PairTables pt;
                buildPairTables(tails, (u32)im->slotBase, &pt, 32, big ? (u32)std::max(1, g_opts.bigSetClasses) : 32);
                im->pairBytes = pt.nClass1 * 4096;
                im->pairRate = pt.modelRate;
                if (getenv("HSB200_TRACE")) {
                    fprintf(stderr, "[hs_b200] class-pair tables: %u x %u classes, modelled %.4f candidates/byte, "
                                    "%zu prefilter keys%s\n", pt.nClass0, pt.nClass1, pt.modelRate, keys.size(),
                            big ? " (large-set layout)" : "");
                }
                table.resize(sizeof(pt.classWord) + sizeof(pt.pair));
                memcpy(table.data(), pt.classWord, sizeof(pt.classWord));
                memcpy(table.data() + sizeof(pt.classWord), pt.pair, sizeof(pt.pair));
                if (keyed) {
                    im->keyBytes = kb;
                    im->bitmapHoles = big ? 0 : 1;
                    u32 bits = 262144;
                    if (big) {
                        /* everything the pair table and 27 queues leave of the 227 KiB */
                        const u32 queues = (u32)scanSmemBytes(FK_PAIR32, 0, 0, 0, 0, 0, 27) - 65536u;
                        const u32 room = (u32)maxSmem - 65536u - im->pairBytes - queues;
                        bits = (room & ~127u) * 8;
                    }
                    im->bitmapBits = bits;
                    buildPairBitmaps(keys, bits, &pairBitmap, &pairBitmap2, &im->bitmap2Shift);
                }
                }
    };
    if (hw->type == HWLM_ENGINE_NOOD) {
        /* single literal: one bucket, slots = the last <= 4 bytes of msk/cmp
         * (first char in the low byte: src/hwlm/noodle_build.cpp:100-118) */
        NoodTable n;
        memcpy(&n, bc + engOff, sizeof(n));
        im->confirmKind = CK_NOODLE;
        im->engineOff = engOff;
        im->kind = FK_BYTE32;
        im->stride = 1;
        table.assign(256 * 4, 0);
        for (u32 b = 0; b < 256; b++) {
            u32 e = 0;
            for (u32 p = 0; p < 4; p++) {
                u8 v = 0xfe; /* buckets 1..7 never match */
                if (p < n.msk_len) {
                    const u32 i = n.msk_len - 1 - p;
                    const u8 m = (u8)(n.msk >> (8 * i)), c = (u8)(n.cmp >> (8 * i));
                    if ((b & m) != c) {
                        v |= 1;
                    }
                }
                e |= (u32)v << (8 * p);
            }
            memcpy(&table[b * 4], &e, 4);
        }
        programsOk = collectProgramReports(bc, h->length, n.id, &im->exhaustible);
    } else if (hw->type == HWLM_ENGINE_FDR) {
        FDR f;
        memcpy(&f, bc + engOff, sizeof(f));
        im->confirmKind = CK_FDR;
        im->confOff = engOff + f.confOffset;
        if (f.engineID == 0) {
            const u32 entries = 1u << f.domain;
            const u8 *src = bc + engOff + FDR_TABLE_OFFSET;
            im->stride = f.stride;
            im->indexMask = f.domainMask;
            int dev = 0, maxSmem = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&maxSmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
            const size_t wideNeed = (size_t)entries * 8 + 48 * 1024;
            programsOk = walkConfirm(bc, h->length, im->confOff, 8, &im->exhaustible, &tails);
            double byteRate = 1;
            std::vector<u8> byteTab;
            if (g_opts.firstStage != 1) {
                byteTab = buildByteTable(tails, &byteRate);
            }
            if (g_opts.wideFdr && wideNeed <= (size_t)maxSmem) {
                im->kind = FK_HASH64;
                table.assign(src, src + (size_t)entries * 8);
            } else if (g_opts.firstStage == 3) {
                pairStage(true);
            } else if (g_opts.firstStage == 2 || (g_opts.firstStage == 0 && byteRate < 0.01)) {
                im->kind = FK_BYTE32;
                im->stride = 1;
                im->slotBase = 0;
                table.swap(byteTab);
            } else if (g_opts.rebuild) {
                u32 minSize = 8, d = f.domain;
                for (const LitTail &t : tails) {
                    minSize = std::min(minSize, t.size);
                }
                if (g_opts.domain >= 9 && g_opts.domain <= 15) {
                    d = (u32)g_opts.domain;
                }
                im->kind = FK_HASH32;
                im->slotBase = minSize >= 2 ? 1 : 0;
                im->indexMask = (1u << d) - 1;
                std::vector<u8> one = rebuildHashTable(tails, d, (u32)im->slotBase);
                /* copies of every entry in adjacent words: lane l reads copy
                 * l & (R-1), so a lookup's lanes fall into R bank groups */
                u32 R = 1;
                const u32 want = g_opts.replicas > 0 ? (u32)g_opts.replicas : 16;
                while (R * 2 <= want && one.size() * R * 2 <= 128u * 1024) {
                    R *= 2;
                }
                im->repShift = (u32)__builtin_ctz(R);
                table.resize(one.size() * R);
                for (size_t i = 0; i < one.size() / 4; i++) {
                    for (u32 g = 0; g < R; g++) {
                        memcpy(&table[(i * R + g) * 4], &one[i * 4], 4);
                    }
                }
            } else {
                im->kind = FK_HASH32; /* FDR suffix slots 0..3 as compiled */
                table.resize((size_t)entries * 4);
                for (u32 i = 0; i < entries; i++) {
                    memcpy(&table[(size_t)i * 4], src + (size_t)i * 8, 4);
                }
            }
        } else if (teddyIdValid(f.engineID)) {
            /* per-byte entry: slot m = lo_m[b & 15] | hi_m[b >> 4]
             * (src/fdr/teddy.c:918-969, teddy_compile.cpp:440-509) */
            const u32 nm = teddyNumMasks(f.engineID);
            const u32 oct = teddyNumBuckets(f.engineID) / 8;
            const u8 *mb = bc + engOff + TEDDY_MASK_OFFSET;
            im->stride = 1;
            im->kind = oct == 2 ? FK_BYTE64 : FK_BYTE32;
            table.assign(256 * 4 * oct, 0);
            for (u32 b = 0; b < 256; b++) {
                for (u32 o = 0; o < oct; o++) {
                    u32 e = 0;
                    for (u32 m = 0; m < nm; m++) {
                        const u8 *lo = mb + ((2 * m) * oct + o) * 16;
                        const u8 *hi = mb + ((2 * m + 1) * oct + o) * 16;
                        e |= (u32)(u8)(lo[b & 15] | hi[b >> 4]) << (8 * m);
                    }
                    memcpy(&table[(b * oct + o) * 4], &e, 4);
                }
            }
            programsOk = walkConfirm(bc, h->length, im->confOff, 8 * oct, &im->exhaustible, &tails);
            if (oct == 2 && g_opts.fatPair && g_opts.split && !tails.empty()) {
                /* 49..96 literals: the class-pair kernel filters them at 3 TB/s where the 64-bit
                 * per-byte entries cost two shared-memory wavefronts a byte; its 8 bucket bits
                 * carry buckets i and i + 8 (confirmKernel unfolds them) */
                table.clear();
                pairStage(false);
                im->bucketFold = 1;
            }
        } else {
            delete im;
            return HS_INVALID;
        }
    } else {
        delete im;
        return HS_INVALID;
    }
    if (!programsOk) {
        /* a literal program uses a state-carrying opcode of roseRunProgram_l that
         * the device interpreter does not implement (delayed literals, SOM,
         * chained / logical reports): refuse here rather than mid-scan */
        delete im;
        return HS_ARCH_ERROR;
    }
    im->tableBytes = (u32)table.size();
    std::vector<u8> bitmap, bitmap2;
    if (im->kind == FK_PAIR32 || im->kind == FK_GRAM4) {
        bitmap.swap(pairBitmap);
        bitmap2.swap(pairBitmap2);
    } else if (g_opts.prefilter) {
        bitmap = buildBitmap(tails, &im->keyBytes, &im->bitmapShift, &bitmap2, &im->bitmap2Shift);
    }
    im->bitmapBytes = (u32)bitmap.size();
    cudaError_t e = cudaMalloc(&im->d_bc, HSB_ROUNDUP(h->length, 16));
    if (e == cudaSuccess && !bitmap.empty()) {
        e = cudaMalloc(&im->d_bitmap, bitmap.size());
        if (e == cudaSuccess) {
            e = cudaMemcpy(im->d_bitmap, bitmap.data(), bitmap.size(), cudaMemcpyHostToDevice);
        }
    }
    if (e == cudaSuccess && !bitmap2.empty()) {
        e = cudaMalloc(&im->d_bitmap2, bitmap2.size());
        if (e == cudaSuccess) {
            e = cudaMemcpy(im->d_bitmap2, bitmap2.data(), bitmap2.size(), cudaMemcpyHostToDevice);
        }
    } else {
        im->bitmap2Shift = 0;
    }
    if (e == cudaSuccess) {
        e = cudaMalloc(&im->d_table, HSB_ROUNDUP(table.size(), 16));
    }
    if (e == cudaSuccess) {
        e = cudaMemcpy(im->d_bc, bc, h->length, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) {
        e = cudaMemcpy(im->d_table, table.data(), table.size(), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        freeImage(im);
        return e == cudaErrorMemoryAllocation ? HS_NOMEM : HS_UNKNOWN_ERROR;
    }
    im->deviceBytes = HSB_ROUNDUP(h->length, 16) + HSB_ROUNDUP(table.size(), 16) + bitmap.size() + bitmap2.size();
    *out = im;
    return HS_SUCCESS;
}

} // namespace

/* ---- corpus handle --------------------------------------------------------- */

struct hs_b200_corpus {
    int device = 0;
    u8 *d_alloc = nullptr;   /* owned allocation (nullptr when wrapping) */
    u8 *d_data = nullptr;    /* corpus position 0 */
    u64 bytes = 0;           /* end of the last block */
    u64 readableEnd = 0;
    u64 *d_off = nullptr;
    u32 *d_len = nullptr;
    size_t nblocks = 0;
    u32 uniformPitch = 0;
    u32 uniformLen = 0;      /* all blocks equally long (and uniformPitch set): tables not needed */
    u64 payload = 0;         /* sum of block lengths */
    size_t capData = 0, capBlocks = 0; /* allocation sizes when reused */
};

/* ---- scratch ------------------------------------------------------------------ */

struct hs_scratch {
    u32 magic;
    u8 in_use;
    int device;
    void *alloc_base;        /* what g_scratch_alloc returned */
    cudaStream_t stream, copyStream;
    cudaStream_t activeStream; /* stream the pending scan was enqueued on */
    cudaEvent_t evStart, evStop;
    cudaEvent_t evDone;       /* counters of the pending scan have landed on the host */
    std::vector<cudaEvent_t> *chunkEvents;
    std::vector<DevImage *> *images;
    DevMatch *d_out;
    u32 outCap;
    bool ringSplit;          /* d_out holds 2 * outCap records: ring + candidate list (split mode) */
    u32 *d_counters;
    u32 *h_counters;         /* pinned */
    hs_b200_corpus *inlineCorpus; /* staging for hs_scan / hs_b200_scan_blocks */
    u8 *h_stage, *h_stage2;  /* pinned pack buffers (unaligned host blocks), alternating */
    size_t h_stageCap, h_stage2Cap;
    cudaEvent_t evStage, evStage2;
    std::vector<u64> *tmpOff;
    const DevImage *lastImage;
    const hs_b200_corpus *lastCorpus;
    /* fused exchange over peer memory (hs_b200_set_peer_exchange) */
    u32 nPeers, myRank, peerCap, blockBase;
    DevMatch *peers[MAX_PEERS];
    bool pending;
    u32 lastCount;
    float lastMs;
    int smCount, maxSmem;
};

namespace {

hs_error_t validDb(const hs_database_t *db) { /* src/database.h:125-137 */
    const DbHeader *h = (const DbHeader *)db;
    if (!h || h->magic != DB_MAGIC) {
        return HS_INVALID;
    }
    if (h->version != DB_VERSION) {
        return HS_DB_VERSION_ERROR;
    }
    return HS_SUCCESS;
}

hs_error_t dbIsValid(const hs_database_t *db) { /* src/database.c:326-350 */
    hs_error_t r = validDb(db);
    if (r != HS_SUCCESS) {
        return r;
    }
    const DbHeader *h = (const DbHeader *)db;
    const u64 known = PLATFORM_NOAVX2 | PLATFORM_NOAVX512 | PLATFORM_NOAVX512VBMI;
    if (h->platform & ~known) {
        return HS_DB_PLATFORM_ERROR;
    }
    if ((uintptr_t)dbRose(db) % 16) {
        return HS_INVALID;
    }
    if (crc32c(0, (const u8 *)dbRose(db), h->length) != h->crc32) {
        return HS_INVALID;
    }
    return HS_SUCCESS;
}

bool markInUse(hs_scratch *s) { /* src/scratch.h:249-271 */
    if (s->in_use) {
        return true;
    }
    s->in_use = 1;
    return false;
}
void unmarkInUse(hs_scratch *s) { s->in_use = 0; }

hs_error_t findImage(hs_scratch *s, const hs_database_t *db, const DevImage **out) {
    const DbHeader *h = (const DbHeader *)db;
    for (DevImage *im : *s->images) {
        if (im->db == db && im->crc == h->crc32 && im->length == h->length) {
            *out = im;
            return HS_SUCCESS;
        }
    }
    DeviceGuard guard(s->device); /* the image is allocated on the scratch's device */
    DevImage *im = nullptr;
    hs_error_t r = buildImage(db, &im);
    if (r != HS_SUCCESS) {
        return r;
    }
    s->images->push_back(im);
    *out = im;
    return HS_SUCCESS;
}

hs_error_t growRing(hs_scratch *s, u32 cap) {
    initOpts();
    const bool split = true; /* second half = candidate list of the split kernels (FK_PAIR32 always) */
    if (cap <= s->outCap && (s->ringSplit || !split)) {
        return HS_SUCCESS;
    }
    cap = std::max(cap, s->outCap);
    DeviceGuard guard(s->device);
    DevMatch *n = nullptr;
    CUDA_TRY(cudaMalloc(&n, (size_t)cap * sizeof(DevMatch) * (split ? 2 : 1)));
    cudaFree(s->d_out);
    s->d_out = n;
    s->outCap = cap;
    s->ringSplit = split;
    return HS_SUCCESS;
}

void freeCorpus(hs_b200_corpus *c) {
    if (!c) {
        return;
    }
    cudaFree(c->d_alloc);
    cudaFree(c->d_off);
    cudaFree(c->d_len);
    delete c;
}

/* (Re)size a corpus handle's device buffers (grow-only). */
hs_error_t reserveCorpus(hs_b200_corpus *c, u64 dataBytes, size_t nblocks) {
    DeviceGuard guard(c->device);
    const size_t need = FRONT_PAD + HSB_ROUNDUP(dataBytes, 16) + 64;
    if (need > c->capData) {
        cudaFree(c->d_alloc);
        c->d_alloc = nullptr;
        c->capData = 0;
        const size_t cap = need + need / 8;
        CUDA_TRY(cudaMalloc(&c->d_alloc, cap));
        CUDA_TRY(cudaMemset(c->d_alloc, 0, FRONT_PAD));
        c->capData = cap;
    }
    c->d_data = c->d_alloc + FRONT_PAD;
    if (nblocks > c->capBlocks) {
        cudaFree(c->d_off);
        cudaFree(c->d_len);
        c->d_off = nullptr;
        c->d_len = nullptr;
        c->capBlocks = 0;
        const size_t cap = nblocks + nblocks / 8 + 16;
        CUDA_TRY(cudaMalloc(&c->d_off, cap * sizeof(u64)));
        CUDA_TRY(cudaMalloc(&c->d_len, cap * sizeof(u32)));
        c->capBlocks = cap;
    }
    return HS_SUCCESS;
}

u32 detectPitch(const u64 *off, const u32 *len, size_t n) {
    if (n == 0) {
        return 0;
    }
    if (n == 1) {
        return off[0] == 0 ? (u32)std::max<u64>(16, HSB_ROUNDUP((u64)len[0], 16)) : 0;
    }
    const u64 pitch = off[1] - off[0];
    if (off[0] != 0 || pitch == 0 || pitch > 0xffffffffu) {
        return 0;
    }
    for (size_t i = 0; i < n; i++) {
        if (off[i] != i * pitch || len[i] > pitch) {
            return 0;
        }
    }
    return (u32)pitch;
}

struct ScanPlan {
    LaunchCfg cfg;
    u32 tileBytes, nstages;
};

hs_error_t planScan(const hs_scratch *s, const DevImage *im, ScanPlan *pl) {
    initOpts();
    if (im->kind == FK_OUTFIX) { /* one launch over all blocks once the corpus has arrived (launchRange) */
        memset(&pl->cfg, 0, sizeof(pl->cfg));
        pl->tileBytes = 1u << 20;
        pl->nstages = 0;
        return HS_SUCCESS;
    }
    const int direct = g_opts.direct ? 1 : 0;
    int warps = g_opts.warps > 0 ? std::min(32, g_opts.warps) : (direct ? 28 : 32);
    u32 tile = (u32)std::max(512, g_opts.tileBytes) & ~511u;
    u32 stages = (u32)std::max(2, std::min(8, g_opts.stages));
    /* shrink until the table + staging fit the opt-in shared memory */
    int stride = im->stride;
    if ((g_opts.stride == 1 || g_opts.stride == 2 || g_opts.stride == 4) &&
        (im->kind == FK_HASH32 || im->kind == FK_HASH64)) {
        stride = g_opts.stride; /* any sampling subset is a sound filter */
    }
    if (im->kind == FK_GRAM4) {
        warps = std::min(warps, 28);
        while (warps > 1 && scanSmemBytes(FK_GRAM4, 0, 0, 0, 0, 0, warps) > (size_t)s->maxSmem) {
            warps--;
        }
        pl->cfg.smemBytes = scanSmemBytes(FK_GRAM4, 0, 0, 0, 0, 0, warps);
        if (pl->cfg.smemBytes > (size_t)s->maxSmem || !s->ringSplit) {
            return HS_NOMEM;
        }
        pl->cfg.kind = im->kind;
        pl->cfg.slotBase = 0;
        pl->cfg.direct = 1;
        pl->cfg.stride = 1;
        pl->cfg.queued = 1;
        pl->cfg.wide = 0;
        pl->cfg.split = 1;
        pl->cfg.grid = s->smCount;
        pl->cfg.warps = warps;
        pl->tileBytes = tile;
        pl->nstages = (u32)std::max(0, std::min(64, g_opts.pfDist));
        return HS_SUCCESS;
    }
    if (im->kind == FK_PAIR32) {
        /* class-pair kernel: direct loads, stride 1, queued candidates, split confirm;
         * as many warps as the queues leave room for (896 threads x 72 registers at most) */
        const u32 contiguous = im->bitmapHoles ? 0 : im->bitmapBytes;
        warps = std::min(warps, 28);
        while (warps > 1 && scanSmemBytes(FK_PAIR32, im->pairBytes, contiguous, 0, 0, 0, warps) > (size_t)s->maxSmem) {
            warps--;
        }
        pl->cfg.smemBytes = scanSmemBytes(FK_PAIR32, im->pairBytes, contiguous, 0, 0, 0, warps);
        if (pl->cfg.smemBytes > (size_t)s->maxSmem || !s->ringSplit) {
            return HS_NOMEM;
        }
        pl->cfg.kind = im->kind;
        pl->cfg.slotBase = im->slotBase;
        pl->cfg.direct = 1;
        pl->cfg.stride = 1;
        /* candidate path: per-lane queue entries while candidates are rare; one entry per
         * word with candidates for sets that saturate the first stage (heavy=2 forces it).
         * The modelled rate assumes independent slots and is ~30x below what is measured:
         * 0.0015 modelled is ~40 candidates per KiB, where the per-word path starts to win
         * (profiles/r02_sweep_candidate_paths.log) */
        pl->cfg.queued = g_opts.heavy == 2 || (g_opts.heavy == 1 && im->pairRate > 0.0015) ? 2 : 1;
        pl->cfg.wide = 0;
        pl->cfg.split = 1;
        pl->cfg.grid = s->smCount;
        pl->cfg.warps = warps;
        pl->tileBytes = tile;
        pl->nstages = (u32)std::max(0, std::min(64, g_opts.pfDist));
        return HS_SUCCESS;
    }
    const bool byteKind = im->kind == FK_BYTE32 || im->kind == FK_BYTE64;
    const int wide = g_opts.wide && direct && stride == 1 && (im->kind == FK_BYTE32 || im->kind == FK_HASH32);
    const int queued = direct && stride == 1 && (g_opts.queue == 1 || (g_opts.queue == 2 && byteKind));
    const int split = wide && g_opts.split && s->ringSplit;
    if (direct && !(wide && split)) {
        warps = std::min(warps, 28); /* direct kernels are built for 896 threads (72 registers); the
                                      * split wide variant also for 1024 (64 registers, spill-free) */
    }
    if (wide) {
        tile = std::max(1024u, tile & ~1023u); /* a warp-iteration covers 1 KiB */
    }
    for (;;) {
        const size_t need = scanSmemBytes(im->kind, im->tableBytes, im->bitmapBytes, direct ? 0 : warps,
                                          stages, tile, wide ? -warps : queued ? warps : 0);
        if (need <= (size_t)s->maxSmem) {
            pl->cfg.smemBytes = need;
            break;
        }
        if (stages > 2) {
            stages--;
        } else if (tile > 1024) {
            tile >>= 1;
        } else if (warps > 4) {
            warps -= 4;
        } else if (tile > 512) {
            tile >>= 1;
        } else if (warps > 1) {
            warps--;
        } else {
            return HS_NOMEM;
        }
    }
    pl->cfg.kind = im->kind;
    pl->cfg.slotBase = im->slotBase;
    pl->cfg.direct = direct;
    pl->cfg.stride = stride;
    pl->cfg.queued = queued;
    pl->cfg.wide = wide;
    pl->cfg.split = split;
    pl->cfg.grid = s->smCount;
    pl->cfg.warps = warps;
    pl->tileBytes = tile;
    pl->nstages = direct ? (u32)std::max(0, std::min(64, g_opts.pfDist)) : stages;
    return HS_SUCCESS;
}

void fillParams(const hs_scratch *s, const DevImage *im, const hs_b200_corpus *c,
                const ScanPlan &pl, ScanParams *p) {
    memset(p, 0, sizeof(*p));
    p->corpus = c->d_data;
    p->corpusBytes = c->bytes;
    p->readableEnd = c->readableEnd;
    p->tileBytes = pl.tileBytes;
    p->nstages = pl.nstages;
    p->blockOff = c->d_off;
    p->blockLen = c->d_len;
    p->nblocks = (u32)c->nblocks;
    p->uniformPitch = c->uniformPitch;
    p->uniformLen = c->uniformLen;
    p->bc = im->d_bc;
    p->table = im->d_table;
    p->tableBytes = im->tableBytes;
    p->indexMask = im->indexMask;
    p->repShift = im->repShift;
    p->bitmap = im->d_bitmap;
    p->bitmapBytes = im->bitmapBytes;
    p->pairBytes = im->pairBytes;
    p->bitmapHoles = im->bitmapHoles;
    p->bucketFold = im->bucketFold;
    p->bitmapBits = im->bitmapBits;
    p->bitmapShift = im->bitmapShift;
    p->keyBytes = im->keyBytes;
    p->bitmap2 = (const u32 *)im->d_bitmap2;
    p->bitmap2Shift = im->d_bitmap2 ? im->bitmap2Shift : 0;
    p->confOff = im->confOff;
    p->engineOff = im->engineOff;
    p->confirmKind = im->confirmKind;
    p->groups = im->groups;
    p->out = s->d_out;
    p->outCap = s->outCap;
    p->counters = s->d_counters;
    p->nPeers = s->nPeers;
    p->myRank = s->myRank;
    p->peerCap = s->peerCap;
    p->blockBase = s->blockBase;
    for (u32 r = 0; r < s->nPeers; r++) {
        p->peers[r] = s->peers[r];
    }
}

/* Launch over tiles [t0, t1) of the corpus on `stream`. */
hs_error_t launchRange(hs_scratch *s, const DevImage *im, const hs_b200_corpus *c,
                       const ScanPlan &pl, u32 t0, u32 t1, cudaStream_t stream) {
    if (t1 <= t0) {
        return HS_SUCCESS;
    }
    if (im->kind == FK_OUTFIX) {
        /* a block is one thread's walk from its first byte: wait for the last range of the
         * corpus, then run the engine over every block */
        const u32 ntiles = (u32)((c->bytes + pl.tileBytes - 1) / pl.tileBytes);
        if (t1 < ntiles) {
            return HS_SUCCESS;
        }
        int smCount = 0, maxSmem = 0;
        cudaDeviceGetAttribute(&smCount, cudaDevAttrMultiProcessorCount, s->device);
        cudaDeviceGetAttribute(&maxSmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, s->device);
        for (DfaParams dp : im->engineLaunches) { /* every engine of one model in one launch */
            dp.corpus = c->d_data;
            dp.readableEnd = c->readableEnd;
            dp.blockOff = c->d_off;
            dp.blockLen = c->d_len;
            dp.nblocks = (u32)c->nblocks;
            dp.uniformPitch = c->uniformPitch;
            dp.uniformLen = c->uniformLen;
            dp.out = s->d_out;
            dp.outCap = s->outCap;
            dp.counters = s->d_counters;
            CUDA_TRY(launchDfa(dp, smCount, maxSmem, stream));
            g_launches++;
        }
        return HS_SUCCESS;
    }
    ScanParams p;
    fillParams(s, im, c, pl, &p);
    p.tileFirst = t0;
    p.ntiles = t1 - t0;
    LaunchCfg cfg = pl.cfg;
    const u32 perCta = (u32)cfg.warps;
    cfg.grid = (int)std::min<u32>((u32)cfg.grid, (p.ntiles + perCta - 1) / perCta);
    if (cfg.split) {
        CUDA_TRY(cudaMemsetAsync(s->d_counters + CTR_CANDQ, 0, sizeof(u32), stream));
    }
    CUDA_TRY(launchScan(cfg, p, stream));
    g_launches++;
    if (cfg.split) {
        CUDA_TRY(launchConfirm(cfg, p, stream));
        g_launches++;
    }
    return HS_SUCCESS;
}

size_t postprocess(const DevImage *im, DevMatch *m, size_t n) {
    return postprocessRecords(im->exhaustible, (MatchRec *)m, n);
}

/* Records of a scan, ordered and with the order-dependent report rules applied (see
 * postprocessRecords).  Single-outfix databases: the kernel's records carry report PROGRAM
 * offsets (and the padding of the lanes' reserved slots); each is replaced by the reports its
 * program raises -- roseReportAdaptor -> roseRunProgram (src/rose/match.c:611-633) -- first. */
hs_error_t postprocessVec(const DevImage *im, std::vector<DevMatch> *v) {
    if (im->kind != FK_OUTFIX) {
        v->resize(postprocess(im, v->data(), v->size()));
        return HS_SUCCESS;
    }
    const u8 *bc = (const u8 *)dbRose((const hs_database_t *)(im->dbCopy.data() + im->dbCopyShift));
    std::vector<DevMatch> outv;
    outv.reserve(v->size());
    for (const DevMatch &m : *v) {
        if (m.id == 0xffffffffu) {
            continue; /* a slot some lane reserved and did not fill */
        }
        auto it = im->progReports.find(m.id);
        if (it == im->progReports.end()) {
            std::vector<ProgReport> reps;
            if (m.id % INSTR_ALIGN || m.id < sizeof(RoseEngine) || m.id >= im->length ||
                !collectProgramReports(bc, im->length, m.id, &im->exhaustible, &reps)) {
                return HS_UNKNOWN_ERROR; /* a program with a state-carrying opcode (or a corrupt record) */
            }
            it = im->progReports.emplace(m.id, std::move(reps)).first;
        }
        for (const ProgReport &rp : it->second) {
            if (m.to < rp.min_bound || m.to > rp.max_bound) {
                continue; /* CHECK_BOUNDS (hs_expr_ext min_offset / max_offset) */
            }
            DevMatch o = m;
            o.id = rp.onmatch;
            o.to = (u64)((long long)m.to + rp.offset_adjust);
            outv.push_back(o);
        }
    }
    outv.resize(postprocess(im, outv.data(), outv.size()));
    v->swap(outv);
    return HS_SUCCESS;
}

hs_error_t finishScan(hs_scratch *s, u32 *count) {
    /* wait for THIS scan only: a later scan may already be queued behind it
     * on the same stream (double-buffered callers) */
    cudaError_t e = cudaEventSynchronize(s->evDone);
    s->pending = false;
    if (e != cudaSuccess) {
        return HS_UNKNOWN_ERROR;
    }
    cudaEventElapsedTime(&s->lastMs, s->evStart, s->evStop);
    if (s->h_counters[CTR_ERROR]) {
        return HS_UNKNOWN_ERROR;
    }
    *count = s->h_counters[CTR_MATCHES];
    s->lastCount = *count;
    return HS_SUCCESS;
}

/* Enqueue: reset counters, scan the whole corpus, read the counters back. */
hs_error_t enqueueScan(hs_scratch *s, const DevImage *im, const hs_b200_corpus *c,
                       cudaStream_t stream) {
    ScanPlan pl;
    hs_error_t r = planScan(s, im, &pl);
    if (r != HS_SUCCESS) {
        return r;
    }
    CUDA_TRY(cudaMemsetAsync(s->d_counters, 0, CTR_COUNT * sizeof(u32), stream));
    CUDA_TRY(cudaEventRecord(s->evStart, stream));
    const u32 ntiles = (u32)((c->bytes + pl.tileBytes - 1) / pl.tileBytes);
    r = launchRange(s, im, c, pl, 0, ntiles, stream);
    if (r != HS_SUCCESS) {
        return r;
    }
    CUDA_TRY(cudaEventRecord(s->evStop, stream));
    if (s->nPeers) {
        ScanParams pp;
        fillParams(s, im, c, pl, &pp);
        CUDA_TRY(launchPublishCount(pp, stream));
        g_launches++;
    }
    CUDA_TRY(cudaMemcpyAsync(s->h_counters, s->d_counters, CTR_COUNT * sizeof(u32),
                             cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaEventRecord(s->evDone, stream));
    s->lastImage = im;
    s->lastCorpus = c;
    s->activeStream = stream;
    s->pending = true;
    return HS_SUCCESS;
}

/* Fill a corpus handle from host blocks.  Returns through *direct whether the
 * caller's buffer could be copied as it lies (all starts 16-byte aligned
 * relative to the first block, ascending, disjoint). */
hs_error_t layoutBlocks(hs_scratch *s, const unsigned long long *offsets,
                        const unsigned *lengths, size_t nblocks, std::vector<u64> *packed,
                        u64 *total, u64 *payload, bool *direct, u32 *uniPitch = nullptr,
                        u32 *uniLen = nullptr) {
    (void)s;
    if (uniPitch) {
        *uniPitch = *uniLen = 0;
        /* fast path (hsbench-style corpora): equally long blocks at a fixed
         * 16-byte aligned pitch -- one tight pass, no packed table at all */
        if (nblocks >= 2 && lengths[0] && offsets[1] > offsets[0]) {
            const u64 base = offsets[0], pitch = offsets[1] - offsets[0];
            const u32 len0 = lengths[0];
            if (pitch % 16 == 0 && pitch <= 0xffffffffu && len0 <= pitch) {
                /* two simple loops the compiler vectorises */
                size_t bad = 0;
                u64 expect = base;
                for (size_t i = 0; i < nblocks; i++, expect += pitch) {
                    bad += offsets[i] != expect;
                }
                for (size_t i = 0; i < nblocks; i++) {
                    bad += lengths[i] != len0;
                }
                if (!bad) {
                    packed->clear();
                    *total = (nblocks - 1) * pitch + len0;
                    *payload = (u64)nblocks * len0;
                    *direct = true;
                    *uniPitch = (u32)pitch;
                    *uniLen = len0;
                    return HS_SUCCESS;
                }
            }
        }
    }
    packed->resize(nblocks);
    bool ok = nblocks > 0;
    u64 pay = 0;
    const u64 base = nblocks ? offsets[0] : 0;
    u64 prevEnd = 0;
    for (size_t i = 0; i < nblocks; i++) {
        pay += lengths[i];
        if (ok) {
            if (offsets[i] < base || (offsets[i] - base) % 16 || offsets[i] - base < prevEnd) {
                ok = false;
            } else {
                (*packed)[i] = offsets[i] - base;
                prevEnd = offsets[i] - base + lengths[i];
            }
        }
    }
    if (!ok) {
        u64 pos = 0;
        for (size_t i = 0; i < nblocks; i++) {
            (*packed)[i] = pos;
            pos += HSB_ROUNDUP((u64)lengths[i], 16);
            if (lengths[i] == 0) {
                pos += 16; /* keep starts distinct */
            }
        }
        prevEnd = nblocks ? (*packed)[nblocks - 1] + lengths[nblocks - 1] : 0;
    }
    *total = prevEnd;
    *payload = pay;
    *direct = ok;
    return HS_SUCCESS;
}

} // namespace

extern "C" {

hs_error_t hs_valid_platform(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        return HS_ARCH_ERROR;
    }
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, 0);
    return major >= 10 ? HS_SUCCESS : HS_ARCH_ERROR;
}

unsigned long long hs_b200_launch_count(void) { return g_launches.load(); }

float hs_b200_last_kernel_ms(const hs_scratch_t *scratch) {
    return scratch ? scratch->lastMs : 0.0f;
}

/* Counters of the last finished scan: [0] raw records, [1] error, [2]
 * first-stage candidates, [3] byte-confirmed literals, [4] candidates that
 * passed the prefilter. */
hs_error_t hs_b200_last_counters(const hs_scratch_t *scratch, unsigned int out[8]) {
    if (!scratch || !out || scratch->pending) {
        return HS_INVALID;
    }
    memcpy(out, scratch->h_counters, CTR_COUNT * sizeof(u32));
    return HS_SUCCESS;
}

hs_error_t hs_b200_set_runtime_option(const char *key, int value) {
    initOpts();
    if (!key) {
        return HS_INVALID;
    }
    struct { const char *n; int *v; } k[] = {
        {"warps", &g_opts.warps},       {"tile_bytes", &g_opts.tileBytes},
        {"stages", &g_opts.stages},     {"wide_fdr", &g_opts.wideFdr},
        {"chunk_mb", &g_opts.chunkMB},  {"initial_ring", &g_opts.initialRing},
        {"stride", &g_opts.stride},     {"prefilter", &g_opts.prefilter},
        {"rebuild", &g_opts.rebuild},   {"domain", &g_opts.domain},
        {"direct", &g_opts.direct},     {"replicas", &g_opts.replicas},
        {"pf_dist", &g_opts.pfDist},    {"queue", &g_opts.queue},
        {"first_stage", &g_opts.firstStage}, {"wide", &g_opts.wide},
        {"split", &g_opts.split},       {"big_set", &g_opts.bigSet},
        {"big_set_classes", &g_opts.bigSetClasses}, {"heavy", &g_opts.heavy},
        {"gram", &g_opts.gram},                {"fat_pair", &g_opts.fatPair},
        {"dfa_ilp", &g_opts.dfaIlp}};
    for (auto &x : k) {
        if (!strcmp(key, x.n)) {
            *x.v = value;
            return HS_SUCCESS;
        }
    }
    return HS_INVALID;
}

/* Acceleration primitives on a host buffer (src/nfa/accel.c:35 run_accel):
 * first position whose byte (pair) is in the class, or len. */
hs_error_t hs_b200_accel_find(unsigned int type, const unsigned char *params,
                              const unsigned char *buf, size_t len, unsigned long long *pos) {
    if (!params || (!buf && len) || !pos) {
        return HS_INVALID;
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        return HS_ARCH_ERROR;
    }
    u8 *d = nullptr;
    u64 *d_res = nullptr;
    CUDA_TRY(cudaMalloc(&d, HSB_ROUNDUP(len, 16) + 64));
    cudaError_t e = cudaMalloc(&d_res, 8);
    if (e == cudaSuccess) e = cudaMemset(d, 0, HSB_ROUNDUP(len, 16) + 64);
    if (e == cudaSuccess && len) e = cudaMemcpy(d, buf, len, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launchAccelFind((int)type, params, d, len, d_res, 0);
    if (e == cudaSuccess) g_launches++;
    unsigned long long r = len;
    if (e == cudaSuccess) e = cudaMemcpy(&r, d_res, 8, cudaMemcpyDeviceToHost);
    cudaFree(d);
    cudaFree(d_res);
    if (e != cudaSuccess) {
        return e == cudaErrorInvalidValue ? HS_INVALID : HS_UNKNOWN_ERROR;
    }
    *pos = r;
    return HS_SUCCESS;
}

/* ---- scratch ---------------------------------------------------------------- */

static hs_error_t newScratch(hs_scratch **out) {
    initOpts();
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        return HS_ARCH_ERROR; /* no CPU scan path exists */
    }
    void *raw = g_scratch_alloc(sizeof(hs_scratch) + 64);
    hs_error_t r = checkAlloc(raw);
    if (r != HS_SUCCESS) {
        g_scratch_free(raw);
        return r;
    }
    hs_scratch *s = (hs_scratch *)HSB_ROUNDUP((uintptr_t)raw, 64);
    memset(s, 0, sizeof(*s));
    s->alloc_base = raw;
    s->magic = SCRATCH_MAGIC;
    cudaGetDevice(&s->device);
    cudaDeviceGetAttribute(&s->smCount, cudaDevAttrMultiProcessorCount, s->device);
    cudaDeviceGetAttribute(&s->maxSmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, s->device);
    s->images = new std::vector<DevImage *>();
    s->chunkEvents = new std::vector<cudaEvent_t>();
    s->tmpOff = new std::vector<u64>();
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->copyStream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&s->evStart);
    if (e == cudaSuccess) e = cudaEventCreate(&s->evStop);
    if (e == cudaSuccess) {
        /* HSB200_BLOCKING_SYNC=1: sleep instead of spinning while a scan is awaited */
        const char *bs = getenv("HSB200_BLOCKING_SYNC");
        e = cudaEventCreateWithFlags(&s->evDone, cudaEventDisableTiming |
                                                      ((bs && *bs == '1') ? cudaEventBlockingSync : 0));
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->evStage, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->evStage2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_counters, CTR_COUNT * sizeof(u32));
    if (e == cudaSuccess) e = cudaMallocHost(&s->h_counters, CTR_COUNT * sizeof(u32));
    if (e == cudaSuccess) {
        memset(s->h_counters, 0, CTR_COUNT * sizeof(u32));
        s->inlineCorpus = new hs_b200_corpus();
        s->inlineCorpus->device = s->device;
    }
    if (e != cudaSuccess || growRing(s, (u32)g_opts.initialRing) != HS_SUCCESS) {
        hs_free_scratch(s);
        return e == cudaErrorMemoryAllocation ? HS_NOMEM : HS_UNKNOWN_ERROR;
    }
    *out = s;
    return HS_SUCCESS;
}

hs_error_t hs_alloc_scratch(const hs_database_t *db, hs_scratch_t **scratch) {
    if (!db || !scratch) {
        return HS_INVALID;
    }
    hs_error_t r = dbIsValid(db);
    if (r != HS_SUCCESS) {
        return r;
    }
    hs_scratch *s = *scratch;
    if (s) {
        if ((uintptr_t)s % 64 || s->magic != SCRATCH_MAGIC) {
            return HS_INVALID;
        }
        if (markInUse(s)) {
            return HS_SCRATCH_IN_USE;
        }
    } else {
        r = newScratch(&s);
        if (r != HS_SUCCESS) {
            *scratch = nullptr;
            return r;
        }
        s->in_use = 1;
    }
    DeviceGuard guard(s->device);
    const DevImage *im = nullptr;
    r = findImage(s, db, &im);
    unmarkInUse(s);
    if (r != HS_SUCCESS) {
        if (!*scratch) {
            hs_free_scratch(s);
        }
        return r;
    }
    *scratch = s;
    return HS_SUCCESS;
}

hs_error_t hs_clone_scratch(const hs_scratch_t *src, hs_scratch_t **dest) {
    if (!dest || !src || (uintptr_t)src % 64 || src->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    *dest = nullptr;
    DeviceGuard guard(src->device); /* the clone lives on the source's device */
    hs_scratch *s = nullptr;
    hs_error_t r = newScratch(&s);
    if (r != HS_SUCCESS) {
        return r;
    }
    for (const DevImage *im : *src->images) {
        const DevImage *mine = nullptr;
        /* rebuild from the source image's own copy of the database: the application may
         * have freed the original (legal in the reference, whose clone never touches it) */
        const hs_database_t *copy = (const hs_database_t *)(im->dbCopy.data() + im->dbCopyShift);
        DevImage *fresh = nullptr;
        r = buildImage(copy, &fresh);
        if (r == HS_SUCCESS) {
            fresh->db = im->db; /* keep the identity the application knows */
            s->images->push_back(fresh);
            mine = fresh;
        }
        if (r != HS_SUCCESS) {
            hs_free_scratch(s);
            return r;
        }
    }
    r = growRing(s, src->outCap);
    if (r != HS_SUCCESS) {
        hs_free_scratch(s);
        return r;
    }
    *dest = s;
    return HS_SUCCESS;
}

hs_error_t hs_scratch_size(const hs_scratch_t *scratch, size_t *size) {
    if (!size || !scratch || (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    size_t n = sizeof(hs_scratch) + 64 + (size_t)scratch->outCap * sizeof(DevMatch);
    for (const DevImage *im : *scratch->images) {
        n += im->deviceBytes;
    }
    if (scratch->inlineCorpus) {
        n += scratch->inlineCorpus->capData;
    }
    *size = n;
    return HS_SUCCESS;
}

hs_error_t hs_free_scratch(hs_scratch_t *s) {
    if (!s) {
        return HS_SUCCESS;
    }
    if ((uintptr_t)s % 64 || s->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    if (markInUse(s)) {
        return HS_SCRATCH_IN_USE;
    }
    DeviceGuard guard(s->device);
    s->magic = 0;
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->images) {
        for (DevImage *im : *s->images) {
            freeImage(im);
        }
        delete s->images;
    }
    if (s->chunkEvents) {
        for (cudaEvent_t ev : *s->chunkEvents) {
            cudaEventDestroy(ev);
        }
        delete s->chunkEvents;
    }
    delete s->tmpOff;
    freeCorpus(s->inlineCorpus);
    cudaFree(s->d_out);
    cudaFree(s->d_counters);
    if (s->h_counters) cudaFreeHost(s->h_counters);
    if (s->h_stage) cudaFreeHost(s->h_stage);
    if (s->h_stage2) cudaFreeHost(s->h_stage2);
    if (s->evStage) cudaEventDestroy(s->evStage);
    if (s->evStage2) cudaEventDestroy(s->evStage2);
    if (s->evStart) cudaEventDestroy(s->evStart);
    if (s->evStop) cudaEventDestroy(s->evStop);
    if (s->evDone) cudaEventDestroy(s->evDone);
    if (s->stream) cudaStreamDestroy(s->stream);
    if (s->copyStream) cudaStreamDestroy(s->copyStream);
    g_scratch_free(s->alloc_base);
    return HS_SUCCESS;
}

/* ---- corpus handles ------------------------------------------------------------ */

static hs_error_t setBlocks(hs_b200_corpus *c, const u64 *packed, const unsigned *lengths,
                            size_t nblocks, u64 total, u64 payload, cudaStream_t stream,
                            u32 uniPitch = 0, u32 uniLen = 0) {
    c->nblocks = nblocks;
    c->bytes = total;
    c->payload = payload;
    if (uniPitch && uniLen) { /* layoutBlocks already proved uniformity: no tables */
        c->uniformPitch = uniPitch;
        c->uniformLen = uniLen;
        return HS_SUCCESS;
    }
    c->uniformPitch = detectPitch(packed, lengths, nblocks);
    c->uniformLen = 0;
    if (c->uniformPitch && nblocks) {
        u32 l0 = lengths[0];
        for (size_t i = 1; i < nblocks && l0; i++) {
            if (lengths[i] != l0) {
                l0 = 0;
            }
        }
        c->uniformLen = l0;
    }
    if (nblocks && !c->uniformLen) {
        CUDA_TRY(cudaMemcpyAsync(c->d_off, packed, nblocks * sizeof(u64), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(c->d_len, lengths, nblocks * sizeof(u32), cudaMemcpyHostToDevice, stream));
    }
    return HS_SUCCESS;
}

hs_error_t hs_b200_corpus_upload(const char *data, const unsigned long long *offsets,
                                 const unsigned int *lengths, size_t nblocks, int device,
                                 hs_b200_corpus_t **corpus) {
    if (!corpus || (nblocks && (!data || !offsets || !lengths)) || nblocks > 0xfffffff0u) {
        return HS_INVALID;
    }
    *corpus = nullptr;
    if (cudaSetDevice(device) != cudaSuccess) {
        return HS_ARCH_ERROR;
    }
    hs_b200_corpus *c = new (std::nothrow) hs_b200_corpus();
    if (!c) {
        return HS_NOMEM;
    }
    c->device = device;
    std::vector<u64> packed;
    u64 total = 0, payload = 0;
    bool direct = false;
    u32 uniPitch = 0, uniLen = 0;
    layoutBlocks(nullptr, offsets, lengths, nblocks, &packed, &total, &payload, &direct, &uniPitch, &uniLen);
    hs_error_t r = reserveCorpus(c, total, nblocks);
    if (r != HS_SUCCESS) {
        freeCorpus(c);
        return r;
    }
    cudaError_t e = cudaSuccess;
    if (direct) {
        e = cudaMemcpy(c->d_data, data + offsets[0], total, cudaMemcpyHostToDevice);
    } else {
        /* pack through a host buffer in 64 MiB pieces */
        std::vector<u8> stage;
        const size_t CH = 64u << 20;
        size_t i = 0;
        while (i < nblocks && e == cudaSuccess) {
            const u64 start = packed[i];
            size_t j = i;
            while (j < nblocks && packed[j] + lengths[j] - start <= CH) {
                j++;
            }
            if (j == i) {
                j = i + 1;
            }
            const u64 end = packed[j - 1] + lengths[j - 1];
            stage.assign(end - start, 0);
            for (size_t k = i; k < j; k++) {
                memcpy(stage.data() + (packed[k] - start), data + offsets[k], lengths[k]);
            }
            e = cudaMemcpy(c->d_data + start, stage.data(), end - start, cudaMemcpyHostToDevice);
            i = j;
        }
    }
    if (e == cudaSuccess) {
        /* zero the tail so the last tile's look-ahead reads defined bytes */
        e = cudaMemset(c->d_data + total, 0, HSB_ROUNDUP(total, 16) + 32 - total);
    }
    c->readableEnd = HSB_ROUNDUP(total, 16) + 16;
    if (e == cudaSuccess) {
        r = setBlocks(c, packed.data(), lengths, nblocks, total, payload, 0, uniPitch, uniLen);
        if (r == HS_SUCCESS && cudaDeviceSynchronize() != cudaSuccess) {
            r = HS_UNKNOWN_ERROR;
        }
    } else {
        r = HS_UNKNOWN_ERROR;
    }
    if (r != HS_SUCCESS) {
        freeCorpus(c);
        return r;
    }
    *corpus = c;
    return HS_SUCCESS;
}

hs_error_t hs_b200_corpus_wrap(const void *d_data, size_t data_bytes,
                               const unsigned long long *offsets, const unsigned int *lengths,
                               size_t nblocks, int device, hs_b200_corpus_t **corpus) {
    if (!corpus || !d_data || (uintptr_t)d_data % 16 || (nblocks && (!offsets || !lengths)) ||
        nblocks > 0xfffffff0u) {
        return HS_INVALID;
    }
    *corpus = nullptr;
    u64 prevEnd = 0, payload = 0;
    for (size_t i = 0; i < nblocks; i++) {
        if (offsets[i] % 16 || offsets[i] < prevEnd || offsets[i] + lengths[i] > data_bytes) {
            return HS_INVALID;
        }
        prevEnd = offsets[i] + lengths[i];
        payload += lengths[i];
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        return HS_ARCH_ERROR;
    }
    hs_b200_corpus *c = new (std::nothrow) hs_b200_corpus();
    if (!c) {
        return HS_NOMEM;
    }
    c->device = device;
    hs_error_t r = HS_SUCCESS;
    if (nblocks) {
        cudaError_t e = cudaMalloc(&c->d_off, nblocks * sizeof(u64));
        if (e == cudaSuccess) e = cudaMalloc(&c->d_len, nblocks * sizeof(u32));
        if (e != cudaSuccess) {
            freeCorpus(c);
            return HS_NOMEM;
        }
        c->capBlocks = nblocks;
    }
    c->d_data = (u8 *)d_data;
    /* the caller's buffer must be readable up to data_bytes rounded up to 16 */
    c->readableEnd = HSB_ROUNDUP((u64)data_bytes, 16);
    std::vector<u64> off(offsets, offsets + nblocks);
    r = setBlocks(c, off.data(), lengths, nblocks, prevEnd, payload, 0);
    if (r == HS_SUCCESS && cudaDeviceSynchronize() != cudaSuccess) {
        r = HS_UNKNOWN_ERROR;
    }
    if (r != HS_SUCCESS) {
        freeCorpus(c);
        return r;
    }
    *corpus = c;
    return HS_SUCCESS;
}

hs_error_t hs_b200_corpus_free(hs_b200_corpus_t *corpus) {
    freeCorpus(corpus);
    return HS_SUCCESS;
}

size_t hs_b200_corpus_bytes(const hs_b200_corpus_t *corpus) {
    return corpus ? (size_t)corpus->payload : 0;
}

/* ---- device-resident scan --------------------------------------------------------- */

static hs_error_t checkScanArgs(const hs_database_t *db, hs_scratch_t *scratch) {
    hs_error_t err = validDb(db);
    if (err != HS_SUCCESS) {
        return err;
    }
    const RoseEngine *rose = dbRose(db);
    if ((uintptr_t)rose % 16) {
        return HS_INVALID;
    }
    if (rose->mode != MODE_BLOCK) {
        return HS_DB_MODE_ERROR;
    }
    if ((uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    return HS_SUCCESS;
}

hs_error_t hs_b200_scan_corpus_async(const hs_database_t *db, const hs_b200_corpus_t *corpus,
                                     hs_scratch_t *scratch, void *cuda_stream) {
    if (!scratch || !corpus) {
        return HS_INVALID;
    }
    hs_error_t r = checkScanArgs(db, scratch);
    if (r != HS_SUCCESS) {
        return r;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    DeviceGuard guard(scratch->device);
    const DevImage *im = nullptr;
    r = findImage(scratch, db, &im);
    if (r == HS_SUCCESS) {
        cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : scratch->stream;
        if (corpus->bytes == 0 || corpus->nblocks == 0) {
            scratch->h_counters[CTR_MATCHES] = 0;
            scratch->h_counters[CTR_ERROR] = 0;
            scratch->lastImage = im;
            scratch->lastCorpus = corpus;
            scratch->pending = false;
            scratch->lastCount = 0;
        } else {
            r = enqueueScan(scratch, im, corpus, st);
        }
    }
    unmarkInUse(scratch);
    return r;
}

hs_error_t hs_b200_scan_corpus_finish(hs_scratch_t *scratch, unsigned long long *nrecords,
                                      const void **d_records) {
    if (!scratch || (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    DeviceGuard guard(scratch->device);
    u32 count = scratch->lastCount;
    if (scratch->pending) {
        hs_error_t r = finishScan(scratch, &count);
        if (r != HS_SUCCESS) {
            return r;
        }
    }
    if (nrecords) {
        *nrecords = count;
    }
    if (d_records) {
        /* on overflow the ring is reallocated below: hand out no pointer */
        *d_records = count > scratch->outCap ? nullptr : scratch->d_out;
    }
    if (count > scratch->outCap) {
        /* ring overflowed: grow so that a re-run succeeds */
        u64 want = (u64)count + count / 4 + 1024;
        if (want > 0xfffffff0ull) {
            want = 0xfffffff0ull;
        }
        hs_error_t r = growRing(scratch, (u32)want);
        if (r != HS_SUCCESS) {
            return r;
        }
        return HS_INSUFFICIENT_SPACE;
    }
    return HS_SUCCESS;
}

/* ---- fused exchange over NVLink peer memory ----------------------------------- */

hs_error_t hs_b200_peer_buffer_alloc(size_t bytes, void **d_ptr, unsigned char handle[64]) {
    if (!d_ptr || !handle || !bytes) {
        return HS_INVALID;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    void *p = nullptr;
    CUDA_TRY(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return HS_UNKNOWN_ERROR;
    }
    memcpy(handle, &h, 64);
    *d_ptr = p;
    return HS_SUCCESS;
}

hs_error_t hs_b200_peer_buffer_open(const unsigned char handle[64], void **d_ptr) {
    if (!handle || !d_ptr) {
        return HS_INVALID;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void *p = nullptr;
    if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        return HS_UNKNOWN_ERROR;
    }
    *d_ptr = p;
    return HS_SUCCESS;
}

hs_error_t hs_b200_peer_buffer_read(const void *d_ptr, void *host_dst, size_t bytes) {
    if (!d_ptr || !host_dst) {
        return HS_INVALID;
    }
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(host_dst, d_ptr, bytes, cudaMemcpyDeviceToHost));
    return HS_SUCCESS;
}

hs_error_t hs_b200_peer_buffer_close(void *d_ptr, int opened) {
    if (!d_ptr) {
        return HS_SUCCESS;
    }
    cudaError_t e = opened ? cudaIpcCloseMemHandle(d_ptr) : cudaFree(d_ptr);
    return e == cudaSuccess ? HS_SUCCESS : HS_UNKNOWN_ERROR;
}

hs_error_t hs_b200_set_peer_exchange(hs_scratch_t *scratch, unsigned int nranks, unsigned int my_rank,
                                     void *const *peer_bases, size_t cap_per_rank,
                                     unsigned int block_base) {
    if (!scratch || (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC || nranks > MAX_PEERS ||
        (nranks && (!peer_bases || my_rank >= nranks || cap_per_rank == 0 || cap_per_rank > 0xfffffff0u))) {
        return HS_INVALID;
    }
    scratch->nPeers = nranks;
    scratch->myRank = my_rank;
    scratch->peerCap = (u32)cap_per_rank;
    scratch->blockBase = block_base;
    for (unsigned r = 0; r < nranks; r++) {
        scratch->peers[r] = (DevMatch *)peer_bases[r];
    }
    return HS_SUCCESS;
}

hs_error_t hs_b200_export_records_async(hs_scratch_t *scratch, void *d_dst, size_t cap,
                                        void *d_count, void *cuda_stream) {
    if (!scratch || !d_dst || !d_count || (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    DeviceGuard guard(scratch->device);
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : scratch->stream;
    const size_t n = std::min<size_t>(cap, scratch->outCap);
    if (n) {
        CUDA_TRY(cudaMemcpyAsync(d_dst, scratch->d_out, n * sizeof(DevMatch), cudaMemcpyDeviceToDevice, st));
    }
    CUDA_TRY(cudaMemcpyAsync(d_count, scratch->d_counters + CTR_MATCHES, sizeof(u32),
                             cudaMemcpyDeviceToDevice, st));
    return HS_SUCCESS;
}

hs_error_t hs_b200_copy_records(hs_scratch_t *scratch, void *d_dst, size_t cap) {
    if (!scratch || !d_dst || scratch->pending) {
        return HS_INVALID;
    }
    DeviceGuard guard(scratch->device);
    const size_t n = std::min<size_t>(cap, std::min<u32>(scratch->lastCount, scratch->outCap));
    if (n) {
        /* the records are final once evDone fired (finish waited for it); use
         * the copy stream so a scan queued behind on the scan stream is not
         * waited for */
        CUDA_TRY(cudaMemcpyAsync(d_dst, scratch->d_out, n * sizeof(DevMatch),
                                 cudaMemcpyDeviceToDevice, scratch->copyStream));
        CUDA_TRY(cudaStreamSynchronize(scratch->copyStream));
    }
    return HS_SUCCESS;
}

hs_error_t hs_b200_fetch_matches(const hs_database_t *db, hs_scratch_t *scratch,
                                 hs_b200_match_t *out, size_t cap,
                                 unsigned long long *nmatches) {
    if (!scratch || !db || scratch->pending) {
        return HS_INVALID;
    }
    DeviceGuard guard(scratch->device);
    const DevImage *im = nullptr;
    hs_error_t r = findImage(scratch, db, &im);
    if (r != HS_SUCCESS) {
        return r;
    }
    const u32 n = std::min(scratch->lastCount, scratch->outCap);
    std::vector<DevMatch> tmp(n);
    if (n) {
        CUDA_TRY(cudaMemcpyAsync(tmp.data(), scratch->d_out, (size_t)n * sizeof(DevMatch),
                                 cudaMemcpyDeviceToHost, scratch->copyStream));
        CUDA_TRY(cudaStreamSynchronize(scratch->copyStream));
    }
    r = postprocessVec(im, &tmp);
    if (r != HS_SUCCESS) {
        return r;
    }
    const size_t m = tmp.size();
    if (nmatches) {
        *nmatches = m;
    }
    if (out) {
        if (cap < m) {
            return HS_INSUFFICIENT_SPACE;
        }
        memcpy(out, tmp.data(), m * sizeof(DevMatch));
    }
    return HS_SUCCESS;
}

/* ---- DFA engines in block mode ------------------------------------------------------
 *
 * nfaExecMcClellan8_B / nfaExecMcClellan16_B / nfaExecSheng_B (src/nfa/mcclellan.c:
 * 937-973, src/nfa/sheng.c:706-739) over every block of a resident corpus, offset 0
 * per block.  The callbacks the reference would fire (report, end offset) come back
 * as records {report, block, to}, ordered by (block, to, report). */
hs_error_t hs_b200_nfa_scan_corpus(const void *nfa, size_t nfa_len, const hs_b200_corpus_t *corpus,
                                   hs_b200_match_t *out, size_t cap, unsigned long long *nmatches,
                                   float *kernel_ms) {
    if (!nfa || nfa_len < sizeof(NFA) + 64 || !corpus || (cap && !out) || !nmatches) {
        return HS_INVALID;
    }
    NFA hdr;
    memcpy(&hdr, nfa, sizeof(hdr));
    if (hdr.length > nfa_len) {
        return HS_INVALID;
    }
    DfaParams p;
    {
        const hs_error_t er = engineParams(nfa, nfa_len, &p);
        if (er != HS_SUCCESS) {
            return er;
        }
    }
    DeviceGuard guard(corpus->device);
    int smCount = 0, maxSmem = 0;
    cudaDeviceGetAttribute(&smCount, cudaDevAttrMultiProcessorCount, corpus->device);
    cudaDeviceGetAttribute(&maxSmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, corpus->device);
    u8 *d_nfa = nullptr; /* the engine's bytes, then its entry of the engine table */
    u32 *d_ctr = nullptr;
    DevMatch *d_out = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    hs_error_t rv = HS_SUCCESS;
    u32 capDev = (u32)std::min<size_t>(std::max<size_t>(cap, 1u << 16), 0xfffffff0u);
    std::vector<DevMatch> host;
    const size_t entryAt = HSB_ROUNDUP(nfa_len, 16);
    cudaError_t e = cudaMalloc(&d_nfa, entryAt + sizeof(DfaEngine));
    if (e == cudaSuccess) e = cudaMemcpy(d_nfa, nfa, nfa_len, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        const DfaEngine entry = {d_nfa, p.tableBytes, p.states, p.squashes, 0};
        e = cudaMemcpy(d_nfa + entryAt, &entry, sizeof(entry), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaMalloc(&d_ctr, CTR_COUNT * sizeof(u32));
    if (e == cudaSuccess) e = cudaEventCreate(&ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&ev1);
    for (int attempt = 0; e == cudaSuccess && attempt < 3; attempt++) {
        e = cudaMalloc(&d_out, (size_t)capDev * sizeof(DevMatch));
        if (e != cudaSuccess) break;
        e = cudaMemset(d_ctr, 0, CTR_COUNT * sizeof(u32));
        p.corpus = corpus->d_data;
        p.readableEnd = corpus->readableEnd;
        p.blockOff = corpus->d_off;
        p.blockLen = corpus->d_len;
        p.nblocks = (u32)corpus->nblocks;
        p.uniformPitch = corpus->uniformPitch;
        p.uniformLen = corpus->uniformLen;
        p.engines = reinterpret_cast<const DfaEngine *>(d_nfa + entryAt);
        p.nengines = 1;
        p.out = d_out;
        p.outCap = capDev;
        p.counters = d_ctr;
        if (e == cudaSuccess) e = cudaEventRecord(ev0, 0);
        if (e == cudaSuccess) e = launchDfa(p, smCount, maxSmem, 0);
        if (e == cudaSuccess) e = cudaEventRecord(ev1, 0);
        g_launches++;
        u32 ctr[CTR_COUNT] = {0};
        if (e == cudaSuccess) e = cudaMemcpy(ctr, d_ctr, sizeof(ctr), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) break;
        if (ctr[CTR_MATCHES] > capDev) { /* grow and run again */
            cudaFree(d_out);
            d_out = nullptr;
            capDev = ctr[CTR_MATCHES] + ctr[CTR_MATCHES] / 8 + 1024;
            continue;
        }
        host.resize(ctr[CTR_MATCHES]); /* reserved slots: the lanes' unused ones carry id 0xffffffff */
        if (!host.empty()) {
            e = cudaMemcpy(host.data(), d_out, host.size() * sizeof(DevMatch), cudaMemcpyDeviceToHost);
        }
        host.erase(std::remove_if(host.begin(), host.end(), [](const DevMatch &m) { return m.id == 0xffffffffu; }),
                   host.end());
        if (kernel_ms && e == cudaSuccess) {
            cudaEventElapsedTime(kernel_ms, ev0, ev1);
        }
        break;
    }
    if (e != cudaSuccess) {
        rv = e == cudaErrorMemoryAllocation ? HS_NOMEM : HS_UNKNOWN_ERROR;
    } else {
        std::sort(host.begin(), host.end(), [](const DevMatch &a, const DevMatch &b) {
            if (a.block != b.block) return a.block < b.block;
            if (a.to != b.to) return a.to < b.to;
            return a.id < b.id;
        });
        *nmatches = host.size();
        memcpy(out, host.data(), std::min(cap, host.size()) * sizeof(DevMatch));
        if (host.size() > cap) {
            rv = HS_INSUFFICIENT_SPACE;
        }
    }
    cudaFree(d_nfa);
    cudaFree(d_ctr);
    cudaFree(d_out);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    return rv;
}

/* ---- host-buffer scans -------------------------------------------------------------- */

/* Copy host blocks into the scratch's inline corpus and scan them, with the
 * host->device copy pipelined against the kernel in chunk_mb pieces. */
static double nowMs() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static hs_error_t scanHostBlocks(const DevImage *im, hs_scratch *s, const char *data,
                                 const unsigned long long *offsets, const unsigned *lengths,
                                 size_t nblocks, std::vector<DevMatch> *matches,
                                 bool countOnly = false) {
    static const bool trace = getenv("HSB200_TRACE") != nullptr;
    DeviceGuard guard(s->device); /* every host-buffer scan (hs_scan, hs_b200_scan_blocks, streams) ends up here */
    const double t0 = nowMs();
    double tLayout = 0, tEnq = 0, tWait = 0, tRec = 0;
    hs_b200_corpus *c = s->inlineCorpus;
    std::vector<u64> &packed = *s->tmpOff;
    u64 total = 0, payload = 0;
    bool direct = false;
    u32 uniPitch = 0, uniLen = 0;
    layoutBlocks(s, offsets, lengths, nblocks, &packed, &total, &payload, &direct, &uniPitch, &uniLen);
    matches->clear();
    if (total == 0) {
        return HS_SUCCESS;
    }
    tLayout = nowMs();
    hs_error_t r = reserveCorpus(c, total, nblocks);
    if (r != HS_SUCCESS) {
        return r;
    }
    c->readableEnd = HSB_ROUNDUP(total, 16) + 16;
    r = setBlocks(c, packed.data(), lengths, nblocks, total, payload, s->copyStream, uniPitch, uniLen);
    if (r != HS_SUCCESS) {
        return r;
    }
    ScanPlan pl;
    r = planScan(s, im, &pl);
    if (r != HS_SUCCESS) {
        return r;
    }
    const u64 chunk = (u64)std::max(1, g_opts.chunkMB) << 20;
    const size_t nchunks = (size_t)((total + chunk - 1) / chunk);
    while (s->chunkEvents->size() < nchunks + 1) {
        cudaEvent_t ev;
        CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        s->chunkEvents->push_back(ev);
    }
    /* a second pass after the record ring grew; split mode may need a third (its
     * candidate list can overflow before the ring does) */
    for (int attempt = 0; attempt < 3; attempt++) {
        CUDA_TRY(cudaMemsetAsync(s->d_counters, 0, CTR_COUNT * sizeof(u32), s->stream));
        CUDA_TRY(cudaEventRecord(s->evStart, s->stream));
        /* zero the look-ahead bytes after the corpus */
        CUDA_TRY(cudaMemsetAsync(c->d_data + total, 0, HSB_ROUNDUP(total, 16) + 32 - total,
                                 s->copyStream));
        u32 tDone = 0;
        size_t blk = 0;
        for (size_t ci = 0; ci < nchunks; ci++) {
            const u64 from = ci * chunk, to = std::min<u64>(total, from + chunk);
            if (attempt == 0) {
                if (direct) {
                    CUDA_TRY(cudaMemcpyAsync(c->d_data + from, data + offsets[0] + from, to - from,
                                             cudaMemcpyHostToDevice, s->copyStream));
                } else {
                    /* unaligned host layout: pack this chunk's blocks (16-byte
                     * aligned starts, zero gaps) into a pinned staging buffer and
                     * send it as one copy; blocks that straddle the chunk edge go
                     * whole with the chunk they start in.  Two buffers alternate. */
                    const size_t b0 = blk;
                    u64 end = from;
                    while (blk < nblocks && packed[blk] < to) {
                        end = std::max<u64>(end, packed[blk] + lengths[blk]);
                        blk++;
                    }
                    if (blk > b0) {
                        const u64 start = packed[b0];
                        const size_t need = (size_t)(end - start);
                        u8 *&stage = (ci & 1) ? s->h_stage2 : s->h_stage;
                        size_t &cap = (ci & 1) ? s->h_stage2Cap : s->h_stageCap;
                        cudaEvent_t ev = (ci & 1) ? s->evStage2 : s->evStage;
                        CUDA_TRY(cudaEventSynchronize(ev)); /* previous use of this buffer has been sent */
                        if (need > cap) {
                            if (stage) cudaFreeHost(stage);
                            stage = nullptr;
                            cap = 0;
                            CUDA_TRY(cudaMallocHost(&stage, need + need / 4 + 4096));
                            cap = need + need / 4 + 4096;
                        }
                        memset(stage, 0, need);
                        for (size_t k = b0; k < blk; k++) {
                            memcpy(stage + (packed[k] - start), data + offsets[k], lengths[k]);
                        }
                        CUDA_TRY(cudaMemcpyAsync(c->d_data + start, stage, need, cudaMemcpyHostToDevice,
                                                 s->copyStream));
                        CUDA_TRY(cudaEventRecord(ev, s->copyStream));
                    }
                }
                CUDA_TRY(cudaEventRecord((*s->chunkEvents)[ci], s->copyStream));
                CUDA_TRY(cudaStreamWaitEvent(s->stream, (*s->chunkEvents)[ci], 0));
            }
            /* tiles wholly inside the copied prefix (plus look-ahead) */
            u32 tEnd;
            if (ci + 1 == nchunks) {
                tEnd = (u32)((total + pl.tileBytes - 1) / pl.tileBytes);
            } else {
                u64 covered = direct ? to : (blk < nblocks ? packed[blk] : total);
                covered = std::min(covered, to);
                tEnd = covered > 16 ? (u32)((covered - 16) / pl.tileBytes) : 0;
            }
            r = launchRange(s, im, c, pl, tDone, tEnd, s->stream);
            if (r != HS_SUCCESS) {
                return r;
            }
            tDone = std::max(tDone, tEnd);
        }
        CUDA_TRY(cudaEventRecord(s->evStop, s->stream));
        CUDA_TRY(cudaMemcpyAsync(s->h_counters, s->d_counters, CTR_COUNT * sizeof(u32),
                                 cudaMemcpyDeviceToHost, s->stream));
        CUDA_TRY(cudaEventRecord(s->evDone, s->stream));
        s->lastImage = im;
        s->lastCorpus = c;
        s->activeStream = s->stream;
        s->pending = true;
        u32 count = 0;
        tEnq = nowMs();
        r = finishScan(s, &count);
        tWait = nowMs();
        if (r != HS_SUCCESS) {
            return r;
        }
        if (count <= s->outCap) {
            matches->resize(count);
            if (count) {
                CUDA_TRY(cudaMemcpyAsync(matches->data(), s->d_out, (size_t)count * sizeof(DevMatch),
                                         cudaMemcpyDeviceToHost, s->stream));
                CUDA_TRY(cudaStreamSynchronize(s->stream));
            }
            tRec = nowMs();
            /* nobody will look at the order, and neither dedupe keys nor
             * exhaustion keys exist: the raw count IS the delivered count */
            const bool plain = countOnly && im->exhaustible.empty() && !im->hasDedupe && im->kind != FK_OUTFIX;
            if (!plain) {
                r = postprocessVec(im, matches);
                if (r != HS_SUCCESS) {
                    return r;
                }
            }
            if (trace) {
                fprintf(stderr, "[hs_b200 trace] host scan: layout %.3f ms, enqueue %.3f, wait %.3f, records %.3f, "
                                "postprocess %.3f (total %.3f, %zu chunks)\n",
                        tLayout - t0, tEnq - tLayout, tWait - tEnq, tRec - tWait, nowMs() - tRec,
                        nowMs() - t0, nchunks);
            }
            return HS_SUCCESS;
        }
        /* record ring overflowed: grow it and scan the resident corpus again */
        u64 want = (u64)count + count / 4 + 1024;
        if (want > 0xfffffff0ull) {
            return HS_NOMEM;
        }
        r = growRing(s, (u32)want);
        if (r != HS_SUCCESS) {
            return r;
        }
    }
    return HS_UNKNOWN_ERROR;
}

hs_error_t hs_b200_scan_blocks(const hs_database_t *db, const char *data,
                               const unsigned long long *offsets, const unsigned int *lengths,
                               size_t nblocks, hs_scratch_t *scratch,
                               hs_b200_block_event_handler onEvent, void *context,
                               unsigned long long *nmatches) {
    if (!scratch || (nblocks && (!data || !offsets || !lengths)) || nblocks > 0xfffffff0u) {
        return HS_INVALID;
    }
    hs_error_t r = checkScanArgs(db, scratch);
    if (r != HS_SUCCESS) {
        return r;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    const DevImage *im = nullptr;
    r = findImage(scratch, db, &im);
    std::vector<DevMatch> matches;
    if (r == HS_SUCCESS) {
        r = scanHostBlocks(im, scratch, data, offsets, lengths, nblocks, &matches, onEvent == nullptr);
    }
    unsigned long long delivered = 0;
    if (r == HS_SUCCESS) {
        if (!onEvent) {
            delivered = matches.size();
        } else {
            u32 stopped = 0xffffffffu;
            for (const DevMatch &m : matches) {
                if (m.block == stopped) {
                    continue;
                }
                delivered++;
                if (onEvent(m.block, m.id, 0, m.to, 0, context)) {
                    stopped = m.block;
                }
            }
        }
    }
    if (nmatches) {
        *nmatches = delivered;
    }
    unmarkInUse(scratch);
    return r;
}

hs_error_t hs_b200_scan_blocks_collect(const hs_database_t *db, const char *data,
                                       const unsigned long long *offsets, const unsigned int *lengths,
                                       size_t nblocks, hs_scratch_t *scratch, hs_b200_match_t *out,
                                       size_t cap, unsigned long long *nmatches) {
    if (!scratch || (nblocks && (!data || !offsets || !lengths)) || nblocks > 0xfffffff0u || (cap && !out)) {
        return HS_INVALID;
    }
    hs_error_t r = checkScanArgs(db, scratch);
    if (r != HS_SUCCESS) {
        return r;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    const DevImage *im = nullptr;
    r = findImage(scratch, db, &im);
    std::vector<DevMatch> matches;
    if (r == HS_SUCCESS) {
        r = scanHostBlocks(im, scratch, data, offsets, lengths, nblocks, &matches, false);
    }
    if (r == HS_SUCCESS) {
        if (nmatches) {
            *nmatches = matches.size();
        }
        static_assert(sizeof(DevMatch) == sizeof(hs_b200_match_t), "record layout");
        memcpy(out, matches.data(), std::min(cap, matches.size()) * sizeof(DevMatch));
        if (matches.size() > cap) {
            r = HS_INSUFFICIENT_SPACE;
        }
    }
    unmarkInUse(scratch);
    return r;
}

hs_error_t hs_scan(const hs_database_t *db, const char *data, unsigned int length,
                   unsigned int flags, hs_scratch_t *scratch, match_event_handler onEvent,
                   void *context) {
    (void)flags;
    if (!scratch || !data) {
        return HS_INVALID;
    }
    hs_error_t r = checkScanArgs(db, scratch);
    if (r != HS_SUCCESS) {
        return r;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    const RoseEngine *rose = dbRose(db);
    if (rose->minWidth > length) { /* src/runtime.c:346-350 */
        unmarkInUse(scratch);
        return HS_SUCCESS;
    }
    const DevImage *im = nullptr;
    r = findImage(scratch, db, &im);
    std::vector<DevMatch> matches;
    if (r == HS_SUCCESS) {
        const unsigned long long off = 0;
        r = scanHostBlocks(im, scratch, data, &off, &length, 1, &matches);
    }
    if (r == HS_SUCCESS && onEvent) {
        for (const DevMatch &m : matches) {
            if (onEvent(m.id, 0, m.to, 0, context)) {
                r = HS_SCAN_TERMINATED; /* src/report.h:324-328 */
                break;
            }
        }
    }
    unmarkInUse(scratch);
    return r;
}

/* ---- streaming mode (src/runtime.c:542-977, pure-literal databases) ------------------
 *
 * A stream carries the last historyRequired (<= 7) bytes it has seen, its
 * offset, a broken/exhausted status and the single-match reports already
 * raised.  hs_scan_stream scans (history ++ write) as one block on the device
 * and delivers the matches that END inside the write, at stream offsets --
 * the restatement of pureLiteralStreamExec / hwlmExecStreaming
 * (src/runtime.c:801-829, src/hwlm/hwlm.c:201-239) with the look-behind made
 * explicit. */

struct hs_stream {
    u32 magic;
    const hs_database_t *db;
    u64 offset;
    u32 hreq, hlen;
    u8 hist[16];
    u8 status; /* 1 = terminated by the callback, 2 = all reports exhausted */
    std::unordered_set<u32> *seen;
};

static const u32 STREAM_MAGIC = 0x4d525453; /* "STRM" */

static bool validStream(const hs_stream *st) { return st && st->magic == STREAM_MAGIC && st->seen; }

static void resetStreamState(hs_stream *st) {
    st->offset = 0;
    st->hlen = 0;
    st->status = 0;
    st->seen->clear();
}

hs_error_t hs_open_stream(const hs_database_t *db, unsigned int flags, hs_stream_t **stream) {
    (void)flags;
    if (!stream) {
        return HS_INVALID;
    }
    *stream = nullptr;
    hs_error_t err = validDb(db);
    if (err != HS_SUCCESS) {
        return err;
    }
    const RoseEngine *rose = dbRose(db);
    if ((uintptr_t)rose % 16) {
        return HS_INVALID;
    }
    if (rose->mode != MODE_STREAM) {
        return HS_DB_MODE_ERROR;
    }
    if (rose->runtimeImpl != RUNTIME_PURE_LITERAL || rose->historyRequired > sizeof(((hs_stream *)0)->hist)) {
        return HS_ARCH_ERROR;
    }
    hs_stream *st = (hs_stream *)g_stream_alloc(sizeof(hs_stream));
    err = checkAlloc(st);
    if (err != HS_SUCCESS) {
        g_stream_free(st);
        return err;
    }
    memset(st, 0, sizeof(*st));
    st->magic = STREAM_MAGIC;
    st->db = db;
    st->hreq = rose->historyRequired;
    st->seen = new (std::nothrow) std::unordered_set<u32>();
    if (!st->seen) {
        g_stream_free(st);
        return HS_NOMEM;
    }
    *stream = st;
    return HS_SUCCESS;
}

/* One write of one stream (hs_scan_stream_internal, src/runtime.c:870-977):
 * scan look-behind ++ write as a block, deliver the matches that end inside the
 * write at stream offsets, roll the history forward.  The scratch is already
 * marked in use by the caller. */
static hs_error_t streamWrite(hs_stream *st, const char *data, unsigned int length, hs_scratch_t *scratch,
                              match_event_handler onEvent, void *context) {
    hs_error_t r = HS_SUCCESS;
    if (st->status & 1) {
        r = HS_SCAN_TERMINATED; /* the stream is broken: src/runtime.c:883-893 */
    } else if (!(st->status & 2) && length != 0) {
        const DevImage *im = nullptr;
        r = findImage(scratch, st->db, &im);
        std::vector<DevMatch> matches;
        std::vector<char> buf;
        if (r == HS_SUCCESS) {
            buf.resize((size_t)st->hlen + length);
            memcpy(buf.data(), st->hist, st->hlen);
            memcpy(buf.data() + st->hlen, data, length);
            const unsigned long long off = 0;
            const unsigned total = (unsigned)buf.size();
            r = scanHostBlocks(im, scratch, buf.data(), &off, &total, 1, &matches);
        }
        if (r == HS_SUCCESS) {
            const RoseEngine *rose = dbRose(st->db);
            for (const DevMatch &m : matches) {
                if (m.to <= st->hlen) {
                    continue; /* ended in the look-behind: raised by an earlier write */
                }
                if (im->exhaustible.count(m.id) && !st->seen->insert(m.id).second) {
                    continue; /* HS_FLAG_SINGLEMATCH: already raised on this stream */
                }
                if (onEvent && onEvent(m.id, 0, st->offset - st->hlen + m.to, 0, context)) {
                    st->status |= 1;
                    r = HS_SCAN_TERMINATED;
                    break;
                }
            }
            if (r == HS_SUCCESS) {
                if (rose->canExhaust && rose->ekeyCount && st->seen->size() >= im->exhaustible.size()) {
                    st->status |= 2;
                }
                /* maintainHistoryBuffer (src/runtime.c:478-508) */
                const size_t keep = std::min<size_t>(buf.size(), st->hreq);
                memcpy(st->hist, buf.data() + buf.size() - keep, keep);
                st->hlen = (u32)keep;
                st->offset += length;
            }
        }
    }
    return r;
}

hs_error_t hs_scan_stream(hs_stream_t *st, const char *data, unsigned int length, unsigned int flags,
                          hs_scratch_t *scratch, match_event_handler onEvent, void *context) {
    (void)flags;
    if (!validStream(st) || !scratch || !data || (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    const hs_error_t r = streamWrite(st, data, length, scratch, onEvent, context);
    unmarkInUse(scratch);
    return r;
}

/* src/runtime.c:1106-1175: a temporary stream, one write per buffer, closed at
 * the end (pure-literal databases have no end-of-data reports). */
hs_error_t hs_scan_vector(const hs_database_t *db, const char *const *data, const unsigned int *length,
                          unsigned int count, unsigned int flags, hs_scratch_t *scratch,
                          match_event_handler onEvent, void *context) {
    (void)flags;
    if (!scratch || !data || !length) {
        return HS_INVALID;
    }
    hs_error_t err = validDb(db);
    if (err != HS_SUCCESS) {
        return err;
    }
    const RoseEngine *rose = dbRose(db);
    if ((uintptr_t)rose % 16) {
        return HS_INVALID;
    }
    if (rose->mode != MODE_VECTORED) {
        return HS_DB_MODE_ERROR;
    }
    if ((uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    if (rose->runtimeImpl != RUNTIME_PURE_LITERAL || rose->historyRequired > sizeof(((hs_stream *)0)->hist)) {
        return HS_ARCH_ERROR;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    std::unordered_set<u32> seen;
    hs_stream st;
    memset(&st, 0, sizeof(st));
    st.magic = STREAM_MAGIC;
    st.db = db;
    st.hreq = rose->historyRequired;
    st.seen = &seen;
    hs_error_t r = HS_SUCCESS;
    for (unsigned int i = 0; i < count && r == HS_SUCCESS; i++) {
        if (!data[i]) {
            r = HS_INVALID; /* hs_scan_stream_internal: src/runtime.c:875 */
            break;
        }
        r = streamWrite(&st, data[i], length[i], scratch, onEvent, context);
    }
    unmarkInUse(scratch);
    return r;
}

hs_error_t hs_close_stream(hs_stream_t *st, hs_scratch_t *scratch, match_event_handler onEvent,
                           void *context) {
    (void)scratch; /* pure-literal databases have no end-of-data work (src/runtime.c:1005-1050) */
    (void)onEvent;
    (void)context;
    if (!validStream(st)) {
        return HS_INVALID;
    }
    st->magic = 0;
    delete st->seen;
    g_stream_free(st);
    return HS_SUCCESS;
}

hs_error_t hs_reset_stream(hs_stream_t *st, unsigned int flags, hs_scratch_t *scratch,
                           match_event_handler onEvent, void *context) {
    (void)flags;
    (void)scratch;
    (void)onEvent;
    (void)context;
    if (!validStream(st)) {
        return HS_INVALID;
    }
    resetStreamState(st);
    return HS_SUCCESS;
}

hs_error_t hs_copy_stream(hs_stream_t **to_id, const hs_stream_t *from_id) {
    if (!to_id) {
        return HS_INVALID;
    }
    *to_id = nullptr;
    if (!validStream(from_id)) {
        return HS_INVALID;
    }
    hs_stream *st = (hs_stream *)g_stream_alloc(sizeof(hs_stream));
    hs_error_t err = checkAlloc(st);
    if (err != HS_SUCCESS) {
        g_stream_free(st);
        return err;
    }
    memcpy(st, from_id, sizeof(*st));
    st->seen = new (std::nothrow) std::unordered_set<u32>(*from_id->seen);
    if (!st->seen) {
        g_stream_free(st);
        return HS_NOMEM;
    }
    *to_id = st;
    return HS_SUCCESS;
}

hs_error_t hs_reset_and_copy_stream(hs_stream_t *to_id, const hs_stream_t *from_id,
                                    hs_scratch_t *scratch, match_event_handler onEvent,
                                    void *context) {
    (void)scratch;
    (void)onEvent;
    (void)context;
    if (!validStream(to_id) || !validStream(from_id) || to_id == from_id) {
        return HS_INVALID;
    }
    if (to_id->db != from_id->db) {
        return HS_INVALID; /* src/runtime.c:758-760: streams of different databases */
    }
    std::unordered_set<u32> *keep = to_id->seen;
    *keep = *from_id->seen;
    memcpy(to_id, from_id, sizeof(*to_id));
    to_id->seen = keep;
    return HS_SUCCESS;
}

/* ---- stream compression (src/runtime.c:1177-1282, src/stream_compress_impl.h) ------
 * Flat form of a hs_stream: header {magic, database crc, status, look-behind
 * length, number of single-match ids already raised, stream offset}, the
 * look-behind bytes, the ids. */

namespace {
const u32 COMPRESS_MAGIC = 0x504d4353; /* "SCMP" */
struct CompressedHeader {
    u32 magic, crc, status, hlen, nseen, reserved;
    u64 offset;
};

size_t compressedSize(const hs_stream *st) {
    return sizeof(CompressedHeader) + st->hlen + 4 * st->seen->size();
}

/* fills *st (whose db, hreq and seen set are already in place) from buf */
bool expandInto(hs_stream *st, const char *buf, size_t size) {
    CompressedHeader h;
    if (size < sizeof(h)) {
        return false;
    }
    memcpy(&h, buf, sizeof(h));
    const DbHeader *dh = (const DbHeader *)st->db;
    if (h.magic != COMPRESS_MAGIC || h.crc != dh->crc32 || h.hlen > st->hreq || h.hlen > sizeof(st->hist) ||
        h.status > 3 || size != sizeof(h) + h.hlen + 4ull * h.nseen) {
        return false;
    }
    st->offset = h.offset;
    st->hlen = h.hlen;
    st->status = (u8)h.status;
    memcpy(st->hist, buf + sizeof(h), h.hlen);
    st->seen->clear();
    for (u32 i = 0; i < h.nseen; i++) {
        u32 id;
        memcpy(&id, buf + sizeof(h) + h.hlen + 4ull * i, 4);
        st->seen->insert(id);
    }
    return true;
}
} // namespace

hs_error_t hs_compress_stream(const hs_stream_t *st, char *buf, size_t buf_space, size_t *used_space) {
    if (!validStream(st) || !used_space || (buf_space && !buf)) {
        return HS_INVALID;
    }
    const size_t need = compressedSize(st);
    *used_space = need;
    if (buf_space < need) {
        return HS_INSUFFICIENT_SPACE;
    }
    CompressedHeader h;
    memset(&h, 0, sizeof(h));
    h.magic = COMPRESS_MAGIC;
    h.crc = ((const DbHeader *)st->db)->crc32;
    h.status = st->status;
    h.hlen = st->hlen;
    h.nseen = (u32)st->seen->size();
    h.offset = st->offset;
    memcpy(buf, &h, sizeof(h));
    memcpy(buf + sizeof(h), st->hist, st->hlen);
    size_t pos = sizeof(h) + st->hlen;
    std::vector<u32> ids(st->seen->begin(), st->seen->end());
    std::sort(ids.begin(), ids.end()); /* equal states compress to equal bytes */
    for (u32 id : ids) {
        memcpy(buf + pos, &id, 4);
        pos += 4;
    }
    return HS_SUCCESS;
}

hs_error_t hs_expand_stream(const hs_database_t *db, hs_stream_t **stream, const char *buf, size_t buf_size) {
    if (!stream || !buf) {
        return HS_INVALID;
    }
    *stream = nullptr;
    hs_stream_t *st = nullptr;
    hs_error_t err = hs_open_stream(db, 0, &st); /* same checks: validity, alignment, mode, engine */
    if (err != HS_SUCCESS) {
        return err;
    }
    if (!expandInto(st, buf, buf_size)) {
        hs_close_stream(st, nullptr, nullptr, nullptr);
        return HS_INVALID;
    }
    *stream = st;
    return HS_SUCCESS;
}

hs_error_t hs_reset_and_expand_stream(hs_stream_t *to_stream, const char *buf, size_t buf_size,
                                      hs_scratch_t *scratch, match_event_handler onEvent, void *context) {
    (void)context;
    if (!validStream(to_stream) || !buf) {
        return HS_INVALID;
    }
    if (onEvent && (!scratch || (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC)) {
        return HS_INVALID; /* pure-literal databases have no end-of-data reports to deliver */
    }
    /* expand into a copy first: a bad buffer must leave the stream as it was */
    hs_stream tmp = *to_stream;
    std::unordered_set<u32> seen;
    tmp.seen = &seen;
    if (!expandInto(&tmp, buf, buf_size)) {
        return HS_INVALID;
    }
    std::unordered_set<u32> *keep = to_stream->seen;
    *keep = seen;
    *to_stream = tmp;
    to_stream->seen = keep;
    return HS_SUCCESS;
}

/* ---- stream sets: many streams, one write each per call, state resident in HBM ------
 * (BASELINE config 4 shape: 16 M x 1 KB streams).  Per stream 16 bytes live in
 * HBM: 7 look-behind bytes + their count, and the 64-bit stream offset.  A scan
 * copies the writes into a pitched corpus (16-byte header per stream), a
 * kernel drops each stream's look-behind into its header, the block kernel
 * scans the lot (blocks = look-behind ++ write, found by division), records
 * come out at stream offsets, and a kernel rolls history and offsets forward. */

struct hs_b200_stream_set {
    const hs_database_t *db;
    int device;
    size_t nstreams;
    u32 histReq;
    u8 *d_hist;     /* 8 bytes per stream */
    u64 *d_offset;
    u32 *d_len;     /* per-write lengths when they differ */
    hs_b200_corpus corpus; /* pitched staging, reused */
    u32 pitchCap;
};

hs_error_t hs_b200_streams_open(const hs_database_t *db, size_t nstreams, int device,
                                hs_b200_stream_set_t **set) {
    if (!set || nstreams == 0 || nstreams > 0xfffffff0u) {
        return HS_INVALID;
    }
    *set = nullptr;
    hs_error_t err = validDb(db);
    if (err != HS_SUCCESS) {
        return err;
    }
    const RoseEngine *rose = dbRose(db);
    if (rose->mode != MODE_STREAM) {
        return HS_DB_MODE_ERROR;
    }
    if (rose->runtimeImpl != RUNTIME_PURE_LITERAL || rose->historyRequired > 7 || rose->ekeyCount) {
        /* HS_FLAG_SINGLEMATCH state per stream is kept only by hs_scan_stream */
        return HS_ARCH_ERROR;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        return HS_ARCH_ERROR;
    }
    hs_b200_stream_set *s = new (std::nothrow) hs_b200_stream_set();
    if (!s) {
        return HS_NOMEM;
    }
    s->db = db;
    s->device = device;
    s->nstreams = nstreams;
    s->histReq = rose->historyRequired;
    s->d_hist = nullptr;
    s->d_offset = nullptr;
    s->d_len = nullptr;
    s->pitchCap = 0;
    cudaError_t e = cudaMalloc(&s->d_hist, nstreams * 8);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_offset, nstreams * 8);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_len, nstreams * 4);
    if (e == cudaSuccess) e = cudaMemset(s->d_hist, 0, nstreams * 8);
    if (e == cudaSuccess) e = cudaMemset(s->d_offset, 0, nstreams * 8);
    if (e != cudaSuccess) {
        hs_b200_streams_close(s);
        return e == cudaErrorMemoryAllocation ? HS_NOMEM : HS_UNKNOWN_ERROR;
    }
    *set = s;
    return HS_SUCCESS;
}

hs_error_t hs_b200_streams_close(hs_b200_stream_set_t *s) {
    if (!s) {
        return HS_SUCCESS;
    }
    DeviceGuard guard(s->device);
    cudaFree(s->d_hist);
    cudaFree(s->d_offset);
    cudaFree(s->d_len);
    cudaFree(s->corpus.d_alloc);
    delete s;
    return HS_SUCCESS;
}

size_t hs_b200_streams_state_bytes(const hs_b200_stream_set_t *s) { return s ? s->nstreams * 16 : 0; }

static hs_error_t streamsScanImpl(hs_b200_stream_set_t *set, const char *data,
                                  const unsigned long long *offsets, const unsigned int *lengths,
                                  hs_scratch_t *scratch, std::vector<DevMatch> &matches) {
    hs_scratch *s = scratch;
    const size_t n = set->nstreams;
    hs_error_t r = HS_SUCCESS;
    if (s->device != set->device) {
        return HS_INVALID; /* the set's state and the scratch's ring must share a device */
    }
    DeviceGuard guard(set->device);
    do {
        const DevImage *im = nullptr;
        r = findImage(s, set->db, &im);
        if (r != HS_SUCCESS) break;
        /* write lengths: uniform (config 4) or per stream */
        u32 maxLen = 0, uni = lengths[0];
        bool contiguous = true;
        for (size_t i = 0; i < n; i++) {
            maxLen = std::max(maxLen, lengths[i]);
            if (lengths[i] != uni) uni = 0;
            if (offsets[i] != offsets[0] + (u64)i * lengths[0]) contiguous = false;
        }
        if (maxLen == 0) break;
        const u32 pitch = 16 + (u32)HSB_ROUNDUP((u64)maxLen, 16);
        hs_b200_corpus *c = &set->corpus;
        const u64 total = (u64)n * pitch;
        c->device = set->device;
        r = reserveCorpus(c, total, 0);
        if (r != HS_SUCCESS) break;
        cudaStream_t st = s->stream;
        cudaError_t e;
        if (uni && contiguous) {
            e = cudaMemcpy2DAsync(c->d_data + 16, pitch, data + offsets[0], uni, uni, n,
                                  cudaMemcpyHostToDevice, st);
        } else {
            /* ragged writes: pack on the host, one copy */
            std::vector<u8> pack((size_t)total, 0);
            for (size_t i = 0; i < n; i++) {
                memcpy(pack.data() + i * pitch + 16, data + offsets[i], lengths[i]);
            }
            e = cudaMemcpyAsync(c->d_data, pack.data(), total, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st); /* `pack` dies at scope end */
            if (e == cudaSuccess && !uni) {
                e = cudaMemcpyAsync(set->d_len, lengths, n * 4, cudaMemcpyHostToDevice, st);
                if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            }
        }
        if (e == cudaSuccess) {
            e = cudaMemsetAsync(c->d_data + total, 0, 48, st);
        }
        if (e == cudaSuccess) e = launchStreamAssemble(c->d_data, set->d_hist, (u32)n, pitch, st);
        if (e != cudaSuccess) { r = HS_UNKNOWN_ERROR; break; }
        g_launches++;
        c->nblocks = n;
        c->bytes = total;
        c->readableEnd = HSB_ROUNDUP(total, 16) + 16;
        c->payload = 0;
        c->uniformPitch = 0;
        c->uniformLen = uni;
        c->d_len = set->d_len;
        ScanPlan pl;
        r = planScan(s, im, &pl);
        if (r != HS_SUCCESS) break;
        for (int attempt = 0; attempt < 2 && r == HS_SUCCESS; attempt++) {
            ScanParams p;
            fillParams(s, im, c, pl, &p);
            p.streamPitch = pitch;
            p.streamHist = set->d_hist;
            p.streamOffset = set->d_offset;
            p.tileFirst = 0;
            p.ntiles = (u32)((total + pl.tileBytes - 1) / pl.tileBytes);
            LaunchCfg cfg = pl.cfg;
            cfg.grid = (int)std::min<u32>((u32)cfg.grid, (p.ntiles + (u32)cfg.warps - 1) / (u32)cfg.warps);
            e = cudaMemsetAsync(s->d_counters, 0, CTR_COUNT * sizeof(u32), st);
            if (e == cudaSuccess) e = cudaEventRecord(s->evStart, st);
            if (e == cudaSuccess) e = launchScan(cfg, p, st);
            if (e == cudaSuccess && cfg.split) {
                e = launchConfirm(cfg, p, st); /* candidate list -> records (counters were just cleared) */
                g_launches++;
            }
            if (e == cudaSuccess) e = cudaEventRecord(s->evStop, st);
            if (e == cudaSuccess) {
                e = cudaMemcpyAsync(s->h_counters, s->d_counters, CTR_COUNT * sizeof(u32),
                                    cudaMemcpyDeviceToHost, st);
            }
            if (e == cudaSuccess) e = cudaEventRecord(s->evDone, st);
            if (e != cudaSuccess) { r = HS_UNKNOWN_ERROR; break; }
            g_launches++;
            s->activeStream = st;
            s->pending = true;
            u32 count = 0;
            r = finishScan(s, &count);
            if (r != HS_SUCCESS) break;
            if (count <= s->outCap) {
                matches.resize(count);
                if (count) {
                    e = cudaMemcpyAsync(matches.data(), s->d_out, (size_t)count * sizeof(DevMatch),
                                        cudaMemcpyDeviceToHost, st);
                    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
                    if (e != cudaSuccess) { r = HS_UNKNOWN_ERROR; break; }
                }
                matches.resize(postprocess(im, matches.data(), count));
                break;
            }
            u64 want = (u64)count + count / 4 + 1024;
            r = want > 0xfffffff0ull ? HS_NOMEM : growRing(s, (u32)want);
        }
        c->d_len = nullptr; /* borrowed */
        if (r != HS_SUCCESS) break;
        e = launchStreamAdvance(c->d_data, set->d_hist, set->d_offset, set->d_len, uni, (u32)n, pitch,
                                set->histReq, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { r = HS_UNKNOWN_ERROR; break; }
        g_launches++;
    } while (0);
    set->corpus.d_len = nullptr;
    return r;
}

hs_error_t hs_b200_streams_scan(hs_b200_stream_set_t *set, const char *data,
                                const unsigned long long *offsets, const unsigned int *lengths,
                                hs_scratch_t *scratch, hs_b200_block_event_handler onEvent,
                                void *context, unsigned long long *nmatches) {
    if (!set || !scratch || !data || !offsets || !lengths || (uintptr_t)scratch % 64 ||
        scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    std::vector<DevMatch> matches;
    hs_error_t r = streamsScanImpl(set, data, offsets, lengths, scratch, matches);
    unsigned long long delivered = 0;
    if (r == HS_SUCCESS) {
        delivered = matches.size();
        if (onEvent) {
            for (const DevMatch &m : matches) {
                onEvent(m.block, m.id, 0, m.to, 0, context);
            }
        }
    }
    if (nmatches) {
        *nmatches = delivered;
    }
    unmarkInUse(scratch);
    return r;
}

hs_error_t hs_b200_streams_scan_collect(hs_b200_stream_set_t *set, const char *data,
                                        const unsigned long long *offsets,
                                        const unsigned int *lengths, hs_scratch_t *scratch,
                                        hs_b200_match_t *out, size_t cap,
                                        unsigned long long *nmatches) {
    if (!set || !scratch || !data || !offsets || !lengths || !nmatches || (cap && !out) ||
        (uintptr_t)scratch % 64 || scratch->magic != SCRATCH_MAGIC) {
        return HS_INVALID;
    }
    if (markInUse(scratch)) {
        return HS_SCRATCH_IN_USE;
    }
    std::vector<DevMatch> matches;
    hs_error_t r = streamsScanImpl(set, data, offsets, lengths, scratch, matches);
    if (r == HS_SUCCESS) {
        *nmatches = matches.size();
        memcpy(out, matches.data(), std::min(cap, matches.size()) * sizeof(DevMatch));
        if (matches.size() > cap) {
            r = HS_INSUFFICIENT_SPACE; /* the stream state HAS advanced; the first cap records are valid */
        }
    }
    unmarkInUse(scratch);
    return r;
}

} /* extern "C" */
