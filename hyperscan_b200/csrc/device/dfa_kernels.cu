/*
 * dfa_kernels.cu -- the reference's DFA engines in block mode on sm_100a:
 * McClellan with 8- and 16-bit states (incl. Sherman states) and Sheng, run
 * over every block of a corpus, straight from the engines' own bytes.
 *
 * Replaces nfaExecMcClellan8_B / nfaExecMcClellan16_B (src/nfa/mcclellan.c:
 * 937-973; inner loops doNormal8 / doNormal16 :122-167,370-444, reports
 * doComplexReport :43-91, Sherman states mcclellan_common_impl.h:61-93) and
 * nfaExecSheng_B (src/nfa/sheng.c:706-739; loop sheng_impl.h:38-100, reports
 * fireReports :116-155) -- the entry points hs_scan uses for the anchored literal
 * table (src/rose/block.c:42-91) and the small-write engine
 * (src/runtime.c:285-315).
 *
 * A DFA run is one dependent table lookup per byte, so the parallelism is across
 * blocks: one thread per block (the configurations scan 10^6..10^7 blocks of
 * ~1 KiB), the 32 blocks of a warp staged through a shared-memory tile (see "staged
 * walk" below).  The transition table sits in shared memory when it fits beside the
 * tiles (McClellan: remap + successor table; Sheng: the 4 KiB of shuffle masks as a
 * byte table), else it is read through L1/L2.  Acceleration schemes
 * (ACCEL_FLAG states, src/nfa/accel.h) are skip-ahead optimisations only and are
 * ignored; wide states (has_wide) are not handled -- the C ABI refuses them.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <type_traits>

#include "kernels.h"

namespace hsb {

namespace {

__device__ __forceinline__ u32 g32(const u8 *p) { return __ldg(reinterpret_cast<const u32 *>(p)); }
__device__ __forceinline__ u16 g16(const u8 *p) { return __ldg(reinterpret_cast<const u16 *>(p)); }

/* Records leave through slots a LANE reserves eight at a time (`cursor` = its next slot;
 * a multiple of 8 = nothing reserved): one atomic on the shared counter per eight records
 * instead of one -- and one dependent L2 round trip -- per record.  Slots a lane reserved
 * but did not fill are written as DFA_NO_RECORD and dropped by the caller; CTR_MATCHES
 * counts reserved slots. */
enum : u32 { DFA_SLOTS = 8, DFA_NO_RECORD = 0xffffffffu };

__device__ __forceinline__ u32 emitDfaMatch(const DfaParams &p, u32 cursor, u32 id, u32 block, u64 to) {
    if ((cursor & (DFA_SLOTS - 1)) == 0) {
        cursor = atomicAdd(p.counters + CTR_MATCHES, (u32)DFA_SLOTS);
    }
    if (cursor < p.outCap) {
        DevMatch m;
        m.id = id;
        m.block = block;
        m.to = to;
        *reinterpret_cast<uint4 *>(p.out + cursor) = *reinterpret_cast<const uint4 *>(&m);
    }
    return cursor + 1;
}

/* struct report_list {u32 count; ReportID report[]} at NFA offset `off` */
__device__ u32 emitReportList(const DfaParams &p, const u8 *nfa, u32 cursor, u32 off, u32 block, u64 to) {
    const u32 n = g32(nfa + off);
    for (u32 i = 0; i < n; i++) {
        cursor = emitDfaMatch(p, cursor, g32(nfa + off + 4 + 4 * i), block, to);
    }
    return cursor;
}

__device__ __forceinline__ u32 ldgState(const u8 *p, u32) { return g32(p); }
__device__ __forceinline__ u64 ldgState(const u8 *p, u64) { return __ldg(reinterpret_cast<const u64 *>(p)); }
__device__ __forceinline__ u32 lowestBit(u32 v) { return (u32)__ffs((int)v) - 1; }
__device__ __forceinline__ u32 lowestBit(u64 v) { return (u32)__ffsll((long long)v) - 1; }
__device__ __forceinline__ u32 rankBelow(u32 mask, u32 bit) { return (u32)__popc(mask & ((1u << bit) - 1)); }
__device__ __forceinline__ u32 rankBelow(u64 mask, u32 bit) { return (u32)__popcll(mask & ((1ull << bit) - 1)); }

/* the LimEx state set: u32 / u64 for the 32- and 64-state models, W 64-bit words for the wider ones (the reference's
 * m128 / m256 / m512); StOps gives both kinds the same few operations */
template <int W> struct alignas(16) WideSt {
    u64 w[W];
};
template <class ST> struct StOps {
    static __device__ __forceinline__ ST zero() { return 0; }
    static __device__ __forceinline__ ST ones() { return ~(ST)0; }
    static __device__ __forceinline__ bool any(ST a) { return a != 0; }
    static __device__ __forceinline__ ST band(ST a, ST b) { return a & b; }
    static __device__ __forceinline__ ST bor(ST a, ST b) { return a | b; }
    static __device__ __forceinline__ bool test(ST a, u32 i) { return (a >> i) & 1; }
    static __device__ __forceinline__ ST clear0(ST a) { return a & ~(ST)1; }
    /* LSHIFT_STATE of the one bit i: the high bits fall off */
    static __device__ __forceinline__ ST shiftedBit(u32 i, u32 amount) { return ((ST)1 << i) << amount; }
    static __device__ __forceinline__ u32 low32(ST a) { return (u32)a; }
    static __device__ __forceinline__ ST fromU32(u32 x) { return x; }
    static __device__ __forceinline__ u32 rank(ST mask, u32 bit) { return rankBelow(mask, bit); }
    static __device__ __forceinline__ ST load(const u8 *p) { return ldgState(p, ST()); }
    template <class F> static __device__ __forceinline__ void forEach(ST on, F f) { /* ascending */
        while (on) {
            f(lowestBit(on));
            on &= on - 1;
        }
    }
};
template <int W> struct StOps<WideSt<W>> {
    typedef WideSt<W> ST;
    static __device__ __forceinline__ ST zero() {
        ST r;
#pragma unroll
        for (int j = 0; j < W; j++) r.w[j] = 0;
        return r;
    }
    static __device__ __forceinline__ ST ones() {
        ST r;
#pragma unroll
        for (int j = 0; j < W; j++) r.w[j] = ~0ull;
        return r;
    }
    static __device__ __forceinline__ bool any(const ST &a) {
        u64 x = 0;
#pragma unroll
        for (int j = 0; j < W; j++) x |= a.w[j];
        return x != 0;
    }
    static __device__ __forceinline__ ST band(const ST &a, const ST &b) {
        ST r;
#pragma unroll
        for (int j = 0; j < W; j++) r.w[j] = a.w[j] & b.w[j];
        return r;
    }
    static __device__ __forceinline__ ST bor(const ST &a, const ST &b) {
        ST r;
#pragma unroll
        for (int j = 0; j < W; j++) r.w[j] = a.w[j] | b.w[j];
        return r;
    }
    static __device__ __forceinline__ bool test(const ST &a, u32 i) {
        u64 x = 0;
#pragma unroll
        for (int j = 0; j < W; j++) x = (i >> 6) == (u32)j ? a.w[j] : x;
        return (x >> (i & 63)) & 1;
    }
    static __device__ __forceinline__ ST clear0(ST a) {
        a.w[0] &= ~1ull;
        return a;
    }
    /* the wide models shift every 64-bit lane on its own (lshift64_m128 ...): a bit never crosses into the next lane */
    static __device__ __forceinline__ ST shiftedBit(u32 i, u32 amount) {
        ST r = zero();
        const u64 v = (1ull << (i & 63)) << amount;
#pragma unroll
        for (int j = 0; j < W; j++) r.w[j] = (i >> 6) == (u32)j ? v : 0;
        return r;
    }
    static __device__ __forceinline__ u32 low32(const ST &a) { return (u32)a.w[0]; }
    static __device__ __forceinline__ ST fromU32(u32 x) {
        ST r = zero();
        r.w[0] = x;
        return r;
    }
    static __device__ __forceinline__ u32 rank(const ST &mask, u32 bit) {
        u32 c = 0;
#pragma unroll
        for (int j = 0; j < W; j++) {
            const u32 lo = 64u * j;
            if (bit >= lo + 64) {
                c += (u32)__popcll(mask.w[j]);
            } else if (bit > lo) {
                c += (u32)__popcll(mask.w[j] & ((1ull << (bit - lo)) - 1));
            }
        }
        return c;
    }
    static __device__ __forceinline__ ST load(const u8 *p) {
        ST r;
#pragma unroll
        for (int j = 0; j < W; j++) r.w[j] = __ldg(reinterpret_cast<const u64 *>(p) + j);
        return r;
    }
    template <class F> static __device__ __forceinline__ void forEach(const ST &on, F f) {
#pragma unroll
        for (int j = 0; j < W; j++) {
            u64 x = on.w[j];
            while (x) {
                f(64u * j + lowestBit(x));
                x &= x - 1;
            }
        }
    }
    /* the same with the word index as a compile-time constant: f(integral_constant<int, j>, bit) */
    template <int J, class F> struct EachWord {
        static __device__ __forceinline__ void run(const ST &on, F &f) {
            u64 x = on.w[J];
            while (x) {
                f(std::integral_constant<int, J>(), 64u * J + lowestBit(x));
                x &= x - 1;
            }
            EachWord<J + 1, F>::run(on, f);
        }
    };
    template <class F> struct EachWord<W, F> {
        static __device__ __forceinline__ void run(const ST &, F &) {}
    };
    template <class F> static __device__ __forceinline__ void forEachWord(const ST &on, F f) {
        EachWord<0, F>::run(on, f);
    }
    /* shared-memory tables of state sets are kept chunk-major -- the k-th 16 bytes of every entry side by side --
     * so that lanes reading DIFFERENT entries hit different banks (entry-major, a 64-byte set per entry would put
     * every entry on the same two bank groups) */
    static __device__ __forceinline__ ST loadChunks(const uint4 *tab, u32 entries, u32 index) {
        ST r;
#pragma unroll
        for (int k = 0; k < W / 2; k++) {
            const uint4 v = tab[k * entries + index];
            r.w[2 * k] = (u64)v.x | ((u64)v.y << 32);
            r.w[2 * k + 1] = (u64)v.z | ((u64)v.w << 32);
        }
        return r;
    }
    static __device__ __forceinline__ void storeChunks(uint4 *tab, u32 entries, u32 index, const ST &v) {
#pragma unroll
        for (int k = 0; k < W / 2; k++) {
            tab[k * entries + index] = make_uint4((u32)v.w[2 * k], (u32)(v.w[2 * k] >> 32), (u32)v.w[2 * k + 1],
                                                  (u32)(v.w[2 * k + 1] >> 32));
        }
    }
};

/* LimEx report list: ReportID[] terminated by MO_INVALID_IDX (limexRunReports, limex_runtime.h:90-103) */
__device__ HSB_NOINLINE u32 emitLimexReports(const DfaParams &p, const u8 *nfa, u32 cursor, u32 listOff, u32 block,
                                             u64 to) {
    const u8 *lx = nfa + sizeof(NFA);
    for (u32 i = 0;; i++) {
        const u32 id = g32(lx + listOff + 4 * i);
        if (id == MO_INVALID_IDX) {
            break;
        }
        cursor = emitDfaMatch(p, cursor, id, block, to);
    }
    return cursor;
}

/* accepts of the states in `found` through an NFAAccept table (PROCESS_ACCEPTS_IMPL_FN,
 * limex_common_impl.h:116-163; the squash of PROCESS_ACCEPTS_FN is dead code there) */
template <class ST>
__device__ HSB_NOINLINE u32 emitLimexAccepts(const DfaParams &p, const u8 *nfa, u32 cursor, ST found, ST mask,
                                             u32 tableOff, u32 block, u64 to) {
    const u8 *lx = nfa + sizeof(NFA);
    StOps<ST>::forEach(found, [&](const u32 bit) {
        const u32 idx = StOps<ST>::rank(mask, bit);
        const u8 *a = lx + tableOff + idx * (u32)sizeof(NFAAccept);
        const u32 reports = g32(a + offsetof(NFAAccept, reports));
        if (__ldg(a + offsetof(NFAAccept, single_report))) {
            cursor = emitDfaMatch(p, cursor, reports, block, to);
        } else {
            cursor = emitLimexReports(p, nfa, cursor, reports, block, to);
        }
    });
    return cursor;
}

__device__ void padReserved(const DfaParams &p, u32 cursor) {
    for (; cursor & (DFA_SLOTS - 1); cursor++) {
        if (cursor < p.outCap) {
            DevMatch m;
            m.id = DFA_NO_RECORD;
            m.block = 0;
            m.to = 0;
            *reinterpret_cast<uint4 *>(p.out + cursor) = *reinterpret_cast<const uint4 *>(&m);
        }
    }
}

struct BlockSpan {
    const u8 *base;
    u32 len;
};

/* 16 corpus bytes at q (16-byte aligned: blocks start aligned); bytes past the readable
 * end read as zero (they lie behind the block's end and are not consumed) */
__device__ HSB_NOINLINE uint4 load16Tail(const u8 *q, const u8 *end) { /* the corpus' last bytes: out of line */
    u32 w[4] = {0, 0, 0, 0};
#pragma unroll 1
    for (u32 i = 0; i < 16 && q + i < end; i++) {
        w[i >> 2] |= (u32)__ldg(q + i) << (8 * (i & 3));
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ uint4 load16(const DfaParams &p, const u8 *q) {
    if (q + 16 <= p.corpus + p.readableEnd) {
        return __ldg(reinterpret_cast<const uint4 *>(q));
    }
    return load16Tail(q, p.corpus + p.readableEnd);
}

__device__ __forceinline__ BlockSpan blockSpan(const DfaParams &p, u32 b) {
    BlockSpan s;
    if (p.uniformPitch && p.uniformLen) {
        s.base = p.corpus + (u64)b * p.uniformPitch;
        s.len = p.uniformLen;
    } else {
        s.base = p.corpus + __ldg(p.blockOff + b);
        s.len = __ldg(p.blockLen + b);
    }
    return s;
}

/* ---- McClellan ---------------------------------------------------------------- */

/* doSherman16 (mcclellan_common_impl.h:61-93): a 32-byte record {type, len, daddy,
 * chars[len], states u16[len]}; a symbol not listed falls through to daddy's row */
__device__ u32 shermanNext(const u8 *nfa, u32 shermanOffset, u32 shermanLimit, u32 s, u32 cprime,
                           const u16 *succ, u32 as) {
    const u8 *rec = nfa + shermanOffset + SHERMAN_FIXED_SIZE * (s - shermanLimit);
    const u32 len = __ldg(rec + SHERMAN_LEN_OFFSET);
    for (u32 i = 0; i < len; i++) {
        if (__ldg(rec + SHERMAN_CHARS_OFFSET + i) == cprime) {
            const u8 *q = rec + SHERMAN_CHARS_OFFSET + len + 2 * i; /* unaligned u16 */
            return (u32)__ldg(q) | ((u32)__ldg(q + 1) << 8);
        }
    }
    const u32 daddy = g16(rec + SHERMAN_DADDY_OFFSET);
    return __ldg(succ + (daddy << as) + cprime);
}

/* ---- staged walk ------------------------------------------------------------------
 *
 * One thread per block means 32 lanes reading 32 different blocks, and a dependent lookup
 * per byte.  Two things decide the speed: how a warp's corpus bytes arrive and how many
 * instructions a byte costs (the first version: 29 per byte, issue bound at 0.5-1.0 TB/s).
 *
 *  - A warp stages its 32 blocks through shared memory: CH bytes of every block per
 *    refill, loaded coalesced (8 lanes x 16 B = 128 contiguous bytes of one block, four
 *    blocks per load instruction) into a tile whose rows are CH + 16 bytes apart -- lane t
 *    then reads ITS row 16 bytes at a time and the eight lanes of a 128-bit shared-memory
 *    wavefront fall into eight disjoint bank groups (row stride 36 words = 4 banks).  No
 *    block-wide barrier in the loop: a tile belongs to one warp.
 *  - The tables are re-laid for the GPU when the CTA starts, from the engine's own bytes:
 *      McClellan-8: tab[s][byte] = succ[(s << alphaShift) + remap[byte]] (<= 64 KiB): the
 *        index is ONE byte permute of the data word and the state, one lookup per byte;
 *      Sheng: 8 copies of the 16 successor bytes of every input byte c (row = c, 128 B;
 *        lane l uses copy l & 7 = banks 4r .. 4r+3), the successor of state s at position
 *        (s + 4c) & 15 of its copy: the four lanes of a copy, which mostly sit in the same
 *        few states, collide only when their bytes agree modulo 4 -- unrotated they met in
 *        one bank (4.75 wavefronts per lookup measured, the shared-memory pipe 92 % busy;
 *        rotating whole rows instead threw all 32 lanes onto 8 banks: slower still);
 *      McClellan-16: remap in shared memory, the successor table where it is (L1/L2), or
 *        in shared memory when it fits beside the tiles.
 *    Full 16-byte pieces run without per-byte bounds or liveness checks (a dead state
 *    stays dead: checked per piece); accepts leave the loop through an out-of-line call. */
template <int CH> struct DfaTile {
    static constexpr u32 ROW = CH + 16;
    static constexpr u32 WARP_BYTES = 32 * ROW;
    static constexpr u32 PIECES = CH / 16;          /* 16-byte pieces per row */
    static constexpr u32 ROWS_PER_LOAD = 32 / PIECES;
};

enum { ENG_MCC8 = 0, ENG_MCC16 = 1, ENG_SHENG = 2, ENG_LIMEX32 = 3, ENG_LIMEX64 = 4, ENG_LIMEX128 = 5, ENG_LIMEX256 = 6,
       ENG_LIMEX512 = 7 };

/* the state of a block's walk: a DFA state id, or the LimEx state set */
template <int ENGINE> struct WalkState { typedef u32 type; };
template <> struct WalkState<ENG_LIMEX64> { typedef u64 type; };
template <> struct WalkState<ENG_LIMEX128> { typedef WideSt<2> type; };
template <> struct WalkState<ENG_LIMEX256> { typedef WideSt<4> type; };
template <> struct WalkState<ENG_LIMEX512> { typedef WideSt<8> type; };
/* the engine structures of the LimEx models share their field names */
template <class ST> struct LimexLayout;
template <> struct LimexLayout<u32> { typedef LimExNFA32 Nfa; typedef NFAException32 Exc; };
template <> struct LimexLayout<u64> { typedef LimExNFA64 Nfa; typedef NFAException64 Exc; };
template <> struct LimexLayout<WideSt<2>> { typedef LimExNFA128 Nfa; typedef NFAException128 Exc; };
template <> struct LimexLayout<WideSt<4>> { typedef LimExNFA256 Nfa; typedef NFAException256 Exc; };
template <> struct LimexLayout<WideSt<8>> { typedef LimExNFA512 Nfa; typedef NFAException512 Exc; };
/* CTA size: the wide state sets need the registers of a 512-thread CTA (and the 512-state tables the room) */
template <int ENGINE> struct StagedThreads { static constexpr int N = ENGINE >= ENG_LIMEX256 ? 512 : 1024; };
/* shared-memory tables of a LimEx engine: the reach mask per byte value, then per state a row of four
 * ST: limited successors, exception successors, squash mask, report list offset */
template <class ST> struct LimexTable { static constexpr u32 BYTES = 256u * sizeof(ST) + 8u * sizeof(ST) * 4u * sizeof(ST); };
/* ... of the wide models: reach, exception successors and squash masks chunk-major (StOps::loadChunks), the
 * report list of every state's exception, then the (up to eight) shift masks and the exception mask as they are */
template <int W> struct LimexTable<WideSt<W>> {
    static constexpr u32 STATES = 64u * W;
    static constexpr u32 REACH = 0, LOCAL = 256u * 8u * W, KEEP = LOCAL + STATES * 8u * W, REP = KEEP + STATES * 8u * W,
                         SHIFT = REP + STATES * 4u, EXC = SHIFT + 8u * 8u * W, BYTES = EXC + 8u * W;
};

enum { SHENG_ROW = 128, SHENG_TABLE_BYTES = 256 * SHENG_ROW };

struct DfaConsts {
    u32 as, single, report, start, auxOffset, shermanOffset, shermanLimit, acceptLimit8, auxSize, stateMask;
};

/* reports of a state that was just entered at offset `to` (doComplexReport, mcclellan.c:43-91;
 * fireReports, sheng_impl.h:116-155).  what = the one report of a single-report engine, else
 * the offset of the state's aux record.  Returns the lane's record cursor. */
__device__ HSB_NOINLINE u32 emitAccept(const DfaParams &p, const u8 *nfa, u32 cursor, u32 single, u32 what, u32 block,
                                       u64 to) {
    if (single) {
        return emitDfaMatch(p, cursor, what, block, to);
    }
    return emitReportList(p, nfa, cursor, g32(nfa + what), block, to);
}

template <int ENGINE, int SMEM_TABLE, int CH, int ILP>
__global__ void __launch_bounds__(StagedThreads<ENGINE>::N, 1) dfaStagedKernel(const HSB_GRID_CONSTANT DfaParams p) {
    HSB_DYNAMIC_SMEM(smem);
    typedef DfaTile<CH> Tile;
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    typedef typename WalkState<ENGINE>::type ST;
    typedef typename LimexLayout<ST>::Nfa LxNfa;
    typedef typename LimexLayout<ST>::Exc LxExc;
    typedef StOps<ST> Ops;
    constexpr bool LIMEX = ENGINE >= ENG_LIMEX32;
    constexpr bool WIDE = ENGINE >= ENG_LIMEX128; /* state sets of several 64-bit words */
    /* the engine the CTA runs (DfaParams.engines[current]) and its constants.  The LimEx walks read its bytes back
     * from the table where a report needs them rather than hold them in registers through the walk (measured
     * faster there; the DFA walks, whose accepts are frequent, are faster with them in a register). */
    u32 current = 0xffffffffu;
    const u8 *dfaBytes = nullptr;
    auto engineBytes = [&]() -> const u8 * { return LIMEX ? p.engines[current].nfa : dfaBytes; }; /* struct NFA */
    u32 squashes = 0;
    DfaConsts k;
    ST lxAccept = Ops::zero(), lxAcceptEod = Ops::zero(), lxStart = Ops::zero();
    u8 *const tile = smem + p.tableArea + warp * (ILP * Tile::WARP_BYTES);
    const u8 *const myRow = tile + lane * Tile::ROW;
    const u16 *succ16 = nullptr;
    const u32 copyOff = (lane & 7) * 16; /* Sheng: this lane's copy of a row */
    const ST *lxReach = reinterpret_cast<const ST *>(smem);
    const ST *lxRows = lxReach + 256;
    ST lxLim0 = Ops::zero(), lxLocal0 = Ops::zero(), lxKeep0 = Ops::ones();
    bool lxRow0Plain = false; /* state 0 raises no reports: its row can be applied without the loop */
    u32 lxShiftCount = 0;
    u64 lxShiftAmounts = 0; /* shiftAmount[0..7], one byte each */
    /* Switch the whole CTA to engine e: its constants, and its tables in shared memory (the caller has made sure
     * that no warp still reads the previous engine's) */
    auto loadEngine = [&](const u32 e) {
        const DfaEngine en = p.engines[e];
        dfaBytes = en.nfa;
        const u8 *const eng = en.nfa + sizeof(NFA); /* struct mcclellan / struct sheng / LimExNFA* */
        const u8 *const succG = eng + sizeof(McClellan);
        squashes = en.squashes;
        k.as = 0;
        k.shermanOffset = 0;
        k.shermanLimit = 0xffffffffu;
        k.acceptLimit8 = 0;
        if (LIMEX) {
            /* eng = struct LimExNFA32 ... 512; a top at offset 0 switches `init` on (moNfaTop) */
            lxStart = Ops::load(eng + offsetof(LxNfa, init));
            k.start = 0;
            k.single = 0;
            k.report = 0;
            k.auxOffset = 0;
            k.auxSize = 0;
            k.stateMask = 0xffffffffu;
            lxAccept = Ops::load(eng + offsetof(LxNfa, accept));
            lxAcceptEod = Ops::load(eng + offsetof(LxNfa, acceptAtEOD));
        } else if (ENGINE == ENG_SHENG) {
            k.start = __ldg(eng + offsetof(Sheng, anchored));
            k.single = __ldg(eng + offsetof(Sheng, flags)) & SHENG_FLAG_SINGLE_REPORT;
            k.report = g32(eng + offsetof(Sheng, report));
            k.auxOffset = g32(eng + offsetof(Sheng, aux_offset));
            k.auxSize = (u32)sizeof(SstateAux);
            k.stateMask = SHENG_STATE_MASK;
        } else {
            k.as = __ldg(eng + offsetof(McClellan, alphaShift));
            k.single = __ldg(eng + offsetof(McClellan, flags)) & MCCLELLAN_FLAG_SINGLE;
            k.report = g32(eng + offsetof(McClellan, arb_report));
            k.start = g16(eng + offsetof(McClellan, start_anchored));
            k.auxOffset = g32(eng + offsetof(McClellan, aux_offset));
            k.shermanOffset = g32(eng + offsetof(McClellan, sherman_offset));
            if (ENGINE == ENG_MCC16) {
                k.shermanLimit = g16(eng + offsetof(McClellan, sherman_limit));
            }
            k.acceptLimit8 = g16(eng + offsetof(McClellan, accept_limit_8));
            k.auxSize = (u32)sizeof(MStateAux);
            k.stateMask = 0xffffffffu;
        }
        if (LIMEX) {
            /* (32- and 64-state models) reach mask by byte value (reach[reachMap[b]]), then ONE row of four ST per state i:
             *   [0] its limited successors: OR over the shifts k with bit i of shift[k] of 1 << (i + shiftAmount[k])
             *   [1] its exception's successors, [2] its squash mask (all ones unless the exception squashes:
             *   LIMEX_SQUASH_CYCLIC / _REPORT), [3] its exception's report list
             * so a byte costs work in proportion to the states that are ON, not eight shift-and-mask rounds */
            const u8 *reach = eng + sizeof(LxNfa);
            const ST excMask = Ops::load(eng + offsetof(LxNfa, exceptionMask));
            const u32 nshift = g32(eng + offsetof(LxNfa, shiftCount));
            const u8 *exc = eng + g32(eng + offsetof(LxNfa, exceptionOffset));
            /* row of state i: limited successors, exception successors, squash mask, report list */
            auto rowOf = [&](const u32 i, ST &lim, ST &local, ST &keep, u32 &rep) {
                lim = Ops::zero(), local = Ops::zero(), keep = Ops::ones(), rep = MO_INVALID_IDX;
                for (u32 q = 0; q < nshift && q < 8; q++) {
                    if (Ops::test(Ops::load(eng + offsetof(LxNfa, shift) + sizeof(ST) * q), i)) {
                        lim = Ops::bor(lim, Ops::shiftedBit(i, __ldg(eng + offsetof(LxNfa, shiftAmount) + q)));
                    }
                }
                if (Ops::test(excMask, i)) {
                    const u8 *x = exc + Ops::rank(excMask, i) * (u32)sizeof(LxExc);
                    const u32 kind = __ldg(x + offsetof(LxExc, hasSquash));
                    local = Ops::load(x + offsetof(LxExc, successors));
                    rep = g32(x + offsetof(LxExc, reports));
                    if (kind == LIMEX_SQUASH_CYCLIC || kind == LIMEX_SQUASH_REPORT) {
                        keep = Ops::load(x + offsetof(LxExc, squash));
                    }
                }
            };
            if constexpr (WIDE) {
                typedef LimexTable<ST> T;
                for (u32 i = threadIdx.x; i < 256; i += blockDim.x) {
                    Ops::storeChunks(reinterpret_cast<uint4 *>(smem + T::REACH), 256, i,
                                     Ops::load(reach + sizeof(ST) * __ldg(eng + offsetof(LxNfa, reachMap) + i)));
                }
                for (u32 i = threadIdx.x; i < T::STATES; i += blockDim.x) {
                    ST lim, local, keep;
                    u32 rep;
                    rowOf(i, lim, local, keep, rep);
                    Ops::storeChunks(reinterpret_cast<uint4 *>(smem + T::LOCAL), T::STATES, i, local);
                    Ops::storeChunks(reinterpret_cast<uint4 *>(smem + T::KEEP), T::STATES, i, keep);
                    reinterpret_cast<u32 *>(smem + T::REP)[i] = rep;
                }
                for (u32 i = threadIdx.x; i < 9; i += blockDim.x) { /* shift masks 0..7, then the exception mask */
                    reinterpret_cast<ST *>(smem + T::SHIFT)[i] =
                        i < 8 ? (i < nshift ? Ops::load(eng + offsetof(LxNfa, shift) + sizeof(ST) * i) : Ops::zero()) : excMask;
                }
            } else {
                ST *d = reinterpret_cast<ST *>(smem);
                for (u32 i = threadIdx.x; i < 256; i += blockDim.x) {
                    d[i] = Ops::load(reach + sizeof(ST) * __ldg(eng + offsetof(LxNfa, reachMap) + i));
                }
                ST *rows = d + 256;
                for (u32 i = threadIdx.x; i < 8 * sizeof(ST); i += blockDim.x) {
                    ST lim, local, keep;
                    u32 rep;
                    rowOf(i, lim, local, keep, rep);
                    rows[4 * i + 0] = lim;
                    rows[4 * i + 1] = local;
                    rows[4 * i + 2] = keep;
                    rows[4 * i + 3] = Ops::fromU32(rep);
                }
            }
        } else if (ENGINE == ENG_SHENG) {
            /* [byte c][copy r][16 successor bytes, the one of state s at position (s + 4c) & 15] */
            for (u32 i = threadIdx.x; i < SHENG_TABLE_BYTES; i += blockDim.x) {
                const u32 c = i >> 7;
                smem[i] = __ldg(eng + c * 16 + (((i & 15) - 4 * c) & 15));
            }
        } else if (ENGINE == ENG_MCC8) {
            const u32 states = g16(eng + offsetof(McClellan, state_count));
            for (u32 i = threadIdx.x; i < states * 256; i += blockDim.x) {
                const u32 cp = __ldg(eng + offsetof(McClellan, remap) + (i & 255));
                smem[i] = __ldg(succG + ((i >> 8) << k.as) + cp);
            }
        } else {
            for (u32 i = threadIdx.x; i < 256; i += blockDim.x) {
                smem[i] = __ldg(eng + offsetof(McClellan, remap) + i);
            }
            if (SMEM_TABLE) {
                u32 *d = reinterpret_cast<u32 *>(smem + 256);
                const u32 *g = reinterpret_cast<const u32 *>(succG);
                for (u32 i = threadIdx.x; i < (en.tableBytes + 3) / 4; i += blockDim.x) {
                    d[i] = __ldg(g + i);
                }
            }
        }
        __syncthreads();
        succ16 = reinterpret_cast<const u16 *>(SMEM_TABLE ? smem + 256 : succG);
        if (LIMEX && !WIDE) { /* (the wide models read it from shared memory like every other row) */
            lxLim0 = lxRows[0];
            lxLocal0 = lxRows[1];
            lxKeep0 = lxRows[2];
            lxRow0Plain = Ops::low32(lxRows[3]) == MO_INVALID_IDX;
        }
        if (WIDE) {
            lxShiftCount = min(g32(eng + offsetof(LxNfa, shiftCount)), 8u);
            lxShiftAmounts = (u64)g32(eng + offsetof(LxNfa, shiftAmount)) | ((u64)g32(eng + offsetof(LxNfa, shiftAmount) + 4) << 32);
        }
    };
    u32 cursor = 0; /* this lane's next record slot (emitDfaMatch) */
    /* one input byte: byte j of data word w, at block offset pos.  DFAs: returns true when the
     * state entered accepts.  LimEx (LOOP_NOACCEL_FN, limex_runtime_impl.h:209-243): the states
     * that are on BEFORE the byte run their exceptions -- reports at offset pos, except at the
     * first byte of the scan (NO_OUTPUT | FIRST_BYTE) -- then succ & reach[byte]. */
    auto step = [&](const u32 w, const u32 j, ST &s, const u32 pos, const u32 blk) -> bool {
        if constexpr (WIDE) {
            /* the reference's own order of work (NFA_EXEC_GET_LIM_SUCC, then processExceptional over the
             * exceptional states only): with many states on, shifting whole 64-bit lanes costs less than a visit
             * per state; the squash masks are read only if the engine has a squashing exception at all */
            typedef LimexTable<ST> T;
            const ST *tShift = reinterpret_cast<const ST *>(smem + T::SHIFT);
            ST lim = Ops::zero(), local = Ops::zero(), keep = Ops::ones();
            for (u32 q = 0; q < lxShiftCount; q++) {
                const ST m = tShift[q];
                const u32 a = (u32)(lxShiftAmounts >> (8 * q)) & 0xff;
#pragma unroll
                for (u32 x = 0; x < sizeof(ST) / 8; x++) {
                    lim.w[x] |= (s.w[x] & m.w[x]) << a; /* LSHIFT_STATE: lane by lane */
                }
            }
            Ops::forEach(Ops::band(s, tShift[8]), [&](const u32 bit) {
                const u32 rep = reinterpret_cast<const u32 *>(smem + T::REP)[bit];
                if (rep != MO_INVALID_IDX && pos != 0) {
                    cursor = emitLimexReports(p, engineBytes(), cursor, rep, blk, pos);
                }
                local = Ops::bor(local, Ops::loadChunks(reinterpret_cast<const uint4 *>(smem + T::LOCAL), T::STATES, bit));
                if (squashes) {
                    keep = Ops::band(keep, Ops::loadChunks(reinterpret_cast<const uint4 *>(smem + T::KEEP), T::STATES, bit));
                }
            });
            s = Ops::band(Ops::bor(Ops::band(lim, keep), local),
                          Ops::loadChunks(reinterpret_cast<const uint4 *>(smem + T::REACH), 256, __byte_perm(w, 0, 0x4440 + j)));
            return false;
        } else if constexpr (LIMEX) {
            /* NFA_EXEC_GET_LIM_SUCC + processExceptional (limex_exceptional.h:190-330, cache
             * aside) over the states that are on, in ascending order: every exception's squash
             * cuts the limited successors only, the exception successors are OR-ed in afterwards */
            /* state 0 first, from registers: in a position automaton it is the floating start,
             * on at every byte -- most bytes of most inputs have nothing else on */
            ST lim = Ops::zero(), local = Ops::zero(), keep = Ops::ones(), on = s;
            if (lxRow0Plain && Ops::test(s, 0)) {
                lim = lxLim0;
                local = lxLocal0;
                keep = lxKeep0;
                on = Ops::clear0(on);
            }
            Ops::forEach(on, [&](const u32 bit) {
                const ST *e = lxRows + 4 * bit;
                const u32 rep = Ops::low32(e[3]);
                if (rep != MO_INVALID_IDX && pos != 0) {
                    cursor = emitLimexReports(p, engineBytes(), cursor, rep, blk, pos);
                }
                lim = Ops::bor(lim, e[0]);
                local = Ops::bor(local, e[1]);
                keep = Ops::band(keep, e[2]);
            });
            s = Ops::band(Ops::bor(Ops::band(lim, keep), local), lxReach[__byte_perm(w, 0, 0x4440 + j)]);
            return false;
        } else if constexpr (ENGINE == ENG_MCC8) {
            s = smem[__byte_perm(w, s, 0x5540 + j)]; /* (s << 8) | byte */
            return s >= k.acceptLimit8;
        } else if constexpr (ENGINE == ENG_SHENG) {
            const u32 ch = __byte_perm(w, 0, 0x4440 + j);
            s = smem[ch * SHENG_ROW + (((s + 4 * ch) & SHENG_STATE_MASK) | copyOff)]; /* pshufb(masks[byte], state) */
            return (s & SHENG_STATE_ACCEPT) != 0;
        } else {
            const u32 cp = smem[__byte_perm(w, 0, 0x4440 + j)];
            u32 e;
            if (s < k.shermanLimit) {
                e = SMEM_TABLE ? succ16[(s << k.as) + cp] : __ldg(succ16 + (s << k.as) + cp);
            } else {
                const u8 *nfa = engineBytes();
                e = shermanNext(nfa, k.shermanOffset, k.shermanLimit, s, cp,
                                reinterpret_cast<const u16 *>(nfa + sizeof(NFA) + sizeof(McClellan)),
                                k.as);
            }
            s = e & MCC_STATE_MASK;
            return (e & MCC_ACCEPT_FLAG) != 0;
        }
    };
    auto acceptWhat = [&](const ST &s) -> u32 {
        return k.single ? k.report : k.auxOffset + k.auxSize * (Ops::low32(s) & k.stateMask);
    };
    auto dead = [&](const ST &s) -> bool {
        return ENGINE == ENG_SHENG ? (Ops::low32(s) & SHENG_STATE_DEAD) != 0 : !Ops::any(s);
    };

    /* a warp takes 32 * ILP consecutive blocks at a time; lane t owns blocks t, t + 32, ...
     * of the group: ILP independent state chains in one instruction stream.  The work of a launch is
     * every engine over every group, in rounds of one engine and nwarps consecutive groups (a warp each),
     * engine-major; CTA c takes rounds c, c + gridDim.x, ... -- with one engine the round-robin over the
     * groups it always was -- and so meets the engines in order, building each one's tables once. */
    const u32 perGroup = 32 * ILP;
    const u32 ngroups = (p.nblocks + perGroup - 1) / perGroup;
    const u32 rounds = (ngroups + nwarps - 1) / nwarps; /* of one engine */
    for (u32 round = blockIdx.x; round < rounds * p.nengines; round += gridDim.x) {
        const u32 e = round / rounds;
        if (e != current) { /* (uniform across the CTA: every warp walks the same rounds) */
            if (current != 0xffffffffu) {
                __syncthreads();
            }
            current = e;
            loadEngine(e);
        }
        const u32 g = (round - e * rounds) * nwarps + warp;
        if (g >= ngroups) {
            continue;
        }
        u32 b[ILP], len[ILP];
        ST s[ILP];
        u64 off[ILP];
        bool live[ILP];
#pragma unroll
        for (int u = 0; u < ILP; u++) {
            b[u] = g * perGroup + 32 * u + lane;
            off[u] = 0;
            len[u] = 0;
            if (b[u] < p.nblocks) {
                const BlockSpan blk = blockSpan(p, b[u]);
                off[u] = (u64)(blk.base - p.corpus);
                len[u] = blk.len;
            }
            s[u] = LIMEX ? lxStart : Ops::fromU32(k.start);
            live[u] = len[u] != 0;
        }
        for (u32 r = 0;; r++) {
            const u32 done = r * CH;
            bool more = false;
#pragma unroll
            for (int u = 0; u < ILP; u++) {
                more |= live[u] && done < len[u];
            }
            if (!__any_sync(0xffffffffu, more)) {
                break;
            }
            /* refill: every load of the tile in flight before the first store */
            uint4 v[ILP * Tile::PIECES];
#pragma unroll
            for (u32 i = 0; i < ILP * Tile::PIECES; i++) {
                const u32 u = i / Tile::PIECES;                                 /* which of the lane's blocks' rows */
                const u32 src = (i % Tile::PIECES) * Tile::ROWS_PER_LOAD + lane / Tile::PIECES; /* owning lane */
                const u32 rOffLo = __shfl_sync(0xffffffffu, (u32)off[u], src);
                const u32 rOffHi = __shfl_sync(0xffffffffu, (u32)(off[u] >> 32), src);
                const u32 rLen = __shfl_sync(0xffffffffu, len[u], src);
                const u32 pos = done + (lane % Tile::PIECES) * 16;
                v[i] = make_uint4(0, 0, 0, 0);
                if (pos < rLen) {
                    v[i] = load16(p, p.corpus + (((u64)rOffHi << 32) | rOffLo) + pos);
                }
            }
#pragma unroll
            for (u32 i = 0; i < ILP * Tile::PIECES; i++) {
                const u32 u = i / Tile::PIECES;
                const u32 src = (i % Tile::PIECES) * Tile::ROWS_PER_LOAD + lane / Tile::PIECES;
                *reinterpret_cast<uint4 *>(tile + (u * 32 + src) * Tile::ROW + (lane % Tile::PIECES) * 16) = v[i];
            }
            __syncwarp();
            u32 n[ILP];
            bool fullAll = true;
#pragma unroll
            for (int u = 0; u < ILP; u++) {
                n[u] = !live[u] || done >= len[u] ? 0u : (len[u] - done < (u32)CH ? len[u] - done : (u32)CH);
            }
            u32 c = 0;
            if (ILP > 1) {
                /* all chains of the lane alive with a full piece ahead: interleaved */
#pragma unroll 1
                for (;; c++) {
                    fullAll = true;
#pragma unroll
                    for (int u = 0; u < ILP; u++) {
                        fullAll &= live[u] && c * 16 + 16 <= n[u];
                    }
                    if (!fullAll) {
                        break;
                    }
                    u32 w[ILP][4];
#pragma unroll
                    for (int u = 0; u < ILP; u++) {
                        const uint4 x = *reinterpret_cast<const uint4 *>(myRow + u * 32 * Tile::ROW + c * 16);
                        w[u][0] = x.x;
                        w[u][1] = x.y;
                        w[u][2] = x.z;
                        w[u][3] = x.w;
                    }
#pragma unroll
                    for (u32 j = 0; j < 16; j++) {
#pragma unroll
                        for (int u = 0; u < ILP; u++) {
                            if (step(w[u][j >> 2], j & 3, s[u], done + c * 16 + j, b[u])) {
                                cursor = emitAccept(p, engineBytes(), cursor, k.single, acceptWhat(s[u]), b[u], (u64)done + c * 16 + j + 1);
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < ILP; u++) {
                        live[u] = !dead(s[u]);
                    }
                }
            }
            /* what is left of each chain's CH bytes, one chain at a time */
#pragma unroll
            for (int u = 0; u < ILP; u++) {
                const u8 *row = myRow + u * 32 * Tile::ROW;
                u32 cc = c;
                if constexpr (WIDE) {
                    /* a step of the wide models is hundreds of instructions: the sixteen unrolled copies of it
                     * (and a second set for the last piece) do not fit the instruction cache -- ncu's first stall
                     * reason was "no instruction" -- so their bytes go through ONE copy of the step */
                    if (live[u]) {
#pragma unroll 1
                        for (u32 j = cc * 16; j < n[u]; j++) {
                            (void)step(row[j], 0, s[u], done + j, b[u]);
                        }
                        live[u] = !dead(s[u]);
                    }
                } else {
#pragma unroll 1
                    for (; live[u] && cc * 16 + 16 <= n[u]; cc++) { /* full pieces: no per-byte checks */
                        const uint4 x = *reinterpret_cast<const uint4 *>(row + cc * 16);
                        const u32 w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                        for (u32 j = 0; j < 16; j++) {
                            if (step(w[j >> 2], j & 3, s[u], done + cc * 16 + j, b[u])) {
                                cursor = emitAccept(p, engineBytes(), cursor, k.single, acceptWhat(s[u]), b[u], (u64)done + cc * 16 + j + 1);
                            }
                        }
                        live[u] = !dead(s[u]);
                    }
                    if (live[u] && cc * 16 < n[u]) { /* the block's last, partial piece */
                        const uint4 x = *reinterpret_cast<const uint4 *>(row + cc * 16);
                        const u32 w[4] = {x.x, x.y, x.z, x.w};
                        const u32 m = n[u] - cc * 16;
#pragma unroll 1
                        for (u32 j = 0; j < m; j++) {
                            if (step(w[j >> 2] >> (8 * (j & 3)), 0, s[u], done + cc * 16 + j, b[u])) {
                                cursor = emitAccept(p, engineBytes(), cursor, k.single, acceptWhat(s[u]), b[u], (u64)done + cc * 16 + j + 1);
                            }
                        }
                        live[u] = !dead(s[u]);
                    }
                }
            }
            __syncwarp();
        }
        /* nfaExec*_B: reports of the final state that fire at end of data */
#pragma unroll
        for (int u = 0; u < ILP; u++) {
            if (LIMEX) {
                if (b[u] < p.nblocks) {
                    /* STREAM_FN's closing accept check (only if the block had bytes to stream),
                     * then nfaExecLimEx*_testEOD (limex_common_impl.h:192-218) */
                    if (len[u] && Ops::any(Ops::band(s[u], lxAccept))) {
                        const u8 *nfa = engineBytes();
                        cursor = emitLimexAccepts<ST>(p, nfa, cursor, Ops::band(s[u], lxAccept), lxAccept,
                                                      g32(nfa + sizeof(NFA) + offsetof(LxNfa, acceptOffset)), b[u], len[u]);
                    }
                    if (Ops::any(Ops::band(s[u], lxAcceptEod))) {
                        const u8 *nfa = engineBytes();
                        cursor = emitLimexAccepts<ST>(p, nfa, cursor, Ops::band(s[u], lxAcceptEod), lxAcceptEod,
                                                      g32(nfa + sizeof(NFA) + offsetof(LxNfa, acceptEodOffset)), b[u],
                                                      len[u]);
                    }
                }
            } else if (b[u] < p.nblocks) {
                const u32 eodOff = ENGINE == ENG_SHENG ? (u32)offsetof(SstateAux, accept_eod)
                                                       : (u32)offsetof(MStateAux, accept_eod);
                const u8 *nfa = engineBytes();
                const u32 eod = g32(nfa + k.auxOffset + k.auxSize * (Ops::low32(s[u]) & k.stateMask) + eodOff);
                if (eod) {
                    cursor = emitReportList(p, nfa, cursor, eod, b[u], len[u]);
                }
            }
        }
    }
    padReserved(p, cursor);
}

template <int ENGINE, int SMEM_TABLE>
cudaError_t launchStaged(const DfaParams &p, int smCount, size_t tableBytes, cudaStream_t stream) {
    /* one CTA of 32 warps per SM: table area + per warp a tile of 32 * ILP rows.
     * ilp 2: two blocks per lane, 64 bytes of each per refill (160 KiB of tiles);
     * ilp 1: one block per lane, 128 bytes per refill (144 KiB) */
    const int threads = StagedThreads<ENGINE>::N;
    const bool two = p.ilp == 2 && ENGINE < ENG_LIMEX128; /* (the wide models walk one block per lane) */
    const size_t tiles = (size_t)(threads / 32) * (two ? 2 * DfaTile<64>::WARP_BYTES : DfaTile<128>::WARP_BYTES);
    const u64 groups = ((u64)p.nblocks + (two ? 63 : 31)) / (two ? 64 : 32);
    const u64 rounds = (groups + threads / 32 - 1) / (threads / 32) * p.nengines; /* (the kernel's) */
    const int grid = (int)std::min<u64>((u64)smCount, rounds);
    void (*kern)(const DfaParams) =
        two ? dfaStagedKernel<ENGINE, SMEM_TABLE, 64, 2> : dfaStagedKernel<ENGINE, SMEM_TABLE, 128, 1>;
    const size_t smem = tableBytes + tiles;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        return e;
    }
    DfaParams q = p;
    q.tableArea = (u32)tableBytes; /* the tiles follow the largest engine's tables */
    HSB_LAUNCH(kern, grid, threads, smem, stream, q);
    return cudaGetLastError();
}

} // namespace

cudaError_t launchDfa(const DfaParams &p, int smCount, int maxSmem, cudaStream_t stream) {
    if (!p.nblocks || !p.nengines) {
        return cudaSuccess;
    }
    const size_t tilesMax = 32 * 2 * DfaTile<64>::WARP_BYTES;
    if (p.kind == NFA_SHENG) {
        return launchStaged<ENG_SHENG, 1>(p, smCount, SHENG_TABLE_BYTES, stream);
    }
    if (p.kind == NFA_LIMEX_32) {
        return launchStaged<ENG_LIMEX32, 1>(p, smCount, LimexTable<u32>::BYTES, stream);
    }
    if (p.kind == NFA_LIMEX_64) {
        return launchStaged<ENG_LIMEX64, 1>(p, smCount, LimexTable<u64>::BYTES, stream);
    }
    if (p.kind == NFA_LIMEX_128) {
        return launchStaged<ENG_LIMEX128, 1>(p, smCount, LimexTable<WideSt<2>>::BYTES, stream);
    }
    if (p.kind == NFA_LIMEX_256) {
        return launchStaged<ENG_LIMEX256, 1>(p, smCount, LimexTable<WideSt<4>>::BYTES, stream);
    }
    if (p.kind == NFA_LIMEX_512) {
        return launchStaged<ENG_LIMEX512, 1>(p, smCount, LimexTable<WideSt<8>>::BYTES, stream);
    }
    if (p.kind == NFA_MCCLELLAN_8) {
        return launchStaged<ENG_MCC8, 1>(p, smCount, (size_t)p.states * 256, stream); /* <= 64 KiB */
    }
    if (p.kind == NFA_MCCLELLAN_16) {
        const size_t inTable = 256 + HSB_ROUNDUP((size_t)p.tableBytes, 16);
        const bool inSmem = p.tableBytes && inTable + tilesMax <= (size_t)maxSmem;
        return inSmem ? launchStaged<ENG_MCC16, 1>(p, smCount, inTable, stream)
                      : launchStaged<ENG_MCC16, 0>(p, smCount, 256, stream);
    }
    return cudaErrorInvalidValue;
}

} // namespace hsb
