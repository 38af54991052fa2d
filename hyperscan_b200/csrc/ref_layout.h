/*
 * ref_layout.h -- byte layouts of the Hyperscan 5.4.2 database ("bytecode")
 * structures that the B200 runtime consumes and the host literal compiler
 * emits.  The serialised database format is the drop-in boundary
 * (BASELINE.json north_star: "serialised database format stays"), so these
 * are restated here field-for-field; every struct cites the reference header
 * it mirrors, and tests/test_layout.py pins each sizeof/offsetof against
 * tests/golden/ref_layout.json, which tools/gen_ref_layout.py produced from
 * the reference's own headers.
 *
 * Usable from host C++ and from CUDA device code (plain PODs, no methods that
 * need a runtime).  All multi-byte fields are little-endian.
 */
#ifndef HSB200_REF_LAYOUT_H
#define HSB200_REF_LAYOUT_H

#include <stddef.h>
#include <stdint.h>

namespace hsb {

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t s32;

#define HSB_ROUNDUP(x, n) ((((x) + (n) - 1) / (n)) * (n))

/* ---- database container: src/database.h:44-113 ------------------------ */

static const u32 DB_MAGIC = 0xdbdbdbdbU;
static const u32 DB_VERSION = (5u << 24) | (4u << 16) | (2u << 8); /* 5.4.2 */

static const u64 PLATFORM_NOAVX2 = 4u << 13;
static const u64 PLATFORM_NOAVX512 = 8u << 13;
static const u64 PLATFORM_NOAVX512VBMI = 0x10u << 13;

struct DbHeader {     /* struct hs_database */
    u32 magic;
    u32 version;
    u32 length;       /* bytes of bytecode */
    u64 platform;
    u32 crc32;        /* raw CRC32C(init 0, no final xor) of the bytecode */
    u32 reserved0;
    u32 reserved1;
    u32 bytecode;     /* offset of bytecode from the start of this struct */
    u32 padding[16];
    /* char bytes[] follows */
};

/* ---- rose engine header: src/rose/rose_internal.h:190-496 -------------- */

struct ScatterPlan {  /* struct scatter_full_plan, src/util/scatter.h:42-51 */
    u32 s_u64a_offset, s_u64a_count, s_u32_offset, s_u32_count;
    u32 s_u16_offset, s_u16_count, s_u8_count, s_u8_offset;
};

struct StateOffsets { /* struct RoseStateOffsets */
    u32 history;
    u32 exhausted;
    u32 exhausted_size;
    u32 logicalVec;
    u32 logicalVec_size;
    u32 combVec;
    u32 combVec_size;
    u32 activeLeafArray;
    u32 activeLeafArray_size;
    u32 activeLeftArray;
    u32 activeLeftArray_size;
    u32 leftfixLagTable;
    u32 anchorState;
    u32 groups;
    u32 groups_size;
    u32 longLitState;
    u32 longLitState_size;
    u32 somLocation;
    u32 somValid;
    u32 somWritable;
    u32 somMultibit_size;
    u32 nfaStateBegin;
    u32 end;
};

struct BoundaryReports { /* struct RoseBoundaryReports */
    u32 reportEodOffset;
    u32 reportZeroOffset;
    u32 reportZeroEodOffset;
};

enum { RUNTIME_FULL_ROSE = 0, RUNTIME_PURE_LITERAL = 1, RUNTIME_SINGLE_OUTFIX = 2 };

static const u32 ROSE_BOUND_INF = 0xffffffffu; /* src/rose/rose_common.h */

/* HS_MODE_* bits, src/hs_compile.h:1156-1171 */
static const u32 MODE_BLOCK = 1, MODE_STREAM = 2, MODE_VECTORED = 4;

struct RoseEngine {
    u8 pureLiteral;
    u8 noFloatingRoots;
    u8 requiresEodCheck;
    u8 hasOutfixesInSmallBlock;
    u8 runtimeImpl;
    u8 mpvTriggeredByLeaf;
    u8 canExhaust;
    u8 hasSom;
    u8 somHorizon;
    u32 mode;
    u32 historyRequired;
    u32 ekeyCount;
    u32 lkeyCount;
    u32 lopCount;
    u32 ckeyCount;
    u32 logicalTreeOffset;
    u32 combInfoMapOffset;
    u32 dkeyCount;
    u32 dkeyLogSize;
    u32 invDkeyOffset;
    u32 somLocationCount;
    u32 somLocationFatbitSize;
    u32 rolesWithStateCount;
    u32 stateSize;
    u32 anchorStateSize;
    u32 tStateSize;
    u32 scratchStateSize;
    u32 smallWriteOffset;
    u32 amatcherOffset;
    u32 ematcherOffset;
    u32 fmatcherOffset;
    u32 drmatcherOffset;
    u32 sbmatcherOffset;
    u32 longLitTableOffset;
    u32 amatcherMinWidth;
    u32 fmatcherMinWidth;
    u32 eodmatcherMinWidth;
    u32 amatcherMaxBiAnchoredWidth;
    u32 fmatcherMaxBiAnchoredWidth;
    u32 reportProgramOffset;
    u32 reportProgramCount;
    u32 delayProgramOffset;
    u32 anchoredProgramOffset;
    u32 activeArrayCount;
    u32 activeLeftCount;
    u32 queueCount;
    u32 activeQueueArraySize;
    u32 eagerIterOffset;
    u32 handledKeyCount;
    u32 handledKeyFatbitSize;
    u32 leftOffset;
    u32 roseCount;
    u32 eodProgramOffset;
    u32 flushCombProgramOffset;
    u32 lastFlushCombProgramOffset;
    u32 lastByteHistoryIterOffset;
    u32 minWidth;
    u32 minWidthExcludingBoundaries;
    u32 maxBiAnchoredWidth;
    u32 anchoredDistance;
    u32 anchoredMinDistance;
    u32 floatingDistance;
    u32 floatingMinDistance;
    u32 smallBlockDistance;
    u32 floatingMinLiteralMatchOffset;
    u32 nfaInfoOffset;
    u64 initialGroups;
    u64 floating_group_mask;
    u32 size;
    u32 delay_count;
    u32 delay_fatbit_size;
    u32 anchored_count;
    u32 anchored_fatbit_size;
    u32 maxFloatingDelayedMatch;
    u32 delayRebuildLength;
    StateOffsets stateOffsets;
    BoundaryReports boundary;
    u32 totalNumLiterals;
    u32 asize;
    u32 outfixBeginQueue;
    u32 outfixEndQueue;
    u32 leftfixBeginQueue;
    u32 initMpvNfa;
    u32 rosePrefixCount;
    u32 activeLeftIterOffset;
    u32 ematcherRegionSize;
    u32 somRevCount;
    u32 somRevOffsetOffset;
    u32 longLitStreamState;
    ScatterPlan state_init;
};

struct NfaInfo { /* src/rose/rose_internal.h:153-166 */
    u32 nfaOffset;
    u32 stateOffset;
    u32 fullStateOffset;
    u32 ekeyListOffset;
    u8 no_retrigger;
    u8 in_sbmatcher;
    u8 eod;
};

/* ---- HWLM + acceleration: src/hwlm/hwlm_internal.h:37-53, nfa/accel.h -- */

enum { HWLM_ENGINE_FDR = 12, HWLM_ENGINE_NOOD = 16 };

enum AccelType {
    ACCEL_NONE = 0, ACCEL_VERM, ACCEL_VERM_NOCASE, ACCEL_DVERM,
    ACCEL_DVERM_NOCASE, ACCEL_RVERM, ACCEL_RVERM_NOCASE, ACCEL_RDVERM,
    ACCEL_RDVERM_NOCASE, ACCEL_REOD, ACCEL_REOD_NOCASE, ACCEL_RDEOD,
    ACCEL_RDEOD_NOCASE, ACCEL_SHUFTI, ACCEL_DSHUFTI, ACCEL_TRUFFLE,
    ACCEL_RED_TAPE, ACCEL_DVERM_MASKED
};

struct alignas(16) AccelAux { /* union AccelAux, 80 bytes, 16-aligned */
    u8 accel_type;
    u8 offset;
    u8 b[14];  /* verm: b[0]=c; dverm: b[0..3]=c1,c2,m1,m2 */
    u8 m0[16]; /* shufti lo / truffle mask1 / dshufti lo1 */
    u8 m1[16]; /* shufti hi / truffle mask2 / dshufti hi1 */
    u8 m2[16]; /* dshufti lo2 */
    u8 m3[16]; /* dshufti hi2 */
};

struct alignas(16) HWLM {
    u8 type;
    u64 accel1_groups;
    AccelAux accel1;
    AccelAux accel0;
};
/* engine follows at ROUNDUP_CL(sizeof(HWLM)) = 192 */
static const u32 HWLM_ENGINE_OFFSET = 192;

struct NoodTable { /* struct noodTable, src/hwlm/noodle_internal.h:38-48 */
    u32 id;
    u64 msk;
    u64 cmp;
    u8 msk_len;
    u8 key_offset;
    u8 nocase;
    u8 single;
    u8 key0;
    u8 key1;
};

/* ---- FDR / Teddy: src/fdr/fdr_internal.h:50-86, teddy_internal.h:57-64 -- */

static const u32 FDR_FLOOD_MAX_IDS = 16;

struct FDRFlood {
    u64 allGroups;
    u32 suffix;
    u16 idCount;
    u32 ids[FDR_FLOOD_MAX_IDS];
    u64 groups[FDR_FLOOD_MAX_IDS];
};

struct alignas(16) FDR {
    u32 engineID;
    u32 size;
    u32 maxStringLen;
    u32 numStrings;
    u32 confOffset;
    u32 floodOffset;
    u8 stride;
    u8 domain;
    u16 domainMask;
    u32 tabSize;
    u8 start[16]; /* m128 initial state */
};
/* table (u64 x 2^domain) at ROUNDUP_CL(sizeof(FDR)) = 64: src/fdr/fdr.c:735 */
static const u32 FDR_TABLE_OFFSET = 64;

struct Teddy { /* first 6 fields shared with FDR */
    u32 engineID;
    u32 size;
    u32 maxStringLen;
    u32 numStrings;
    u32 confOffset;
    u32 floodOffset;
};
/* nibble masks at ROUNDUP_CL(sizeof(Teddy)) = 64: teddy_runtime_common.h:441 */
static const u32 TEDDY_MASK_OFFSET = 64;
/* engine ids: src/fdr/teddy_engine_description.cpp:55-72 */
static inline bool teddyIdValid(u32 id) { return id >= 3 && id <= 18; }
static inline u32 teddyNumMasks(u32 id) { return ((id - 3) % 8) / 2 + 1; }
static inline u32 teddyNumBuckets(u32 id) { return id <= 10 ? 16 : 8; }

/* confirm: src/fdr/fdr_confirm.h:36-94 */
static const u64 CONF_HASH_MULT = 0x0b4e0ef37bc32127ULL;
static const u8 FDR_LIT_FLAG_NOREPEAT = 1;

struct LitInfo {
    u64 v;
    u64 msk;
    u64 groups;
    u32 id;
    u8 size;
    u8 flags;
    u8 next;
};

struct FDRConfirm {
    u64 andmsk;
    u64 mult;
    u32 nBits;
    u64 groups;
    /* u32 litIndex[1 << nBits] follows, then LitInfo chains */
};

/* ---- rose programs: src/rose/rose_program.h:40-724 --------------------- */

enum RoseOp {
    OP_END = 0,
    OP_CHECK_GROUPS = 3,
    OP_CHECK_BOUNDS = 5,
    OP_CHECK_MASK = 9,
    OP_CHECK_MASK_32 = 10,
    OP_CHECK_BYTE = 11,
    OP_DEDUPE = 28,
    OP_REPORT = 33,
    OP_REPORT_EXHAUST = 34,
    OP_DEDUPE_AND_REPORT = 37,
    OP_FINAL_REPORT = 38,
    OP_CHECK_EXHAUSTED = 39,
    OP_ENGINES_EOD = 48,
    OP_SQUASH_GROUPS = 43,
    OP_CHECK_LONG_LIT = 51,
    OP_CHECK_LONG_LIT_NOCASE = 52,
    OP_CHECK_MED_LIT = 53,
    OP_CHECK_MED_LIT_NOCASE = 54,
    OP_CLEAR_WORK_DONE = 55,
    OP_INCLUDED_JUMP = 61,
    OP_SET_EXHAUST = 65,
    OP_CHECK_MASK_64 = 69,
    OP_LAST = 69
};

static const u32 INSTR_ALIGN = 8;
static const u32 INVALID_EKEY = 0xffffffffu; /* src/util/report.h */
static const u32 INVALID_DKEY = 0xffffffffu; /* MO_INVALID_IDX */

struct InstrEnd { u8 code; };
struct InstrCheckGroups { u8 code; u64 groups; };
struct InstrCheckMask { u8 code; u64 and_mask, cmp_mask, neg_mask; s32 offset; u32 fail_jump; };
struct InstrCheckMask32 { u8 code; u8 and_mask[32]; u8 cmp_mask[32]; u32 neg_mask; s32 offset; u32 fail_jump; };
struct InstrCheckMask64 { u8 code; u8 and_mask[64]; u8 cmp_mask[64]; u64 neg_mask; s32 offset; u32 fail_jump; };
struct InstrCheckByte { u8 code, and_mask, cmp_mask, negation; s32 offset; u32 fail_jump; };
struct InstrCheckBounds { u8 code; u64 min_bound; u64 max_bound; u32 fail_jump; }; /* on the match end, before any offset_adjust */
struct InstrDedupe { u8 code, quash_som; u32 dkey; s32 offset_adjust; u32 fail_jump; };
struct InstrReport { u8 code; u32 onmatch; s32 offset_adjust; };
struct InstrReportExhaust { u8 code; u32 onmatch; s32 offset_adjust; u32 ekey; };
struct InstrDedupeAndReport { u8 code, quash_som; u32 dkey; u32 onmatch; s32 offset_adjust; u32 fail_jump; };
struct InstrFinalReport { u8 code; u32 onmatch; s32 offset_adjust; };
struct InstrCheckExhausted { u8 code; u32 ekey; u32 fail_jump; };
struct InstrSquashGroups { u8 code; u64 groups; };
struct InstrCheckLit { u8 code; u32 lit_offset; u32 lit_length; u32 fail_jump; }; /* MED + LONG */
struct InstrIncludedJump { u8 code, squash; u32 child_offset; };
struct InstrSetExhaust { u8 code; u32 ekey; };
struct InstrEnginesEod { u8 code; u32 iter_offset; }; /* the queues of a sparse iterator at EOD */

/* one record of a sparse multibit iterator (src/util/multibit_internal.h:59-62) */
struct MmbitSparseIter { u64 mask; u32 val; };

/* ---- NFA engines (DFA subset): src/nfa/nfa_internal.h:53-126,
 *      src/nfa/mcclellan_internal.h:36-106 -------------------------------- */

enum { NFA_LIMEX_32 = 0, NFA_LIMEX_64 = 1, NFA_LIMEX_128 = 2, NFA_LIMEX_256 = 3, NFA_LIMEX_384 = 4, NFA_LIMEX_512 = 5, NFA_MCCLELLAN_8 = 6, NFA_MCCLELLAN_16 = 7, NFA_SHENG = 17 };

struct alignas(64) NFA {
    u32 flags;
    u32 length;
    u8 type;
    u8 rAccelType;
    u8 rAccelOffset;
    u8 maxBiAnchoredWidth;
    u16 rAccelData;
    u32 queueIndex;
    u32 nPositions;
    u32 scratchStateSize;
    u32 streamStateSize;
    u32 maxWidth;
    u32 minWidth;
    u32 maxOffset;
};
static const u32 NFA_ACCEPTS_EOD = 1; /* src/nfa/nfa_internal.h:128 */

struct MStateAux { u32 accept; u32 accept_eod; u16 top; u32 accel_offset; };

static const u16 MCC_ACCEPT_FLAG = 0x8000, MCC_ACCEL_FLAG = 0x4000, MCC_STATE_MASK = 0x3fff;
static const u8 MCCLELLAN_FLAG_SINGLE = 1;

struct McClellan {
    u16 state_count;
    u32 length;
    u16 start_anchored;
    u16 start_floating;
    u32 aux_offset;
    u32 sherman_offset;
    u32 sherman_end;
    u16 accel_limit_8;
    u16 accept_limit_8;
    u16 sherman_limit;
    u16 wide_limit;
    u8 alphaShift;
    u8 flags;
    u8 has_accel;
    u8 has_wide;
    u8 remap[256];
    u32 arb_report;
    u32 accel_offset;
    u32 haig_offset;
    u32 wide_offset;
};

/* ---- LimEx NFA, 32-state model: src/nfa/limex_internal.h:102-203 (CREATE_NFA_LIMEX(32)).
 *      The reach table (u32 per reach class) follows the struct; the other tables sit at
 *      the offsets it names, all relative to the start of the LimExNFA32. ------------- */
struct NFAException32 {
    u32 squash;       /* mask of states to leave on */
    u32 successors;   /* mask of states to switch on */
    u32 reports;      /* offset of a MO_INVALID_IDX-terminated report list, or MO_INVALID_IDX */
    u32 repeatOffset; /* offset of NFARepeatInfo, or MO_INVALID_IDX */
    u8 hasSquash;     /* enum LimExSquash */
    u8 trigger;       /* enum LimExTrigger */
};
struct NFAAccept {
    u8 single_report; /* 1: `reports` is the report id itself */
    u32 reports;      /* else offset of a MO_INVALID_IDX-terminated list */
    u32 squash;       /* offset of a squash mask, or MO_INVALID_IDX */
};
struct LimExNFA32 {
    u8 reachMap[256];
    u32 reachSize, accelCount, accelTableOffset, accelAuxCount, accelAuxOffset;
    u32 acceptCount, acceptOffset, acceptEodCount, acceptEodOffset;
    u32 exceptionCount, exceptionOffset, repeatCount, repeatOffset;
    u32 squashOffset, squashCount, topCount, topOffset, stateSize, flags;
    u32 init, initDS, accept, acceptAtEOD, accel, accelPermute, accelCompare, accel_and_friends;
    u32 compressMask, exceptionMask, repeatCyclicMask, zombieMask;
    u32 shift[8];
    u32 shiftCount;
    u8 shiftAmount[8];
    alignas(64) u8 exceptionShufMask[64];
    alignas(64) u8 exceptionBitMask[64];
    alignas(64) u8 exceptionAndMask[64];
};
/* ... and the 64-state model (CREATE_NFA_LIMEX(64): the same fields over u64) */
struct NFAException64 {
    u64 squash, successors;
    u32 reports, repeatOffset;
    u8 hasSquash, trigger;
};
struct LimExNFA64 {
    u8 reachMap[256];
    u32 reachSize, accelCount, accelTableOffset, accelAuxCount, accelAuxOffset;
    u32 acceptCount, acceptOffset, acceptEodCount, acceptEodOffset;
    u32 exceptionCount, exceptionOffset, repeatCount, repeatOffset;
    u32 squashOffset, squashCount, topCount, topOffset, stateSize, flags;
    u64 init, initDS, accept, acceptAtEOD, accel, accelPermute, accelCompare, accel_and_friends;
    u64 compressMask, exceptionMask, repeatCyclicMask, zombieMask;
    u64 shift[8];
    u32 shiftCount;
    u8 shiftAmount[8];
    alignas(64) u8 exceptionShufMask[64];
    alignas(64) u8 exceptionBitMask[64];
    alignas(64) u8 exceptionAndMask[64];
};
/* ... and the 128-, 256- and 512-state models (CREATE_NFA_LIMEX(128 / 256 / 512)): the same fields over m128 /
 * m256 / m512, which are restated here as arrays of 64-bit words with the vector types' alignment (the 384-state
 * model is not emitted: an automaton of 257-384 states takes the 512-state one) */
template <unsigned BYTES> struct alignas(BYTES) StateWordT {
    u64 w[BYTES / 8];
};
typedef StateWordT<16> StateWord128;
typedef StateWordT<32> StateWord256;
typedef StateWordT<64> StateWord512;
template <class T> struct NFAExceptionW {
    T squash, successors;
    u32 reports, repeatOffset;
    u8 hasSquash, trigger;
};
template <class T> struct LimExNFAW {
    u8 reachMap[256];
    u32 reachSize, accelCount, accelTableOffset, accelAuxCount, accelAuxOffset;
    u32 acceptCount, acceptOffset, acceptEodCount, acceptEodOffset;
    u32 exceptionCount, exceptionOffset, repeatCount, repeatOffset;
    u32 squashOffset, squashCount, topCount, topOffset, stateSize, flags;
    T init, initDS, accept, acceptAtEOD, accel, accelPermute, accelCompare, accel_and_friends;
    T compressMask, exceptionMask, repeatCyclicMask, zombieMask;
    T shift[8];
    u32 shiftCount;
    u8 shiftAmount[8];
    alignas(64) u8 exceptionShufMask[64];
    alignas(64) u8 exceptionBitMask[64];
    alignas(64) u8 exceptionAndMask[64];
};
typedef NFAExceptionW<StateWord128> NFAException128;
typedef NFAExceptionW<StateWord256> NFAException256;
typedef NFAExceptionW<StateWord512> NFAException512;
typedef LimExNFAW<StateWord128> LimExNFA128;
typedef LimExNFAW<StateWord256> LimExNFA256;
typedef LimExNFAW<StateWord512> LimExNFA512;
static const u32 MO_INVALID_IDX = 0xffffffffu;            /* src/ue2common.h */
static const u32 LIMEX_FLAG_CANNOT_DIE = 4;               /* limex_internal.h:89 */
static const u8 LIMEX_SQUASH_NONE = 0, LIMEX_SQUASH_CYCLIC = 1, LIMEX_SQUASH_TUG = 2, LIMEX_SQUASH_REPORT = 3;
static const u8 LIMEX_TRIGGER_NONE = 0;

/* ---- small-write engine header: src/smallwrite/smallwrite_internal.h:35-39 (the
 *      struct NFA of a McClellan / Sheng DFA follows at the next cache line) ------ */
struct alignas(64) SmallWriteEngine {
    u32 largestBuffer; /* buffers shorter than this go through the DFA instead of rose */
    u32 start_offset;
    u32 size;          /* of the engine in bytes, including the NFA */
};

/* ---- Sheng: src/nfa/sheng_internal.h:36-79 ------------------------------ */

static const u8 SHENG_STATE_ACCEPT = 0x10, SHENG_STATE_DEAD = 0x20, SHENG_STATE_ACCEL = 0x40,
                SHENG_STATE_MASK = 0xf;
static const u8 SHENG_FLAG_SINGLE_REPORT = 1, SHENG_FLAG_CAN_DIE = 2, SHENG_FLAG_HAS_ACCEL = 4;

struct SstateAux { u32 accept; u32 accept_eod; u32 accel; u32 top; };

struct alignas(16) Sheng {
    u8 shuffle_masks[256][16]; /* m128 per input byte: next state (with flags) of each of the 16 states */
    u32 length;
    u32 aux_offset;
    u32 report_offset;
    u32 accel_offset;
    u8 n_states;
    u8 anchored;
    u8 floating;
    u8 flags;
    u32 report;
};

/* Sherman state record (src/nfa/mcclellan_internal.h:43-49): 32 bytes */
static const u32 SHERMAN_FIXED_SIZE = 32, SHERMAN_TYPE_OFFSET = 0, SHERMAN_LEN_OFFSET = 1,
                 SHERMAN_DADDY_OFFSET = 2, SHERMAN_CHARS_OFFSET = 4;
static const u8 SHERMAN_STATE = 1;

/* ---- multibit sizing: src/util/multibit_build.cpp:49-73 ---------------- */

static inline u32 mmbitSize(u32 total_bits) {
    if (total_bits <= 256) {
        return HSB_ROUNDUP(total_bits, 8) / 8;
    }
    u64 level = 1, total = 0;
    while (level * 64 < total_bits) {
        total += level;
        level <<= 6;
    }
    total += ((u64)total_bits + 63) / 64;
    return (u32)(total * 8);
}
/* src/util/fatbit_build.cpp:40-42 (sizeof(struct fatbit) == 32) */
static inline u32 fatbitSize(u32 total_bits) {
    u32 m = mmbitSize(total_bits);
    return m < 32 ? 32 : m;
}

} // namespace hsb

#endif
