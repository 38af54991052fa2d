/*
 * rose_build.cpp -- assembles the RoseEngine bytecode of a pure-literal
 * database: one role program per literal fragment, the dedupe-key table and
 * the floating HWLM table, behind a RoseEngine header whose fields are set the
 * way the reference's back end sets them for ROSE_RUNTIME_PURE_LITERAL
 * databases (src/rose/rose_build_bytecode.cpp:259-305 isPureFloating,
 * :382-465 fillStateOffsets, :3609-3888 buildFinalEngine).
 *
 * Program shapes follow src/rose/rose_build_program.cpp:525-710 (makeReport)
 * and :780-829 (makeCheckLiteralInstruction):
 *
 *   per pattern P of the fragment            (fail_jump -> next pattern / END)
 *     |P| > 8            CHECK_MED_LIT[_NOCASE]  lit bytes live in the blob
 *     SINGLEMATCH        CHECK_EXHAUSTED, [DEDUPE,] REPORT_EXHAUST
 *     shared report id   DEDUPE_AND_REPORT
 *     otherwise          REPORT
 *   END
 *
 * Literals longer than 8 bytes reach the literal matcher as their 8-byte
 * suffix (src/rose/rose_build_matchers.cpp:717-720); patterns with equal
 * suffix/case share one HWLM literal ("fragment") whose id is the byte offset
 * of its program in the bytecode (src/rose/match.c:238).
 */
#include "rose_build.h"
#include "dfa_build.h"
#include "limex_build.h"
#include "regex_nfa.h"
#include "../../../include/hs_b200.h"

#include <algorithm>
#include <cstring>
#include <map>
#include <tuple>
#include <set>
#include <stdexcept>

namespace hsb {

namespace {

struct Blob {
    std::vector<u8> bytes; /* starts at RoseEngine offset `base` */
    u32 base;
    explicit Blob(u32 b) : base(b) {}
    u32 reserve(size_t len, size_t align) {
        size_t pos = HSB_ROUNDUP(base + bytes.size(), align);
        bytes.resize(pos - base + len, 0);
        return (u32)pos;
    }
    u32 add(const void *p, size_t len, size_t align) {
        u32 off = reserve(len, align);
        memcpy(bytes.data() + (off - base), p, len);
        return off;
    }
    u8 *at(u32 off) { return bytes.data() + (off - base); }
};

template <class T> u32 instrSize() { return (u32)HSB_ROUNDUP(sizeof(T), INSTR_ALIGN); }

struct PatInfo {
    const LitPattern *p;
    std::string folded; /* upper-cased if caseless */
    bool anyAlpha;
    u32 ekey, dkey;
};

u32 blockSize(const PatInfo &pi) {
    u32 sz = 0;
    if (pi.p->s.size() > 8) {
        sz += instrSize<InstrCheckLit>();
    }
    if (pi.ekey != INVALID_EKEY) {
        sz += instrSize<InstrCheckExhausted>();
        if (pi.dkey != INVALID_DKEY) {
            sz += instrSize<InstrDedupe>();
        }
        sz += instrSize<InstrReportExhaust>();
    } else if (pi.dkey != INVALID_DKEY) {
        sz += instrSize<InstrDedupeAndReport>();
    } else {
        sz += instrSize<InstrReport>();
    }
    return sz;
}

/* What the header needs to know about the literal set. */
struct RoseTail {
    u32 minLen, maxLen, ekeyCount, dkeyCount, invDkeyOffset;
    bool canExhaust;
    u32 smallWriteOffset = 0;
};

/* A database whose only matcher is ONE engine run as an outfix over the whole block
 * (ROSE_RUNTIME_SINGLE_OUTFIX: hs_scan -> soleOutfixBlockExec, src/runtime.c:245-280): queue 0,
 * no literal matchers.  What the reference's compiler emits for a pattern set that is all
 * engine and no literal (rose_build_bytecode.cpp:3672-3690 pickRuntimeImpl); here it is built
 * for literal sets on request, so that the DFA / NFA engines run inside a real database. */
std::vector<u8> finishOutfixRose(Blob &blob, const std::vector<u8> &nfa, const RoseTail &t, const CompileOpts &opts) {
    NFA hdr;
    memcpy(&hdr, nfa.data(), sizeof(hdr));
    const u32 nfaOffset = blob.add(nfa.data(), nfa.size(), 64);
    RoseEngine r;
    memset(&r, 0, sizeof(r));
    r.pureLiteral = 0;
    r.runtimeImpl = RUNTIME_SINGLE_OUTFIX;
    r.canExhaust = t.canExhaust ? 1 : 0;
    r.mode = MODE_BLOCK;
    r.ekeyCount = t.ekeyCount;
    r.dkeyCount = t.dkeyCount;
    r.dkeyLogSize = fatbitSize(r.dkeyCount);
    r.invDkeyOffset = t.invDkeyOffset;
    r.somLocationFatbitSize = fatbitSize(0);
    r.activeArrayCount = 1;
    r.queueCount = 1;
    r.activeQueueArraySize = fatbitSize(1);
    r.handledKeyFatbitSize = fatbitSize(0);
    r.minWidth = t.minLen;
    r.minWidthExcludingBoundaries = t.minLen;
    r.maxBiAnchoredWidth = ROSE_BOUND_INF;
    r.floatingDistance = ROSE_BOUND_INF;
    r.initialGroups = 0;
    r.delay_fatbit_size = fatbitSize(0);
    r.anchored_fatbit_size = fatbitSize(0);
    r.outfixBeginQueue = 0;
    r.outfixEndQueue = 1;
    r.leftfixBeginQueue = 1;
    r.initMpvNfa = 0xffffffffu;
    r.scratchStateSize = (u32)HSB_ROUNDUP(hdr.scratchStateSize, 64); /* the queue's full state, in scratch */
    StateOffsets &so = r.stateOffsets;
    u32 cur = 1; /* status byte; no roles */
    so.activeLeafArray = cur;
    so.activeLeafArray_size = mmbitSize(1);
    cur += so.activeLeafArray_size;
    so.activeLeftArray = so.longLitState = so.leftfixLagTable = so.anchorState = cur;
    so.groups = cur;
    so.groups_size = 0;
    so.history = cur;
    so.exhausted = cur;
    so.exhausted_size = mmbitSize(r.ekeyCount);
    cur += so.exhausted_size;
    so.logicalVec = so.combVec = cur;
    so.nfaStateBegin = cur;
    NfaInfo ni;
    memset(&ni, 0, sizeof(ni));
    ni.nfaOffset = nfaOffset;
    ni.stateOffset = cur;
    ni.fullStateOffset = 0;
    cur += hdr.streamStateSize;
    so.end = cur;
    r.stateSize = cur;
    r.nfaInfoOffset = blob.add(&ni, sizeof(ni), 4);
    const u32 total = (u32)HSB_ROUNDUP(blob.base + blob.bytes.size(), 64);
    r.size = total;
    (void)opts;
    std::vector<u8> out(total, 0);
    memcpy(out.data(), &r, sizeof(r));
    memcpy(out.data() + blob.base, blob.bytes.data(), blob.bytes.size());
    return out;
}

/* uncompressed state alignment of an engine in scratch (NFATraits<>::stateAlign, src/nfa/nfa_build_util.cpp:174-230:
 * LimEx models max(alignof(state set), alignof(RepeatControl) = 8)) */
u32 engineStateAlign(u8 type) {
    switch (type) {
    case NFA_MCCLELLAN_16: return 2;
    case NFA_LIMEX_32: return 8;
    case NFA_LIMEX_64:
    case NFA_LIMEX_128: return 16;
    case NFA_LIMEX_256: return 32;
    case NFA_LIMEX_512: return 64;
    default: return 1;
    }
}

/* A database of several engines, each run as an outfix over the whole block, and nothing else: what the
 * reference's back end emits for a set of outfixes without literals (ROSE_RUNTIME_FULL_ROSE; buildFinalEngine,
 * src/rose/rose_build_bytecode.cpp:3609-3888).  hs_scan -> roseBlockExec (src/rose/block.c:345-422): every queue
 * starts in blockInitSufPQ and runs to the end under catch-up; engines that accept at EOD are listed in the EOD
 * program [ENGINES_EOD iter] END (makeEodProgram, :3334-3349; buildEodNfaIterator, :2276-2294). */
std::vector<u8> finishEnginesRose(Blob &blob, const std::vector<std::vector<u8>> &engines, const RoseTail &t) {
    const u32 n = (u32)engines.size();
    std::vector<NfaInfo> infos(n);
    memset(infos.data(), 0, sizeof(NfaInfo) * n);
    std::vector<u32> eodQueues;
    for (u32 q = 0; q < n; q++) {
        std::vector<u8> eng = engines[q];
        NFA hdr;
        memcpy(&hdr, eng.data(), sizeof(hdr));
        hdr.queueIndex = q; /* the engine knows its queue (buildOutfixes sets it) */
        memcpy(eng.data(), &hdr, sizeof(hdr));
        infos[q].nfaOffset = blob.add(eng.data(), eng.size(), 64);
        if (hdr.flags & NFA_ACCEPTS_EOD) {
            eodQueues.push_back(q);
        }
    }
    RoseEngine r;
    memset(&r, 0, sizeof(r));
    r.runtimeImpl = RUNTIME_FULL_ROSE;
    r.canExhaust = t.canExhaust ? 1 : 0;
    r.mode = MODE_BLOCK;
    r.ekeyCount = t.ekeyCount;
    r.dkeyCount = t.dkeyCount;
    r.dkeyLogSize = fatbitSize(r.dkeyCount);
    r.invDkeyOffset = t.invDkeyOffset;
    r.somLocationFatbitSize = fatbitSize(0);
    r.activeArrayCount = n;
    r.queueCount = n;
    r.activeQueueArraySize = fatbitSize(n);
    r.handledKeyFatbitSize = fatbitSize(0);
    r.minWidth = t.minLen;
    r.minWidthExcludingBoundaries = t.minLen;
    r.maxBiAnchoredWidth = ROSE_BOUND_INF;
    r.floatingDistance = ROSE_BOUND_INF;
    r.delay_fatbit_size = fatbitSize(0);
    r.anchored_fatbit_size = fatbitSize(0);
    r.outfixBeginQueue = 0;
    r.outfixEndQueue = n;
    r.leftfixBeginQueue = n;
    r.initMpvNfa = 0xffffffffu;
    r.hasOutfixesInSmallBlock = 1; /* hasNonSmallBlockOutfix: none of them is in a small-block matcher */
    if (!eodQueues.empty()) {
        const std::vector<MmbitSparseIter> it = sparseIterator(eodQueues, n);
        const u32 iterOffset = blob.add(it.data(), it.size() * sizeof(MmbitSparseIter), 8);
        const u32 sz = instrSize<InstrEnginesEod>() + instrSize<InstrEnd>();
        const u32 pc = blob.reserve(sz, INSTR_ALIGN);
        InstrEnginesEod ee;
        memset(&ee, 0, sizeof(ee));
        ee.code = OP_ENGINES_EOD;
        ee.iter_offset = iterOffset;
        memcpy(blob.at(pc), &ee, sizeof(ee));
        InstrEnd e;
        e.code = OP_END;
        memcpy(blob.at(pc + instrSize<InstrEnginesEod>()), &e, sizeof(e));
        r.eodProgramOffset = pc;
        r.requiresEodCheck = 1;
    }
    StateOffsets &so = r.stateOffsets;
    u32 cur = 1; /* status byte; no roles */
    so.activeLeafArray = cur;
    so.activeLeafArray_size = mmbitSize(n);
    cur += so.activeLeafArray_size;
    so.activeLeftArray = so.longLitState = so.leftfixLagTable = so.anchorState = cur;
    so.groups = cur;
    so.groups_size = 0;
    so.history = cur;
    so.exhausted = cur;
    so.exhausted_size = mmbitSize(r.ekeyCount);
    cur += so.exhausted_size;
    so.logicalVec = so.combVec = cur;
    so.nfaStateBegin = cur;
    /* allocateStateSpace (:2078-2099): stream state packed after rose's, full state in scratch, aligned */
    u32 full = 0;
    for (u32 q = 0; q < n; q++) {
        NFA hdr;
        memcpy(&hdr, engines[q].data(), sizeof(hdr));
        infos[q].stateOffset = cur;
        cur += hdr.streamStateSize;
        full = HSB_ROUNDUP(full, engineStateAlign(hdr.type));
        infos[q].fullStateOffset = full;
        full += hdr.scratchStateSize;
    }
    so.end = cur;
    r.stateSize = cur;
    r.scratchStateSize = full;
    r.nfaInfoOffset = blob.add(infos.data(), infos.size() * sizeof(NfaInfo), 4);
    const u32 total = (u32)HSB_ROUNDUP(blob.base + blob.bytes.size(), 64);
    r.size = total;
    std::vector<u8> out(total, 0);
    memcpy(out.data(), &r, sizeof(r));
    memcpy(out.data() + blob.base, blob.bytes.data(), blob.bytes.size());
    return out;
}

/* An expression of a set, with its report programs, and whether its own automaton determinises within 1 024 states */
struct RegexMember {
    const RegexPattern *p;
    u32 report, reportBeforeNewline;
    bool ownDfa;
};

/* The engines of a set whose expressions do not fit one automaton.  DFA groups first, since the DFA kernels scan
 * several times faster than the wide LimEx models: in input order, a group takes the next expression while their
 * union still determinises within 1 024 states.  The expressions whose own DFA is larger go to LimEx groups, each
 * filled up to the 512-state model.  regexDfa = false: LimEx groups only. */
std::vector<std::vector<u8>> partitionEngines(const std::vector<RegexMember> &members, bool regexDfa) {
    std::vector<std::vector<u8>> engines;
    auto add = [](RawNfa *nfa, const RegexMember &m) -> bool { /* false: the automaton would outgrow the model */
        RawNfa trial = *nfa;
        try {
            regexNfaAdd(&trial, m.p->re.c_str(), m.p->flags, m.report, m.reportBeforeNewline, m.p->minLength);
        } catch (const RegexError &) {
            return false;
        }
        *nfa = std::move(trial);
        return true;
    };
    std::vector<const RegexMember *> nfaOnly;
    RawNfa group;
    RawDfa groupDfa;
    u32 count = 0;
    auto closeDfa = [&]() {
        if (count) {
            minimizeDfa(&groupDfa);
            engines.push_back(emitDfa(groupDfa, groupDfa.size() <= 256 ? DFA_MCCLELLAN8 : DFA_MCCLELLAN16, true));
        }
        regexNfaInit(&group);
        count = 0;
    };
    regexNfaInit(&group);
    for (const RegexMember &m : members) {
        if (!regexDfa || !m.ownDfa) {
            nfaOnly.push_back(&m);
            continue;
        }
        RawNfa trial = group;
        RawDfa d;
        if (add(&trial, m) && determinize(trial, 1024, &d)) {
            group = std::move(trial);
            groupDfa = std::move(d);
            count++;
            continue;
        }
        closeDfa();
        if (add(&group, m) && determinize(group, 1024, &groupDfa)) {
            count = 1;
        } else {
            regexNfaInit(&group);
            nfaOnly.push_back(&m);
        }
    }
    closeDfa();
    for (const RegexMember *m : nfaOnly) {
        if (add(&group, *m)) {
            count++;
            continue;
        }
        engines.push_back(emitLimEx(group));
        regexNfaInit(&group);
        count = 0;
        if (!add(&group, *m)) {
            throw std::runtime_error("an expression outgrows the NFA model on its own");
        }
        count = 1;
    }
    if (count) {
        engines.push_back(emitLimEx(group));
    }
    return engines;
}

/* Floating literal matcher + RoseEngine header around a finished program blob. */
std::vector<u8> finishRose(Blob &blob, const std::vector<HwlmLit> &hl, const RoseTail &t,
                           const CompileOpts &opts, HwlmBuildInfo *info) {
    std::vector<u8> hwlm;
    try {
        hwlm = buildHwlm(hl, opts.hwlm, info);
    } catch (const std::runtime_error &e) {
        throw CompileError{std::string("Unable to build literal matcher: ") + e.what(), -1};
    }
    const u32 fmatcherOffset = blob.add(hwlm.data(), hwlm.size(), 64);
    const u32 total = (u32)HSB_ROUNDUP(blob.base + blob.bytes.size(), 64);

    /* --- header --- */
    RoseEngine r;
    memset(&r, 0, sizeof(r));
    r.pureLiteral = opts.pureLiteralApi ? 1 : 0;
    r.runtimeImpl = RUNTIME_PURE_LITERAL;
    r.canExhaust = t.canExhaust ? 1 : 0;
    /* src/rose/rose_build_bytecode.cpp:3615-3622 */
    r.mode = !opts.streaming ? MODE_BLOCK : opts.vectored ? MODE_VECTORED : MODE_STREAM;
    /* matches may start in earlier writes: keep the last maxLen-1 bytes
     * (calcHistoryRequired, src/rose/rose_build_misc.cpp; updated by HWLM) */
    const u32 historyRequired = opts.streaming && t.maxLen > 1 ? t.maxLen - 1 : 0;
    r.historyRequired = historyRequired;
    r.ekeyCount = t.ekeyCount;
    r.dkeyCount = t.dkeyCount;
    r.dkeyLogSize = fatbitSize(r.dkeyCount);
    r.invDkeyOffset = t.invDkeyOffset;
    r.somLocationFatbitSize = fatbitSize(0);
    r.fmatcherOffset = fmatcherOffset;
    r.smallWriteOffset = t.smallWriteOffset;
    r.fmatcherMinWidth = t.minLen;
    r.activeQueueArraySize = fatbitSize(0);
    r.handledKeyFatbitSize = fatbitSize(0);
    r.minWidth = t.minLen;
    r.minWidthExcludingBoundaries = t.minLen;
    r.maxBiAnchoredWidth = ROSE_BOUND_INF;
    r.floatingDistance = ROSE_BOUND_INF;
    r.floatingMinLiteralMatchOffset = t.minLen;
    r.initialGroups = 1;
    r.floating_group_mask = 1;
    r.size = total;
    r.delay_fatbit_size = fatbitSize(0);
    r.anchored_fatbit_size = fatbitSize(0);
    r.totalNumLiterals = (u32)hl.size();
    r.initMpvNfa = 0xffffffffu; /* MO_INVALID_IDX: no MPV outfix */
    StateOffsets &so = r.stateOffsets;
    u32 cur = 1;                 /* status byte; role multibit is empty */
    so.activeLeafArray = so.activeLeftArray = so.longLitState = cur;
    so.leftfixLagTable = so.anchorState = cur;
    so.groups = cur;
    so.groups_size = 1;
    cur += so.groups_size;
    so.history = cur;
    cur += historyRequired;
    so.exhausted = cur;
    so.exhausted_size = mmbitSize(r.ekeyCount);
    cur += so.exhausted_size;
    so.logicalVec = so.combVec = cur;
    so.nfaStateBegin = so.end = cur;

    std::vector<u8> out(total, 0);
    memcpy(out.data(), &r, sizeof(r));
    memcpy(out.data() + blob.base, blob.bytes.data(), blob.bytes.size());
    return out;
}

} // namespace

/* mmbBuildSparseIterator (src/util/multibit_build.cpp:156-190): one record per node of the multibit's 64-ary tree
 * that holds a key, level by level, each level in key order.  A record's mask has the bits of its children; its val
 * is where those children's records start, on the last level the count of keys before it. */
std::vector<MmbitSparseIter> sparseIterator(const std::vector<u32> &keys, u32 totalBits) {
    u32 ks = 0; /* mmbit_keyshift: 6 bits per level below the root */
    for (u64 cap = 64; totalBits > 1 && cap < totalBits; cap <<= 6) {
        ks += 6;
    }
    std::vector<MmbitSparseIter> out;
    std::vector<size_t> levelStart;
    for (u32 d = 0; d * 6 <= ks; d++) {
        levelStart.push_back(out.size());
        std::map<u32, u64> nodes; /* path above the level -> mask */
        for (u32 k : keys) {
            nodes[(u32)((u64)k >> (ks - 6 * d + 6))] |= 1ull << ((k >> (ks - 6 * d)) & 63);
        }
        for (const auto &n : nodes) {
            MmbitSparseIter it;
            memset(&it, 0, sizeof(it));
            it.mask = n.second;
            out.push_back(it);
        }
    }
    levelStart.push_back(out.size());
    for (size_t l = 0; l + 1 < levelStart.size(); l++) {
        const bool last = l + 2 == levelStart.size();
        u32 population = 0;
        for (size_t i = levelStart[l]; i < levelStart[l + 1]; i++) {
            out[i].val = (last ? 0 : (u32)levelStart[l + 1]) + population;
            population += (u32)__builtin_popcountll(out[i].mask);
        }
    }
    return out;
}

std::vector<u8> buildLiteralRose(const std::vector<LitPattern> &patsIn,
                                 const CompileOpts &opts, HwlmBuildInfo *info) {
    if (patsIn.empty()) {
        throw CompileError{"Invalid parameter: elements is zero", -1};
    }
    if (patsIn.size() > LIMIT_LITERAL_COUNT) {
        throw CompileError{"Number of patterns too large", -1};
    }

    /* --- validate, fold case, drop exact duplicates, assign ekeys/dkeys --- */
    std::vector<PatInfo> pats;
    std::map<u32, std::pair<bool, u32>> idHighlander; /* report -> (flag, first index) */
    std::set<std::tuple<std::string, bool, u32>> seen;
    for (const LitPattern &p : patsIn) {
        if (p.s.empty()) {
            throw CompileError{"Pure literal API doesn't support empty string.", (int)p.index};
        }
        if (p.s.size() > LIMIT_PATTERN_LENGTH) {
            throw CompileError{"Pattern length exceeds limit.", (int)p.index};
        }
        if (p.s.size() > LIMIT_LITERAL_LENGTH) {
            throw CompileError{"Resource limit exceeded.", (int)p.index};
        }
        if (opts.streaming && p.s.size() > 8) {
            /* in streaming mode literals beyond the literal matcher's 8 bytes need
             * the long-literal table and the full rose runtime
             * (src/rose/rose_build_bytecode.cpp:292-296 isPureFloating) */
            throw CompileError{"Streaming and vectored modes in this build support literals of up to 8 "
                               "bytes; longer literals need the long literal table.", (int)p.index};
        }
        auto it = idHighlander.find(p.report);
        if (it == idHighlander.end()) {
            idHighlander[p.report] = {p.singlematch, p.index};
        } else if (it->second.first != p.singlematch) {
            std::string m = "Expression (index " + std::to_string(p.index) +
                            ") with match ID " + std::to_string(p.report) + " ";
            m += p.singlematch ? "specified " : "did not specify ";
            m += "HS_FLAG_SINGLEMATCH whereas previous expression (index " +
                 std::to_string(it->second.second) + ") with the same match ID did";
            m += p.singlematch ? " not." : ".";
            throw CompileError{m, (int)p.index};
        }
        PatInfo pi;
        pi.p = &p;
        pi.folded = p.s;
        pi.anyAlpha = false;
        for (char &c : pi.folded) {
            if (isAsciiAlpha((u8)c)) {
                pi.anyAlpha = true;
                if (p.caseless) {
                    c = (char)asciiUpper((u8)c);
                }
            }
        }
        bool effNocase = p.caseless && pi.anyAlpha;
        if (!seen.insert(std::make_tuple(pi.folded, effNocase, p.report)).second) {
            continue; /* identical literal + report: one report source */
        }
        pi.ekey = pi.dkey = INVALID_EKEY;
        pats.push_back(pi);
    }
    std::map<u32, u32> perReport;
    for (const auto &pi : pats) {
        perReport[pi.p->report]++;
    }
    std::map<u32, u32> ekeys, dkeys;
    bool allHighlander = true;
    for (auto &pi : pats) {
        const u32 r = pi.p->report;
        if (pi.p->singlematch) {
            auto it = ekeys.find(r);
            if (it == ekeys.end()) {
                it = ekeys.emplace(r, (u32)ekeys.size()).first;
            }
            pi.ekey = it->second;
        } else {
            allHighlander = false;
        }
        if (perReport[r] > 1) {
            auto it = dkeys.find(r);
            if (it == dkeys.end()) {
                it = dkeys.emplace(r, (u32)dkeys.size()).first;
            }
            pi.dkey = it->second;
        }
    }

    if (opts.outfixKind) {
        /* --- single-outfix database: report programs ([CHECK_EXHAUSTED] [DEDUPE] REPORT_EXHAUST |
         * DEDUPE_AND_REPORT | REPORT, END -- run by roseReportAdaptor / roseRunProgram), one engine
         * over the whole literals whose reports are those programs' offsets --- */
        if (opts.streaming) {
            throw CompileError{"Single-engine databases are built for block mode only.", -1};
        }
        Blob blob((u32)HSB_ROUNDUP(sizeof(RoseEngine), 64));
        std::vector<DfaLiteral> dl;
        u32 minLen = ~0u, maxLen = 0;
        for (const PatInfo &pi : pats) {
            minLen = std::min<u32>(minLen, (u32)pi.p->s.size());
            maxLen = std::max<u32>(maxLen, (u32)pi.p->s.size());
            const u32 sz = blockSize(pi) - (pi.p->s.size() > 8 ? instrSize<InstrCheckLit>() : 0) + instrSize<InstrEnd>();
            u32 pc = blob.reserve(sz, INSTR_ALIGN);
            const u32 prog = pc, endAt = pc + sz - instrSize<InstrEnd>();
            if (pi.ekey != INVALID_EKEY) {
                InstrCheckExhausted ce;
                memset(&ce, 0, sizeof(ce));
                ce.code = OP_CHECK_EXHAUSTED;
                ce.ekey = pi.ekey;
                ce.fail_jump = endAt - pc;
                memcpy(blob.at(pc), &ce, sizeof(ce));
                pc += instrSize<InstrCheckExhausted>();
                if (pi.dkey != INVALID_DKEY) {
                    InstrDedupe dd;
                    memset(&dd, 0, sizeof(dd));
                    dd.code = OP_DEDUPE;
                    dd.dkey = pi.dkey;
                    dd.fail_jump = endAt - pc;
                    memcpy(blob.at(pc), &dd, sizeof(dd));
                    pc += instrSize<InstrDedupe>();
                }
                InstrReportExhaust re;
                memset(&re, 0, sizeof(re));
                re.code = OP_REPORT_EXHAUST;
                re.onmatch = pi.p->report;
                re.ekey = pi.ekey;
                memcpy(blob.at(pc), &re, sizeof(re));
            } else if (pi.dkey != INVALID_DKEY) {
                InstrDedupeAndReport dr;
                memset(&dr, 0, sizeof(dr));
                dr.code = OP_DEDUPE_AND_REPORT;
                dr.dkey = pi.dkey;
                dr.onmatch = pi.p->report;
                dr.fail_jump = endAt - pc;
                memcpy(blob.at(pc), &dr, sizeof(dr));
            } else {
                InstrReport rr;
                memset(&rr, 0, sizeof(rr));
                rr.code = OP_REPORT;
                rr.onmatch = pi.p->report;
                memcpy(blob.at(pc), &rr, sizeof(rr));
            }
            InstrEnd e;
            e.code = OP_END;
            memcpy(blob.at(endAt), &e, sizeof(e));
            DfaLiteral l;
            l.s = pi.p->s;
            l.caseless = pi.p->caseless && pi.anyAlpha;
            l.report = prog;
            dl.push_back(l);
        }
        RoseTail t;
        t.minLen = minLen;
        t.maxLen = maxLen;
        t.ekeyCount = (u32)ekeys.size();
        t.dkeyCount = (u32)dkeys.size();
        t.invDkeyOffset = 0;
        if (!dkeys.empty()) {
            std::vector<u32> inv(dkeys.size());
            for (const auto &d : dkeys) {
                inv[d.second] = d.first;
            }
            t.invDkeyOffset = blob.add(inv.data(), inv.size() * sizeof(u32), 4);
        }
        t.canExhaust = allHighlander;
        std::vector<u8> nfa;
        try {
            if (opts.outfixKind == OUTFIX_LIMEX32) {
                nfa = emitLimEx(nfaFromLiterals(dl));
            } else {
                const DfaKind k = opts.outfixKind == OUTFIX_MCCLELLAN8    ? DFA_MCCLELLAN8
                                  : opts.outfixKind == OUTFIX_MCCLELLAN16 ? DFA_MCCLELLAN16
                                  : opts.outfixKind == OUTFIX_SHENG       ? DFA_SHENG
                                                                          : DFA_AUTO;
                nfa = emitDfa(dfaFromLiterals(dl, false), k, false);
            }
        } catch (const std::runtime_error &e) {
            throw CompileError{std::string("Unable to build the engine: ") + e.what(), -1};
        }
        if (info) {
            memset(info, 0, sizeof(*info));
        }
        return finishOutfixRose(blob, nfa, t, opts);
    }

    /* --- group into fragments by (8-byte suffix, effective nocase) --- */
    struct Fragment {
        std::string suffix;
        bool nocase;
        std::vector<u32> pats;
        u32 program = 0;
    };
    std::vector<Fragment> frags;
    std::map<std::pair<std::string, bool>, u32> fragIndex;
    u32 minLen = ~0u;
    for (u32 i = 0; i < pats.size(); i++) {
        const std::string &f = pats[i].folded;
        minLen = std::min<u32>(minLen, (u32)f.size());
        std::string suf = f.size() > 8 ? f.substr(f.size() - 8) : f;
        bool nc = false;
        if (pats[i].p->caseless) {
            for (char c : suf) {
                nc |= isAsciiAlpha((u8)c);
            }
        }
        auto key = std::make_pair(suf, nc);
        auto it = fragIndex.find(key);
        if (it == fragIndex.end()) {
            it = fragIndex.emplace(key, (u32)frags.size()).first;
            frags.push_back({suf, nc, {}, 0});
        }
        frags[it->second].pats.push_back(i);
    }

    /* --- programs --- */
    const u32 blobBase = (u32)HSB_ROUNDUP(sizeof(RoseEngine), 64);
    Blob blob(blobBase);
    struct PendingLit {
        u32 instrOff;
        std::string bytes;
    };
    std::vector<PendingLit> pendingLits;
    for (Fragment &fr : frags) {
        u32 total = instrSize<InstrEnd>();
        for (u32 pi : fr.pats) {
            total += blockSize(pats[pi]);
        }
        const u32 start = blob.reserve(total, INSTR_ALIGN);
        fr.program = start;
        u32 pc = start;
        for (size_t k = 0; k < fr.pats.size(); k++) {
            const PatInfo &pi = pats[fr.pats[k]];
            const u32 next = pc + blockSize(pi); /* next pattern's block or END */
            const u32 report = pi.p->report;
            if (pi.p->s.size() > 8) {
                InstrCheckLit in;
                memset(&in, 0, sizeof(in));
                bool nc = pi.p->caseless && pi.anyAlpha;
                in.code = nc ? OP_CHECK_MED_LIT_NOCASE : OP_CHECK_MED_LIT;
                in.lit_length = (u32)pi.folded.size();
                in.fail_jump = next - pc;
                memcpy(blob.at(pc), &in, sizeof(in));
                pendingLits.push_back({pc, pi.folded});
                pc += instrSize<InstrCheckLit>();
            }
            if (pi.ekey != INVALID_EKEY) {
                InstrCheckExhausted ce;
                memset(&ce, 0, sizeof(ce));
                ce.code = OP_CHECK_EXHAUSTED;
                ce.ekey = pi.ekey;
                ce.fail_jump = next - pc;
                memcpy(blob.at(pc), &ce, sizeof(ce));
                pc += instrSize<InstrCheckExhausted>();
                if (pi.dkey != INVALID_DKEY) {
                    InstrDedupe d;
                    memset(&d, 0, sizeof(d));
                    d.code = OP_DEDUPE;
                    d.dkey = pi.dkey;
                    d.fail_jump = next - pc;
                    memcpy(blob.at(pc), &d, sizeof(d));
                    pc += instrSize<InstrDedupe>();
                }
                InstrReportExhaust re;
                memset(&re, 0, sizeof(re));
                re.code = OP_REPORT_EXHAUST;
                re.onmatch = report;
                re.ekey = pi.ekey;
                memcpy(blob.at(pc), &re, sizeof(re));
                pc += instrSize<InstrReportExhaust>();
            } else if (pi.dkey != INVALID_DKEY) {
                InstrDedupeAndReport dr;
                memset(&dr, 0, sizeof(dr));
                dr.code = OP_DEDUPE_AND_REPORT;
                dr.dkey = pi.dkey;
                dr.onmatch = report;
                dr.fail_jump = next - pc;
                memcpy(blob.at(pc), &dr, sizeof(dr));
                pc += instrSize<InstrDedupeAndReport>();
            } else {
                InstrReport r;
                memset(&r, 0, sizeof(r));
                r.code = OP_REPORT;
                r.onmatch = report;
                memcpy(blob.at(pc), &r, sizeof(r));
                pc += instrSize<InstrReport>();
            }
        }
        InstrEnd e;
        e.code = OP_END;
        memcpy(blob.at(pc), &e, sizeof(e));
    }
    for (const PendingLit &pl : pendingLits) {
        u32 off = blob.add(pl.bytes.data(), pl.bytes.size(), 1);
        InstrCheckLit in;
        memcpy(&in, blob.at(pl.instrOff), sizeof(in));
        in.lit_offset = off;
        memcpy(blob.at(pl.instrOff), &in, sizeof(in));
    }

    /* --- dkey -> external report id table (rose_internal.h:354) --- */
    u32 invDkeyOffset = 0;
    if (!dkeys.empty()) {
        std::vector<u32> inv(dkeys.size());
        for (const auto &d : dkeys) {
            inv[d.second] = d.first;
        }
        invDkeyOffset = blob.add(inv.data(), inv.size() * sizeof(u32), 4);
    }

    /* --- floating literal matcher --- */
    std::vector<HwlmLit> hl;
    for (const Fragment &fr : frags) {
        HwlmLit l;
        l.s = fr.suffix;
        l.nocase = fr.nocase;
        l.noruns = false;
        l.id = fr.program;
        l.groups = 1;
        hl.push_back(l);
    }
    u32 maxLen = 0;
    for (const auto &pi : pats) {
        maxLen = std::max<u32>(maxLen, (u32)pi.folded.size());
    }
    RoseTail t;
    t.minLen = minLen;
    t.maxLen = maxLen;
    t.ekeyCount = (u32)ekeys.size();
    t.dkeyCount = (u32)dkeys.size();
    t.invDkeyOffset = invDkeyOffset;
    t.canExhaust = allHighlander;

    /* --- small-write engine (src/smallwrite/smallwrite_build.cpp; used by hs_scan for
     * buffers shorter than largestBuffer, src/runtime.c:401-413): one DFA over the WHOLE
     * literals whose reports are the offsets of report programs -- the literal's program
     * without the literal check, which the DFA has already done -- run through
     * roseReportAdaptor (src/rose/match.c:611-633).  Only while the automaton stays small
     * (12 000 literal bytes, 16 K states); otherwise no engine, like the reference when its
     * DFA limits are exceeded. --- */
    if (opts.smallWrite && !opts.streaming) {
        const u32 LARGEST_BUFFER = 70; /* Grey::smallWriteLargestBuffer, src/grey.cpp:135 */
        std::vector<DfaLiteral> dl;
        size_t budget = 0;
        bool ok = true;
        for (const PatInfo &pi : pats) {
            if (pi.p->s.size() >= LARGEST_BUFFER) {
                continue; /* cannot match in a buffer that short */
            }
            const bool nc = pi.p->caseless && pi.anyAlpha;
            budget += pi.p->s.size();
            if (budget > 12000) { /* positions of the automaton; it may still grow past 16 K states */
                ok = false;
                break;
            }
            /* report program: [CHECK_EXHAUSTED] [DEDUPE] REPORT_EXHAUST | DEDUPE_AND_REPORT | REPORT, END */
            const u32 sz = blockSize(pi) - (pi.p->s.size() > 8 ? instrSize<InstrCheckLit>() : 0) + instrSize<InstrEnd>();
            u32 pc = blob.reserve(sz, INSTR_ALIGN);
            const u32 prog = pc, endAt = pc + sz - instrSize<InstrEnd>();
            if (pi.ekey != INVALID_EKEY) {
                InstrCheckExhausted ce;
                memset(&ce, 0, sizeof(ce));
                ce.code = OP_CHECK_EXHAUSTED;
                ce.ekey = pi.ekey;
                ce.fail_jump = endAt - pc;
                memcpy(blob.at(pc), &ce, sizeof(ce));
                pc += instrSize<InstrCheckExhausted>();
                if (pi.dkey != INVALID_DKEY) {
                    InstrDedupe dd;
                    memset(&dd, 0, sizeof(dd));
                    dd.code = OP_DEDUPE;
                    dd.dkey = pi.dkey;
                    dd.fail_jump = endAt - pc;
                    memcpy(blob.at(pc), &dd, sizeof(dd));
                    pc += instrSize<InstrDedupe>();
                }
                InstrReportExhaust re;
                memset(&re, 0, sizeof(re));
                re.code = OP_REPORT_EXHAUST;
                re.onmatch = pi.p->report;
                re.ekey = pi.ekey;
                memcpy(blob.at(pc), &re, sizeof(re));
            } else if (pi.dkey != INVALID_DKEY) {
                InstrDedupeAndReport dr;
                memset(&dr, 0, sizeof(dr));
                dr.code = OP_DEDUPE_AND_REPORT;
                dr.dkey = pi.dkey;
                dr.onmatch = pi.p->report;
                dr.fail_jump = endAt - pc;
                memcpy(blob.at(pc), &dr, sizeof(dr));
            } else {
                InstrReport rr;
                memset(&rr, 0, sizeof(rr));
                rr.code = OP_REPORT;
                rr.onmatch = pi.p->report;
                memcpy(blob.at(pc), &rr, sizeof(rr));
            }
            InstrEnd e;
            e.code = OP_END;
            memcpy(blob.at(endAt), &e, sizeof(e));
            DfaLiteral l;
            l.s = pi.p->s;
            l.caseless = nc;
            l.report = prog;
            dl.push_back(l);
        }
        if (ok && !dl.empty()) {
            try {
                const std::vector<u8> nfa = emitDfa(dfaFromLiterals(dl, false), DFA_AUTO, false);
                SmallWriteEngine sw;
                memset(&sw, 0, sizeof(sw));
                sw.largestBuffer = LARGEST_BUFFER;
                sw.start_offset = 0;
                sw.size = (u32)(sizeof(SmallWriteEngine) + nfa.size());
                t.smallWriteOffset = blob.add(&sw, sizeof(sw), 64);
                blob.add(nfa.data(), nfa.size(), 64);
            } catch (const std::runtime_error &) {
                /* automaton too large: no small-write engine */
            }
        }
    }
    return finishRose(blob, hl, t, opts, info);
}

std::vector<u8> buildRegexRose(const std::vector<RegexPattern> &pats, const CompileOpts &opts) {
    if (pats.empty()) {
        throw CompileError{"Invalid parameter: elements is zero", -1};
    }
    if (opts.streaming) {
        throw CompileError{"Expressions that need an NFA engine are compiled for block mode only in this build.", -1};
    }
    /* report keys: one exhaustion key per HS_FLAG_SINGLEMATCH report id; one dedupe key per report
     * id, always -- several accepting positions (or expressions) may raise one id at one offset and
     * the reference delivers a report once (dedupe, src/report.h:55-119) */
    std::map<u32, std::pair<bool, u32>> highlander;
    std::map<u32, u32> ekeys, dkeys;
    bool allHighlander = true;
    for (const RegexPattern &p : pats) {
        const bool single = (p.flags & HS_FLAG_SINGLEMATCH) != 0;
        auto it = highlander.find(p.report);
        if (it == highlander.end()) {
            highlander[p.report] = {single, p.index};
        } else if (it->second.first != single) {
            std::string m = "Expression (index " + std::to_string(p.index) + ") with match ID " +
                            std::to_string(p.report) + " ";
            m += single ? "specified " : "did not specify ";
            m += "HS_FLAG_SINGLEMATCH whereas previous expression (index " + std::to_string(it->second.second) +
                 ") with the same match ID did";
            m += single ? " not." : ".";
            throw CompileError{m, (int)p.index};
        }
        if (single) {
            ekeys.emplace(p.report, (u32)ekeys.size());
        } else {
            allHighlander = false;
        }
        dkeys.emplace(p.report, (u32)dkeys.size());
    }
    Blob blob((u32)HSB_ROUNDUP(sizeof(RoseEngine), 64));
    RawNfa nfa;
    regexNfaInit(&nfa);
    u32 minLen = ~0u;
    std::map<std::tuple<u32, int, u64, u64>, u32> progOf; /* (report id, offset_adjust, bounds) -> its report program */
    auto program = [&](const RegexPattern &p, int adjust) -> u32 {
        const auto key = std::make_tuple(p.report, adjust, p.minOffset, p.maxOffset);
        auto pit = progOf.find(key);
        if (pit != progOf.end()) {
            return pit->second;
        }
        const bool single = (p.flags & HS_FLAG_SINGLEMATCH) != 0;
        const bool bounded = p.minOffset > 0 || p.maxOffset != ~0ull;
        u32 sz = instrSize<InstrEnd>() + (bounded ? instrSize<InstrCheckBounds>() : 0);
        sz += single ? instrSize<InstrCheckExhausted>() + instrSize<InstrDedupe>() + instrSize<InstrReportExhaust>()
                     : instrSize<InstrDedupeAndReport>();
        u32 pc = blob.reserve(sz, INSTR_ALIGN);
        const u32 prog = pc;
        const u32 endAt = pc + sz - instrSize<InstrEnd>();
        if (bounded) {
            /* makeReport (src/rose/rose_build_program.cpp:533-538): the bounds come first, and they are on the raw
             * match end -- min_offset / max_offset less the report's offset_adjust (ng_extparam.cpp:199-211) */
            InstrCheckBounds cb;
            memset(&cb, 0, sizeof(cb));
            cb.code = OP_CHECK_BOUNDS;
            cb.min_bound = p.minOffset - (u64)(long long)adjust;
            cb.max_bound = p.maxOffset == ~0ull ? ~0ull : p.maxOffset - (u64)(long long)adjust;
            cb.fail_jump = endAt - pc;
            memcpy(blob.at(pc), &cb, sizeof(cb));
            pc += instrSize<InstrCheckBounds>();
        }
        if (single) {
            InstrCheckExhausted ce;
            memset(&ce, 0, sizeof(ce));
            ce.code = OP_CHECK_EXHAUSTED;
            ce.ekey = ekeys[p.report];
            ce.fail_jump = endAt - pc;
            memcpy(blob.at(pc), &ce, sizeof(ce));
            pc += instrSize<InstrCheckExhausted>();
            InstrDedupe dd;
            memset(&dd, 0, sizeof(dd));
            dd.code = OP_DEDUPE;
            dd.dkey = dkeys[p.report];
            dd.offset_adjust = adjust;
            dd.fail_jump = endAt - pc;
            memcpy(blob.at(pc), &dd, sizeof(dd));
            pc += instrSize<InstrDedupe>();
            InstrReportExhaust re;
            memset(&re, 0, sizeof(re));
            re.code = OP_REPORT_EXHAUST;
            re.onmatch = p.report;
            re.offset_adjust = adjust;
            re.ekey = ekeys[p.report];
            memcpy(blob.at(pc), &re, sizeof(re));
        } else {
            InstrDedupeAndReport dr;
            memset(&dr, 0, sizeof(dr));
            dr.code = OP_DEDUPE_AND_REPORT;
            dr.dkey = dkeys[p.report];
            dr.onmatch = p.report;
            dr.offset_adjust = adjust;
            dr.fail_jump = endAt - pc;
            memcpy(blob.at(pc), &dr, sizeof(dr));
        }
        InstrEnd e;
        e.code = OP_END;
        memcpy(blob.at(endAt), &e, sizeof(e));
        progOf[key] = prog;
        return prog;
    };
    std::vector<RegexMember> members;
    bool overflow = false; /* the set's positions exceed one automaton: it is split into several engines */
    for (const RegexPattern &p : pats) {
        try {
            const RegexInfo ri = regexInfo(p.re.c_str(), p.flags);
            /* extended parameters no match can satisfy (src/nfagraph/ng_extparam.cpp:820-880) */
            if (p.minLength && ri.maxLen != 0xffffffffu && p.minLength > ri.maxLen) {
                throw CompileError{"Expression has min_length=" + std::to_string(p.minLength) + " but can only produce matches of length " +
                                       std::to_string(ri.maxLen) + " bytes at most.", (int)p.index};
            }
            if (p.maxOffset != ~0ull && ri.minLen > p.maxOffset) {
                throw CompileError{"Expression has max_offset=" + std::to_string(p.maxOffset) + " but requires " +
                                       std::to_string(ri.minLen) + " bytes to match.", (int)p.index};
            }
            if (ri.anchored && p.minOffset && ri.maxLen != 0xffffffffu && p.minOffset > ri.maxLen) {
                throw CompileError{"Expression is anchored and cannot satisfy min_offset=" + std::to_string(p.minOffset) +
                                       " as it can only produce matches of length " + std::to_string(ri.maxLen) + " bytes at most.",
                                   (int)p.index};
            }
            if (p.minLength || p.maxOffset != ~0ull) {
                /* ... and taken together: some alternative must have a match that is long enough and can end early
                 * enough (the reference prunes the graph by the parameters and reports what is left) */
                bool some = false;
                for (const auto &w : ri.armWidths) {
                    some |= (w.second == 0xffffffffu || w.second >= p.minLength) &&
                            std::max<u64>(w.first, p.minLength) <= p.maxOffset;
                }
                if (!some) {
                    throw CompileError{"Extended parameter constraints can not be satisfied for any match from this "
                                       "expression.", (int)p.index};
                }
            }
            bool ownDfa = false;
            {
                /* "Pattern can never match." (can_never_match after resolveAsserts, src/nfagraph/ng.cpp:330-350): the
                 * expression's own automaton, determinised and minimised, is the dead state alone */
                RawNfa own;
                regexNfaInit(&own);
                regexNfaAdd(&own, p.re.c_str(), p.flags, 1, ri.needsAdjust ? 2 : 0, p.minLength);
                RawDfa d;
                ownDfa = determinize(own, 1024, &d);
                if (ownDfa) {
                    minimizeDfa(&d);
                    if (d.size() < 2) {
                        throw CompileError{"Pattern can never match.", (int)p.index};
                    }
                }
            }
            minLen = std::min<u32>(minLen, (u32)std::max<u64>(ri.minLen, std::min<u64>(p.minLength, 0xffffffffu)));
            if (!overflow) {
                try {
                    regexNfaAdd(&nfa, p.re.c_str(), p.flags, program(p, 0), ri.needsAdjust ? program(p, -1) : 0, p.minLength);
                } catch (const RegexError &) {
                    overflow = true; /* the expression alone fits (its own automaton was built above): the set does not */
                }
            }
            const u32 report = program(p, 0); /* (made above while the set fits: the same programs) */
            members.push_back({&p, report, ri.needsAdjust ? program(p, -1) : 0, ownDfa});
        } catch (const RegexError &e) {
            throw CompileError{e.msg, (int)p.index};
        }
    }
    RoseTail t;
    t.minLen = minLen;
    t.maxLen = 0;
    t.ekeyCount = (u32)ekeys.size();
    t.dkeyCount = (u32)dkeys.size();
    std::vector<u32> inv(dkeys.size());
    for (const auto &d : dkeys) {
        inv[d.second] = d.first;
    }
    t.invDkeyOffset = blob.add(inv.data(), inv.size() * sizeof(u32), 4);
    t.canExhaust = allHighlander;
    if (overflow) {
        std::vector<std::vector<u8>> engines;
        try {
            engines = partitionEngines(members, opts.regexDfa);
        } catch (const std::runtime_error &e) {
            throw CompileError{std::string("Unable to build the NFA: ") + e.what(), -1};
        }
        return finishEnginesRose(blob, engines, t);
    }
    std::vector<u8> eng;
    try {
        /* small automata run as DFAs, as in the reference (ng_mcclellan before LimEx); the report programs are
         * the same either way */
        RawDfa dfa;
        bool asDfa = opts.regexDfa && determinize(nfa, 1024, &dfa);
        if (asDfa) {
            minimizeDfa(&dfa);
            /* (nothing left but the dead state: an expression set that cannot match; it stays an NFA) */
            asDfa = dfa.size() >= 2 && dfa.size() <= 1024;
        }
        if (asDfa) {
            eng = emitDfa(dfa, dfa.size() <= 256 ? DFA_MCCLELLAN8 : DFA_MCCLELLAN16, true);
        } else {
            eng = emitLimEx(nfa);
        }
    } catch (const std::runtime_error &e) {
        throw CompileError{std::string("Unable to build the NFA: ") + e.what(), -1};
    }
    return finishOutfixRose(blob, eng, t, opts);
}

/* Test hook (hs_b200_test_compile_programs): a pure-literal block database whose
 * literal programs are given as raw instruction bytes -- the way to reach every
 * opcode of roseRunProgram_l (src/rose/program_runtime.c:3101-3522) that this
 * compiler does not emit itself.  lits[i].id = offset of its program inside
 * `area`, which is placed at programAreaBase(); absolute offsets inside the
 * programs (lit_offset, child_offset) are the caller's business. */
u32 programAreaBase() { return (u32)HSB_ROUNDUP(sizeof(RoseEngine), 64); }

std::vector<u8> buildRawProgramRose(std::vector<HwlmLit> lits, const std::vector<u8> &area,
                                    u32 ekeyCount, const std::vector<u32> &invDkey,
                                    const CompileOpts &opts, HwlmBuildInfo *info) {
    if (lits.empty()) {
        throw CompileError{"Invalid parameter: elements is zero", -1};
    }
    Blob blob(programAreaBase());
    blob.add(area.data(), area.size(), INSTR_ALIGN);
    RoseTail t;
    t.minLen = ~0u;
    t.maxLen = 0;
    for (HwlmLit &l : lits) {
        if (l.s.empty() || l.s.size() > 8 || l.id >= area.size() || (l.id % INSTR_ALIGN)) {
            throw CompileError{"bad literal or program offset", -1};
        }
        l.id += blob.base;
        t.minLen = std::min<u32>(t.minLen, (u32)l.s.size());
        t.maxLen = std::max<u32>(t.maxLen, (u32)l.s.size());
    }
    t.ekeyCount = ekeyCount;
    t.dkeyCount = (u32)invDkey.size();
    t.invDkeyOffset = invDkey.empty() ? 0 : blob.add(invDkey.data(), invDkey.size() * sizeof(u32), 4);
    t.canExhaust = false;
    return finishRose(blob, lits, t, opts, info);
}

} // namespace hsb
