/* db_walk.cpp -- see db_walk.h */
#include "db_walk.h"

#include <algorithm>
#include <cstring>

#include "api_internal.h"
#include "rose_build.h"

namespace hsb {

/* Linear walk over one literal program.  A program is a sequence of blocks, each
 * ending in END or FINAL_REPORT; later blocks are reached through the fail_jump
 * of a check in an earlier one (src/rose/rose_build_program.cpp:525-829), so
 * the walk continues past a terminator while a jump target lies beyond it.
 * Returns false on an opcode the device interpreter (scan_kernels.cu
 * runProgram) does not implement -- the state-carrying ones of
 * roseRunProgram_l: PUSH_DELAYED, CATCH_UP*, SOM_*, TRIGGER_SUFFIX, REPORT_CHAIN,
 * REPORT_SOM*, SET_LOGICAL, SET_COMBINATION, FLUSH_COMBINATION, SET_EXHAUST. */
bool outfixesOnly(const RoseEngine *r, u32 bcLen) {
    const u32 n = r->queueCount;
    const BoundaryReports &br = r->boundary;
    if (r->runtimeImpl != RUNTIME_FULL_ROSE || r->mode != MODE_BLOCK || !n || r->activeArrayCount != n ||
        r->outfixBeginQueue != 0 || r->outfixEndQueue != n || r->leftfixBeginQueue != n || !r->nfaInfoOffset ||
        r->initMpvNfa != 0xffffffffu || r->hasSom || r->somLocationCount || r->somRevCount || r->amatcherOffset ||
        r->ematcherOffset || r->fmatcherOffset || r->drmatcherOffset || r->sbmatcherOffset || r->longLitTableOffset ||
        r->smallWriteOffset || r->rolesWithStateCount || r->activeLeftCount || r->roseCount || r->rosePrefixCount ||
        r->activeLeftIterOffset || r->eagerIterOffset || r->lastByteHistoryIterOffset || r->delayProgramOffset ||
        r->anchoredProgramOffset || r->delay_count || r->anchored_count || r->handledKeyCount || r->lkeyCount ||
        r->lopCount || r->ckeyCount || r->flushCombProgramOffset || r->lastFlushCombProgramOffset ||
        br.reportEodOffset || br.reportZeroOffset || br.reportZeroEodOffset ||
        (u64)r->nfaInfoOffset + (u64)n * sizeof(NfaInfo) > bcLen) {
        return false;
    }
    const u8 *bc = (const u8 *)r;
    std::vector<u32> eod;
    for (u32 q = 0; q < n; q++) {
        NfaInfo ni;
        memcpy(&ni, bc + r->nfaInfoOffset + q * sizeof(NfaInfo), sizeof(ni));
        if ((u64)ni.nfaOffset + sizeof(NFA) > bcLen) {
            return false;
        }
        NFA nh;
        memcpy(&nh, bc + ni.nfaOffset, sizeof(nh));
        if (nh.flags & NFA_ACCEPTS_EOD) {
            eod.push_back(q);
        }
    }
    if (eod.empty() || !r->eodProgramOffset) {
        return eod.empty() && !r->eodProgramOffset;
    }
    const u32 pc = r->eodProgramOffset;
    const u32 endAt = pc + (u32)HSB_ROUNDUP(sizeof(InstrEnginesEod), INSTR_ALIGN);
    if (!r->requiresEodCheck || pc % INSTR_ALIGN || (u64)endAt + sizeof(InstrEnd) > bcLen) {
        return false;
    }
    InstrEnginesEod ee;
    memcpy(&ee, bc + pc, sizeof(ee));
    const std::vector<MmbitSparseIter> want = sparseIterator(eod, n);
    const size_t iterBytes = want.size() * sizeof(MmbitSparseIter);
    if (ee.code != OP_ENGINES_EOD || bc[endAt] != OP_END || (u64)ee.iter_offset + iterBytes > bcLen) {
        return false;
    }
    for (size_t i = 0; i < want.size(); i++) {
        MmbitSparseIter it;
        memcpy(&it, bc + ee.iter_offset + i * sizeof(it), sizeof(it));
        if (it.mask != want[i].mask || it.val != want[i].val) {
            return false;
        }
    }
    return true;
}

bool collectProgramReports(const u8 *bc, u32 bcLen, u32 prog, std::unordered_set<u32> *ex,
                           std::vector<ProgReport> *reports) {
    u32 pc = prog, furthest = prog;
    /* CHECK_BOUNDS guards the instructions up to its fail_jump target */
    struct Guard { u32 until; u64 lo, hi; };
    std::vector<Guard> guards;
    auto report = [&](u32 onmatch, s32 adjust) {
        u64 lo = 0, hi = ~0ull;
        for (const Guard &g : guards) {
            if (pc < g.until) {
                lo = std::max(lo, g.lo);
                hi = std::min(hi, g.hi);
            }
        }
        reports->push_back({onmatch, adjust, lo, hi});
    };
    auto jump = [&](u32 from, u32 rel) { furthest = std::max(furthest, from + rel); };
#define STEP(T) pc += (u32)HSB_ROUNDUP(sizeof(T), INSTR_ALIGN)
#define STEP_JUMP(T)                                \
    do {                                            \
        T in;                                       \
        memcpy(&in, bc + pc, sizeof(in));           \
        jump(pc, in.fail_jump);                     \
        STEP(T);                                    \
    } while (0)
    for (int guard = 0; guard < 65536; guard++) {
        if (pc + 8 > bcLen) {
            return false;
        }
        const u8 code = bc[pc];
        switch (code) {
        case OP_END:
            if (furthest <= pc) {
                return true;
            }
            STEP(InstrEnd);
            break;
        case OP_FINAL_REPORT: {
            if (reports) {
                InstrFinalReport in;
                memcpy(&in, bc + pc, sizeof(in));
                report(in.onmatch, in.offset_adjust);
            }
            if (furthest <= pc) {
                return true;
            }
            STEP(InstrFinalReport);
            break;
        }
        case OP_CHECK_GROUPS: STEP(InstrCheckGroups); break;
        case OP_CHECK_BOUNDS: {
            InstrCheckBounds in;
            memcpy(&in, bc + pc, sizeof(in));
            guards.push_back({pc + in.fail_jump, in.min_bound, in.max_bound});
            STEP_JUMP(InstrCheckBounds);
            break;
        }
        case OP_CHECK_MASK: STEP_JUMP(InstrCheckMask); break;
        case OP_CHECK_MASK_32: STEP_JUMP(InstrCheckMask32); break;
        case OP_CHECK_MASK_64: STEP_JUMP(InstrCheckMask64); break;
        case OP_CHECK_BYTE: STEP_JUMP(InstrCheckByte); break;
        case OP_CHECK_MED_LIT:
        case OP_CHECK_MED_LIT_NOCASE:
        case OP_CHECK_LONG_LIT:
        case OP_CHECK_LONG_LIT_NOCASE: STEP_JUMP(InstrCheckLit); break;
        case OP_CHECK_EXHAUSTED: STEP_JUMP(InstrCheckExhausted); break;
        case OP_DEDUPE: STEP_JUMP(InstrDedupe); break;
        case OP_REPORT: {
            if (reports) {
                InstrReport in;
                memcpy(&in, bc + pc, sizeof(in));
                report(in.onmatch, in.offset_adjust);
            }
            STEP(InstrReport);
            break;
        }
        case OP_REPORT_EXHAUST: {
            InstrReportExhaust in;
            memcpy(&in, bc + pc, sizeof(in));
            ex->insert(in.onmatch);
            if (reports) {
                report(in.onmatch, in.offset_adjust);
            }
            STEP(InstrReportExhaust);
            break;
        }
        case OP_DEDUPE_AND_REPORT: {
            if (reports) {
                InstrDedupeAndReport in;
                memcpy(&in, bc + pc, sizeof(in));
                report(in.onmatch, in.offset_adjust);
            }
            STEP_JUMP(InstrDedupeAndReport);
            break;
        }
        case OP_SQUASH_GROUPS: STEP(InstrSquashGroups); break;
        case OP_CLEAR_WORK_DONE: pc += INSTR_ALIGN; break;
        case OP_INCLUDED_JUMP: STEP(InstrIncludedJump); break;
        default:
            return false;
        }
    }
#undef STEP
#undef STEP_JUMP
    return false;
}

/* Walk the hash-confirm structures to enumerate literal programs
 * (src/fdr/fdr_confirm.h:36-94). */
bool walkConfirm(const u8 *bc, u32 bcLen, u32 confOff, u32 nBuckets,
                 std::unordered_set<u32> *ex, std::vector<LitTail> *tails) {
    bool ok = true;
    const u8 *confBase = bc + confOff;
    for (u32 b = 0; b < nBuckets; b++) {
        u32 cf;
        memcpy(&cf, confBase + 4 * b, 4);
        if (!cf) {
            continue;
        }
        const u8 *fc = confBase + cf;
        FDRConfirm h;
        memcpy(&h, fc, sizeof(h));
        const u32 n = 1u << h.nBits;
        for (u32 c = 0; c < n; c++) {
            u32 start;
            memcpy(&start, fc + sizeof(FDRConfirm) + 4 * c, 4);
            if (!start) {
                continue;
            }
            const u8 *li = fc + start;
            for (;;) {
                LitInfo x;
                memcpy(&x, li, sizeof(x));
                ok &= collectProgramReports(bc, bcLen, x.id, ex);
                tails->push_back({x.v, x.msk, x.size, b});
                if (!x.next) {
                    break;
                }
                li += sizeof(LitInfo);
            }
        }
    }
    return ok;
}

hs_error_t collectExhaustible(const hs_database_t *db, std::unordered_set<u32> *ex) {
    const DbHeader *h = (const DbHeader *)db;
    if (!h || h->magic != DB_MAGIC) {
        return HS_INVALID;
    }
    const RoseEngine *r = dbRose(db);
    const u8 *bc = (const u8 *)r;
    if (r->runtimeImpl != RUNTIME_PURE_LITERAL || !r->fmatcherOffset) {
        return HS_ARCH_ERROR;
    }
    const HWLM *hw = (const HWLM *)(bc + r->fmatcherOffset);
    const u32 engOff = r->fmatcherOffset + HWLM_ENGINE_OFFSET;
    if (hw->type == HWLM_ENGINE_NOOD) {
        NoodTable n;
        memcpy(&n, bc + engOff, sizeof(n));
        return collectProgramReports(bc, h->length, n.id, ex) ? HS_SUCCESS : HS_ARCH_ERROR;
    }
    FDR f;
    memcpy(&f, bc + engOff, sizeof(f));
    const u32 nb = f.engineID == 0 ? 8 : teddyNumBuckets(f.engineID);
    std::vector<LitTail> tails;
    return walkConfirm(bc, h->length, engOff + f.confOffset, nb, ex, &tails) ? HS_SUCCESS : HS_ARCH_ERROR;
}

size_t postprocessRecords(const std::unordered_set<u32> &exhaustible, MatchRec *m, size_t n) {
    std::sort(m, m + n, [](const MatchRec &a, const MatchRec &b) {
        if (a.block != b.block) return a.block < b.block;
        if (a.to != b.to) return a.to < b.to;
        return a.id < b.id;
    });
    size_t w = 0;
    std::unordered_set<u32> seen;
    u32 curBlock = 0xffffffffu;
    const bool anyEx = !exhaustible.empty();
    for (size_t i = 0; i < n; i++) {
        if (w && m[w - 1].block == m[i].block && m[w - 1].to == m[i].to && m[w - 1].id == m[i].id) {
            continue;
        }
        if (anyEx) {
            if (m[i].block != curBlock) {
                curBlock = m[i].block;
                seen.clear();
            }
            if (exhaustible.count(m[i].id) && !seen.insert(m[i].id).second) {
                continue;
            }
        }
        m[w++] = m[i];
    }
    return w;
}

} // namespace hsb

extern "C" hs_error_t hs_b200_postprocess_matches(const hs_database_t *db, hs_b200_match_t *recs,
                                                  size_t n, unsigned long long *nout) {
    if (!db || (n && !recs) || !nout) {
        return HS_INVALID;
    }
    std::unordered_set<hsb::u32> ex;
    hs_error_t r = hsb::collectExhaustible(db, &ex);
    if (r != HS_SUCCESS) {
        return r;
    }
    static_assert(sizeof(hsb::MatchRec) == sizeof(hs_b200_match_t), "record layout");
    *nout = hsb::postprocessRecords(ex, (hsb::MatchRec *)recs, n);
    return HS_SUCCESS;
}
