/*
 * db_walk.h -- host-side walks over a literal database's bytecode: enumerate
 * the literal tails held in the hash-confirm structures
 * (src/fdr/fdr_confirm.h:36-94), find the reports that carry an exhaustion key
 * (HS_FLAG_SINGLEMATCH; REPORT_EXHAUST, src/rose/rose_program.h:485), and apply
 * the order-dependent report rules to a list of raw match records.
 */
#ifndef HSB200_DB_WALK_H
#define HSB200_DB_WALK_H

#include <unordered_set>
#include <utility>
#include <vector>

#include "../../../include/hs_b200.h"
#include "../ref_layout.h"

namespace hsb {

struct LitTail {
    u64 v, msk;
    u32 size;
    u32 bucket;
};

struct MatchRec { /* == hs_b200_match_t */
    u32 id;
    u32 block;
    u64 to;
};

/* Both return false if a program holds an opcode the device does not implement
 * (callers refuse the database with HS_ARCH_ERROR instead of failing mid-scan). */
/* a report instruction of a program: what it raises, and the bounds on the match end (CHECK_BOUNDS,
 * src/rose/program_runtime.c:2319-2326) under which the program reaches it */
struct ProgReport {
    u32 onmatch;
    s32 offset_adjust;
    u64 min_bound, max_bound;
};
bool collectProgramReports(const u8 *bc, u32 bcLen, u32 prog, std::unordered_set<u32> *ex,
                           std::vector<ProgReport> *reports = nullptr); /* every report instruction, in program order */

bool walkConfirm(const u8 *bc, u32 bcLen, u32 confOff, u32 nBuckets,
                 std::unordered_set<u32> *ex, std::vector<LitTail> *tails);

/** Reports compiled with HS_FLAG_SINGLEMATCH in a pure-literal database. */
hs_error_t collectExhaustible(const hs_database_t *db, std::unordered_set<u32> *ex);

/** A FULL_ROSE database whose only contents are outfix engines (queues [0, queueCount), no matchers, roles,
 * leftfixes, MPV, SOM, delays, boundary reports or logical combinations), with an EOD program that is absent or
 * [ENGINES_EOD iter] END over exactly the queues whose engine accepts at EOD: what the device runs as it is. */
bool outfixesOnly(const RoseEngine *r, u32 bcLen);

/** Order records for delivery and apply the order-dependent report rules the
 * device skipped: one report per (block, id, to) (dedupe, src/report.h:55-119)
 * and, for HS_FLAG_SINGLEMATCH reports, only the first match per block
 * (exhaustion keys, src/report.h:121-147, program_runtime.c:464-481).
 * Returns the number of records kept (in place, sorted by (block, to, id)). */
size_t postprocessRecords(const std::unordered_set<u32> &exhaustible, MatchRec *m, size_t n);

} // namespace hsb
#endif
