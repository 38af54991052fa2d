/*
 * rose_build.h -- host-side assembly of a pure-literal RoseEngine bytecode
 * (programs + floating literal matcher) and the hs_database container.
 * Stands where the reference's RoseBuildImpl::buildFinalEngine + dbCreate stand
 * (src/rose/rose_build_bytecode.cpp:3609-3888, src/compiler/compiler.cpp:476-
 * 536), restricted to databases whose runtimeImpl is ROSE_RUNTIME_PURE_LITERAL.
 */
#ifndef HSB200_ROSE_BUILD_H
#define HSB200_ROSE_BUILD_H

#include <string>
#include <vector>

#include "hwlm_build.h"

namespace hsb {

struct CompileError {
    std::string msg;
    int index; /* expression index or -1 */
};

struct LitPattern {
    std::string s;      /* raw bytes of the literal */
    bool caseless = false;
    bool singlematch = false;
    u32 report = 0;     /* user-visible id */
    u32 index = 0;      /* position in the caller's expression array */
};

struct CompileOpts {
    bool pureLiteralApi = false; /* hs_compile_lit*: sets RoseEngine.pureLiteral */
    bool streaming = false;      /* HS_MODE_STREAM / HS_MODE_VECTORED: history + per-stream state
                                  * (literals <= 8 bytes); src/util/compile_context.h:47-48 */
    bool vectored = false;       /* HS_MODE_VECTORED: a streaming database stamped for hs_scan_vector */
    bool smallWrite = true;      /* block mode: also emit the small-write DFA (src/smallwrite/) for buffers
                                  * shorter than 70 bytes when the literal set's automaton stays small */
    int outfixKind = 0;          /* != 0: no literal matcher, ONE engine over the whole literals run as an
                                  * outfix (ROSE_RUNTIME_SINGLE_OUTFIX): see enum OutfixKind */
    bool regexDfa = true;        /* regex route: determinise the position automaton when the DFA stays small
                                  * (McClellan-8 up to 256 states, McClellan-16 up to 1024), else LimEx */
    u64 platform = PLATFORM_NOAVX2 | PLATFORM_NOAVX512 | PLATFORM_NOAVX512VBMI;
    HwlmBuildOpts hwlm;
};

enum OutfixKind { OUTFIX_NONE = 0, OUTFIX_DFA_AUTO = 1, OUTFIX_MCCLELLAN8 = 2, OUTFIX_MCCLELLAN16 = 3, OUTFIX_SHENG = 4,
                  OUTFIX_LIMEX32 = 5 };

/* grey-box limits mirrored from src/grey.cpp:40-160 */
static const size_t LIMIT_PATTERN_LENGTH = 16000;
static const size_t LIMIT_LITERAL_LENGTH = 1600;
static const size_t LIMIT_LITERAL_COUNT = 8000000;

/** Build the RoseEngine bytecode for a set of literal patterns. */
std::vector<u8> buildLiteralRose(const std::vector<LitPattern> &pats,
                                 const CompileOpts &opts, HwlmBuildInfo *info);

/** Expressions that need an NFA (regex_nfa.h): ONE engine over all of them (McClellan-8 / -16 when the automaton
 * determinises small enough, else LimEx), run as the database's single outfix (ROSE_RUNTIME_SINGLE_OUTFIX).  A set
 * whose positions do not fit one 512-state automaton is split into several engines, each an outfix of a
 * FULL_ROSE database that holds nothing else.  Block mode only.  Throws CompileError. */
struct RegexPattern {
    std::string re;
    unsigned flags = 0;
    u32 report = 0;
    u32 index = 0;
    u64 minOffset = 0, maxOffset = ~0ull; /* hs_expr_ext: bounds on the match end (CHECK_BOUNDS in the report programs) */
    u64 minLength = 0;                    /* hs_expr_ext: shortest match that counts (regex_nfa.cpp) */
};
std::vector<u8> buildRegexRose(const std::vector<RegexPattern> &pats, const CompileOpts &opts);

/** The sparse iterator over `keys` of a multibit of totalBits bits, as the reference lays it out
 * (mmbBuildSparseIterator): what an ENGINES_EOD instruction walks. */
std::vector<MmbitSparseIter> sparseIterator(const std::vector<u32> &keys, u32 totalBits);

/** Test hook: pure-literal block database from raw literal programs (`area`
 * is placed at programAreaBase(); lits[i].id = its program's offset in area). */
u32 programAreaBase();
std::vector<u8> buildRawProgramRose(std::vector<HwlmLit> lits, const std::vector<u8> &area,
                                    u32 ekeyCount, const std::vector<u32> &invDkey,
                                    const CompileOpts &opts, HwlmBuildInfo *info);

} // namespace hsb
#endif
