/*
 * kernels.h -- launch interface between the C-ABI shim (api_device.cu) and the
 * sm_100a scan kernels (scan_kernels.cu).  Plain PODs only.
 */
#ifndef HSB200_KERNELS_H
#define HSB200_KERNELS_H

#include <cuda_runtime.h>

#include "../ref_layout.h"

/* Kernel launches and the dynamic shared-memory window are spelled through two
 * macros so that the same sources also compile as plain C++ for the SIMT
 * emulator of tests/emu (TEST infrastructure, -DHSB_HOST_EMU: kernel logic under
 * `pytest -m "not gpu"`).  In the product build they are exactly the CUDA forms;
 * libhs_b200.so contains no emulator and has no CPU scan path. */
#ifdef HSB_HOST_EMU
#define HSB_LAUNCH(kern, grid, block, smem, stream, ...) \
    hsb_emu::launch(dim3(grid), dim3(block), smem, [=]() { kern(__VA_ARGS__); })
#define HSB_DYNAMIC_SMEM(name) u8 *name = hsb_emu::dynamicSmem()
#define HSB_NOINLINE __attribute__((noinline))
#define HSB_GRID_CONSTANT
#else
#define HSB_LAUNCH(kern, grid, block, smem, stream, ...) kern<<<grid, block, smem, stream>>>(__VA_ARGS__)
#define HSB_DYNAMIC_SMEM(name) extern __shared__ __align__(128) u8 name[]
#define HSB_NOINLINE __noinline__
/* kernel parameters whose address is taken (passed by reference into the out-of-line
 * candidate path) stay in the constant bank instead of being copied to every
 * thread's stack */
#define HSB_GRID_CONSTANT __grid_constant__
#endif

namespace hsb {

/* One match record as the device writes it: identical to hs_b200_match_t
 * (include/hs_b200.h). */
struct DevMatch {
    u32 id;
    u32 block;
    u64 to;
};

/* First-stage ("shift-OR") filter variants.  An entry read at sampled position
 * x holds SLOTS bytes; byte p has bit b SET iff no literal of bucket b can end
 * at position x+p given the bytes at x (FDR: src/fdr/fdr.c:157-327; Teddy:
 * src/fdr/teddy.c:918-969 -- see DESIGN.md section 3 for the derivation). */
enum FilterKind {
    FK_BYTE32 = 0, /* index = 1 byte; u32 entry (4 slots x 8 buckets); table
                      replicated per lane (bank-conflict free). Teddy, noodle, and
                      FDR sets whose tails keep the per-byte filter sparse */
    FK_BYTE64 = 1, /* index = 1 byte; 2 x u32 (4 slots x 16 buckets). Fat Teddy */
    FK_HASH32 = 2, /* index = 2-byte FDR hash; u32 entry (slots 0..3 of FDR) */
    FK_HASH64 = 3, /* index = 2-byte FDR hash; u64 entry (all 8 FDR slots)   */
    FK_PAIR32 = 4, /* index = (class of byte 0, class of byte 1), 5 bits each, classes
                      from a per-lane byte table; u32 entry; both tables replicated per
                      lane (bank-conflict free).  FDR sets.  Table image: 256 class words
                      (c0 << 7 | c1 << 12), then 1024 pair entries */
    FK_GRAM4 = 5,  /* index = classes of the FOUR bytes ending at a position (5 bits each) into
                      a 1 Mbit bitmap in shared memory; no buckets.  Large FDR sets whose
                      literals are all >= 4 bytes.  Table image: 256 class words
                      (4 * c); ScanParams.bitmap = the bitmap (bitmapBytes), bit c[e] of word
                      c[e-3] + 33 c[e-2] + 1025 c[e-1] */
    FK_OUTFIX = 6, /* no literal first stage at all: a single-outfix database, its one engine runs on
                      the DFA / NFA kernels (dfa_kernels.cu) */
};

enum ConfirmKind {
    CK_FDR = 0,    /* hash confirm: FDRConfirm / LitInfo (src/fdr/fdr_confirm.h) */
    CK_NOODLE = 1, /* single literal: noodTable msk/cmp (src/hwlm/noodle_internal.h) */
};

enum { MAX_PEERS = 8 };
enum { CTR_MATCHES = 0, CTR_ERROR = 1, CTR_CANDIDATES = 2, CTR_CONFIRMED = 3,
       CTR_PREFILTER_PASS = 4, CTR_CANDQ = 5 /* split mode: candidates handed to the confirm kernel */,
       CTR_COUNT = 8 };

/* Split mode (opt-in): the scan kernel stops at the prefilter and appends the
 * surviving candidates to a list in HBM; confirmKernel finishes them, one thread
 * per candidate.  The list is the SECOND half of the record ring the scratch
 * allocated (records [outCap, 2 * outCap) of ScanParams.out), so no launch
 * parameter changes; if it overflows, the record count is raised above outCap
 * and the caller's grow-and-rescan path takes over. */
struct DevCand {
    u64 g;       /* corpus position of the candidate's last byte */
    u32 buckets; /* first-stage bucket bits */
    u32 pad;
};
enum { ERR_BAD_OPCODE = 1, ERR_INTERNAL = 2 };

struct ScanParams {
    /* corpus: position 0 = first byte of the packed corpus; bytes
     * [-16, paddedBytes + 16) are readable; blocks start 16-byte aligned */
    const u8 *corpus;
    u64 corpusBytes;       /* end of the last block */
    u64 readableEnd;       /* multiple of 16, >= corpusBytes: TMA may read up to here */
    u32 tileFirst;         /* tiles [tileFirst, tileFirst + ntiles) are scanned */
    u32 ntiles;
    u32 tileBytes;         /* multiple of 512 */
    u32 nstages;           /* per-warp TMA ring depth */
    const u64 *blockOff;   /* ascending, 16-byte aligned */
    const u32 *blockLen;
    u32 nblocks;
    u32 uniformPitch;      /* != 0: blockOff[i] == i * uniformPitch */
    u32 uniformLen;        /* != 0 (with uniformPitch): every block has this length; no table reads */
    /* stream sets (hs_b200_streams_*): stream b's write at b * streamPitch + 16,
     * preceded by its look-behind; 8 bytes of state per stream (7 history bytes,
     * right-aligned, + their count) and the stream offset live in HBM */
    u32 streamPitch;
    const u8 *streamHist;
    const u64 *streamOffset;
    /* database image */
    const u8 *bc;          /* RoseEngine bytecode (device copy) */
    const u8 *table;       /* first-stage table in HBM (copied to smem) */
    u32 tableBytes;
    u32 indexMask;         /* FK_HASH*: FDR domainMask */
    u32 repShift;          /* FK_HASH32: log2 of the copies per entry (bank partition) */
    const u8 *bitmap;      /* second-stage prefilter (copied to smem), may be null */
    u32 bitmapBytes;       /* power of two >= 16, or 0 = no prefilter */
    u32 bitmapShift;       /* 32 - log2(bits) */
    u32 keyBytes;          /* 1..4: literal tail bytes hashed into the bitmap */
    u32 pairBytes;         /* FK_PAIR32: shared-memory bytes of the pair table = 4 KiB x classes of the
                            * second byte (<= 128 KiB) */
    u32 bitmapHoles;       /* FK_PAIR32: 1 = the (32 KiB) bitmap sits in the class rows' upper halves;
                            * 0 = bitmapBytes contiguous bytes after the pair table (large sets) */
    u32 bitmapBits;        /* FK_PAIR32: bits of the first-level bitmap; index = mulhi(key * K, bits) */
    u32 bucketFold;        /* 1 = 16 confirm buckets (fat Teddy) behind 8 first-stage bits: bit i of a
                            * candidate stands for buckets i and i + 8 */
    const u32 *bitmap2;    /* optional second-level bitmap in HBM/L2 (large literal sets) */
    u32 bitmap2Shift;      /* 32 - log2(bits); 0 = none */
    u32 confOff;           /* CK_FDR: offset of the confirm base in bc */
    u32 engineOff;         /* CK_NOODLE: offset of the noodTable in bc */
    u32 confirmKind;
    u64 groups;
    /* output */
    DevMatch *out;
    u32 outCap;
    u32 *counters;
    /* fused exchange (multi-GPU): every record is also stored, over NVLink,
     * into slot [myRank][1 + i] of each peer's exchange buffer (peer-mapped
     * pointers; layout [nPeers][peerCap + 1] records, slot 0 = count) */
    u32 nPeers;
    u32 myRank;
    u32 peerCap;
    u32 blockBase;           /* added to block indices in exchanged records */
    DevMatch *peers[MAX_PEERS];
};

struct LaunchCfg {
    int kind;      /* FilterKind */
    int stride;    /* 1, 2, 4 */
    int slotBase;  /* FK_HASH32: 0 = slots 0..3 (reference numbering), 1 = slots 1..4 */
    int direct;    /* 1: corpus loaded straight into registers; 0: TMA-staged tiles */
    int queued;    /* 1 (direct, stride 1 only): candidates go through the per-warp queue */
    int wide;      /* 1 (direct, stride 1, FK_BYTE32 / FK_HASH32, tileBytes % 1024 == 0): 32-byte lanes */
    int split;     /* 1 (wide only): candidates go to the list in HBM, confirmKernel finishes them */
    int grid;      /* CTAs (one per SM) */
    int warps;     /* per CTA */
    size_t smemBytes;
};

/* Dynamic shared memory the kernel needs (warps = warps with TMA stages, 0 in
 * direct mode; queueWarps = warps with a candidate queue, 0 without, negative =
 * that many warps of the wide-step variant). */
size_t scanSmemBytes(int kind, u32 tableBytes, u32 bitmapBytes, int warps, u32 nstages,
                     u32 tileBytes, int queueWarps);

cudaError_t launchScan(const LaunchCfg &cfg, const ScanParams &p, cudaStream_t stream);

/* Split mode: finish the candidates the scan kernel left in the list (same stream, after it). */
cudaError_t launchConfirm(const LaunchCfg &cfg, const ScanParams &p, cudaStream_t stream);

/* Publish the record count of a finished scan into slot 0 of this rank's
 * region in every peer's exchange buffer (runs after the scan on its stream). */
cudaError_t launchPublishCount(const ScanParams &p, cudaStream_t stream);

/* stream-set helpers: write every stream's look-behind in front of its write /
 * roll history and offsets forward after a scan */
cudaError_t launchStreamAssemble(u8 *corpus, const u8 *hist, u32 nstreams, u32 pitch, cudaStream_t stream);
cudaError_t launchStreamAdvance(const u8 *corpus, u8 *hist, u64 *offsets, const u32 *lens, u32 uniformLen,
                                u32 nstreams, u32 pitch, u32 histReq, cudaStream_t stream);

/* One engine of a DFA / NFA launch: its own bytes (struct NFA first) in device memory. */
struct DfaEngine {
    const u8 *nfa;
    u32 tableBytes;  /* McClellan: bytes of the successor table (staged in shared memory if it fits) */
    u32 states;      /* McClellan-8: state_count (<= 256): rows of the byte-indexed table built in shared memory */
    u32 squashes;    /* LimEx: some exception squashes (LIMEX_SQUASH_CYCLIC / _REPORT): the kernel reads the squash masks */
    u32 pad;
};

/* DFA / NFA engines in block mode (dfa_kernels.cu): McClellan 8 / 16, Sheng, LimEx-32 ... -512, one thread per
 * block.  One launch runs every engine of the table over every block; they are all of one model (`kind`), and
 * tableBytes / states / squashes are the largest (any) over them, which size the launch's shared memory. */
struct DfaParams {
    const u8 *corpus;
    u64 readableEnd;
    const u64 *blockOff;
    const u32 *blockLen;
    u32 nblocks;
    u32 uniformPitch, uniformLen;
    const DfaEngine *engines; /* device memory */
    u32 nengines;
    u32 kind;        /* NFA.type: NFA_MCCLELLAN_8 / NFA_MCCLELLAN_16 / NFA_SHENG / NFA_LIMEX_* */
    u32 tableBytes;
    u32 ilp;         /* blocks walked by one lane at a time: 1 or 2 (runtime option dfa_ilp) */
    u32 states;
    u32 squashes;
    u32 tableArea;   /* set by launchDfa: shared-memory bytes of the tables, the tiles follow */
    DevMatch *out;   /* {report, block, offset after the last byte} */
    u32 outCap;
    u32 *counters;   /* CTR_MATCHES */
};
cudaError_t launchDfa(const DfaParams &p, int smCount, int maxSmem, cudaStream_t stream);

/* accel primitives (src/nfa/shufti.c, truffle.c, vermicelli.h): first
 * position in [0,len) whose byte is in the class, or len. */
cudaError_t launchAccelFind(int type, const u8 *params, const u8 *d_buf, u64 len,
                            u64 *d_result, cudaStream_t stream);

} // namespace hsb
#endif
