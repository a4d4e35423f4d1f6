/* include/megapath_b200.h -- C-ABI of libmegapath_b200.so
 *
 * Drop-in boundary for the soap4 alignment hot path of HKU-BAL/MegaPath, B200 (sm_100a).
 * The reference has no FFI layer (one statically linked C++ binary, SURVEY.md section 8b);
 * every entry point below replaces the C++ seam named beside it, so that the reference's
 * host code (SOAP4.cpp driver, IniParam, QueryParser, output) could call the GPU path
 * instead of its CPU engines.  Plain C: pointers, sizes, PODs.  No exceptions cross the
 * boundary; every call returns 0 on success or a negative mp_status and sets
 * mp_last_error().  One context per GPU; calls on one context are single-threaded
 * (the reference dispatcher is single-threaded too, DV-DPfunctions.cpp:3222-3277).
 *
 * All file:line citations are relative to the reference's soap4/ directory.
 */
#ifndef MEGAPATH_B200_H
#define MEGAPATH_B200_H
#include <stdint.h>
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct mp_context mp_context;

enum mp_status {
    MP_OK = 0,
    MP_ERR_CUDA = -1,       /* CUDA runtime failure (no device, OOM, launch error) */
    MP_ERR_IO = -2,         /* index file missing / malformed */
    MP_ERR_ARG = -3,        /* invalid argument */
    MP_ERR_STATE = -4,      /* call out of order (no index / no batch uploaded) */
    MP_ERR_CAPACITY = -5    /* internal buffer bound exceeded */
};

/* [MMP] section of soap4.ini -- MmpProperties (PEAlgnmt.h:374-384, IniParam.cpp:427-435) */
typedef struct mp_mmp_params {
    int32_t seedSAsizeThreshold;
    int32_t seedMinLength;
    int32_t uniqThreshold;
    int32_t indelFuzz;
    int32_t goodSeedLen;
    int32_t reseedLen;
    double  reseedRLTratio;
    int32_t reseedAbsDiff;
    double  shortSeedRatio;
} mp_mmp_params;

/* DPParameters subset that is live on this path (PEAlgnmt.h:386-405) + pairing options */
typedef struct mp_align_params {
    mp_mmp_params mmp;
    int32_t matchScore;        /* must be 1  (CPU_DP.cpp:199-208) */
    int32_t mismatchScore;     /* -4..-2, and > 2 * openGapScore (see mp_align_pairs) */
    int32_t openGapScore;      /* -6..-2 : cost of the first gap base */
    int32_t extendGapScore;    /* must be -1 */
    int32_t softClipLeft;      /* [Clipping] MaxFrontLenClipped */
    int32_t softClipRight;     /* [Clipping] MaxEndLenClipped */
    int32_t insert_low;        /* -v, after the first-batch clamp (SOAP4.cpp:465-474) */
    int32_t insert_high;       /* -u */
    int32_t peStrandLeftLeg;   /* 1 = '+', 2 = '-' ; only 1/2 ("+/-") is supported */
    int32_t peStrandRightLeg;
    int32_t skipDefaultDP;     /* [OtherSettings] SkipDefaultDP */
    int32_t maxReadLength;     /* -L : batch read-length bound (reads are < maxReadLength) */
} mp_align_params;

/* SeedPos (SeedPool.h:52-57) */
typedef struct mp_seed_pos { uint64_t pos; uint32_t strand_readID; uint32_t paired_seedLength; } mp_seed_pos;
/* DeepDP_Space::CandidateInfo at the pairing seam (DV-DPfunctions.h:1232-1240) */
typedef struct mp_candidate { uint32_t readIDLeft; uint32_t pad; uint64_t pos[2]; } mp_candidate;

/* One paired alignment -- DeepDPAlignResult (PEAlgnmt.h:509-545).  CIGAR strings live in a
 * flat char arena owned by the library (mp_results.cigars + offset), NUL terminated, in the
 * reference's "special" alphabet (M match, m mismatch, I, D, S). */
typedef struct mp_pair_result {
    uint32_t readID;           /* even read id of the pair */
    int32_t  insertSize;
    uint64_t algnmt_1, algnmt_2;
    int32_t  score_1, score_2;
    int32_t  editdist_1, editdist_2;
    int32_t  num_sameScore_1, num_sameScore_2;
    uint8_t  strand_1, strand_2; uint16_t pad; /* pad: 1 on the best pair of its read pair (first maximal score_1 + score_2,
                                                * OutputDPResult.cpp:156-232), chosen on the device for stage-S1 results; else 0 */
    uint32_t cigar_1, cigar_2; /* offsets into mp_results.cigars */
    uint64_t startPos_1, startPos_2;
    uint32_t refDpLength_1, refDpLength_2;
    uint32_t peLeftAnchor_1, peLeftAnchor_2, peRightAnchor_1, peRightAnchor_2;
} mp_pair_result;

/* One single-end alignment -- SingleAlgnmtResult (PEAlgnmt.h:549-575) */
typedef struct mp_single_result {
    uint32_t readID;
    uint32_t cigar;
    uint64_t algnmt;
    int32_t  score, editdist, num_sameScore;
    uint8_t  strand; uint8_t pad[3];
    uint32_t seedAlignmentLength;
    uint64_t startPos;
    uint32_t refDpLength; uint32_t peLeftAnchor;   /* peRightAnchor is always 0 here (DV-DPfunctions.cpp:437-438) */
} mp_single_result;

/* Result set of one mp_align_pairs call; owned by the library until mp_results_release. */
typedef struct mp_results {
    /* stage S1 (deep DP) and S3 (default DP / mate rescue): paired results, grouped by pair,
     * each group sorted and de-duplicated as OutputBuffer::ready does (DV-DPfunctions.h:198-243) */
    const mp_pair_result *pairs;      uint64_t n_pairs;
    const mp_pair_result *rescued;    uint64_t n_rescued;
    /* stage S2: single-end results of pairs S1 left unaligned, sorted by readID */
    const mp_single_result *singles;  uint64_t n_singles;
    const char *cigars;               uint64_t cigar_bytes;
    /* counters the reference prints (alignment.cpp:114-135, SOAP4.cpp:599-613) */
    uint64_t numDPAlignedPair, numDPAlignment;          /* deep DP */
    uint64_t numSingleDPAligned, numSingleDPAlignment;  /* single-end DP */
    uint64_t numRescuedPair, numRescuedAlignment;       /* default DP */
} mp_results;

/* Work counters and device timings of a context's last mp_align_pairs call (instrumentation for bench.py and the roofline
 * accounting; not part of the result set).  mp_last_stats copies them out. */
typedef struct mp_stats {
    /* algorithmic work of this call (SURVEY.md 8d): occ evaluations of the backward search, on-spot
     * occ evaluations of the SA walks (LF steps), SA lookups, LKT jumps, DP cells (sum of
     * dnaLen*readLen over required tasks), DP tasks */
    uint64_t n_occ, n_lf, n_sa, n_lkt, dp_cells, dp_tasks;
    /* gathers the seeding kernel actually issued beyond those: K-mer filter probes (8 B each) and text-compare
     * steps (each replaces the two occ evaluations the reference makes for the same step, counted in n_occ) */
    uint64_t n_probe, n_text;
    /* device time of the main kernels in this call, milliseconds (CUDA events) */
    float ms_seed, ms_sa, ms_pair, ms_dp, ms_total;
    /* host wall clock of the whole mp_align_pairs call, milliseconds */
    float ms_wall;
    /* summed device time of the DP fill / traceback kernels of this call (CUDA events around every launch) */
    float ms_fill, ms_tb;
    /* DP tasks answered by the exact-occurrence test instead of the DP kernels (bit-identical results, see mp_dp.cu), and the cells the
     * fill kernel really computed (dp_cells counts what the reference computes) */
    uint64_t dp_tasks_exact, dp_cells_filled;
    /* summed device time of that test and of compacting the remaining tasks */
    float ms_exact, reserved_;
} mp_stats;

/* ---- context ---- */
int  mp_init(int device, mp_context **ctx);
void mp_destroy(mp_context *ctx);
/* second context on the same GPU that shares the resident index (and K-mer filter) of `src` without owning it: own stream,
 * own batch / work buffers.  Two contexts driven by two host threads overlap one batch's host-side list plumbing and
 * latency-bound traceback with the other batch's compute-bound kernels (the reference double-buffers batches the same
 * way, SOAP4.cpp:424-441, 576-585).  `src` must outlive the clone. */
int  mp_clone(mp_context *src, mp_context **ctx);
const char *mp_last_error(void);
/* number of this library's own CUDA kernels launched so far in the process (bench.py "gpu_launches") */
uint64_t mp_launch_count(void);

/* ---- index: replaces INDEXLoad / INDEXFree (IndexHandler.cpp:49-99, 196-249) ----
 * Host reads <prefix>.{bwt,fmv,sa,lkt,pac}; the library owns the HBM copies (re-laid out).
 * .ann/.amb/.tra (chromosome translation) stay with the caller: they are host-side output data. */
int  mp_index_load(mp_context *ctx, const char *prefix);
int  mp_index_info(mp_context *ctx, uint64_t *textLength, uint64_t *inverseSa0, uint64_t cumFreq[5], uint64_t *hbmBytes);
/* ---- index built in HBM from a packed text (GPU index builder; replaces 2bwt-builder,
 *      2bwt-lib/2BWT-Builder.c, for the bench/synthetic path).  text2bit: 4 bases per byte,
 *      first base in the top 2 bits (.pac order). */
int  mp_index_build(mp_context *ctx, const uint8_t *text2bit, uint64_t textLength);
/* writes the resident index back in the reference's file formats (so the reference binary can
 * be timed on the same index) */
int  mp_index_save(mp_context *ctx, const char *prefix);
/* .ann/.amb/.tra of a text without ambiguity runs (HSP.c:569-699), host only */
int  mp_index_save_annotation(const char *prefix, uint64_t textLength, uint32_t numSeq, const char *const *names,
                              const uint64_t *starts, const uint64_t *lengths);

/* builds the per-parameter acceleration structures of the resident index now (the K-mer presence filter for
 * params->mmp.seedMinLength) instead of lazily in the first mp_seed_pairs call; call it before mp_clone so that the
 * clones share them */
int  mp_index_prepare(mp_context *ctx, const mp_align_params *params);

/* sizes the context's per-batch device buffers and pinned result arenas for batches of up to nReads reads (of up to
 * params->maxReadLength - 1 bases) now instead of on first use: the double-buffered driver (SOAP4.cpp:424-441) calls it for every
 * context before the batch loop so that no batch pays for allocations (which stall every context of the GPU while they run) */
int  mp_reserve(mp_context *ctx, const mp_align_params *params, uint32_t nReads);

/* index primitives, for parity tests against BWTOccValue / BWTSaValue / LT (2bwt-lib/BWT.c:597,968) */
int  mp_occ(mp_context *ctx, const uint64_t *idx, const uint32_t *c, uint64_t *out, uint64_t n);
int  mp_sa(mp_context *ctx, const uint64_t *saIndex, uint64_t *out, uint64_t n);
int  mp_lkt(mp_context *ctx, const uint32_t *key, uint64_t *l, uint64_t *r, uint64_t n);

/* ---- read batch: the buffers appendToQueryArrays fills (QueryParser.cpp:184-233) ----
 * queries: 2-bit reads, 16 bases per word LSB-first, 32-read interleaved
 *          (word j of read r at queries[(r/32*32)*wordPerQuery + r%32 + 32*j]);
 * caller keeps ownership, library copies to HBM.  nReads must be even (mate1, mate2, ...). */
int  mp_batch_upload(mp_context *ctx, const uint32_t *queries, const uint32_t *readLengths,
                     uint32_t nReads, uint32_t wordPerQuery);

/* ---- seeding + pairing: replaces PairEndSeedingEngine::performMmpSeeding
 *      (DV-DPfunctions.h:1366-1379; .cpp:2617-2687) for all pairs of the uploaded batch.
 *      Outputs stay device resident; the download calls exist for parity checks and return
 *      the arrays exactly as the reference builds them (two sentinels included). */
int  mp_seed_pairs(mp_context *ctx, const mp_align_params *params);
int  mp_download_seedpos(mp_context *ctx, mp_seed_pos **readPos, uint64_t *nReadPos,
                         mp_seed_pos **matePos, uint64_t *nMatePos);      /* free with mp_free */
int  mp_download_candidates(mp_context *ctx, mp_candidate **cands, uint64_t *nCands);
void mp_free(void *p);

/* ---- DP batch: the old GPU-kernel wrapper signature, SemiGlobalAligner::performAlignment
 *      (CPU_DPfunctions.h:103-111 -> callDP, CPU_DP.cpp:881-978).  Caller-owned arrays in the
 *      reference's layout: sequences 2-bit MSB-first, 1-based, 32-task interleaved
 *      (PairEndAlgnBatch::packRead/repackDNA, DV-DPfunctions.cpp:3009-3073);
 *      pattern has numOfThreads*(maxDNALength+maxReadLength) bytes.  As in the reference the
 *      whole batch uses clipLtSizes[0] / clipRtSizes[0] (CPU_DPfunctions.cpp:300). */
int  mp_dp_batch(mp_context *ctx,
                 const uint32_t *packedDNASequence, const uint32_t *DNALengths, uint32_t maxDNALength,
                 const uint32_t *packedReadSequence, const uint32_t *readLengths, uint32_t maxReadLength,
                 const int32_t *cutoffThresholds, int32_t *scores, uint32_t *hitLocs,
                 uint32_t *maxScoreCounts, uint8_t *pattern, uint32_t numOfThreads,
                 const uint32_t *clipLtSizes, const uint32_t *clipRtSizes,
                 int32_t mismatchScore, int32_t openGapScore);

/* ---- whole stage sequence for the uploaded batch: replaces soap3_dp_pair_align's engines
 *      (alignment.cpp:29-355): PairEndAlignmentEngine / SingleEndAlignmentEngine /
 *      HalfEndAlignmentEngine::performAlignment (DV-DPfunctions.h:1558-1576, 976-991, 1205-1221).
 *      Runs seeding (if not done), deep DP, single-end DP and default DP on the device and
 *      returns host-resident result arrays.  Host buffers in, host buffers out: this is the
 *      end-to-end call. */
int  mp_align_pairs(mp_context *ctx, const mp_align_params *params, mp_results *out);
void mp_results_release(mp_context *ctx, mp_results *res);
int  mp_last_stats(mp_context *ctx, mp_stats *stats);

/* ---- FASTQ ingest and annotated-FASTQ egress on the device (the two host loops either side of the hot path) ----
 * Ingest replaces loadPairReadsKseq + appendToQueryArrays (QueryParser.cpp:160-260, kseq.h) for plain four-line FASTQ text:
 * the caller hands over the raw bytes of exactly nPairs records of each mate file; record boundaries, name / comment split
 * (kseq: name up to the first blank), the "/<digit>" name trim, the length clamp to maxReadLength - 1 (QueryParser.cpp:188) and
 * the 2-bit packing are done by kernels.  The batch is then uploaded exactly as mp_batch_upload leaves it, and the text stays
 * resident for mp_format_fastq.  Returns MP_ERR_FORMAT (no batch uploaded) when the text is anything but
 * strict four-line FASTQ ('\r', NUL bytes, multi-line records, quality of another length, a record count other than nPairs):
 * the caller then parses with its own kseq-style parser and calls mp_batch_upload.
 * *readLengths (optional): host copy of the clamped lengths, owned by the context until the next upload. */
#define MP_ERR_FORMAT (-6)
int  mp_fastq_upload(mp_context *ctx, const char *text1, uint64_t bytes1, const char *text2, uint64_t bytes2,
                     uint32_t nPairs, uint32_t wordPerQuery, uint32_t maxReadLength, const uint32_t **readLengths);

/* sizes a context's ingest / egress buffers for batches of nPairs pairs and textBytes of FASTQ text (both mates) before the batch loop */
int  mp_fastq_reserve(mp_context *ctx, uint64_t textBytes, uint32_t nPairs);

/* chromosome translation tables of the index (.ann names, .tra grid + translate table; HSP.c:57-330): what getChrAndPos /
 * decideTargetChr (BGS-IO.cpp:163-190, 1312-1341) read.  Copied to the device once per context. */
typedef struct mp_annotation {
    uint64_t dnaLength;
    uint32_t numSeq, gridEntries, numTranslate, reserved_;
    const uint32_t *grid;               /* gridEntries */
    const uint64_t *trStartPos;         /* numTranslate */
    const uint32_t *trChrID;            /* numTranslate, 1-based */
    const char     *names;              /* the .ann name lines, concatenated */
    const uint64_t *nameOffsets;        /* numSeq + 1 offsets into names */
} mp_annotation;
int  mp_annotation_upload(mp_context *ctx, const mp_annotation *ann);

/* Egress replaces pairDeepDPOutputFastqAPI / unproperlypairDPOutputFastqAPI with getMappingFromHeader and decideTargetChr
 * (BGS-IO.cpp:1312-1446, 1966-2091; OutputDPResult.cpp:65-265) for the batch a context has just aligned (mp_fastq_upload +
 * mp_align_pairs): the whole stdout text of the batch -- deep-DP pairs, rescued pairs, then every other pair, each read as
 * "@name\tSCORE:<best>;<score>,<sequence name>;...<kept entries of the previous comment>\n<bases>\n+\n<qualities>\n" -- is
 * composed on the device.  mp_format_fastq returns its size, mp_format_fetch copies it into caller memory (pinned memory from
 * mp_host_alloc makes that a single DMA). */
typedef struct mp_format_params {
    double  top;                /* -top / 100 */
    int32_t megapathMode;       /* 1 = -F, 2 = -P */
    int32_t ignoreComments;     /* -nc */
} mp_format_params;
int  mp_format_fastq(mp_context *ctx, const mp_format_params *fmt, uint64_t *bytes);
/* on != 0: mp_align_pairs leaves the result arrays on the device (for mp_format_fastq) and returns the counters only --
 * mp_results.pairs / rescued / singles / cigars are empty.  Saves the device-to-host copies when the caller prints nothing else. */
int  mp_results_on_device(mp_context *ctx, int on);
int  mp_format_fetch(mp_context *ctx, char *dst, uint64_t bytes);
/* page-locked host memory for the two calls above */
void *mp_host_alloc(uint64_t bytes);
void  mp_host_free(void *p);

/* ---- BGZF compression on the device: replaces the zlib deflate behind BgzfWriter (bgzf_write / bgzf_flush of samtools 0.1.18,
 *      which the reference links for -b).  Any byte string in, a run of complete BGZF members out: each covers the next piece of at
 *      most 0xff00 input bytes with the gzip header and its "BC" extra subfield (BSIZE), one final raw DEFLATE block (dynamic Huffman,
 *      fixed Huffman or stored, whichever is smallest), CRC-32 and ISIZE.  No EOF marker: the writer appends it when it closes the
 *      file.  The output depends on the input bytes only (the same on every call, context and GPU).
 *      src and dst are host memory; page-locked memory from mp_host_alloc makes each copy one DMA.  Everything runs on the context's
 *      stream and ends with a synchronise of that stream; no index or batch is needed and a resident batch or result set is left as it
 *      is.  n == 0 writes nothing (*outBytes = 0); dstCap below MP_BGZF_BOUND(n) returns MP_ERR_ARG before anything is written. */
#define MP_BGZF_BOUND(n) ((((uint64_t)(n) + 0xff00u - 1) / 0xff00u) * 65536u)
int  mp_bgzf_compress(mp_context *ctx, const uint8_t *src, uint64_t n, uint8_t *dst, uint64_t dstCap, uint64_t *outBytes);
/* sizes the context's compression buffers for calls of up to maxBytes input bytes before the batch loop (like mp_reserve: an
 * allocation inside the loop stalls every context of the GPU while it runs); larger inputs are best fed in pieces of maxBytes */
int  mp_bgzf_reserve(mp_context *ctx, uint64_t maxBytes);

/* ---- gzip inflated on the device: replaces gzread for regular .gz read files.  Single- and multi-member streams (gzip, pigz,
 *      bgzip / BGZF, concatenated files).  Each call cuts its compressed bytes into chunks of MP_GUNZIP_CHUNK bytes, finds in every
 *      chunk after the first the first bit offset where a dynamic-Huffman block header is valid (exactly as zlib's inflate accepts
 *      one), decodes the chunks in parallel from there into slots of MP_GUNZIP_SLOT symbols, and keeps a chunk's output only when
 *      it starts where the verified chunk before it ended; otherwise the chunk is decoded again from that end.  Every byte returned
 *      was therefore decoded from a true block boundary, whatever the CRC says.  CRC-32 and ISIZE are checked per member.
 *      src holds the file's next n bytes, starting at the previous call's *consumed (the bit offset inside the first byte is kept in
 *      the handle); fin != 0: these bytes reach the end of the file.  At most dstCap (>= MP_GUNZIP_MIN_DST) bytes are written.
 *      *done = 1: the end of the file was reached and every member's CRC-32 and ISIZE verified.  Bytes after the last member that
 *      do not start with the gzip magic are ignored, as gzread ignores them.  The call makes progress whenever n >= 64 KiB or fin.
 *      MP_ERR_FORMAT: anything zlib refuses (bad magic, method or flags, header CRC, an invalid code, a distance too far back, a
 *      CRC-32 or ISIZE mismatch, a truncated member when fin is set); *produced then holds exactly the bytes zlib delivers before
 *      the error, and later calls on the handle return MP_ERR_FORMAT.  Host buffers in and out; the call runs on the context's stream
 *      and leaves a resident batch or result set as it is. */
#define MP_GUNZIP_CHUNK 65536u          /* compressed bytes per chunk; the block search covers the chunk's bit offsets */
#define MP_GUNZIP_SLOT (1u << 20)       /* decoded bytes a chunk holds before it stops (slot overflow) and is resumed */
#define MP_GUNZIP_EVENTS (MP_GUNZIP_CHUNK / 16u + 8u)   /* member starts / ends a chunk records before it stops the same way */
#define MP_GUNZIP_MIN_DST 65536u
#define MP_GUNZIP_MAX_IN (1ull << 30)   /* largest maxIn of mp_gunzip_open: 16384 chunks, 32 GiB of slots */
typedef struct mp_gunzip mp_gunzip;      /* one gzip file being inflated by the kernels of one context */
typedef struct mp_gunzip_stats_t {       /* counters of the last mp_gunzip_run call */
    uint64_t in_bytes, out_bytes;        /* compressed bytes consumed, decompressed bytes produced */
    uint64_t chunks;                     /* chunks the input was cut into */
    uint64_t candidates_tested;          /* bit offsets examined by the block search (up to and including the accepted one) */
    uint64_t candidates;                 /* chunks where the search accepted a block start */
    uint64_t false_candidates;           /* accepted starts the verified chain did not reach: those chunks were decoded again */
    uint64_t merged;                     /* chunks without a candidate, decoded as part of the chunk before */
    uint64_t overflows;                  /* times a verified chunk filled its slot (or event list) and was resumed */
    uint64_t rounds;                     /* decode launches: 1 + repairs + resumes */
    uint64_t members;                    /* gzip members whose CRC-32 and ISIZE were verified */
    float ms_total, reserved_;           /* host wall clock of the call */
} mp_gunzip_stats_t;
int  mp_gunzip_open(mp_context *ctx, uint64_t maxIn, mp_gunzip **g);   /* sizes the device buffers for calls of up to maxIn bytes */
int  mp_gunzip_run(mp_gunzip *g, const uint8_t *src, uint64_t n, int fin,
                   uint8_t *dst, uint64_t dstCap, uint64_t *consumed, uint64_t *produced, int *done);
int  mp_gunzip_stats(mp_gunzip *g, mp_gunzip_stats_t *s);
void mp_gunzip_close(mp_gunzip *g);

/* ---- roofline denominators measured on the spot (bench.py): kind 0 = random 32-byte gathers over an 8 GB table,
 *      1 = random 64-byte gathers (GB/s of requested bytes), 2 = packed 16-bit DPX issue rate (1e9 thread-instr/s) ---- */
int  mp_microbench(mp_context *ctx, int kind, double *result);

/* default parameters = soap4.ini (nt2 != 0: soap4-nt2.ini) */
void mp_default_params(mp_align_params *p, int nt2);

#ifdef __cplusplus
}
#endif
#endif
