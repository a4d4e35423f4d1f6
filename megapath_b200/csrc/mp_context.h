// mp_context.h -- library-internal context (one per GPU) and helpers.
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include <chrono>
#include <atomic>
#include "../../include/megapath_b200.h"
#include "mp_index.cuh"

void mp_set_error(const char *fmt, ...);
extern std::atomic<unsigned long long> g_mp_launches;
static inline double mp_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
// MP_TRACE=1: wall-clock phase marks on stderr
struct MpTrace {
    bool on, sync; double t0, last;      // MP_TRACE=1: marks + extra stream syncs at phase ends; MP_TRACE=2: marks only
    MpTrace() { const char *e = getenv("MP_TRACE"); on = e && *e && *e != '0'; sync = on && *e == '1'; t0 = last = mp_now_ms(); }
    void mark(const char *what) { if (!on) return; double t = mp_now_ms(); fprintf(stderr, "[mp_trace] %-28s +%9.3f ms (%9.3f)\n", what, t - last, t - t0); last = t; }
};     // kernels of this library launched so far (mp_launch_count)

#define MP_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    mp_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); \
    return MP_ERR_CUDA; } } while (0)

// growable device buffer
struct DevBuf {
    void *p = nullptr; size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { mp_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return MP_ERR_CUDA; }
        cap = want; return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

// growable pinned host array (results are DMA'd straight into it; cudaMallocHost memory is plain host memory for the caller)
template <class T> struct PinnedBuf {
    T *p = nullptr; size_t n = 0, cap = 0;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    T *data() { return p; }
    const T *data() const { return p; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    void clear() { n = 0; }
    T &operator[](size_t i) { return p[i]; }
    const T &operator[](size_t i) const { return p[i]; }
    T *begin() { return p; }
    T *end() { return p + n; }
    int reserve(size_t want) {
        if (want <= cap) return 0;
        size_t nc = cap ? cap : 1024;
        while (nc < want) nc += nc / 2 + 1024;
        T *q = nullptr;
        if (cudaMallocHost((void **)&q, nc * sizeof(T)) != cudaSuccess) { mp_set_error("cudaMallocHost(%zu) failed", nc * sizeof(T)); return MP_ERR_CUDA; }
        if (n) memcpy((void *)q, (const void *)p, n * sizeof(T));
        if (p) cudaFreeHost(p);
        p = q; cap = nc; return 0;
    }
    int resize(size_t want) { if (reserve(want)) return MP_ERR_CUDA; n = want; return 0; }
    int push_back(const T &v) { if (n == cap && reserve(n + 1)) return MP_ERR_CUDA; p[n++] = v; return 0; }
};

// ---- seeding records (device) ----
struct MpSeed {            // SeedSAalign (DV-DPfunctions.cpp:2161-2171) + owner
    uint64_t sa_l;
    uint32_t strandIdx;    // read * 2 + (strand == '-')
    uint32_t hitBase;      // first slot of this seed in the hit-stub list
    uint16_t query_offset, seed_len, sa_diff, pad;
};
struct MpHit {             // SeedAlign (DV-DPfunctions.cpp:2144-2159)
    uint64_t offset;       // target text position (u64, wraps like the reference)
    uint16_t length, query_offset, multiplicity;
    uint16_t strand;       // 0 '+', 1 '-'
};
struct MpDpTask {          // one semi-global DP instance
    uint64_t refStart;     // window start in the text
    uint32_t refLen;       // DNALength
    uint32_t readID;
    uint16_t readLen;
    uint8_t  strand;       // 1 '+', 2 '-' (read is reverse-complemented)
    uint8_t  valid;
    int32_t  cutoff;
    int16_t  diag;         // expected window offset of the read's first base (the seed's diagonal), -1 = unknown; only a hint:
    uint16_t pad_;         // k_dp_fill derives a lower bound of the best score from it, results do not depend on it
};
struct MpDpOut {
    int32_t score; uint32_t hitLoc; uint32_t count; uint32_t patLen;
    // the special CIGAR of the pattern (CigarStringEncoder, DV-DPfunctions.h:344-427), built by the traceback while it emits: text length,
    // the encoder's statistics, and whether the text itself sits at the end of the task's pattern row ([patStride - cigLen, patStride))
    uint16_t cigLen, nI, nD, nS; int16_t gapPenalty; uint8_t cigStored, pad_[5];
};

struct mp_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8];
    // event pairs around the DP kernels of one mp_align_pairs call (kind 0 = fill, 1 = traceback)
    std::vector<cudaEvent_t> evPool; std::vector<int> evKind; size_t evUsed = 0;
    cudaEvent_t ev_begin(int kind) {
        if (evUsed + 2 > evPool.size()) { cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b); evPool.push_back(a); evPool.push_back(b); evKind.push_back(kind); }
        evKind[evUsed / 2] = kind;
        cudaEventRecord(evPool[evUsed], stream);
        return evPool[evUsed + 1];
    }
    void ev_end(cudaEvent_t stop) { cudaEventRecord(stop, stream); evUsed += 2; }
    void ev_collect(float &msFill, float &msTb, float &msExact) {       // after a stream sync; kinds 0 fill, 1 traceback, 2 exact-occurrence test
        msFill = msTb = msExact = 0;
        for (size_t i = 0; i + 1 < evUsed; i += 2) {
            float t = 0; cudaEventElapsedTime(&t, evPool[i], evPool[i + 1]);
            (evKind[i / 2] == 0 ? msFill : evKind[i / 2] == 1 ? msTb : msExact) += t;
        }
        evUsed = 0;
    }
    // index
    bool hasIndex = false, sharedIndex = false;   // sharedIndex: index buffers belong to another context (mp_clone)
    MpIndexView ix;
    DevBuf dBlocks, dSuper, dSa, dSa32, dSa40Lo, dSa40Hi, dLkt, dPac, dBloom;
    int bloomK = 0, bloomStride = 1, bloomSeedMin = 0; uint64_t bloomWords = 0; const void *bloomFor = nullptr;   // K-mer presence filter (mp_seed.cu)
    uint64_t hbmBytes = 0;
    std::vector<uint64_t> hSa; uint64_t saInterval = 16;   // kept for mp_index_save
    // batch
    bool hasBatch = false, seeded = false;
    uint32_t nReads = 0, wpq = 0, maxLenBatch = 0;       // maxLenBatch: longest read of the uploaded batch
    DevBuf dReadsIl, dReads, dLens;
    // seeding
    DevBuf dCounters;                 // u64[16]: 0 seeds, 1 hit stubs, 2 occ, 3 sa, 4 lkt, 5 lf, 6 work-queue
    DevBuf dSeeds, dStubs, dHitsPerRead, dHitStart, dCursor, dHits, dHits2, dSeedPos, dNPos, dNNeg;
    DevBuf dCandCount, dCandStart, dCands, dScanTmp;
    uint64_t nSeeds = 0, nHits = 0, nCands = 0;
    uint64_t capSeeds = 0, capStubs = 0;
    mp_align_params seedParams;
    // DP
    DevBuf dTasks, dRefSeq, dReadSeq, dTable, dFill, dPattern, dDpOut;
    DevBuf dHintTest;                                                             // MP_DP_TEST_HINT (mp_dp.cu)
    DevBuf dExFlag, dExPos, dExIdx;                                              // exact-occurrence test: flags, scan, active slots (mp_dp.cu)
    DevBuf dLT, dRT, dLO, dRO, dLP, dRP, dOk, dBytes, dIdx, dOff, dRes, dCig;   // stage S1 chunk buffers (kept across calls)
    DevBuf dRes2, dKeep, dKeepPos, dTotals;                                      // stage S1 per-pair dedup / best pick (k_pair_ready)
    mp_stats stats = {};                    // work counters / timings of the last mp_align_pairs call (mp_last_stats)
    // results (host, owned until release)
    PinnedBuf<mp_pair_result> hPairs;
    PinnedBuf<mp_pair_result> hRescued;
    PinnedBuf<mp_single_result> hSingles;
    PinnedBuf<char> hCigars;
    std::vector<uint32_t> hLens;            // host copy of the batch's read lengths (stages S2/S3)
    DevBuf dAligned, dGather;               // per-pair "placed by deep DP" flags; (dGather: unused scratch kept for mp_reserve)
    DevBuf dS2Counts, dS2Start, dS2Tasks, dS2Res;   // stage S2 on the device: kept seeds per read, task offsets, tasks, results
    DevBuf dRsSlotTasks, dRsSlotInfo, dRsFlag, dRsPos, dRsTasks, dRsInfo, dRsRec, dRsOut, dRsKeep, dRsKeepPos;   // stage S3 (mate rescue) on the device
    // results of the last mp_align_pairs call that are still resident: dRes2[0], dRsOut[1], dS2Res[2] (mp_format_fastq reads them)
    uint64_t resCount[3] = { 0, 0, 0 }; bool resValid = false;
    bool resultsOnDevice = false;           // mp_results_on_device: mp_align_pairs skips the device-to-host copies of the result arrays
    // FASTQ ingest / egress on the device (mp_fastq.cu)
    bool fqBatch = false;                   // the uploaded batch came through mp_fastq_upload: text + record index are resident
    uint64_t fqBase[2] = { 0, 0 }, fqBytes[2] = { 0, 0 };
    DevBuf dFqText, dFqCnt, dFqCntPos, dFqLines, dFqRec, dFqFlags;
    bool hasAnn = false; uint64_t annDnaLength = 0; uint32_t annGridEntries = 0, annNumTr = 0, annNumSeq = 0;
    DevBuf dAnnGrid, dAnnTrStart, dAnnTrChr, dAnnNames, dAnnNameOff;
    DevBuf dFmtKeys, dFmtGroups, dFmtRecLen, dFmtTail, dFmtTailText, dFmtSeg, dFmtDst, dFmtLen, dFmtOff, dFmtOut;
    uint64_t fmtBytes = 0; bool fmtReady = false;
    // BGZF compression (mp_bgzf.cu): input, one 64 KiB member slot per 0xff00-byte piece, the packed stream, member sizes / offsets,
    // and a match row per resident CTA
    DevBuf dBgzfIn, dBgzfSlots, dBgzfOut, dBgzfSizes, dBgzfOffs, dBgzfScratch;
};

// mp_index.cu
int mpi_load(mp_context *ctx, const char *prefix);
int mpi_finish_sa(mp_context *ctx);      // texts >= 2^32: 40-bit SA samples at the densest rate the HBM budget allows
int mpi_build_from_words(mp_context *ctx, const uint32_t *hBwtWords, uint64_t n, uint64_t inverseSa0, const uint64_t cum[5]);
// mp_seed.cu
int mps_seed_pairs(mp_context *ctx, const mp_align_params *P);
// mp_dp.cu
struct MpDpParams { int clipLt, clipRt, mismatch, open; int cigText = 1; };      // cigText = 0: never keep the CIGAR text in the pattern row (test hook MP_CIG_TEXT=0)
// tasks (device) -> outs (device); sequences are extracted from the index / uploaded reads
int mpd_run_tasks(mp_context *ctx, const MpDpTask *dTasks, uint32_t nTasks, uint32_t maxRefLen, uint32_t maxReadLen,
                  const MpDpParams &P, MpDpOut *dOuts, uint8_t *dPatterns, uint32_t patStride);
// mp_stages.cu: single-end DP + default DP for the pairs stage S1 left unaligned
int mps_single_and_rescue(mp_context *ctx, const mp_align_params *P, mp_results *out, uint64_t &cells, uint64_t &tasksRun);
// explicit sequences (one byte per base, stride maxRefLen / maxReadLen)
int mpd_run_explicit(mp_context *ctx, const uint8_t *dRef, const uint32_t *dRefLens, uint32_t maxRefLen,
                     const uint8_t *dRead, const uint32_t *dReadLens, uint32_t maxReadLen, const int32_t *dCutoffs,
                     uint32_t nTasks, const MpDpParams &P, MpDpOut *dOuts, uint8_t *dPatterns, uint32_t patStride);
