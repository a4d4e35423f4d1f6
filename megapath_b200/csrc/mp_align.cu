// mp_align.cu -- stage orchestration on the device + the C-ABI entry points.
//
// Stage S1 "deep DP" (alignment.cpp:91-137 -> DPForUnalignPairs2 -> DeepDPWrapper):
//   task packing   PairEndAlgnBatch::packLeft / packRight        DV-DPfunctions.cpp:2857-3007
//   result assembly DP2CPUAlgnThread + CigarStringEncoder         DV-DPfunctions.cpp:3391-3540, .h:344-427
//   per-pair dedup  OutputBuffer::ready / ResultCompare           DV-DPfunctions.h:198-243, .cpp:253-258
#include "mp_context.h"
#include "mp_cigar.h"
#include <cub/device/device_scan.cuh>
#include <algorithm>
#include <tuple>
#include <string.h>
#include <stdlib.h>

int mps_upload(mp_context *ctx, const uint32_t *queries, const uint32_t *readLengths, uint32_t nReads, uint32_t wpq);
int mps_download_seedpos(mp_context *ctx, mp_seed_pos **readPos, uint64_t *nReadPos, mp_seed_pos **matePos, uint64_t *nMatePos);


// ---- packLeft (DV-DPfunctions.cpp:2857-2924) ----
// adds (cells, tasks) of a warp's lanes to counters[11], counters[12] (work accounting, SURVEY 8d)
__device__ __forceinline__ void account_work(unsigned long long cells, unsigned long long tasks, unsigned long long *__restrict__ counters)
{
#pragma unroll
    for (int d = 16; d; d >>= 1) { cells += __shfl_xor_sync(0xffffffffu, cells, d); tasks += __shfl_xor_sync(0xffffffffu, tasks, d); }
    if ((threadIdx.x & 31) == 0 && tasks) { atomicAdd(&counters[11], cells); atomicAdd(&counters[12], tasks); }
}

__global__ void k_left_tasks(const mp_candidate *__restrict__ cands, uint32_t n, const uint32_t *__restrict__ lens,
                             uint64_t fullLen, int strandLeft, MpDpTask *__restrict__ tasks, unsigned long long *__restrict__ counters)
{
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) { account_work(0, 0, counters); return; }
    mp_candidate ci = cands[c];
    uint32_t readLength = lens[ci.readIDLeft];
    uint32_t margin = MP_MARGIN(readLength);
    uint64_t start = ci.pos[0] - margin;
    if (start >= fullLen) start = 0;
    uint32_t dnaLen = readLength + margin * 2;
    if (start + dnaLen > fullLen) dnaLen = (uint32_t)(fullLen - start);
    MpDpTask t; t.refStart = start; t.refLen = dnaLen; t.readID = ci.readIDLeft; t.readLen = (uint16_t)readLength;
    t.strand = (uint8_t)strandLeft; t.valid = 1; t.cutoff = dp_cutoff(readLength);
    t.diag = (int16_t)min((uint64_t)ci.pos[0] - start, (uint64_t)0x7fff); t.pad_ = 0;     // the seed's diagonal inside the window (hint only)
    tasks[c] = t;
    account_work((unsigned long long)dnaLen * readLength, 1, counters);
}
// ---- packRight (DV-DPfunctions.cpp:2926-3007) ----
__global__ void k_right_tasks(const mp_candidate *__restrict__ cands, uint32_t n, const uint32_t *__restrict__ lens,
                              uint64_t fullLen, int strandRight, int insert_high, const MpDpTask *__restrict__ left,
                              const MpDpOut *__restrict__ leftOut, MpDpTask *__restrict__ tasks, unsigned long long *__restrict__ counters)
{
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) { account_work(0, 0, counters); return; }
    mp_candidate ci = cands[c];
    MpDpTask t; memset(&t, 0, sizeof t);
    if (leftOut[c].score >= left[c].cutoff) {
        uint32_t readIDRight = ci.readIDLeft ^ 1u;
        uint32_t readLength = lens[readIDRight];
        uint32_t margin = MP_MARGIN(readLength);
        uint64_t start = ci.pos[1] - margin;
        if (start >= fullLen) start = 0;
        uint32_t dnaLen = readLength + margin * 2;
        if (start + dnaLen > fullLen) dnaLen = (uint32_t)(fullLen - start);
        uint64_t hitPosLeft = left[c].refStart + leftOut[c].hitLoc;
        uint64_t bounded = hitPosLeft + (uint64_t)(int64_t)insert_high - start;     // restrict maximum insert size
        if (bounded < dnaLen) dnaLen = (uint32_t)bounded;
        t.refStart = start; t.refLen = dnaLen; t.readID = readIDRight; t.readLen = (uint16_t)readLength;
        t.strand = (uint8_t)strandRight; t.valid = 1; t.cutoff = dp_cutoff(readLength);
        t.diag = (int16_t)min((uint64_t)ci.pos[1] - start, (uint64_t)0x7fff);
    }
    tasks[c] = t;
    account_work(t.valid ? (unsigned long long)t.refLen * t.readLen : 0ull, t.valid ? 1ull : 0ull, counters);
}

__global__ void k_assemble_measure(uint32_t n, const MpDpTask *__restrict__ lt, const MpDpOut *__restrict__ lo,
                                   const MpDpTask *__restrict__ rt, const MpDpOut *__restrict__ ro,
                                   uint32_t *__restrict__ okFlag, uint32_t *__restrict__ cigBytes, uint32_t *__restrict__ leftLen)
{
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    bool ok = lo[c].score >= lt[c].cutoff && rt[c].valid && ro[c].score >= rt[c].cutoff;
    uint32_t bytes = 0;
    if (ok) {
        bytes = (uint32_t)lo[c].cigLen + 1 + ro[c].cigLen + 1;
        leftLen[c] = lo[c].cigLen;
    }
    okFlag[c] = ok; cigBytes[c] = bytes;
}

struct AsmParams { int match, mm, open, ext, strandLeft, strandRight, insert_low; uint32_t maxDNALength; };

__global__ void k_assemble_write(uint32_t n, const mp_candidate *__restrict__ cands, const MpDpTask *__restrict__ lt,
                                 const MpDpOut *__restrict__ lo, const MpDpTask *__restrict__ rt, const MpDpOut *__restrict__ ro,
                                 const uint8_t *__restrict__ lpat, const uint8_t *__restrict__ rpat, uint32_t patStride,
                                 AsmParams A, const uint32_t *__restrict__ okFlag, const uint32_t *__restrict__ outIdx,
                                 const uint32_t *__restrict__ cigOff, const uint32_t *__restrict__ leftLen, uint32_t *__restrict__ totals, uint32_t cigCap,
                                 mp_pair_result *__restrict__ res, char *__restrict__ cig, uint8_t *__restrict__ alignedPair)
{
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || !okFlag[c]) return;
    // results and CIGAR text of all chunks of a batch go to one device arena each; totals[0] / totals[1] hold what earlier chunks used
    // (k_add_totals), so no host round trip is needed between chunks
    const uint32_t resBase = totals[0], cigBase = totals[1];
    if ((uint64_t)cigBase + cigOff[c + 1] > cigCap) { totals[4] = 1; return; }            // arena too small: the host re-runs the stage with room
    // index 0 = left leg, 1 = right leg (DV-DPfunctions.cpp:3432-3530)
    const uint8_t *pat[2] = { lpat + (size_t)c * patStride, rpat + (size_t)c * patStride };
    const MpDpTask *tk[2] = { lt + c, rt + c };
    const MpDpOut *ou[2] = { lo + c, ro + c };
    int editdist[2], DIS[2]; uint32_t cigPos[2];
    uint32_t off = cigBase + cigOff[c];
    const int lengths_i = rt[c].readLen;                // batch->lengths[i] was overwritten by packRight
    for (int s = 0; s < 2; ++s) {
        const CigStats m = leg_stats(*ou[s]);
        leg_text(*ou[s], pat[s], patStride, A.open, A.ext, cig + off);
        cig[off + m.textLen] = 0;
        cigPos[s] = off;
        off += m.textLen + 1;
        int L = lengths_i - m.nI - m.nS;
        int numMis = (L * A.match + m.gapPenalty - ou[s]->score) / (A.match - A.mm);
        editdist[s] = m.nI + m.nD + numMis;
        DIS[s] = m.nD - m.nI - m.nS;
    }
    uint32_t readIDLeft = cands[c].readIDLeft;
    int readSide = readIDLeft & 1, mateSide = 1 - readSide;
    mp_pair_result r; memset(&r, 0, sizeof r);
    r.readID = readIDLeft - readSide;
    r.strand_1 = (uint8_t)(readSide == 0 ? A.strandLeft : A.strandRight);
    r.strand_2 = (uint8_t)(mateSide == 0 ? A.strandLeft : A.strandRight);
    r.algnmt_1 = tk[readSide]->refStart + ou[readSide]->hitLoc;
    r.algnmt_2 = tk[mateSide]->refStart + ou[mateSide]->hitLoc;
    r.cigar_1 = cigPos[readSide]; r.cigar_2 = cigPos[mateSide];
    r.score_1 = ou[readSide]->score; r.score_2 = ou[mateSide]->score;
    r.editdist_1 = editdist[readSide]; r.editdist_2 = editdist[mateSide];
    r.startPos_1 = (uint32_t)tk[readSide]->refStart;      // unsigned int in the reference (PEAlgnmt.h:521)
    r.startPos_2 = tk[mateSide]->refStart;
    r.refDpLength_1 = tk[readSide]->refLen; r.refDpLength_2 = tk[mateSide]->refLen;
    // anchors (DV-DPfunctions.cpp:2885-2886, 2987-2990)
    uint64_t hitPosLeft = lt[c].refStart + lo[c].hitLoc;
    long long rightAnchor = (long long)(hitPosLeft + (uint64_t)(int64_t)A.insert_low - rt[c].refStart);
    uint32_t la[2] = { A.maxDNALength, A.maxDNALength }, ra[2] = { 0u, (uint32_t)(rightAnchor > 0 ? rightAnchor : 0) };
    r.peLeftAnchor_1 = la[readSide]; r.peLeftAnchor_2 = la[mateSide];
    r.peRightAnchor_1 = ra[readSide]; r.peRightAnchor_2 = ra[mateSide];
    if (r.algnmt_1 < r.algnmt_2) r.insertSize = (int32_t)(r.algnmt_2 - r.algnmt_1 + (uint64_t)(int64_t)lengths_i + (uint64_t)(int64_t)DIS[1]);
    else r.insertSize = (int32_t)(r.algnmt_1 - r.algnmt_2 + (uint64_t)(int64_t)lengths_i + (uint64_t)(int64_t)DIS[1]);
    r.num_sameScore_1 = (int32_t)ou[readSide]->count; r.num_sameScore_2 = (int32_t)ou[mateSide]->count;
    res[resBase + outIdx[c]] = r;
    alignedPair[r.readID >> 1] = 1;
}
// totals: [0] results so far, [1] CIGAR bytes so far, [2] results kept after dedup, [3] pairs with a result, [4] arena overflow flag
__global__ void k_add_totals(const uint32_t *__restrict__ idxTotal, const uint32_t *__restrict__ offTotal, uint32_t *__restrict__ totals)
{
    totals[0] += *idxTotal; totals[1] += *offTotal;
}

// ---- per pair: OutputBuffer::ready (DV-DPfunctions.h:198-243 -> arrayCopyNRemoveDuplicate :167-196, ResultCompare .cpp:253-258):
//      stable sort of the pair's results by (algnmt_1, algnmt_2, score_1, score_2), exact duplicates dropped; then the best-hit choice
//      of outputDeepDPResult2 (OutputDPResult.cpp:156-232, alignmentType ALL_VALID): the FIRST result with the maximal score_1 + score_2
//      is marked (pad = 1).  One thread per pair group (groups are contiguous: candidates are sorted by read id); a group is a handful
//      of records, so an in-place insertion sort is the right tool. ----
__device__ __forceinline__ bool pair_key_less(const mp_pair_result &a, const mp_pair_result &b)
{
    if (a.algnmt_1 != b.algnmt_1) return a.algnmt_1 < b.algnmt_1;
    if (a.algnmt_2 != b.algnmt_2) return a.algnmt_2 < b.algnmt_2;
    if (a.score_1 != b.score_1) return a.score_1 < b.score_1;
    return a.score_2 < b.score_2;
}
__global__ void k_pair_ready(mp_pair_result *__restrict__ res, uint32_t *__restrict__ totals, uint32_t *__restrict__ keep)
{
    const uint32_t total = totals[0];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t pairs = 0, kept = 0;
    if (i < total && (i == 0 || res[i - 1].readID != res[i].readID)) {
        uint32_t e = i + 1;
        while (e < total && res[e].readID == res[i].readID) ++e;
        for (uint32_t a = i + 1; a < e; ++a) {                 // stable insertion sort
            mp_pair_result key = res[a]; uint32_t b = a;
            while (b > i && pair_key_less(key, res[b - 1])) { res[b] = res[b - 1]; --b; }
            if (b != a) res[b] = key;
        }
        uint32_t lastKept = i, best = i; int bestSum = res[i].score_1 + res[i].score_2;
        keep[i] = 1; kept = 1;
        for (uint32_t a = i + 1; a < e; ++a) {
            const bool k = pair_key_less(res[lastKept], res[a]);
            keep[a] = k;
            if (k) {
                lastKept = a; ++kept;
                const int sum = res[a].score_1 + res[a].score_2;
                if (sum > bestSum) { bestSum = sum; best = a; }
            }
        }
        for (uint32_t a = i; a < e; ++a) res[a].pad = a == best ? 1 : 0;
        pairs = 1;
    }
    pairs = __reduce_add_sync(0xffffffffu, pairs); kept = __reduce_add_sync(0xffffffffu, kept);
    if ((threadIdx.x & 31) == 0 && pairs) { atomicAdd(&totals[3], pairs); atomicAdd(&totals[2], kept); }
}
__global__ void k_pair_compact(const mp_pair_result *__restrict__ res, const uint32_t *__restrict__ totals, const uint32_t *__restrict__ keep,
                               const uint32_t *__restrict__ pos, mp_pair_result *__restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < totals[0] && keep[i]) out[pos[i]] = res[i];
}

static int scan_u32(mp_context *ctx, const uint32_t *in, uint32_t *out, uint64_t n)
{
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, (int64_t)n, ctx->stream);
    if (ctx->dScanTmp.reserve(tb)) return MP_ERR_CUDA;
    cub::DeviceScan::ExclusiveSum(ctx->dScanTmp.p, tb, in, out, (int64_t)n, ctx->stream);
    return 0;
}

// ---- stage S1 over all candidates, in chunks ----
static int deep_dp(mp_context *ctx, const mp_align_params *P, mp_results *out, uint64_t &cells, uint64_t &tasksRun)
{
    cudaStream_t st = ctx->stream;
    const uint64_t nC = ctx->nCands;
    const uint32_t inputMax = (uint32_t)P->maxReadLength;
    const uint32_t maxReadLength = (inputMax / 4 + 1) * 4;                       // DV-DPfunctions.cpp:3166-3167
    const uint32_t maxDNALength = maxReadLength + 2 * MP_MARGIN(inputMax) + 8;
    const uint32_t patStride = (maxDNALength + maxReadLength + 3) & ~3u;         // word-aligned rows: k_dp_tb stores four pattern bytes at a time
    MpDpParams dpl, dpr;
    // softClipLtSizes/RtSizes per leg (DV-DPfunctions.cpp:2908-2911, 2994-2997); callDP uses task 0's pair
    dpl.mismatch = dpr.mismatch = P->mismatchScore; dpl.open = dpr.open = P->openGapScore;
    dpl.clipLt = P->peStrandLeftLeg == 1 ? P->softClipLeft : P->softClipRight;
    dpl.clipRt = P->peStrandLeftLeg == 1 ? P->softClipRight : P->softClipLeft;
    dpr.clipLt = P->peStrandRightLeg == 1 ? P->softClipLeft : P->softClipRight;
    dpr.clipRt = P->peStrandRightLeg == 1 ? P->softClipRight : P->softClipLeft;
    AsmParams A; A.match = P->matchScore; A.mm = P->mismatchScore; A.open = P->openGapScore; A.ext = P->extendGapScore;
    A.strandLeft = P->peStrandLeftLeg; A.strandRight = P->peStrandRightLeg; A.insert_low = P->insert_low; A.maxDNALength = maxDNALength;

    const uint32_t CH = 1u << 18;
    DevBuf &dLT = ctx->dLT, &dRT = ctx->dRT, &dLO = ctx->dLO, &dRO = ctx->dRO, &dLP = ctx->dLP, &dRP = ctx->dRP, &dOk = ctx->dOk,
           &dBytes = ctx->dBytes, &dIdx = ctx->dIdx, &dOff = ctx->dOff, &dRes = ctx->dRes, &dCig = ctx->dCig;
    // full-size chunk buffers unless the whole batch is small: batch-to-batch variation must not re-allocate
    uint32_t chunkCap = (uint32_t)std::min<uint64_t>(CH, std::max<uint64_t>((nC + nC / 4 + 1024), 1));
    const size_t resCap = (size_t)nC + nC / 8 + 1024;                         // one result per candidate at most
    if (dLT.reserve((size_t)chunkCap * sizeof(MpDpTask)) || dRT.reserve((size_t)chunkCap * sizeof(MpDpTask)) ||
        dLO.reserve((size_t)chunkCap * sizeof(MpDpOut)) || dRO.reserve((size_t)chunkCap * sizeof(MpDpOut)) ||
        dLP.reserve((size_t)chunkCap * patStride) || dRP.reserve((size_t)chunkCap * patStride) ||
        dOk.reserve(((size_t)chunkCap + 1) * 4) || dBytes.reserve(((size_t)chunkCap + 1) * 4 * 2) ||
        dIdx.reserve(((size_t)chunkCap + 1) * 4) || dOff.reserve(((size_t)chunkCap + 1) * 4) ||
        dRes.reserve(resCap * sizeof(mp_pair_result)) || ctx->dRes2.reserve(resCap * sizeof(mp_pair_result)) ||
        ctx->dKeep.reserve((resCap + 1) * 4) || ctx->dKeepPos.reserve((resCap + 1) * 4) || ctx->dTotals.reserve(8 * 4)) return MP_ERR_CUDA;
    PinnedBuf<mp_pair_result> &H = ctx->hPairs;
    PinnedBuf<char> &HC = ctx->hCigars;
    unsigned long long *dCnt = ctx->dCounters.as<unsigned long long>();
    uint32_t *dTot = ctx->dTotals.as<uint32_t>();
    if (ctx->dAligned.reserve((size_t)ctx->nReads / 2 + 8)) return MP_ERR_CUDA;
    const uint64_t fullLen = ctx->ix.n;
    MpTrace tr;
    // CIGAR arena of the batch: ~12 bytes per result on clean reads, a few dozen on divergent ones.  If a batch needs more, the stage
    // is run again with the size it asked for (the DP patterns of earlier chunks are gone by then).
    size_t cigCap = std::max<size_t>(ctx->dCig.cap, std::max<size_t>((size_t)resCap * 40, (size_t)1 << 20));
    uint32_t tot[8] = { 0 };
    for (int attempt = 0; attempt < 3; ++attempt) {
        if (cigCap > 0xFFFFFFF0ull) { mp_set_error("CIGAR arena of one batch exceeds 4 GB; use smaller batches"); return MP_ERR_CAPACITY; }
        if (dCig.reserve(cigCap)) return MP_ERR_CUDA;
        MP_CUDA(cudaMemsetAsync(dTot, 0, 8 * 4, st));
        MP_CUDA(cudaMemsetAsync(ctx->dAligned.p, 0, (size_t)ctx->nReads / 2 + 8, st));
        MP_CUDA(cudaMemsetAsync(dCnt + 11, 0, 16, st));                        // work accounting of k_left_tasks / k_right_tasks
        for (uint64_t base = 0; base < nC; base += CH) {
            uint32_t n = (uint32_t)std::min<uint64_t>(CH, nC - base);
            const mp_candidate *cands = ctx->dCands.as<mp_candidate>() + base;
            unsigned g = (n + 127) / 128;
            (++g_mp_launches), k_left_tasks<<<g, 128, 0, st>>>(cands, n, ctx->dLens.as<uint32_t>(), fullLen, P->peStrandLeftLeg, dLT.as<MpDpTask>(), dCnt);
            if (int rc = mpd_run_tasks(ctx, dLT.as<MpDpTask>(), n, maxDNALength, maxReadLength, dpl, dLO.as<MpDpOut>(), dLP.as<uint8_t>(), patStride)) return rc;
            (++g_mp_launches), k_right_tasks<<<g, 128, 0, st>>>(cands, n, ctx->dLens.as<uint32_t>(), fullLen, P->peStrandRightLeg, P->insert_high,
                                             dLT.as<MpDpTask>(), dLO.as<MpDpOut>(), dRT.as<MpDpTask>(), dCnt);
            if (int rc = mpd_run_tasks(ctx, dRT.as<MpDpTask>(), n, maxDNALength, maxReadLength, dpr, dRO.as<MpDpOut>(), dRP.as<uint8_t>(), patStride)) return rc;
            if (tr.sync) cudaStreamSynchronize(st);
            tr.mark(" dp left+right (enqueue)");
            MP_CUDA(cudaMemsetAsync(dOk.p, 0, ((size_t)n + 1) * 4, st));
            MP_CUDA(cudaMemsetAsync(dBytes.p, 0, ((size_t)n + 1) * 4, st));
            (++g_mp_launches), k_assemble_measure<<<g, 128, 0, st>>>(n, dLT.as<MpDpTask>(), dLO.as<MpDpOut>(), dRT.as<MpDpTask>(), dRO.as<MpDpOut>(),
                                                  dOk.as<uint32_t>(), dBytes.as<uint32_t>(), dBytes.as<uint32_t>() + chunkCap + 1);
            if (scan_u32(ctx, dOk.as<uint32_t>(), dIdx.as<uint32_t>(), (uint64_t)n + 1)) return MP_ERR_CUDA;
            if (scan_u32(ctx, dBytes.as<uint32_t>(), dOff.as<uint32_t>(), (uint64_t)n + 1)) return MP_ERR_CUDA;
            (++g_mp_launches), k_assemble_write<<<g, 128, 0, st>>>(n, cands, dLT.as<MpDpTask>(), dLO.as<MpDpOut>(), dRT.as<MpDpTask>(), dRO.as<MpDpOut>(),
                                                dLP.as<uint8_t>(), dRP.as<uint8_t>(), patStride, A, dOk.as<uint32_t>(), dIdx.as<uint32_t>(),
                                                dOff.as<uint32_t>(), dBytes.as<uint32_t>() + chunkCap + 1, dTot, (uint32_t)cigCap, dRes.as<mp_pair_result>(), dCig.as<char>(),
                                                ctx->dAligned.as<uint8_t>());
            (++g_mp_launches), k_add_totals<<<1, 1, 0, st>>>(dIdx.as<uint32_t>() + n, dOff.as<uint32_t>() + n, dTot);
            MP_CUDA(cudaGetLastError());
            tr.mark(" assemble (enqueue)");
        }
        // ---- per pair: sort, drop exact duplicates, mark the best pair; compact ----
        if (nC) {
            const unsigned g = (unsigned)((nC + 127) / 128);
            MP_CUDA(cudaMemsetAsync(ctx->dKeep.p, 0, (resCap + 1) * 4, st));
            (++g_mp_launches), k_pair_ready<<<g, 128, 0, st>>>(dRes.as<mp_pair_result>(), dTot, ctx->dKeep.as<uint32_t>());
            if (scan_u32(ctx, ctx->dKeep.as<uint32_t>(), ctx->dKeepPos.as<uint32_t>(), (uint64_t)nC + 1)) return MP_ERR_CUDA;
            (++g_mp_launches), k_pair_compact<<<g, 128, 0, st>>>(dRes.as<mp_pair_result>(), dTot, ctx->dKeep.as<uint32_t>(), ctx->dKeepPos.as<uint32_t>(),
                                                                 ctx->dRes2.as<mp_pair_result>());
            MP_CUDA(cudaGetLastError());
        }
        MP_CUDA(cudaMemcpyAsync(tot, dTot, sizeof tot, cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaStreamSynchronize(st));                                    // the one host round trip of stage S1
        tr.mark(" s1 device work");
        if (!tot[4]) break;
        cigCap = (size_t)tot[1] + tot[1] / 8 + (1 << 20);                       // the arena was too small: run the stage again with room
        if (attempt == 2) { mp_set_error("CIGAR arena overflowed repeatedly"); return MP_ERR_CAPACITY; }
    }
    const uint32_t nKept = tot[2], nBytes = tot[1];
    if (H.resize(nKept) || HC.resize(nBytes)) return MP_ERR_CUDA;
    if (nKept && !ctx->resultsOnDevice) MP_CUDA(cudaMemcpyAsync(H.data(), ctx->dRes2.p, (size_t)nKept * sizeof(mp_pair_result), cudaMemcpyDeviceToHost, st));
    if (nBytes && !ctx->resultsOnDevice) MP_CUDA(cudaMemcpyAsync(HC.data(), dCig.p, nBytes, cudaMemcpyDeviceToHost, st));
    {   // cells / tasks counted on the device by k_left_tasks / k_right_tasks
        unsigned long long hc2[2];
        MP_CUDA(cudaMemcpyAsync(hc2, dCnt + 11, sizeof hc2, cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaStreamSynchronize(st));
        cells += hc2[0]; tasksRun += hc2[1];
    }
    tr.mark(" s1 download");
    out->numDPAlignedPair = tot[3]; out->numDPAlignment = nKept;
    return 0;
}

// =====================================================================================
// C-ABI
// =====================================================================================
extern "C" int mp_init(int device, mp_context **pctx)
{
    if (!pctx) { mp_set_error("mp_init: null argument"); return MP_ERR_ARG; }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) { mp_set_error("mp_init: no CUDA device (%s); there is no CPU fallback", cudaGetErrorString(e)); return MP_ERR_CUDA; }
    if (device < 0 || device >= count) { mp_set_error("mp_init: device %d out of range (%d devices)", device, count); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(device));
    {   // MP_L2_FETCH=32|64|128: optional L2 fill-granularity hint (measured: no effect on the scattered-read kernels here)
        const char *e = getenv("MP_L2_FETCH");
        size_t g = e ? (size_t)atoi(e) : 0;
        if (g == 32 || g == 64 || g == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, g);
    }
    mp_context *ctx = new mp_context;
    memset(&ctx->ix, 0, sizeof ctx->ix);
    for (int i = 0; i < 8; ++i) ctx->ev[i] = nullptr;
    ctx->device = device;
    cudaError_t ce = cudaStreamCreate(&ctx->stream);
    for (int i = 0; i < 8 && ce == cudaSuccess; ++i) ce = cudaEventCreate(&ctx->ev[i]);
    if (ce != cudaSuccess) {
        mp_set_error("mp_init: CUDA error %s: %s", cudaGetErrorName(ce), cudaGetErrorString(ce));
        for (int i = 0; i < 8; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return MP_ERR_CUDA;
    }
    *pctx = ctx;
    return 0;
}
extern "C" int mp_clone(mp_context *src, mp_context **pctx)
{
    if (!src || !pctx) { mp_set_error("mp_clone: null argument"); return MP_ERR_ARG; }
    if (!src->hasIndex) { mp_set_error("mp_clone: the source context has no index"); return MP_ERR_STATE; }
    if (int rc = mp_init(src->device, pctx)) return rc;
    mp_context *c = *pctx;
    c->ix = src->ix; c->saInterval = src->saInterval; c->hbmBytes = src->hbmBytes;
    c->hasIndex = true; c->sharedIndex = true;
    c->bloomK = src->bloomK; c->bloomStride = src->bloomStride; c->bloomSeedMin = src->bloomSeedMin; c->bloomWords = src->bloomWords; c->bloomFor = src->bloomFor;
    c->dBloom.p = src->dBloom.p; c->dBloom.cap = 0;          // borrowed: never freed or grown by the clone
    return 0;
}
extern "C" void mp_destroy(mp_context *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->sharedIndex && ctx->dBloom.cap == 0) ctx->dBloom.p = nullptr;
    for (cudaEvent_t e : ctx->evPool) cudaEventDestroy(e);
    DevBuf *bufs[] = { &ctx->dBlocks, &ctx->dSuper, &ctx->dSa, &ctx->dSa32, &ctx->dSa40Lo, &ctx->dSa40Hi, &ctx->dBloom, &ctx->dLkt, &ctx->dPac, &ctx->dReadsIl, &ctx->dReads, &ctx->dLens,
                       &ctx->dCounters, &ctx->dSeeds, &ctx->dStubs, &ctx->dHitsPerRead, &ctx->dHitStart, &ctx->dCursor, &ctx->dHits, &ctx->dHits2,
                       &ctx->dSeedPos, &ctx->dNPos, &ctx->dNNeg, &ctx->dCandCount, &ctx->dCandStart, &ctx->dCands, &ctx->dScanTmp,
                       &ctx->dTasks, &ctx->dRefSeq, &ctx->dReadSeq, &ctx->dTable, &ctx->dFill, &ctx->dPattern, &ctx->dDpOut,
                       &ctx->dLT, &ctx->dRT, &ctx->dLO, &ctx->dRO, &ctx->dLP, &ctx->dRP, &ctx->dOk, &ctx->dBytes, &ctx->dIdx, &ctx->dOff,
                       &ctx->dRes, &ctx->dCig, &ctx->dExFlag, &ctx->dExPos, &ctx->dExIdx, &ctx->dAligned, &ctx->dGather, &ctx->dHintTest, &ctx->dRes2, &ctx->dKeep, &ctx->dKeepPos, &ctx->dTotals, &ctx->dS2Counts, &ctx->dS2Start, &ctx->dS2Tasks, &ctx->dS2Res,
                       &ctx->dRsSlotTasks, &ctx->dRsSlotInfo, &ctx->dRsFlag, &ctx->dRsPos, &ctx->dRsTasks, &ctx->dRsInfo, &ctx->dRsRec, &ctx->dRsOut, &ctx->dRsKeep, &ctx->dRsKeepPos,
                       &ctx->dFqText, &ctx->dFqCnt, &ctx->dFqCntPos, &ctx->dFqLines, &ctx->dFqRec, &ctx->dFqFlags, &ctx->dAnnGrid, &ctx->dAnnTrStart, &ctx->dAnnTrChr,
                       &ctx->dAnnNames, &ctx->dAnnNameOff, &ctx->dFmtKeys, &ctx->dFmtGroups, &ctx->dFmtRecLen, &ctx->dFmtTail, &ctx->dFmtTailText, &ctx->dFmtSeg, &ctx->dFmtDst, &ctx->dFmtLen, &ctx->dFmtOff, &ctx->dFmtOut,
                       &ctx->dBgzfIn, &ctx->dBgzfSlots, &ctx->dBgzfOut, &ctx->dBgzfSizes, &ctx->dBgzfOffs, &ctx->dBgzfScratch };
    for (DevBuf *b : bufs) b->release();
    for (int i = 0; i < 8; ++i) cudaEventDestroy(ctx->ev[i]);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}
extern "C" int mp_index_load(mp_context *ctx, const char *prefix)
{
    if (!ctx || !prefix) { mp_set_error("mp_index_load: null argument"); return MP_ERR_ARG; }
    return mpi_load(ctx, prefix);
}
extern "C" int mp_index_info(mp_context *ctx, uint64_t *textLength, uint64_t *inverseSa0, uint64_t cumFreq[5], uint64_t *hbmBytes)
{
    if (!ctx || !ctx->hasIndex) { mp_set_error("mp_index_info: no index loaded"); return MP_ERR_STATE; }
    if (textLength) *textLength = ctx->ix.n;
    if (inverseSa0) *inverseSa0 = ctx->ix.inverseSa0;
    if (cumFreq) for (int i = 0; i < 5; ++i) cumFreq[i] = ctx->ix.cum[i];
    if (hbmBytes) *hbmBytes = ctx->hbmBytes;
    return 0;
}
extern "C" int mp_batch_upload(mp_context *ctx, const uint32_t *queries, const uint32_t *readLengths, uint32_t nReads, uint32_t wordPerQuery)
{
    if (!ctx || !queries || !readLengths) { mp_set_error("mp_batch_upload: null argument"); return MP_ERR_ARG; }
    if (nReads == 0 || (nReads & 1) || wordPerQuery == 0) { mp_set_error("mp_batch_upload: nReads must be even and non-zero"); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(ctx->device));
    return mps_upload(ctx, queries, readLengths, nReads, wordPerQuery);
}
extern "C" int mp_seed_pairs(mp_context *ctx, const mp_align_params *params)
{
    if (!ctx || !params) { mp_set_error("mp_seed_pairs: null argument"); return MP_ERR_ARG; }
    if (!ctx->hasIndex || !ctx->hasBatch) { mp_set_error("mp_seed_pairs: index and batch must be loaded first"); return MP_ERR_STATE; }
    if (params->peStrandLeftLeg != 1 || params->peStrandRightLeg != 2) { mp_set_error("only StrandArrangement +/- is supported"); return MP_ERR_ARG; }
    if ((int64_t)ctx->maxLenBatch >= (int64_t)params->maxReadLength) {          // the reference truncates reads to -L - 1 (QueryParser.cpp:188)
        mp_set_error("the batch holds a read of %u bases but maxReadLength is %d (reads must be shorter)", ctx->maxLenBatch, params->maxReadLength);
        return MP_ERR_ARG;
    }
    MP_CUDA(cudaSetDevice(ctx->device));
    return mps_seed_pairs(ctx, params);
}
extern "C" int mp_download_seedpos(mp_context *ctx, mp_seed_pos **readPos, uint64_t *nReadPos, mp_seed_pos **matePos, uint64_t *nMatePos)
{
    if (!ctx || !ctx->seeded) { mp_set_error("mp_download_seedpos: mp_seed_pairs has not run"); return MP_ERR_STATE; }
    return mps_download_seedpos(ctx, readPos, nReadPos, matePos, nMatePos);
}
extern "C" int mp_download_candidates(mp_context *ctx, mp_candidate **cands, uint64_t *nCands)
{
    if (!ctx || !ctx->seeded) { mp_set_error("mp_download_candidates: mp_seed_pairs has not run"); return MP_ERR_STATE; }
    *nCands = ctx->nCands;
    *cands = (mp_candidate *)malloc((ctx->nCands + 1) * sizeof(mp_candidate));
    if (ctx->nCands) MP_CUDA(cudaMemcpy(*cands, ctx->dCands.p, ctx->nCands * sizeof(mp_candidate), cudaMemcpyDeviceToHost));
    return 0;
}
extern "C" void mp_free(void *p) { free(p); }

extern "C" void mp_default_params(mp_align_params *p, int nt2)
{
    memset(p, 0, sizeof *p);
    p->mmp.seedSAsizeThreshold = 30; p->mmp.seedMinLength = nt2 ? 17 : 22; p->mmp.uniqThreshold = 6; p->mmp.indelFuzz = 5;
    p->mmp.goodSeedLen = 27; p->mmp.reseedLen = nt2 ? 18 : 23; p->mmp.reseedRLTratio = 0.7; p->mmp.reseedAbsDiff = 4;
    p->mmp.shortSeedRatio = 0.5;
    p->matchScore = 1; p->mismatchScore = -2; p->openGapScore = -3; p->extendGapScore = -1;
    p->softClipLeft = 130; p->softClipRight = 130;
    p->insert_low = 1; p->insert_high = 500;
    p->peStrandLeftLeg = 1; p->peStrandRightLeg = 2; p->skipDefaultDP = 0; p->maxReadLength = 120;
}

// SemiGlobalAligner::performAlignment seam (CPU_DPfunctions.h:103-111)
extern "C" int mp_dp_batch(mp_context *ctx,
                           const uint32_t *packedDNA, const uint32_t *DNALengths, uint32_t maxDNALength,
                           const uint32_t *packedRead, const uint32_t *readLengths, uint32_t maxReadLength,
                           const int32_t *cutoffs, int32_t *scores, uint32_t *hitLocs, uint32_t *maxScoreCounts,
                           uint8_t *pattern, uint32_t n, const uint32_t *clipLt, const uint32_t *clipRt,
                           int32_t mismatchScore, int32_t openGapScore)
{
    if (!ctx || !packedDNA || !DNALengths || !packedRead || !readLengths || !cutoffs || !scores || !hitLocs || !maxScoreCounts || !pattern || !clipLt || !clipRt) {
        mp_set_error("mp_dp_batch: null argument"); return MP_ERR_ARG;
    }
    if (mismatchScore > -2 || mismatchScore <= openGapScore * 2 || mismatchScore < -4 || openGapScore < -6 || openGapScore >= -1) {
        mp_set_error("mp_dp_batch: score parameters outside the supported range (CPU_DP.cpp:199-208; mismatch = -1 divides by zero at CPU_DP.cpp:310, and for mismatch == 2 * open the reference traceback prefers I over D where the plain recurrence ties: unpinned, refused)"); return MP_ERR_ARG;
    }
    if (n == 0) return 0;
    for (uint32_t t = 0; t < n; ++t)
        if (DNALengths[t] > maxDNALength || readLengths[t] > maxReadLength) {
            mp_set_error("mp_dp_batch: task %u has lengths (%u, %u) above the stated maxima (%u, %u)", t, DNALengths[t], readLengths[t], maxDNALength, maxReadLength);
            return MP_ERR_ARG;
        }
    MP_CUDA(cudaSetDevice(ctx->device));
    const uint32_t wDNA = (maxDNALength + 15) >> 4, wRead = (maxReadLength + 15) >> 4;
    // un-interleave into one byte per base (host side of the seam; the kernels take bytes)
    std::vector<uint8_t> hRef((size_t)n * maxDNALength), hRead((size_t)n * maxReadLength);
    for (uint32_t t = 0; t < n; ++t) {
        size_t dT = (size_t)(t / 32) * 32 * wDNA + (t % 32), rT = (size_t)(t / 32) * 32 * wRead + (t % 32);
        for (uint32_t i = 1; i <= DNALengths[t] && i <= maxDNALength; ++i)
            hRef[(size_t)t * maxDNALength + i - 1] = (packedDNA[dT + ((i >> 4) << 5)] >> ((15 - (i & 15)) << 1)) & 3;
        for (uint32_t i = 1; i <= readLengths[t] && i <= maxReadLength; ++i)
            hRead[(size_t)t * maxReadLength + i - 1] = (packedRead[rT + ((i >> 4) << 5)] >> ((15 - (i & 15)) << 1)) & 3;
    }
    DevBuf dRef, dRead, dRL, dDL, dCo, dOut, dPat;
    const uint32_t patStride = maxDNALength + maxReadLength;
    if (dRef.reserve(hRef.size()) || dRead.reserve(hRead.size()) || dRL.reserve((size_t)n * 4) || dDL.reserve((size_t)n * 4) ||
        dCo.reserve((size_t)n * 4) || dOut.reserve((size_t)n * sizeof(MpDpOut)) || dPat.reserve((size_t)n * patStride)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpy(dRef.p, hRef.data(), hRef.size(), cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(dRead.p, hRead.data(), hRead.size(), cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(dDL.p, DNALengths, (size_t)n * 4, cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(dRL.p, readLengths, (size_t)n * 4, cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(dCo.p, cutoffs, (size_t)n * 4, cudaMemcpyHostToDevice));
    MpDpParams P; P.clipLt = (int)clipLt[0]; P.clipRt = (int)clipRt[0]; P.mismatch = mismatchScore; P.open = openGapScore;
    int rc = mpd_run_explicit(ctx, dRef.as<uint8_t>(), dDL.as<uint32_t>(), maxDNALength, dRead.as<uint8_t>(), dRL.as<uint32_t>(),
                              maxReadLength, dCo.as<int32_t>(), n, P, dOut.as<MpDpOut>(), dPat.as<uint8_t>(), patStride);
    if (rc) return rc;
    std::vector<MpDpOut> ho(n);
    std::vector<uint8_t> hp((size_t)n * patStride);
    MP_CUDA(cudaMemcpyAsync(ho.data(), dOut.p, (size_t)n * sizeof(MpDpOut), cudaMemcpyDeviceToHost, ctx->stream));
    MP_CUDA(cudaMemcpyAsync(hp.data(), dPat.p, hp.size(), cudaMemcpyDeviceToHost, ctx->stream));
    MP_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->evUsed = 0;
    for (uint32_t t = 0; t < n; ++t) {
        scores[t] = ho[t].score; hitLocs[t] = ho[t].hitLoc; maxScoreCounts[t] = ho[t].count;
        if (ho[t].patLen) memcpy(pattern + (size_t)t * patStride, hp.data() + (size_t)t * patStride, ho[t].patLen + 1);
    }
    dRef.release(); dRead.release(); dRL.release(); dDL.release(); dCo.release(); dOut.release(); dPat.release();
    return 0;
}

// Sizes every per-batch buffer for batches of up to nReads reads now.  All of them grow on demand anyway; but the first batch of a
// context would otherwise pay for a few dozen cudaMalloc / cudaMallocHost calls (tens of GB of traceback tables, pinned result
// arenas), and every one of them stalls the kernels of the other contexts on the same GPU while it runs.
extern "C" int mp_reserve(mp_context *ctx, const mp_align_params *P, uint32_t nReads)
{
    if (!ctx || !P || nReads == 0) { mp_set_error("mp_reserve: bad argument"); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(ctx->device));
    const uint32_t inputMax = (uint32_t)P->maxReadLength, wpq = (inputMax + 15) / 16;
    const uint64_t nPad = ((uint64_t)nReads + 31) / 32 * 32, nStrands = (uint64_t)nReads * 2, nPairs = nReads / 2;
    const uint32_t maxReadLength = (inputMax / 4 + 1) * 4, maxDNALength = maxReadLength + 2 * MP_MARGIN(inputMax) + 8;
    const uint32_t patStride = (maxDNALength + maxReadLength + 3) & ~3u;
    const uint32_t CH = (uint32_t)std::min<uint64_t>(1u << 18, nPairs + nPairs / 4 + 1024);
    const size_t resCap = (size_t)(nPairs + nPairs / 4) + 1024, hitSlots = (size_t)nReads * 3;
    if (ctx->capSeeds < nStrands * 4) ctx->capSeeds = nStrands * 4;
    if (ctx->capStubs < nStrands * 8) ctx->capStubs = nStrands * 8;
    const int K = maxReadLength <= 160 ? 5 : maxReadLength <= 256 ? 8 : 10;
    const size_t tableStride = (size_t)(((int)maxDNALength + 44) & ~3) * 32 * K;
    size_t freeB = 0, totalB = 0; cudaMemGetInfo(&freeB, &totalB);
    // stage S3 (mate rescue) aligns windows of up to insert_high + L bases: wider rows for the sequence / pattern buffers, and a
    // traceback table per task three to four times the size of a stage-S1 one.  Sized here for both, so that the first batch with many
    // rescue tasks does not free and re-allocate tens of GB (a cudaFree stalls every context of the GPU).
    const uint32_t maxDNALengthR = (uint32_t)std::max(P->insert_high, 0) + inputMax + 1, rStride = (maxDNALengthR + maxReadLength + 3) & ~3u;
    const uint32_t CH3 = (uint32_t)std::min<uint64_t>(1u << 17, (uint64_t)nReads + 1024);
    const bool big = CH >= (1u << 15);
    const size_t tableWant = std::min<size_t>(big ? (size_t)24 << 30 : (size_t)(CH + 1) * tableStride, std::min<size_t>((size_t)24 << 30, freeB / 2));
    const size_t refSeqWant = std::max<size_t>((((size_t)CH * maxDNALength + 15) & ~(size_t)15) + (size_t)CH * 14 + 16,
                                               big && !P->skipDefaultDP ? (((size_t)CH3 * maxDNALengthR + 15) & ~(size_t)15) + (size_t)CH3 * 14 + 16 : 0);
    const size_t patWant = std::max<size_t>((size_t)CH * patStride, big && !P->skipDefaultDP ? (size_t)CH3 * rStride : 0);
    if (ctx->dReadsIl.reserve(nPad * wpq * 4) || ctx->dReads.reserve(nPad * wpq * 4 + 64) || ctx->dLens.reserve((size_t)nReads * 4) ||
        ctx->dCounters.reserve(16 * 8) || ctx->dHitsPerRead.reserve(((size_t)nReads + 1) * 4) || ctx->dHitStart.reserve(((size_t)nReads + 1) * 4) ||
        ctx->dCursor.reserve(((size_t)nReads + 1) * 4) || ctx->dNPos.reserve((size_t)nReads * 4) || ctx->dNNeg.reserve((size_t)nReads * 4) ||
        ctx->dSeeds.reserve(ctx->capSeeds * sizeof(MpSeed)) || ctx->dStubs.reserve(ctx->capStubs * 4) ||
        ctx->dHits.reserve(hitSlots * sizeof(MpHit)) || ctx->dHits2.reserve(hitSlots * sizeof(MpHit)) || ctx->dSeedPos.reserve(hitSlots * sizeof(mp_seed_pos)) ||
        ctx->dCandCount.reserve(((size_t)nPairs + 1) * 4) || ctx->dCandStart.reserve(((size_t)nPairs + 1) * 4) ||
        ctx->dCands.reserve((size_t)nPairs * 2 * sizeof(mp_candidate)) ||
        ctx->dLT.reserve((size_t)CH * sizeof(MpDpTask)) || ctx->dRT.reserve((size_t)CH * sizeof(MpDpTask)) ||
        ctx->dLO.reserve((size_t)CH * sizeof(MpDpOut)) || ctx->dRO.reserve((size_t)CH * sizeof(MpDpOut)) ||
        ctx->dLP.reserve(patWant) || ctx->dRP.reserve((size_t)CH * patStride) ||
        ctx->dOk.reserve(((size_t)CH + 1) * 4) || ctx->dBytes.reserve(((size_t)CH + 1) * 8) || ctx->dIdx.reserve(((size_t)CH + 1) * 4) ||
        ctx->dOff.reserve(((size_t)CH + 1) * 4) || ctx->dRes.reserve(resCap * sizeof(mp_pair_result)) || ctx->dRes2.reserve(resCap * sizeof(mp_pair_result)) ||
        ctx->dKeep.reserve((resCap + 1) * 4) || ctx->dKeepPos.reserve((resCap + 1) * 4) || ctx->dTotals.reserve(16 * 4) ||
        ctx->dCig.reserve(std::max<size_t>(resCap * 40, (size_t)1 << 20)) || ctx->dAligned.reserve((size_t)nPairs + 8) ||
        ctx->dRefSeq.reserve(refSeqWant) || ctx->dReadSeq.reserve((size_t)CH * maxReadLength) ||
        ctx->dFill.reserve((size_t)CH * 16) || ctx->dExFlag.reserve(((size_t)CH + 1) * 4) || ctx->dExPos.reserve(((size_t)CH + 1) * 4) ||
        ctx->dExIdx.reserve(((size_t)CH + 1) * 4) || ctx->dScanTmp.reserve((size_t)1 << 20) || ctx->dS2Counts.reserve(((size_t)nReads + 1) * 4) || ctx->dS2Start.reserve(((size_t)nReads + 1) * 4) ||
        (ctx->dTable.cap < tableWant && ctx->dTable.reserve(tableWant))) return MP_ERR_CUDA;
    // stages S2 / S3: a guess (one pair in eight unplaced, a few tasks each); they grow on demand like everything else
    const size_t s2 = big ? (size_t)nReads / 4 : 0;
    if (s2 && (ctx->dS2Tasks.reserve(s2 * sizeof(MpDpTask)) || ctx->dS2Res.reserve(s2 * sizeof(mp_single_result)) ||
               ctx->dRsSlotTasks.reserve(s2 * sizeof(MpDpTask)) || ctx->dRsSlotInfo.reserve(s2 * 8) || ctx->dRsFlag.reserve((s2 + 1) * 4) ||
               ctx->dRsPos.reserve((s2 + 1) * 4) || ctx->dRsTasks.reserve(s2 * sizeof(MpDpTask)) || ctx->dRsInfo.reserve(s2 * 8) ||
               ctx->dRsRec.reserve(s2 * sizeof(mp_pair_result)) || ctx->dRsOut.reserve(s2 * sizeof(mp_pair_result)) ||
               ctx->dRsKeep.reserve((s2 + 1) * 4) || ctx->dRsKeepPos.reserve((s2 + 1) * 4))) return MP_ERR_CUDA;
    if (ctx->hPairs.reserve(resCap) || ctx->hCigars.reserve(resCap * 40) || (s2 && (ctx->hSingles.reserve(s2) || ctx->hRescued.reserve(s2 / 2)))) return MP_ERR_CUDA;
    return 0;
}

extern "C" int mp_align_pairs(mp_context *ctx, const mp_align_params *params, mp_results *out)
{
    if (!ctx || !params || !out) { mp_set_error("mp_align_pairs: null argument"); return MP_ERR_ARG; }
    if (!ctx->hasIndex || !ctx->hasBatch) { mp_set_error("mp_align_pairs: index and batch must be loaded first"); return MP_ERR_STATE; }
    if (params->matchScore != 1 || params->extendGapScore != -1 || params->mismatchScore > -2 || params->mismatchScore <= params->openGapScore * 2 ||
        params->mismatchScore < -4 || params->openGapScore < -6 || params->openGapScore >= -1) {
        mp_set_error("mp_align_pairs: score parameters outside the supported range (CPU_DP.cpp:199-208; mismatch = -1 divides by zero at CPU_DP.cpp:310, and for mismatch == 2 * open the reference traceback prefers I over D where the plain recurrence ties: unpinned, refused)"); return MP_ERR_ARG;
    }
    if ((int64_t)ctx->maxLenBatch >= (int64_t)params->maxReadLength) {
        mp_set_error("the batch holds a read of %u bases but maxReadLength is %d (reads must be shorter)", ctx->maxLenBatch, params->maxReadLength);
        return MP_ERR_ARG;
    }
    MP_CUDA(cudaSetDevice(ctx->device));
    const double wall0 = mp_now_ms();
    MpTrace tr;
    memset(out, 0, sizeof *out);
    ctx->resValid = false; ctx->fmtReady = false;
    ctx->hPairs.clear(); ctx->hRescued.clear(); ctx->hSingles.clear(); ctx->hCigars.clear();
    ctx->evUsed = 0;
    MP_CUDA(cudaEventRecord(ctx->ev[4], ctx->stream));
    if (!ctx->seeded) { if (int rc = mp_seed_pairs(ctx, params)) return rc; }
    MP_CUDA(cudaEventRecord(ctx->ev[5], ctx->stream));
    tr.mark("seed_pairs");
    uint64_t cells = 0, tasksRun = 0;
    if (int rc = deep_dp(ctx, params, out, cells, tasksRun)) return rc;
    tr.mark("deep_dp");
    if (int rc = mps_single_and_rescue(ctx, params, out, cells, tasksRun)) return rc;
    MP_CUDA(cudaEventRecord(ctx->ev[6], ctx->stream));
    // (on the context's own stream: a cudaMemcpy on the legacy default stream would wait for the work queued by every other context of
    // the GPU -- their batches' kernels and, with device-side FASTQ I/O, transfers of hundreds of MB)
    unsigned long long hc[16];
    MP_CUDA(cudaMemcpyAsync(hc, ctx->dCounters.p, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    MP_CUDA(cudaStreamSynchronize(ctx->stream));
    tr.mark("single+default dp");
    mp_stats &S = ctx->stats;
    memset(&S, 0, sizeof S);
    S.n_occ = hc[2]; S.n_lf = hc[5] + hc[8]; S.n_sa = hc[3]; S.n_lkt = hc[4]; S.n_probe = hc[9]; S.n_text = hc[10];
    ctx->ev_collect(S.ms_fill, S.ms_tb, S.ms_exact);
    S.dp_cells = cells; S.dp_tasks = tasksRun; S.dp_tasks_exact = hc[14]; S.dp_cells_filled = hc[15];
    cudaEventElapsedTime(&S.ms_seed, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_sa, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_pair, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&S.ms_dp, ctx->ev[5], ctx->ev[6]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[4], ctx->ev[6]);
    out->pairs = ctx->hPairs.data(); out->n_pairs = ctx->hPairs.size();
    out->rescued = ctx->hRescued.data(); out->n_rescued = ctx->hRescued.size();
    out->singles = ctx->hSingles.data(); out->n_singles = ctx->hSingles.size();
    out->cigars = ctx->hCigars.data(); out->cigar_bytes = ctx->hCigars.size();
    ctx->seeded = false;       // the batch has been consumed
    ctx->resCount[0] = out->n_pairs; ctx->resCount[1] = out->n_rescued; ctx->resCount[2] = out->n_singles; ctx->resValid = true;
    if (ctx->resultsOnDevice) {            // nothing was copied: the caller gets the counters only
        out->pairs = nullptr; out->rescued = nullptr; out->singles = nullptr; out->cigars = nullptr;
        out->n_pairs = out->n_rescued = out->n_singles = out->cigar_bytes = 0;
    }
    S.ms_wall = (float)(mp_now_ms() - wall0);
    tr.mark("finish");
    return 0;
}
extern "C" int mp_results_on_device(mp_context *ctx, int on)
{
    if (!ctx) { mp_set_error("mp_results_on_device: null argument"); return MP_ERR_ARG; }
    ctx->resultsOnDevice = on != 0;
    return 0;
}
extern "C" int mp_last_stats(mp_context *ctx, mp_stats *stats)
{
    if (!ctx || !stats) { mp_set_error("mp_last_stats: null argument"); return MP_ERR_ARG; }
    *stats = ctx->stats;
    return 0;
}
extern "C" void mp_results_release(mp_context *ctx, mp_results *res)
{
    if (!ctx) return;
    ctx->hPairs.clear(); ctx->hRescued.clear(); ctx->hSingles.clear(); ctx->hCigars.clear();
    if (res) memset(res, 0, sizeof *res);
}

