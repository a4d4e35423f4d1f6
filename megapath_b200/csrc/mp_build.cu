// mp_build.cu -- FM-index construction in HBM from a packed text, and index export in the
// reference's on-disk formats.  Replaces the offline builder of the reference
//   2bwt-lib/2BWT-Builder.c (driver), BWTConstruct.c (incremental BWT + occ tables,
//   BWTGenerateOccValueFromBwt :994-1204, BWTGenerateSaValue :1250-1313, BWTSaveBwtCodeAndOcc
//   :1206-1236, BWTSaveSaValue :1370-1393), LTConstruct.c:46-96 (13-mer lookup table),
//   HSP.c:354-699 (.pac/.ann/.amb/.tra)
// for ACGT-only texts (no ambiguity runs; SURVEY.md 8f-1).  The reference inserts the text
// incrementally into a dynamic BWT on one CPU thread (22 s per 50 Mbp); here the suffix array
// is built by prefix doubling with device-wide radix sorts:
//   round 0   key = first 21 symbols (3 bits each, 0 = past the end) of every suffix, one
//             64-bit radix sort of all n+1 suffixes
//   round k   only suffixes still sharing their group are re-sorted by
//             (rank[i], rank[i + h]), h = 21 * 2^(k-1); ranks are group-head positions so
//             resolved suffixes never move (Larsson-Sadakane refinement)
// then BWT[j] = T[SA[j]-1], occurrence blocks (mp_index.cu relayout), SA samples, LKT.
#include "mp_context.h"
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <string.h>
#include <stdlib.h>
#include <string>
#include <vector>

int mpi_relayout_words(mp_context *ctx, const uint32_t *dWords, uint64_t n);
int mpb_build_large(mp_context *ctx, uint64_t n);       // mp_build_large.cu

#define SYM_PER_KEY 21

__device__ __forceinline__ uint32_t pac_base(const uint8_t *__restrict__ pac, uint64_t pos)
{
    return (pac[pos >> 2] >> ((3 - (pos & 3)) << 1)) & 3;
}

__global__ void k_init_keys(const uint8_t *__restrict__ pac, uint64_t n, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    uint64_t key = 0;
#pragma unroll
    for (int s = 0; s < SYM_PER_KEY; ++s) {
        uint64_t p = i + s;
        uint64_t code = p < n ? pac_base(pac, p) + 1 : 0;
        key = (key << 3) | code;
    }
    keys[i] = key;
    vals[i] = (uint32_t)i;
}

// headPos[j] = j+1 if element j starts a new key group, else 0 (slot == nullptr: slot[j] = j)
__global__ void k_heads(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ slot, uint64_t m, uint32_t *__restrict__ headPos)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    bool head = t == 0 || keys[t] != keys[t - 1];
    uint32_t s = slot ? slot[t] : (uint32_t)t;
    headPos[t] = head ? s + 1 : 0;
}
// scatter the sorted subset back: SA[slot[t]] = suf[t], rankOf[suf[t]] = rank[t]; flag non-singletons
__global__ void k_scatter(const uint32_t *__restrict__ suf, const uint32_t *__restrict__ slot, const uint32_t *__restrict__ rank, uint64_t m,
                          uint32_t *__restrict__ sa, uint32_t *__restrict__ rankOf, uint32_t *__restrict__ unresFlag)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    uint32_t s = slot ? slot[t] : (uint32_t)t;
    uint32_t i = suf[t], r = rank[t];
    if (slot) sa[s] = i;
    rankOf[i] = r;
    bool head = r == s + 1;
    bool nextHead = true;
    if (t + 1 < m) { uint32_t s1 = slot ? slot[t + 1] : (uint32_t)(t + 1); nextHead = rank[t + 1] == s1 + 1; }
    unresFlag[t] = (head && nextHead) ? 0u : 1u;
}
__global__ void k_compact(const uint32_t *__restrict__ suf, const uint32_t *__restrict__ slot, const uint32_t *__restrict__ flag,
                          const uint32_t *__restrict__ dst, uint64_t m, uint32_t *__restrict__ outSuf, uint32_t *__restrict__ outSlot)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m || !flag[t]) return;
    uint32_t d = dst[t];
    outSuf[d] = suf[t];
    outSlot[d] = slot ? slot[t] : (uint32_t)t;
}
__global__ void k_pair_keys(const uint32_t *__restrict__ suf, uint64_t m, const uint32_t *__restrict__ rankOf, uint64_t n, uint64_t h,
                            uint64_t *__restrict__ keys)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    uint64_t i = suf[t];
    uint64_t r2 = i + h <= n ? rankOf[i + h] : 0;
    keys[t] = ((uint64_t)rankOf[i] << 32) | r2;
}
// BWT words (16 symbols per u32, first symbol in the top bits), '$' skipped (BWT.c:132-157)
__global__ void k_bwt_words(const uint8_t *__restrict__ pac, const uint32_t *__restrict__ sa, uint64_t n, uint64_t inverseSa0,
                            uint32_t *__restrict__ words, uint64_t nWords)
{
    uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nWords) return;
    uint32_t word = 0;
#pragma unroll
    for (int s = 0; s < 16; ++s) {
        uint64_t jj = w * 16 + s;
        if (jj < n) {
            uint64_t j = jj + (jj >= inverseSa0);
            uint64_t i = sa[j];
            word |= pac_base(pac, i - 1) << ((15 - s) << 1);
        }
    }
    words[w] = word;
}
__global__ void k_sa_sample(const uint32_t *__restrict__ sa, uint64_t nSamples, uint32_t shift, uint64_t *__restrict__ out)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nSamples) out[t] = t == 0 ? ~0ull : (uint64_t)sa[t << shift];     // "saValue[0] = -1" (BWT.c:241)
}
// 13-mer histogram; windows past the end are padded with 'A' (LTConstruct.c:46-96)
__global__ void k_lkt_hist(const uint8_t *__restrict__ pac, uint64_t n, unsigned long long *__restrict__ hist)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t key = 0;
#pragma unroll
    for (int s = 0; s < 13; ++s) {
        uint64_t p = i + s;
        key = (key << 2) | (p < n ? pac_base(pac, p) : 0u);
    }
    atomicAdd(&hist[key], 1ull);
}
__global__ void k_count_syms(const uint32_t *__restrict__ words, uint64_t nWords, unsigned long long *__restrict__ cnt)
{
    uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    if (w < nWords) {
        uint32_t x = words[w];
        c0 = mp_word_count(x, 0, 16); c1 = mp_word_count(x, 1, 16); c2 = mp_word_count(x, 2, 16); c3 = mp_word_count(x, 3, 16);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        c0 += __shfl_xor_sync(0xffffffffu, c0, d); c1 += __shfl_xor_sync(0xffffffffu, c1, d);
        c2 += __shfl_xor_sync(0xffffffffu, c2, d); c3 += __shfl_xor_sync(0xffffffffu, c3, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (c0) atomicAdd(&cnt[0], (unsigned long long)c0);
        if (c1) atomicAdd(&cnt[1], (unsigned long long)c1);
        if (c2) atomicAdd(&cnt[2], (unsigned long long)c2);
        if (c3) atomicAdd(&cnt[3], (unsigned long long)c3);
    }
}

__global__ void k_sa_subsample(const uint64_t *__restrict__ in, uint64_t nOut, uint64_t step, uint64_t *__restrict__ out)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nOut) out[t] = in[t * step];
}
// the same from the 40-bit sample arrays of a text >= 2^32 (entry 0 is overwritten by the caller)
__global__ void k_sa40_subsample(const uint32_t *__restrict__ lo, const uint8_t *__restrict__ hi, uint64_t nOut, uint64_t step, uint64_t *__restrict__ out)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nOut) out[t] = (uint64_t)lo[t * step] | ((uint64_t)hi[t * step] << 32);
}

struct MaxU32 { __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; } };

static inline unsigned grid_for(uint64_t n, unsigned block) { return (unsigned)((n + block - 1) / block); }

extern "C" int mp_index_build(mp_context *ctx, const uint8_t *text2bit, uint64_t n)
{
    if (!ctx || !text2bit || n < 32) { mp_set_error("mp_index_build: null argument or text shorter than 32 bases"); return MP_ERR_ARG; }
    // texts of 2^32 bases and more take the bucketed builder of mp_build_large.cu (MP_BUILD_LARGE=1 forces it: parity tests on small texts)
    const bool large = n + 1 >= 0xFFFFFFF0ull || (getenv("MP_BUILD_LARGE") && getenv("MP_BUILD_LARGE")[0] == '1');
    MP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ctx->hasIndex = false; ctx->bloomK = 0; ctx->ix.sa32 = nullptr; ctx->dSa32.release(); ctx->hbmBudget = 0;
    const uint64_t N = n + 1;                       // suffixes incl. the '$' suffix
    const uint64_t pacBytes = (n + 3) / 4;
    // ---- packed text (kept as the index's .pac) ----
    if (ctx->dPac.reserve(pacBytes + 64)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemsetAsync(ctx->dPac.p, 0, pacBytes + 64, st));
    MP_CUDA(cudaMemcpyAsync(ctx->dPac.p, text2bit, pacBytes, cudaMemcpyHostToDevice, st));
    if (n & 3) {                                    // clear the unused low bits of the last byte
        uint8_t last = text2bit[pacBytes - 1] & (uint8_t)(0xFF << ((4 - (n & 3)) * 2));
        MP_CUDA(cudaMemcpyAsync(ctx->dPac.as<uint8_t>() + pacBytes - 1, &last, 1, cudaMemcpyHostToDevice, st));
        MP_CUDA(cudaStreamSynchronize(st));
    }
    const uint8_t *pac = ctx->dPac.as<uint8_t>();
    if (large) { MP_CUDA(cudaStreamSynchronize(st)); return mpb_build_large(ctx, n); }

    DevBuf keysA, keysB, valsA, valsB, rankOf, tmpRank, tmpFlag, tmpDst, sortTmp, scanTmp;
    auto fail = [&](int rc) { keysA.release(); keysB.release(); valsA.release(); valsB.release(); rankOf.release(); tmpRank.release();
                              tmpFlag.release(); tmpDst.release(); sortTmp.release(); scanTmp.release(); return rc; };
    if (keysA.reserve(N * 8) || keysB.reserve(N * 8) || valsA.reserve(N * 4) || valsB.reserve(N * 4) || rankOf.reserve(N * 4 + 4) ||
        tmpRank.reserve(N * 4) || tmpFlag.reserve(N * 4) || tmpDst.reserve(N * 4 + 4)) return fail(MP_ERR_CUDA);
    size_t sortBytes = 0, scanBytes = 0, b2 = 0;
    {
        cub::DoubleBuffer<uint64_t> dk(keysA.as<uint64_t>(), keysB.as<uint64_t>());
        cub::DoubleBuffer<uint32_t> dv(valsA.as<uint32_t>(), valsB.as<uint32_t>());
        cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, dk, dv, (int64_t)N, 0, 64, st);
        cub::DeviceScan::InclusiveScan(nullptr, scanBytes, tmpRank.as<uint32_t>(), tmpRank.as<uint32_t>(), MaxU32(), (int64_t)N, st);
        cub::DeviceScan::ExclusiveSum(nullptr, b2, tmpFlag.as<uint32_t>(), tmpDst.as<uint32_t>(), (int64_t)N, st);
        if (b2 > scanBytes) scanBytes = b2;
    }
    if (sortTmp.reserve(sortBytes) || scanTmp.reserve(scanBytes)) return fail(MP_ERR_CUDA);

    // ---- round 0: all suffixes by their first 21 symbols ----
    ++g_mp_launches; k_init_keys<<<grid_for(N, 256), 256, 0, st>>>(pac, n, keysA.as<uint64_t>(), valsA.as<uint32_t>());
    cub::DoubleBuffer<uint64_t> dk(keysA.as<uint64_t>(), keysB.as<uint64_t>());
    cub::DoubleBuffer<uint32_t> dv(valsA.as<uint32_t>(), valsB.as<uint32_t>());
    cub::DeviceRadixSort::SortPairs(sortTmp.p, sortBytes, dk, dv, (int64_t)N, 0, 63, st);
    MP_CUDA(cudaGetLastError());
    uint32_t *sa = dv.Current();                    // the full suffix array lives here from now on
    uint32_t *spare32 = dv.Alternate();             // N u32 of scratch
    uint64_t *keyCur = dk.Current(), *keyAlt = dk.Alternate();
    ++g_mp_launches; k_heads<<<grid_for(N, 256), 256, 0, st>>>(keyCur, nullptr, N, tmpRank.as<uint32_t>());
    cub::DeviceScan::InclusiveScan(scanTmp.p, scanBytes, tmpRank.as<uint32_t>(), tmpRank.as<uint32_t>(), MaxU32(), (int64_t)N, st);
    ++g_mp_launches; k_scatter<<<grid_for(N, 256), 256, 0, st>>>(sa, nullptr, tmpRank.as<uint32_t>(), N, sa, rankOf.as<uint32_t>(), tmpFlag.as<uint32_t>());
    cub::DeviceScan::ExclusiveSum(scanTmp.p, scanBytes, tmpFlag.as<uint32_t>(), tmpDst.as<uint32_t>(), (int64_t)N, st);
    uint32_t lastDst = 0, lastFlag = 0;
    MP_CUDA(cudaMemcpyAsync(&lastDst, tmpDst.as<uint32_t>() + (N - 1), 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaMemcpyAsync(&lastFlag, tmpFlag.as<uint32_t>() + (N - 1), 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    uint64_t m = (uint64_t)lastDst + lastFlag;
    // unresolved (suffix, slot) lists; ping-pong between two pairs of arrays carved from the key buffers
    // (after round 0 the 64-bit key buffers are only needed for m <= N/2 ... N entries of the subset)
    DevBuf uSufA, uSlotA, uSufB, uSlotB;
    auto fail2 = [&](int rc) { uSufA.release(); uSlotA.release(); uSufB.release(); uSlotB.release(); return fail(rc); };
    if (m) {
        if (uSufA.reserve(m * 4) || uSlotA.reserve(m * 4) || uSufB.reserve(m * 4) || uSlotB.reserve(m * 4)) return fail2(MP_ERR_CUDA);
        ++g_mp_launches; k_compact<<<grid_for(N, 256), 256, 0, st>>>(sa, nullptr, tmpFlag.as<uint32_t>(), tmpDst.as<uint32_t>(), N,
                                                                     uSufA.as<uint32_t>(), uSlotA.as<uint32_t>());
    }
    (void)spare32;
    uint32_t *uSuf = uSufA.as<uint32_t>(), *uSlot = uSlotA.as<uint32_t>(), *vSuf = uSufB.as<uint32_t>(), *vSlot = uSlotB.as<uint32_t>();
    uint64_t h = SYM_PER_KEY;
    int rounds = 1;
    while (m) {
        if (rounds > 64) { mp_set_error("mp_index_build: prefix doubling did not converge"); return fail2(MP_ERR_STATE); }
        ++g_mp_launches; k_pair_keys<<<grid_for(m, 256), 256, 0, st>>>(uSuf, m, rankOf.as<uint32_t>(), n, h, keyCur);
        cub::DoubleBuffer<uint64_t> k2(keyCur, keyAlt);
        cub::DoubleBuffer<uint32_t> v2(uSuf, vSuf);
        cub::DeviceRadixSort::SortPairs(sortTmp.p, sortBytes, k2, v2, (int64_t)m, 0, 64, st);
        uint64_t *ks = k2.Current();
        uint32_t *sortedSuf = v2.Current(), *otherSuf = v2.Alternate();
        ++g_mp_launches; k_heads<<<grid_for(m, 256), 256, 0, st>>>(ks, uSlot, m, tmpRank.as<uint32_t>());
        cub::DeviceScan::InclusiveScan(scanTmp.p, scanBytes, tmpRank.as<uint32_t>(), tmpRank.as<uint32_t>(), MaxU32(), (int64_t)m, st);
        ++g_mp_launches; k_scatter<<<grid_for(m, 256), 256, 0, st>>>(sortedSuf, uSlot, tmpRank.as<uint32_t>(), m, sa, rankOf.as<uint32_t>(), tmpFlag.as<uint32_t>());
        cub::DeviceScan::ExclusiveSum(scanTmp.p, scanBytes, tmpFlag.as<uint32_t>(), tmpDst.as<uint32_t>(), (int64_t)m, st);
        MP_CUDA(cudaMemcpyAsync(&lastDst, tmpDst.as<uint32_t>() + (m - 1), 4, cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaMemcpyAsync(&lastFlag, tmpFlag.as<uint32_t>() + (m - 1), 4, cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaStreamSynchronize(st));
        uint64_t m2 = (uint64_t)lastDst + lastFlag;
        if (m2) {
            ++g_mp_launches; k_compact<<<grid_for(m, 256), 256, 0, st>>>(sortedSuf, uSlot, tmpFlag.as<uint32_t>(), tmpDst.as<uint32_t>(), m, otherSuf, vSlot);
        }
        // next round reads (otherSuf, vSlot); the buffer holding sortedSuf becomes the sort's alternate
        uSuf = otherSuf; vSuf = sortedSuf;
        uint32_t *ts = uSlot; uSlot = vSlot; vSlot = ts;
        m = m2; h *= 2; ++rounds;
    }
    MP_CUDA(cudaGetLastError());
    uSufA.release(); uSlotA.release(); uSufB.release(); uSlotB.release();
    // ---- inverseSa0 = SA position of suffix 0 ----
    uint32_t r0 = 0;
    MP_CUDA(cudaMemcpyAsync(&r0, rankOf.as<uint32_t>(), 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    const uint64_t inverseSa0 = (uint64_t)r0 - 1;
    tmpRank.release(); tmpFlag.release(); tmpDst.release(); rankOf.release();
    // ---- BWT words, padded with zero words to whole occ blocks ----
    const uint64_t nBlocks = n / MP_BLK_SYMS + 1, nWords = (n + 15) / 16;
    uint32_t *dWords = (uint32_t *)keyAlt;          // N*8 bytes of scratch >= nBlocks*48
    if (nBlocks * 48 > N * 8) { mp_set_error("mp_index_build: scratch too small"); return fail(MP_ERR_STATE); }
    MP_CUDA(cudaMemsetAsync(dWords, 0, nBlocks * 48, st));
    ++g_mp_launches; k_bwt_words<<<grid_for(nWords, 256), 256, 0, st>>>(pac, sa, n, inverseSa0, dWords, nWords);
    // ---- symbol counts -> cumFreq ----
    unsigned long long *dCnt = (unsigned long long *)keyCur;
    MP_CUDA(cudaMemsetAsync(dCnt, 0, 32, st));
    ++g_mp_launches; k_count_syms<<<grid_for(nWords, 256), 256, 0, st>>>(dWords, nWords, dCnt);
    unsigned long long hc[4];
    MP_CUDA(cudaMemcpyAsync(hc, dCnt, 32, cudaMemcpyDeviceToHost, st));
    // ---- SA samples (every 16th SA index; saValue[0] = -1 as after BWTLoad) ----
    const uint32_t saShift = 4;
    const uint64_t nSa = (n + 16) / 16;
    if (ctx->dSa.reserve(nSa * 8)) return fail(MP_ERR_CUDA);
    ++g_mp_launches; k_sa_sample<<<grid_for(nSa, 256), 256, 0, st>>>(sa, nSa, saShift, ctx->dSa.as<uint64_t>());
    MP_CUDA(cudaStreamSynchronize(st));
    hc[0] -= nWords * 16 - n;                        // zero padding of the last word was counted as 'A'
    ctx->ix.n = n; ctx->ix.inverseSa0 = inverseSa0;
    ctx->ix.cum[0] = 0;
    for (int c = 0; c < 4; ++c) ctx->ix.cum[c + 1] = ctx->ix.cum[c] + hc[c];
    if (ctx->ix.cum[4] != n) { mp_set_error("mp_index_build: symbol counts do not add up"); return fail(MP_ERR_STATE); }
    ctx->ix.sa = ctx->dSa.as<uint64_t>(); ctx->ix.saShift = saShift; ctx->saInterval = 16;
    // ---- occurrence blocks ----
    if (int rc = mpi_relayout_words(ctx, dWords, n)) return fail(rc);
    // keep the full suffix array as the dense SA of the resident index (the buffer changes owner)
    {
        DevBuf &owner = (sa == valsA.as<uint32_t>()) ? valsA : valsB;
        ctx->dSa32.release();
        ctx->dSa32 = owner; owner.p = nullptr; owner.cap = 0;
        ctx->ix.sa32 = ctx->dSa32.as<uint32_t>();
    }
    valsA.release(); valsB.release(); keysA.release(); keysB.release(); sortTmp.release();
    // ---- LKT: inclusive cumulative 13-mer counts ----
    const uint64_t nLkt = 1ull << 26;
    if (ctx->dLkt.reserve(nLkt * 8)) return fail(MP_ERR_CUDA);
    MP_CUDA(cudaMemsetAsync(ctx->dLkt.p, 0, nLkt * 8, st));
    ++g_mp_launches; k_lkt_hist<<<grid_for(n, 256), 256, 0, st>>>(pac, n, ctx->dLkt.as<unsigned long long>());
    {
        size_t tb = 0;
        cub::DeviceScan::InclusiveSum(nullptr, tb, ctx->dLkt.as<uint64_t>(), ctx->dLkt.as<uint64_t>(), (int64_t)nLkt, st);
        if (scanTmp.reserve(tb)) return fail(MP_ERR_CUDA);
        cub::DeviceScan::InclusiveSum(scanTmp.p, tb, ctx->dLkt.as<uint64_t>(), ctx->dLkt.as<uint64_t>(), (int64_t)nLkt, st);
    }
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaStreamSynchronize(st));
    scanTmp.release();
    ctx->ix.lkt = ctx->dLkt.as<uint64_t>();
    ctx->ix.pac = pac;
    ctx->hbmBytes = ctx->dBlocks.cap + ctx->dSuper.cap + ctx->dSa.cap + ctx->dSa32.cap + ctx->dLkt.cap + ctx->dPac.cap;
    ctx->hasIndex = true; ctx->hasBatch = false; ctx->seeded = false;
    return 0;
}

// =====================================================================================
// export in the reference's file formats
// =====================================================================================
static int write_all(const std::string &path, const void *hdr, size_t hdrBytes, const void *body, size_t bodyBytes,
                     const void *tail = nullptr, size_t tailBytes = 0)
{
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) { mp_set_error("cannot create %s", path.c_str()); return MP_ERR_IO; }
    bool ok = (hdrBytes == 0 || fwrite(hdr, 1, hdrBytes, f) == hdrBytes) && (bodyBytes == 0 || fwrite(body, 1, bodyBytes, f) == bodyBytes) &&
              (tailBytes == 0 || fwrite(tail, 1, tailBytes, f) == tailBytes);
    if (fclose(f) != 0) ok = false;
    if (!ok) { mp_set_error("short write to %s", path.c_str()); return MP_ERR_IO; }
    return 0;
}

extern "C" int mp_index_save(mp_context *ctx, const char *prefix)
{
    if (!ctx || !prefix) { mp_set_error("mp_index_save: null argument"); return MP_ERR_ARG; }
    if (!ctx->hasIndex) { mp_set_error("mp_index_save: no index resident"); return MP_ERR_STATE; }
    if (ctx->saInterval > 16 || (ctx->saInterval & (ctx->saInterval - 1))) { mp_set_error("mp_index_save: saInterval %llu cannot be exported as the 1/16 samples of the .sa format", (unsigned long long)ctx->saInterval); return MP_ERR_STATE; }
    MP_CUDA(cudaSetDevice(ctx->device));
    const std::string p(prefix);
    const uint64_t n = ctx->ix.n, nBlocks = ctx->ix.nBlocks;
    uint64_t hdr[5] = { ctx->ix.inverseSa0, ctx->ix.cum[1], ctx->ix.cum[2], ctx->ix.cum[3], ctx->ix.cum[4] };
    // ---- .bwt : the BWT words sit in bytes [16, 64) of every occ block ----
    const uint64_t nWords = (n + 15) / 16;
    std::vector<uint32_t> words(nBlocks * 12);
    {
        std::vector<uint32_t> blk(nBlocks * 16);
        MP_CUDA(cudaMemcpy(blk.data(), ctx->dBlocks.p, nBlocks * 64, cudaMemcpyDeviceToHost));
        for (uint64_t b = 0; b < nBlocks; ++b) memcpy(&words[b * 12], &blk[b * 16 + 4], 48);
    }
    if (int rc = write_all(p + ".bwt", hdr, 40, words.data(), nWords * 4)) return rc;
    // ---- .fmv : BWTGenerateOccValueFromBwt (BWTConstruct.c:994-1204).  Sample k counts the symbols of
    //      the zero-padded BWT in [0, 256k) relative to the major sample of its 65536-symbol group; two
    //      samples per word (even sample in the high half); the padding counts as 'A'. ----
    {
        const uint64_t nOcc = (n + 255) / 256 + 1;
        const uint64_t minorWords = (nOcc + 1) / 2 * 4, majorEntries = (nOcc + 255) / 256 * 4;
        std::vector<uint32_t> minor(minorWords, 0);
        std::vector<uint64_t> major(majorEntries, 0);
        uint64_t tot[4] = { 0, 0, 0, 0 };
        uint32_t rel[4] = { 0, 0, 0, 0 };
        for (uint64_t k = 0; k < nOcc; ++k) {
            if (k % 256 == 0) {
                for (int c = 0; c < 4; ++c) { major[(k / 256) * 4 + c] = tot[c]; rel[c] = 0; }
            }
            for (int c = 0; c < 4; ++c) {
                if (k & 1) minor[(k / 2) * 4 + c] |= rel[c] & 0xFFFFu;
                else minor[(k / 2) * 4 + c] = rel[c] << 16;
            }
            // symbols [256k, 256k+256): 16 words, zero beyond the stored words
            uint32_t add[4] = { 0, 0, 0, 0 };
            for (uint64_t w = k * 16; w < k * 16 + 16; ++w) {
                uint32_t x = w < words.size() ? words[w] : 0u;
                uint32_t c1 = __builtin_popcount(~(x ^ 0x55555555u) & ~((x ^ 0x55555555u) >> 1) & 0x55555555u);
                uint32_t c2 = __builtin_popcount(~(x ^ 0xAAAAAAAAu) & ~((x ^ 0xAAAAAAAAu) >> 1) & 0x55555555u);
                uint32_t c3 = __builtin_popcount(x & (x >> 1) & 0x55555555u);
                add[1] += c1; add[2] += c2; add[3] += c3; add[0] += 16 - c1 - c2 - c3;
            }
            for (int c = 0; c < 4; ++c) { tot[c] += add[c]; rel[c] += add[c]; }
        }
        if (nOcc & 1) for (int c = 0; c < 4; ++c) minor[(nOcc / 2) * 4 + c] |= (minor[(nOcc / 2) * 4 + c] >> 16);   // lone even sample is repeated
        if (int rc = write_all(p + ".fmv", hdr, 40, minor.data(), minor.size() * 4, major.data(), major.size() * 8)) return rc;
    }
    words.clear(); words.shrink_to_fit();
    // ---- .sa : BWTSaveSaValue (BWTConstruct.c:1370-1393): entry 0 is written as textLength ----
    {
        const uint64_t nSa = (n + 16) / 16;
        std::vector<uint64_t> sa(nSa + 6);
        memcpy(sa.data(), hdr, 40);
        sa[5] = 16;
        if (ctx->ix.sa40lo) {                       // 40-bit samples (texts >= 2^32) -> the file's u64 samples
            DevBuf tmp;
            if (tmp.reserve(nSa * 8)) return MP_ERR_CUDA;
            (++g_mp_launches), k_sa40_subsample<<<grid_for(nSa, 256), 256>>>(ctx->ix.sa40lo, ctx->ix.sa40hi, nSa, 16 / ctx->saInterval, tmp.as<uint64_t>());
            MP_CUDA(cudaMemcpy(sa.data() + 6, tmp.p, nSa * 8, cudaMemcpyDeviceToHost));
            tmp.release();
        } else if (ctx->saInterval == 16) MP_CUDA(cudaMemcpy(sa.data() + 6, ctx->dSa.p, nSa * 8, cudaMemcpyDeviceToHost));
        else {                                       // the resident index samples more densely: every (16 / interval)-th sample goes to the file
            DevBuf tmp;
            if (tmp.reserve(nSa * 8)) return MP_ERR_CUDA;
            (++g_mp_launches), k_sa_subsample<<<grid_for(nSa, 256), 256>>>(ctx->dSa.as<uint64_t>(), nSa, 16 / ctx->saInterval, tmp.as<uint64_t>());
            MP_CUDA(cudaMemcpy(sa.data() + 6, tmp.p, nSa * 8, cudaMemcpyDeviceToHost));
            tmp.release();
        }
        sa[6] = n;
        if (int rc = write_all(p + ".sa", nullptr, 0, sa.data(), sa.size() * 8)) return rc;
    }
    // ---- .lkt ----
    {
        const uint64_t nLkt = 1ull << 26;
        std::vector<uint64_t> lkt(nLkt);
        MP_CUDA(cudaMemcpy(lkt.data(), ctx->dLkt.p, nLkt * 8, cudaMemcpyDeviceToHost));
        int32_t ts = 13;
        if (int rc = write_all(p + ".lkt", &ts, 4, lkt.data(), nLkt * 8)) return rc;
    }
    // ---- .pac : 4 bases per byte + trailer (HSP.c:560-565) ----
    {
        const uint64_t pacBytes = (n + 3) / 4;
        std::vector<uint8_t> pac(pacBytes + 2);
        MP_CUDA(cudaMemcpy(pac.data(), ctx->dPac.p, pacBytes, cudaMemcpyDeviceToHost));
        size_t len = pacBytes;
        if (n % 4 == 0) pac[len++] = 0;
        pac[len++] = (uint8_t)(n % 4);
        if (int rc = write_all(p + ".pac", nullptr, 0, pac.data(), len)) return rc;
    }
    return 0;
}

// .ann / .amb / .tra for a text without ambiguity runs (HSP.c:569-699): one translate entry per sequence
extern "C" int mp_index_save_annotation(const char *prefix, uint64_t textLength, uint32_t numSeq, const char *const *names,
                                        const uint64_t *starts, const uint64_t *lengths)
{
    if (!prefix || !names || !starts || !lengths || numSeq == 0) { mp_set_error("mp_index_save_annotation: bad argument"); return MP_ERR_ARG; }
    const std::string p(prefix);
    FILE *f = fopen((p + ".ann").c_str(), "w");
    if (!f) { mp_set_error("cannot create %s.ann", prefix); return MP_ERR_IO; }
    fprintf(f, "%llu %u %u\n", (unsigned long long)textLength, numSeq, 0u);
    for (uint32_t i = 0; i < numSeq; ++i) {
        fprintf(f, "%u %s\n", 0u, names[i]);
        fprintf(f, "%llu %llu 0\n", (unsigned long long)starts[i], (unsigned long long)lengths[i]);
    }
    fclose(f);
    f = fopen((p + ".amb").c_str(), "w");
    if (!f) { mp_set_error("cannot create %s.amb", prefix); return MP_ERR_IO; }
    fprintf(f, "%llu %u %u\n", (unsigned long long)textLength, numSeq, 0u);
    fclose(f);
    f = fopen((p + ".tra").c_str(), "w");
    if (!f) { mp_set_error("cannot create %s.tra", prefix); return MP_ERR_IO; }
    const uint64_t GRID = 262144;
    const uint32_t gridEntries = (uint32_t)(textLength / GRID) + 1;
    std::vector<uint32_t> grid(gridEntries, 0);
    for (uint32_t i = 0; i < numSeq; ++i) grid[starts[i] / GRID] += 1;
    for (uint32_t j = 1; j < gridEntries; ++j) grid[j] += grid[j - 1];
    fprintf(f, "%llu %u %u %u\n", (unsigned long long)textLength, numSeq, 0u, gridEntries);
    for (uint32_t j = 0; j < gridEntries; ++j) fprintf(f, "%u\n", grid[j] - 1);
    for (uint32_t i = 0; i < numSeq; ++i)
        fprintf(f, "%llu %u %llu\n", (unsigned long long)starts[i], i + 1, (unsigned long long)(starts[i] - 1));
    for (uint32_t i = 0; i < numSeq; ++i)
        fprintf(f, "%llu %llu\n", (unsigned long long)starts[i], (unsigned long long)lengths[i]);
    fclose(f);
    return 0;
}
