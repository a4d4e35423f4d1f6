// mp_index.cu -- index loader: reads the reference's 2BWT index files and re-lays them out
// in HBM (see mp_index.cuh).  Replaces INDEXLoad (IndexHandler.cpp:49-99, 101-148):
// BWTLoad (2bwt-lib/BWT.c:100-250), LTLoad (2bwt-flex/LT.c:34-57), DNALoadPacked
// (2bwt-lib/TextConverter.c:427-479).  Only the forward BWT is used, as in the reference
// (rev BWT/LKT loads are commented out at IndexHandler.cpp:111,140-142).
#include "mp_context.h"
#include <cub/device/device_scan.cuh>
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>

static thread_local char g_err[1024] = "";
void mp_set_error(const char *fmt, ...)
{
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
}
extern "C" const char *mp_last_error(void) { return g_err; }
std::atomic<unsigned long long> g_mp_launches(0);
extern "C" uint64_t mp_launch_count(void) { return g_mp_launches.load(); }

// ---- file -> device in bounded chunks ----
static int upload_region(FILE *f, uint64_t fileOff, uint64_t bytes, void *dst)
{
    const size_t CH = 256u << 20;
    void *h = nullptr;
    if (cudaMallocHost(&h, CH) != cudaSuccess) { mp_set_error("cudaMallocHost failed"); return MP_ERR_CUDA; }
    if (fseeko(f, (off_t)fileOff, SEEK_SET) != 0) { cudaFreeHost(h); mp_set_error("seek failed"); return MP_ERR_IO; }
    uint64_t done = 0;
    while (done < bytes) {
        size_t want = (size_t)((bytes - done) < CH ? (bytes - done) : CH);
        size_t got = fread(h, 1, want, f);
        if (got != want) { cudaFreeHost(h); mp_set_error("short read (%zu of %zu)", got, want); return MP_ERR_IO; }
        cudaError_t e = cudaMemcpy((char *)dst + done, h, want, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { cudaFreeHost(h); mp_set_error("H2D copy failed: %s", cudaGetErrorString(e)); return MP_ERR_CUDA; }
        done += want;
    }
    cudaFreeHost(h);
    return 0;
}

static FILE *open_idx(const std::string &path)
{
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) mp_set_error("cannot open index file %s", path.c_str());
    return f;
}

// ---- relayout kernels ----
// per-block symbol counts; block b = .bwt words [12b, 12b+12); symbols at or beyond n are not counted
__global__ void k_block_counts(const uint32_t *__restrict__ words, uint64_t n, uint64_t nBlocks, uint32_t c,
                               uint64_t *__restrict__ out)
{
    uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nBlocks) return;
    uint64_t base = b * MP_BLK_SYMS;
    uint32_t total = 0;
    if (base < n) {
        uint64_t rem = n - base;
        uint32_t lim = rem < MP_BLK_SYMS ? (uint32_t)rem : MP_BLK_SYMS;
        for (uint32_t w = 0; w < 12 && w * 16 < lim; ++w) {
            uint32_t r = lim - w * 16; if (r > 16) r = 16;
            total += mp_word_count(words[b * 12 + w], c, r);
        }
    }
    out[b] = total;
}
__global__ void k_super(const uint64_t *__restrict__ scan, uint64_t nBlocks, uint32_t c, uint64_t *__restrict__ super)
{
    uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t nSuper = (nBlocks >> MP_SUPER_SHIFT) + 1;
    if (s < nSuper) super[s * 4 + c] = scan[min(s << MP_SUPER_SHIFT, nBlocks - 1)];
}
__global__ void k_build_blocks(const uint32_t *__restrict__ words, const uint64_t *__restrict__ scan,
                               const uint64_t *__restrict__ super, uint64_t nBlocks, uint32_t c, uint32_t *__restrict__ blocks)
{
    uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nBlocks) return;
    uint32_t *o = blocks + b * 16;
    o[c] = (uint32_t)(scan[b] - super[(b >> MP_SUPER_SHIFT) * 4 + c]);
    if (c == 0) {
#pragma unroll
        for (int w = 0; w < 12; ++w) o[4 + w] = words[b * 12 + w];
    }
}

// dWords: device .bwt words, padded to 12 * nBlocks words (zero filled)
static int relayout(mp_context *ctx, const uint32_t *dWords, uint64_t n)
{
    uint64_t nBlocks = n / MP_BLK_SYMS + 1;
    uint64_t nSuper = (nBlocks >> MP_SUPER_SHIFT) + 1;
    if (ctx->dBlocks.reserve(nBlocks * 64)) return MP_ERR_CUDA;
    if (ctx->dSuper.reserve(nSuper * 4 * 8)) return MP_ERR_CUDA;
    DevBuf cnt, scan, tmp;
    if (cnt.reserve(nBlocks * 8) || scan.reserve(nBlocks * 8)) return MP_ERR_CUDA;
    size_t tmpBytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, cnt.as<uint64_t>(), scan.as<uint64_t>(), (int64_t)nBlocks);
    if (tmp.reserve(tmpBytes)) return MP_ERR_CUDA;
    unsigned g = (unsigned)((nBlocks + 255) / 256);
    for (uint32_t c = 0; c < 4; ++c) {
        (++g_mp_launches), k_block_counts<<<g, 256>>>(dWords, n, nBlocks, c, cnt.as<uint64_t>());
        cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, cnt.as<uint64_t>(), scan.as<uint64_t>(), (int64_t)nBlocks);
        (++g_mp_launches), k_super<<<(unsigned)((nSuper + 255) / 256), 256>>>(scan.as<uint64_t>(), nBlocks, c, ctx->dSuper.as<uint64_t>());
        (++g_mp_launches), k_build_blocks<<<g, 256>>>(dWords, scan.as<uint64_t>(), ctx->dSuper.as<uint64_t>(), nBlocks, c, ctx->dBlocks.as<uint32_t>());
    }
    MP_CUDA(cudaDeviceSynchronize());
    cnt.release(); scan.release(); tmp.release();
    ctx->ix.blocks = ctx->dBlocks.as<uint4>();
    ctx->ix.nBlocks = nBlocks;
    ctx->ix.super = ctx->dSuper.as<uint64_t>();
    return 0;
}

int mpi_relayout_words(mp_context *ctx, const uint32_t *dWords, uint64_t n) { return relayout(ctx, dWords, n); }

int mpi_build_from_words(mp_context *ctx, const uint32_t *hBwtWords, uint64_t n, uint64_t inverseSa0, const uint64_t cum[5])
{
    uint64_t nBlocks = n / MP_BLK_SYMS + 1;
    DevBuf raw;
    if (raw.reserve(nBlocks * 48)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemset(raw.p, 0, nBlocks * 48));
    MP_CUDA(cudaMemcpy(raw.p, hBwtWords, ((n + 15) / 16) * 4, cudaMemcpyHostToDevice));
    ctx->ix.n = n; ctx->ix.inverseSa0 = inverseSa0;
    for (int i = 0; i < 5; ++i) ctx->ix.cum[i] = cum[i];
    int rc = relayout(ctx, raw.as<uint32_t>(), n);
    raw.release();
    return rc;
}

__global__ void k_densify_sa(MpIndexView ix, uint32_t *__restrict__ out, uint64_t count)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = (uint32_t)mp_sa(ix, i);      // ix.sa32 is still null here: sampled walk
}
// texts of 2^32 bases and more: no 32-bit array; 40-bit samples (u32 + u8) at a denser rate than the resident u64 ones
__global__ void k_sa40_build(MpIndexView ix, uint32_t *__restrict__ lo, uint8_t *__restrict__ hi, uint64_t count, uint32_t newShift)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint64_t v = i == 0 ? 0 : mp_sa(ix, i << newShift);          // entry 0 (SA[0] = -1) is special-cased by mp_sa_sample
    lo[i] = (uint32_t)v; hi[i] = (uint8_t)(v >> 32);
}

// bytes of the resident index this context owns (the K-mer filter is counted by mp_index_prepare)
uint64_t mpi_index_bytes(const mp_context *ctx)
{
    return ctx->dBlocks.cap + ctx->dSuper.cap + ctx->dSa.cap + ctx->dSa32.cap + ctx->dSa40Lo.cap + ctx->dSa40Hi.cap + ctx->dLkt.cap + ctx->dPac.cap;
}
static uint64_t devbuf_bytes(uint64_t bytes) { return bytes + bytes / 8 + 256; }     // what DevBuf::reserve(bytes) allocates

// Called once the u64 samples (ctx->dSa, ix.saShift) are resident.  Texts shorter than 2^32 keep them (the dense u32 array is built
// by the callers); longer texts get 40-bit samples at the densest rate whose arrays fit 35 % of the free HBM -- every SA index
// when possible (8 Gbp: 40 GB), so that an SA lookup is two small gathers instead of an LF walk -- and the u64 array is released.
// With an HBM budget (mp_index_load_budget) and no dense u32 array, any text gets the densest 40-bit samples that keep the index
// within the budget, or keeps the file's samples.
// MP_DENSE_SA=0 keeps the file's samples; MP_SA40=<shift> forces the 40-bit arrays at that shift whatever the text length (tests).
int mpi_finish_sa(mp_context *ctx)
{
    ctx->ix.sa40lo = nullptr; ctx->ix.sa40hi = nullptr; ctx->dSa40Lo.release(); ctx->dSa40Hi.release();
    const uint64_t n = ctx->ix.n, budget = ctx->hbmBudget;
    const char *dense = getenv("MP_DENSE_SA"), *force = getenv("MP_SA40");
    if (dense && dense[0] == '0') return 0;
    if (ctx->ix.sa32) return 0;
    if (!force && !budget && n + 1 < 0xFFFFFFF0ull) return 0;
    const uint64_t rest = mpi_index_bytes(ctx) - ctx->dSa.cap;      // what stays resident beside the 40-bit arrays
    size_t freeB = 0, totalB = 0; cudaMemGetInfo(&freeB, &totalB);
    for (uint32_t sh = 0; sh <= ctx->ix.saShift; ++sh) {
        if (force ? sh != (uint32_t)atoi(force) : (sh == ctx->ix.saShift && sh > 0)) continue;
        const uint64_t cnt = (n >> sh) + 1;
        if (!force && budget && rest + devbuf_bytes(cnt * 4) + devbuf_bytes(cnt) > budget) continue;
        if (!force && !budget && (double)cnt * 5.0 > 0.35 * (double)freeB) continue;
        if (ctx->dSa40Lo.reserve(cnt * 4) || ctx->dSa40Hi.reserve(cnt)) return MP_ERR_CUDA;
        (++g_mp_launches), k_sa40_build<<<(unsigned)((cnt + 255) / 256), 256>>>(ctx->ix, ctx->dSa40Lo.as<uint32_t>(), ctx->dSa40Hi.as<uint8_t>(), cnt, sh);
        MP_CUDA(cudaGetLastError());
        MP_CUDA(cudaDeviceSynchronize());
        ctx->dSa.release(); ctx->ix.sa = nullptr;
        ctx->ix.sa40lo = ctx->dSa40Lo.as<uint32_t>(); ctx->ix.sa40hi = ctx->dSa40Hi.as<uint8_t>();
        ctx->ix.saShift = sh; ctx->saInterval = 1ull << sh;
        break;
    }
    return 0;
}

int mpi_load(mp_context *ctx, const char *prefix)
{
    std::string p(prefix);
    MP_CUDA(cudaSetDevice(ctx->device));
    ctx->hasIndex = false; ctx->bloomK = 0;
    // ---- .bwt ----
    FILE *f = open_idx(p + ".bwt");
    if (!f) return MP_ERR_IO;
    uint64_t hdr[5];
    if (fread(hdr, 8, 5, f) != 5) { fclose(f); mp_set_error("%s.bwt: short header", prefix); return MP_ERR_IO; }
    uint64_t n = hdr[4];
    ctx->ix.inverseSa0 = hdr[0];
    ctx->ix.cum[0] = 0;
    for (int i = 1; i <= 4; ++i) ctx->ix.cum[i] = hdr[i];
    ctx->ix.n = n;
    uint64_t nBlocks = n / MP_BLK_SYMS + 1;
    uint64_t fileWords = (n + 15) / 16;
    {
        DevBuf raw;
        if (raw.reserve(nBlocks * 48)) { fclose(f); return MP_ERR_CUDA; }
        MP_CUDA(cudaMemset(raw.p, 0, nBlocks * 48));
        int rc = upload_region(f, 40, fileWords * 4, raw.p);
        fclose(f);
        if (rc) return rc;
        rc = relayout(ctx, raw.as<uint32_t>(), n);
        raw.release();
        if (rc) return rc;
    }
    // ---- .fmv is not needed: the occurrence counts are rebuilt into the 64-byte blocks; its
    //      header is checked like BWTLoad does (BWT.c:139-152) ----
    f = open_idx(p + ".fmv");
    if (!f) return MP_ERR_IO;
    uint64_t h2[5];
    if (fread(h2, 8, 5, f) != 5 || memcmp(h2, hdr, 40) != 0) { fclose(f); mp_set_error("%s.fmv: header does not match .bwt", prefix); return MP_ERR_IO; }
    fclose(f);
    // ---- .sa ----
    f = open_idx(p + ".sa");
    if (!f) return MP_ERR_IO;
    uint64_t h3[6];
    if (fread(h3, 8, 6, f) != 6 || memcmp(h3, hdr, 40) != 0) { fclose(f); mp_set_error("%s.sa: header does not match .bwt", prefix); return MP_ERR_IO; }
    uint64_t saInterval = h3[5];
    if (saInterval == 0 || (saInterval & (saInterval - 1))) { fclose(f); mp_set_error("%s.sa: saInterval %llu is not a power of two", prefix, (unsigned long long)saInterval); return MP_ERR_IO; }
    uint64_t nSa = (n + saInterval) / saInterval;
    if (ctx->dSa.reserve(nSa * 8)) { fclose(f); return MP_ERR_CUDA; }
    {
        int rc = upload_region(f, 48, nSa * 8, ctx->dSa.p);
        fclose(f);
        if (rc) return rc;
        uint64_t minus1 = ~0ull;                      // "saValue[0] = -1" (BWT.c:241)
        MP_CUDA(cudaMemcpy(ctx->dSa.p, &minus1, 8, cudaMemcpyHostToDevice));
    }
    ctx->saInterval = saInterval;
    ctx->ix.sa = ctx->dSa.as<uint64_t>();
    ctx->ix.saShift = 0;
    while ((1ull << ctx->ix.saShift) < saInterval) ++ctx->ix.saShift;
    // ---- .lkt ----
    f = open_idx(p + ".lkt");
    if (!f) return MP_ERR_IO;
    int32_t ts = 0;
    if (fread(&ts, 4, 1, f) != 1 || ts != 13) { fclose(f); mp_set_error("%s.lkt: table size %d != 13", prefix, ts); return MP_ERR_IO; }
    uint64_t nLkt = 1ull << 26;
    if (ctx->dLkt.reserve(nLkt * 8)) { fclose(f); return MP_ERR_CUDA; }
    {
        int rc = upload_region(f, 4, nLkt * 8, ctx->dLkt.p);
        fclose(f);
        if (rc) return rc;
    }
    ctx->ix.lkt = ctx->dLkt.as<uint64_t>();
    // ---- .pac ----
    f = open_idx(p + ".pac");
    if (!f) return MP_ERR_IO;
    uint64_t pacBytes = (n + 3) / 4;
    if (ctx->dPac.reserve(pacBytes + 64)) { fclose(f); return MP_ERR_CUDA; }
    MP_CUDA(cudaMemset(ctx->dPac.p, 0, pacBytes + 64));
    {
        int rc = upload_region(f, 0, pacBytes, ctx->dPac.p);
        fclose(f);
        if (rc) return rc;
    }
    ctx->ix.pac = ctx->dPac.as<uint8_t>();
    const uint64_t fixed = mpi_index_bytes(ctx), budget = ctx->hbmBudget;      // BWT blocks, LKT, text and the file's SA samples
    if (budget && fixed > budget) {
        DevBuf *bufs[] = { &ctx->dBlocks, &ctx->dSuper, &ctx->dSa, &ctx->dLkt, &ctx->dPac };
        for (DevBuf *b : bufs) b->release();
        memset(&ctx->ix, 0, sizeof ctx->ix);
        mp_set_error("%s: the index needs %llu bytes of HBM without a dense SA, the budget is %llu", prefix, (unsigned long long)fixed, (unsigned long long)budget);
        return MP_ERR_CAPACITY;
    }
    // ---- dense SA: resolve every SA index once at load time (LF walks to the file's 1/16 samples) so that
    //      lookups on the hot path are a single gather.  MP_DENSE_SA=0 keeps the sampled array only. ----
    ctx->ix.sa32 = nullptr; ctx->dSa32.release();
    const char *dense = getenv("MP_DENSE_SA");
    size_t freeB = 0, totalB = 0; cudaMemGetInfo(&freeB, &totalB);
    const bool fits = budget ? fixed + devbuf_bytes((n + 1) * 4) <= budget : (n + 1) * 4 < freeB / 2;
    if (!(dense && dense[0] == '0') && !getenv("MP_SA40") && n + 1 < 0xFFFFFFF0ull && fits) {
        if (ctx->dSa32.reserve((n + 1) * 4)) return MP_ERR_CUDA;
        (++g_mp_launches), k_densify_sa<<<(unsigned)((n + 1 + 255) / 256), 256>>>(ctx->ix, ctx->dSa32.as<uint32_t>(), n + 1);
        MP_CUDA(cudaGetLastError());
        MP_CUDA(cudaDeviceSynchronize());
        ctx->ix.sa32 = ctx->dSa32.as<uint32_t>();
    }
    if (int rc = mpi_finish_sa(ctx)) return rc;
    ctx->hbmBytes = mpi_index_bytes(ctx);
    ctx->hasIndex = true;
    return 0;
}

// ---- primitive kernels for parity tests ----
__global__ void k_occ(MpIndexView ix, const uint64_t *idx, const uint32_t *c, uint64_t *out, uint64_t n)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = mp_occ(ix, idx[i], c[i]);
}
__global__ void k_sa(MpIndexView ix, const uint64_t *idx, uint64_t *out, uint64_t n)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = mp_sa(ix, idx[i]);
}
__global__ void k_lkt(MpIndexView ix, const uint32_t *key, uint64_t *l, uint64_t *r, uint64_t n)
{
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { uint32_t k = key[i]; l[i] = k == 0 ? 1 : ix.lkt[k - 1] + 1; r[i] = ix.lkt[k]; }
}

extern "C" int mp_occ(mp_context *ctx, const uint64_t *idx, const uint32_t *c, uint64_t *out, uint64_t n)
{
    if (!ctx || !ctx->hasIndex) { mp_set_error("mp_occ: no index loaded"); return MP_ERR_STATE; }
    DevBuf a, b, o;
    if (a.reserve(n * 8) || b.reserve(n * 4) || o.reserve(n * 8)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpy(a.p, idx, n * 8, cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(b.p, c, n * 4, cudaMemcpyHostToDevice));
    (++g_mp_launches), k_occ<<<(unsigned)((n + 255) / 256), 256>>>(ctx->ix, a.as<uint64_t>(), b.as<uint32_t>(), o.as<uint64_t>(), n);
    MP_CUDA(cudaMemcpy(out, o.p, n * 8, cudaMemcpyDeviceToHost));
    a.release(); b.release(); o.release();
    return 0;
}
extern "C" int mp_sa(mp_context *ctx, const uint64_t *idx, uint64_t *out, uint64_t n)
{
    if (!ctx || !ctx->hasIndex) { mp_set_error("mp_sa: no index loaded"); return MP_ERR_STATE; }
    DevBuf a, o;
    if (a.reserve(n * 8) || o.reserve(n * 8)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpy(a.p, idx, n * 8, cudaMemcpyHostToDevice));
    (++g_mp_launches), k_sa<<<(unsigned)((n + 255) / 256), 256>>>(ctx->ix, a.as<uint64_t>(), o.as<uint64_t>(), n);
    MP_CUDA(cudaMemcpy(out, o.p, n * 8, cudaMemcpyDeviceToHost));
    a.release(); o.release();
    return 0;
}
extern "C" int mp_lkt(mp_context *ctx, const uint32_t *key, uint64_t *l, uint64_t *r, uint64_t n)
{
    if (!ctx || !ctx->hasIndex) { mp_set_error("mp_lkt: no index loaded"); return MP_ERR_STATE; }
    DevBuf a, o1, o2;
    if (a.reserve(n * 4) || o1.reserve(n * 8) || o2.reserve(n * 8)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpy(a.p, key, n * 4, cudaMemcpyHostToDevice));
    (++g_mp_launches), k_lkt<<<(unsigned)((n + 255) / 256), 256>>>(ctx->ix, a.as<uint32_t>(), o1.as<uint64_t>(), o2.as<uint64_t>(), n);
    MP_CUDA(cudaMemcpy(l, o1.p, n * 8, cudaMemcpyDeviceToHost));
    MP_CUDA(cudaMemcpy(r, o2.p, n * 8, cudaMemcpyDeviceToHost));
    a.release(); o1.release(); o2.release();
    return 0;
}
