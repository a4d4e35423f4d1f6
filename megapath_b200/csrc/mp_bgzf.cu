// mp_bgzf.cu -- BGZF (the blocked gzip container of BAM files) compressed on the device: mp_bgzf_reserve / mp_bgzf_compress.
//
// The input is cut into consecutive pieces of at most 0xff00 bytes; every piece becomes one complete BGZF member -- the gzip header
// with the "BC" extra subfield and BSIZE, one final raw DEFLATE block, CRC-32 and ISIZE -- exactly the framing
// BgzfWriter::compress_block (host/bam_out.h) writes with zlib.  Members are independent, so their concatenation is a valid stream
// and a reader decodes the same bytes whatever encoder made them.
//
// k_bgzf_member: one 512-thread CTA per piece (persistent: a CTA loops over pieces), the piece in shared memory.
//   crc        every thread takes the CRC-32 of its 128-byte slice; one thread combines the slices with x^(8n) mod P shifts
//              (zlib's crc32_combine) while another parses.
//   match      positions are matched in tiles of 512: each position looks up the last earlier-tile position with the same 3-byte and
//              4-byte hash (two head tables, updated with atomicMax after every tile, so the result does not depend on thread order),
//              keeps the longer match (3..258 bytes, distance <= 32768, the DEFLATE window) and writes (length, distance) to a
//              per-CTA scratch row in global memory.
//   parse      greedy: one thread walks next = i + max(1, len[i]) over the lengths in shared memory and flags the token starts.
//   trees      a shared-memory histogram of the tokens; one thread builds length-limited Huffman codes (15 bits, 7 for the
//              code-length code; at least two codes per tree, as zlib's trees.c does), run-length codes the code lengths with 16/17/18
//              and counts the exact bits of the dynamic, fixed and stored encodings.  The smallest is emitted.
//   emit       every thread sizes the tokens that start in its slice, a block scan gives each slice its bit offset, and the slices are
//              OR'ed into the piece's 64 KiB output slot (zeroed first).
// A scan of the member sizes and k_bgzf_gather then pack the slots into one contiguous stream.
// Every tie (hash heads, equal-length matches, equal frequencies in the Huffman construction) is broken by position or symbol
// number, so the output depends on the input bytes only.
#include "mp_context.h"
#include "mp_crc32.h"
#include <cub/cub.cuh>

namespace {

constexpr int BG_THREADS = 512;
constexpr uint32_t BG_PIECE = 0xff00;           // input bytes per member, as BgzfWriter::compress_all cuts them
constexpr uint32_t BG_SLOT = 65536;             // a member never exceeds this: a stored block is 0xff00 + 5 + 26 bytes
constexpr int BG_HASH_BITS = 14;
constexpr uint32_t BG_WINDOW = 32768;

__constant__ uint16_t c_lenBase[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258 };
__constant__ uint8_t c_lenExtra[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
__constant__ uint16_t c_distBase[30] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
                                         4097, 6145, 8193, 12289, 16385, 24577 };
__constant__ uint8_t c_distExtra[30] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };
__constant__ uint8_t c_clOrder[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

typedef cub::BlockScan<uint32_t, BG_THREADS> BgScan;

struct BgSmem {
    uint8_t bytes[BG_PIECE + 16];
    // matching: two hash-head tables (position + 1, 0 = none); from the parse on: the match length of every position (u16, bit 15 =
    // token start)
    uint32_t region[2u << BG_HASH_BITS];
    uint32_t crcTab[256];
    uint32_t sliceCrc[BG_THREADS];
    uint32_t litFreq[288], distFreq[32], clFreq[20];
    uint16_t litCode[288], distCode[32], clCode[20];
    uint8_t litLen[288], distLen[32], clLen[20];
    uint8_t lenLut[256], distLut[512];
    // Huffman construction (one thread)
    unsigned long long sortKey[288];
    uint32_t moff[288];
    uint16_t rle[320];                           // run-length coded code lengths: symbol | extra << 5
    uint8_t allLens[320];
    int hcount[33], hnext[16];
    typename BgScan::TempStorage scan;
    uint32_t nRle, hlit, hdist, hclen, mode, headerBits, crc, totalBits;
};

__device__ __forceinline__ void bg_or_byte(uint32_t *slot, uint32_t at, uint32_t v) { atomicOr(slot + (at >> 2), (v & 0xffu) << ((at & 3) * 8)); }

// LSB-first bit writer into a zeroed slot, by 32-bit atomicOr (neighbouring slices share their boundary words)
struct BgBits {
    uint32_t *slot; uint64_t acc; uint32_t word; int n;
    __device__ BgBits(uint32_t *s, uint32_t bitPos) : slot(s), acc(0), word(bitPos >> 5), n((int)(bitPos & 31)) {}
    __device__ __forceinline__ void put(uint32_t v, int len) {
        acc |= (uint64_t)v << n; n += len;
        while (n >= 32) { atomicOr(slot + word, (uint32_t)acc); acc >>= 32; n -= 32; ++word; }
    }
    __device__ __forceinline__ void flush() { if (n > 0) atomicOr(slot + word, (uint32_t)acc); }
};

__device__ __forceinline__ uint32_t bg_rev(uint32_t code, int len) { return __brev(code) >> (32 - len); }

// Code lengths limited to `limit` bits for symbols 0..n-1 of freq[] (zero-frequency symbols get 0; at least two symbols get a code, the
// lowest-numbered unused ones standing in, as trees.c does).  In-place minimum-redundancy lengths (Moffat & Katajainen) over the
// symbols sorted by (frequency, symbol), then the length-limiting and length assignment of miniz's tdefl_optimize_huffman_table.
__device__ void bg_build_lengths(BgSmem &S, const uint32_t *freqIn, int n, int limit, uint8_t *lens)
{
    int used = 0;
    for (int s = 0; s < n; ++s) { lens[s] = 0; if (freqIn[s]) S.sortKey[used++] = ((unsigned long long)freqIn[s] << 16) | (unsigned)s; }
    for (int s = 0; used < 2 && s < n; ++s) if (!freqIn[s]) S.sortKey[used++] = (1ull << 16) | (unsigned)s;
    for (int i = 1; i < used; ++i) {                                            // insertion sort (at most 286 keys)
        const unsigned long long k = S.sortKey[i]; int j = i - 1;
        while (j >= 0 && S.sortKey[j] > k) { S.sortKey[j + 1] = S.sortKey[j]; --j; }
        S.sortKey[j + 1] = k;
    }
    uint32_t *A = S.moff;
    for (int i = 0; i < used; ++i) A[i] = (uint32_t)(S.sortKey[i] >> 16);
    {
        int root = 0, leaf = 2, next;
        A[0] += A[1];
        for (next = 1; next < used - 1; ++next) {
            if (leaf >= used || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = (uint32_t)next; } else A[next] = A[leaf++];
            if (leaf >= used || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = (uint32_t)next; } else A[next] += A[leaf++];
        }
        A[used - 2] = 0;
        for (next = used - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
        int avbl = 1, u = 0, dpth = 0; root = used - 2; next = used - 1;
        while (avbl > 0) {
            while (root >= 0 && (int)A[root] == dpth) { ++u; --root; }
            while (avbl > u) { A[next--] = (uint32_t)dpth; --avbl; }
            avbl = 2 * u; ++dpth; u = 0;
        }
    }
    int *count = S.hcount;
    for (int i = 0; i <= 32; ++i) count[i] = 0;
    for (int i = 0; i < used; ++i) ++count[A[i] > 32 ? 32 : A[i]];
    for (int i = limit + 1; i <= 32; ++i) { count[limit] += count[i]; count[i] = 0; }
    uint32_t total = 0;
    for (int i = limit; i > 0; --i) total += (uint32_t)count[i] << (limit - i);
    while (total != (1u << limit)) {
        --count[limit];
        for (int i = limit - 1; i > 0; --i) if (count[i]) { --count[i]; count[i + 1] += 2; break; }
        --total;
    }
    for (int i = 1, j = used; i <= limit; ++i)
        for (int l = count[i]; l > 0; --l) lens[S.sortKey[--j] & 0xffff] = (uint8_t)i;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first writer
__device__ void bg_codes(BgSmem &S, const uint8_t *lens, int n, uint16_t *codes)
{
    int *cnt = S.hcount, *next = S.hnext;
    for (int i = 0; i < 16; ++i) cnt[i] = 0;
    for (int s = 0; s < n; ++s) ++cnt[lens[s]];
    cnt[0] = 0;
    int code = 0;
    for (int b = 1; b < 16; ++b) { code = (code + cnt[b - 1]) << 1; next[b] = code; }
    for (int s = 0; s < n; ++s) codes[s] = lens[s] ? (uint16_t)bg_rev((uint32_t)next[lens[s]]++, lens[s]) : 0;
}

__device__ __forceinline__ int bg_dist_code(const BgSmem &S, uint32_t d) { return S.distLut[d <= 256 ? d - 1 : 256 + ((d - 1) >> 7)]; }

// Trees, costs and the choice of encoding for one piece (thread 0).  Sets S.mode (0 stored, 1 fixed, 2 dynamic), the code tables and,
// for the dynamic block, the run-length coded header.
__device__ __noinline__ void bg_plan(BgSmem &S, uint32_t n)
{
    uint64_t extraBits = 0;
    for (int c = 0; c < 29; ++c) extraBits += (uint64_t)S.litFreq[257 + c] * c_lenExtra[c];
    for (int c = 0; c < 30; ++c) extraBits += (uint64_t)S.distFreq[c] * c_distExtra[c];
    // fixed
    uint64_t fixedBits = 3 + extraBits;
    for (int s = 0; s < 286; ++s) fixedBits += (uint64_t)S.litFreq[s] * (s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8);
    for (int c = 0; c < 30; ++c) fixedBits += (uint64_t)S.distFreq[c] * 5;
    // dynamic
    bg_build_lengths(S, S.litFreq, 286, 15, S.litLen);
    bg_build_lengths(S, S.distFreq, 30, 15, S.distLen);
    int hlit = 286, hdist = 30;
    while (hlit > 257 && !S.litLen[hlit - 1]) --hlit;
    while (hdist > 1 && !S.distLen[hdist - 1]) --hdist;
    const int nl = hlit + hdist;
    for (int i = 0; i < hlit; ++i) S.allLens[i] = S.litLen[i];
    for (int i = 0; i < hdist; ++i) S.allLens[hlit + i] = S.distLen[i];
    for (int i = 0; i < 19; ++i) S.clFreq[i] = 0;
    int nr = 0;
    for (int i = 0; i < nl;) {
        const uint8_t v = S.allLens[i];
        int r = 1;
        while (i + r < nl && S.allLens[i + r] == v) ++r;
        i += r;
        if (v == 0) {
            while (r >= 11) { const int k = r < 138 ? r : 138; S.rle[nr++] = (uint16_t)(18 | (k - 11) << 5); ++S.clFreq[18]; r -= k; }
            if (r >= 3) { S.rle[nr++] = (uint16_t)(17 | (r - 3) << 5); ++S.clFreq[17]; r = 0; }
        } else {
            S.rle[nr++] = v; ++S.clFreq[v]; --r;
            while (r >= 3) { const int k = r < 6 ? r : 6; S.rle[nr++] = (uint16_t)(16 | (k - 3) << 5); ++S.clFreq[16]; r -= k; }
        }
        while (r > 0) { S.rle[nr++] = v; ++S.clFreq[v]; --r; }
    }
    bg_build_lengths(S, S.clFreq, 19, 7, S.clLen);
    int hclen = 19;
    while (hclen > 4 && !S.clLen[c_clOrder[hclen - 1]]) --hclen;
    uint64_t dynBits = 3 + 5 + 5 + 4 + 3 * (uint64_t)hclen + extraBits;
    for (int k = 0; k < nr; ++k) { const int s = S.rle[k] & 31; dynBits += S.clLen[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0); }
    for (int s = 0; s < 286; ++s) dynBits += (uint64_t)S.litFreq[s] * S.litLen[s];
    for (int c = 0; c < 30; ++c) dynBits += (uint64_t)S.distFreq[c] * S.distLen[c];
    const uint64_t storedBits = (5ull + n) * 8;
    S.nRle = (uint32_t)nr; S.hlit = (uint32_t)hlit; S.hdist = (uint32_t)hdist; S.hclen = (uint32_t)hclen;
    if (dynBits <= fixedBits && dynBits < storedBits) {
        S.mode = 2;
        bg_codes(S, S.litLen, 286, S.litCode); bg_codes(S, S.distLen, 30, S.distCode); bg_codes(S, S.clLen, 19, S.clCode);
        S.headerBits = 3 + 14 + 3 * hclen;
        for (int k = 0; k < nr; ++k) { const int s = S.rle[k] & 31; S.headerBits += S.clLen[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0); }
    } else if (fixedBits < storedBits) {
        S.mode = 1;
        for (int s = 0; s < 288; ++s) S.litLen[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
        for (int c = 0; c < 30; ++c) S.distLen[c] = 5;
        bg_codes(S, S.litLen, 288, S.litCode); bg_codes(S, S.distLen, 30, S.distCode);
        S.headerBits = 3;
    } else {
        S.mode = 0; S.headerBits = 0;
    }
}

__device__ __forceinline__ uint32_t bg_token_bits(const BgSmem &S, const uint32_t *scr, uint32_t p, uint32_t v)
{
    const uint32_t L = v & 0x7fff;
    if (!L) return S.litLen[S.bytes[p]];
    const int lc = S.lenLut[L - 3], dc = bg_dist_code(S, scr[p] & 0xffff);
    return S.litLen[257 + lc] + c_lenExtra[lc] + S.distLen[dc] + c_distExtra[dc];
}

__global__ void __launch_bounds__(BG_THREADS, 1)
k_bgzf_member(const uint8_t *__restrict__ src, uint64_t n, uint32_t nPieces, uint8_t *__restrict__ slots, unsigned long long *__restrict__ sizes,
              uint32_t *__restrict__ scratch)
{
    extern __shared__ __align__(16) uint8_t bg_smem_raw[];
    BgSmem &S = *reinterpret_cast<BgSmem *>(bg_smem_raw);
    const int t = threadIdx.x;
    uint32_t *scr = scratch + (size_t)blockIdx.x * BG_PIECE;
    if (t < 256) {
        uint32_t c = (uint32_t)t;
        for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        S.crcTab[t] = c;
        int lc = 28; while (c_lenBase[lc] > t + 3) --lc;
        S.lenLut[t] = (uint8_t)lc;
    }
    if (t < 512) {
        const uint32_t d = t < 256 ? (uint32_t)t + 1 : ((uint32_t)(t - 256) << 7) + 1;
        int dc = 29; while (c_distBase[dc] > d) --dc;
        S.distLut[t] = (uint8_t)dc;
    }
    for (uint32_t piece = blockIdx.x; piece < nPieces; piece += gridDim.x) {
        const uint64_t base = (uint64_t)piece * BG_PIECE;
        const uint32_t len = (uint32_t)(n - base < BG_PIECE ? n - base : BG_PIECE);
        uint32_t *slot = reinterpret_cast<uint32_t *>(slots + (size_t)piece * BG_SLOT);
        // ---- load, zero the slot and the head tables, histograms ----
        for (uint32_t i = t; i < len; i += BG_THREADS) S.bytes[i] = src[base + i];
        if (t < 16) S.bytes[len + t] = 0;
        for (uint32_t i = t; i < BG_SLOT / 16; i += BG_THREADS) reinterpret_cast<uint4 *>(slot)[i] = make_uint4(0, 0, 0, 0);
        for (uint32_t i = t; i < (2u << BG_HASH_BITS); i += BG_THREADS) S.region[i] = 0;
        for (int i = t; i < 288; i += BG_THREADS) S.litFreq[i] = 0;
        if (t < 32) S.distFreq[t] = 0;
        __syncthreads();
        const uint32_t per = (len + BG_THREADS - 1) / BG_THREADS, lo = min(len, t * per), hi = min(len, lo + per);
        {
            uint32_t c = 0xffffffffu;
            for (uint32_t i = lo; i < hi; ++i) c = S.crcTab[(c ^ S.bytes[i]) & 0xff] ^ (c >> 8);
            S.sliceCrc[t] = ~c;
        }
        // ---- matching, tile by tile ----
        uint32_t *head3 = S.region, *head4 = S.region + (1u << BG_HASH_BITS);
        for (uint32_t tile = 0; tile < len; tile += BG_THREADS) {
            const uint32_t i = tile + t;
            uint32_t h3 = 0, h4 = 0, best = 0;
            const bool ok3 = i + 3 <= len, ok4 = i + 4 <= len;
            if (ok3) {
                const uint32_t w3 = S.bytes[i] | (uint32_t)S.bytes[i + 1] << 8 | (uint32_t)S.bytes[i + 2] << 16;
                h3 = (w3 * 2654435761u) >> (32 - BG_HASH_BITS);
                h4 = ((w3 | (uint32_t)S.bytes[i + 3] << 24) * 2246822519u) >> (32 - BG_HASH_BITS);
                const uint32_t maxL = min(258u, len - i);
                uint32_t bestL = 0, bestD = 0;
                const uint32_t cand[2] = { ok4 ? head4[h4] : 0u, head3[h3] };
                for (int k = 0; k < 2; ++k) {
                    if (!cand[k] || (k == 1 && cand[1] == cand[0])) continue;
                    const uint32_t c = cand[k] - 1, d = i - c;
                    if (d > BG_WINDOW) continue;
                    uint32_t L = 0;
                    while (L < maxL && S.bytes[c + L] == S.bytes[i + L]) ++L;
                    if (L > bestL) { bestL = L; bestD = d; }
                }
                if (bestL >= 3) best = bestL << 16 | bestD;
            }
            if (i < len) scr[i] = best;
            __syncthreads();
            if (ok3) atomicMax(head3 + h3, i + 1);
            if (ok4) atomicMax(head4 + h4, i + 1);
            __syncthreads();
        }
        // ---- greedy parse (thread 0) beside the CRC combination (thread 32) ----
        uint16_t *lens = reinterpret_cast<uint16_t *>(S.region);
        for (uint32_t i = t; i < len; i += BG_THREADS) lens[i] = (uint16_t)(scr[i] >> 16);
        __syncthreads();
        if (t == 0) {
            for (uint32_t p = 0; p < len;) { const uint32_t v = lens[p]; lens[p] = (uint16_t)(v | 0x8000); p += v ? v : 1; }
        } else if (t == 32) {
            uint32_t c = S.sliceCrc[0];
            const uint32_t shiftPer = mp_crc32_x8n(per);
            for (uint32_t k = 1; k < BG_THREADS; ++k) {
                const uint32_t a = min(len, k * per), b = min(len, a + per);
                if (b == a) break;
                c = mp_crc32_mulmod(b - a == per ? shiftPer : mp_crc32_x8n(b - a), c) ^ S.sliceCrc[k];
            }
            S.crc = c;
        }
        __syncthreads();
        // ---- histogram ----
        for (uint32_t p = lo; p < hi; ++p) {
            const uint32_t v = lens[p];
            if (!(v & 0x8000)) continue;
            const uint32_t L = v & 0x7fff;
            if (!L) atomicAdd(&S.litFreq[S.bytes[p]], 1u);
            else { atomicAdd(&S.litFreq[257 + S.lenLut[L - 3]], 1u); atomicAdd(&S.distFreq[bg_dist_code(S, scr[p] & 0xffff)], 1u); }
        }
        __syncthreads();
        if (t == 0) { S.litFreq[256] = 1; bg_plan(S, len); }
        __syncthreads();
        const uint32_t mode = S.mode;
        uint32_t clen;
        if (mode == 0) {
            uint8_t *o = reinterpret_cast<uint8_t *>(slot);
            for (uint32_t i = t; i < len; i += BG_THREADS) o[23 + i] = S.bytes[i];
            if (t == 0) { o[18] = 1; o[19] = len & 0xff; o[20] = len >> 8; o[21] = ~len & 0xff; o[22] = (~len >> 8) & 0xff; }
            clen = len + 5;
            __syncthreads();
        } else {
            uint32_t bits = 0;
            for (uint32_t p = lo; p < hi; ++p) { const uint32_t v = lens[p]; if (v & 0x8000) bits += bg_token_bits(S, scr, p, v); }
            uint32_t off;
            BgScan(S.scan).ExclusiveSum(bits, off);
            if (t == BG_THREADS - 1) S.totalBits = S.headerBits + off + bits;
            BgBits w(slot, 18 * 8 + S.headerBits + off);
            for (uint32_t p = lo; p < hi; ++p) {
                const uint32_t v = lens[p];
                if (!(v & 0x8000)) continue;
                const uint32_t L = v & 0x7fff;
                if (!L) { const uint8_t b = S.bytes[p]; w.put(S.litCode[b], S.litLen[b]); continue; }
                const int lc = S.lenLut[L - 3];
                w.put(S.litCode[257 + lc], S.litLen[257 + lc]);
                if (c_lenExtra[lc]) w.put(L - c_lenBase[lc], c_lenExtra[lc]);
                const uint32_t d = scr[p] & 0xffff;
                const int dc = bg_dist_code(S, d);
                w.put(S.distCode[dc], S.distLen[dc]);
                if (c_distExtra[dc]) w.put(d - c_distBase[dc], c_distExtra[dc]);
            }
            w.flush();
            __syncthreads();
            if (t == 0) {
                BgBits h(slot, 18 * 8);
                h.put(1, 1);
                if (mode == 1) h.put(1, 2);
                else {
                    h.put(2, 2); h.put(S.hlit - 257, 5); h.put(S.hdist - 1, 5); h.put(S.hclen - 4, 4);
                    for (uint32_t k = 0; k < S.hclen; ++k) h.put(S.clLen[c_clOrder[k]], 3);
                    for (uint32_t k = 0; k < S.nRle; ++k) {
                        const int s = S.rle[k] & 31, x = S.rle[k] >> 5;
                        h.put(S.clCode[s], S.clLen[s]);
                        if (s >= 16) h.put((uint32_t)x, s == 16 ? 2 : s == 17 ? 3 : 7);
                    }
                }
                h.flush();
                BgBits e(slot, 18 * 8 + S.totalBits);
                e.put(S.litCode[256], S.litLen[256]);
                e.flush();
            }
            clen = (S.totalBits + S.litLen[256] + 7) / 8;
        }
        // ---- gzip framing ----
        if (t == 0) {
            const uint32_t size = clen + 26;
            const uint8_t hdr[18] = { 31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0, (uint8_t)((size - 1) & 0xff), (uint8_t)((size - 1) >> 8) };
            for (int k = 0; k < 18; ++k) bg_or_byte(slot, k, hdr[k]);
            for (int k = 0; k < 4; ++k) { bg_or_byte(slot, 18 + clen + k, S.crc >> (8 * k)); bg_or_byte(slot, 22 + clen + k, len >> (8 * k)); }
            sizes[piece] = size;
        }
        __syncthreads();
    }
}

__global__ void k_bgzf_gather(const uint8_t *__restrict__ slots, const unsigned long long *__restrict__ offs, uint32_t nPieces, uint8_t *__restrict__ out)
{
    const uint32_t piece = blockIdx.x;
    if (piece >= nPieces) return;
    const uint64_t at = offs[piece], size = offs[piece + 1] - at;
    const uint8_t *s = slots + (size_t)piece * BG_SLOT;
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) out[at + i] = s[i];
}

int bg_reserve(mp_context *ctx, uint64_t maxBytes)
{
    const uint64_t nPieces = (maxBytes + BG_PIECE - 1) / BG_PIECE;
    int sms = 0;
    MP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    const uint64_t grid = nPieces < (uint64_t)sms ? nPieces : (uint64_t)sms;
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int64_t)(nPieces + 1), ctx->stream);
    if (ctx->dBgzfIn.reserve(maxBytes) || ctx->dBgzfSlots.reserve(nPieces * BG_SLOT) || ctx->dBgzfOut.reserve(nPieces * BG_SLOT) ||
        ctx->dBgzfSizes.reserve((nPieces + 1) * 8) || ctx->dBgzfOffs.reserve((nPieces + 1) * 8) || ctx->dBgzfScratch.reserve(grid * BG_PIECE * 4) ||
        ctx->dScanTmp.reserve(tb)) return MP_ERR_CUDA;
    return 0;
}

}  // namespace

extern "C" int mp_bgzf_reserve(mp_context *ctx, uint64_t maxBytes)
{
    if (!ctx || maxBytes == 0) { mp_set_error("mp_bgzf_reserve: bad argument"); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(ctx->device));
    return bg_reserve(ctx, maxBytes);
}

extern "C" int mp_bgzf_compress(mp_context *ctx, const uint8_t *src, uint64_t n, uint8_t *dst, uint64_t dstCap, uint64_t *outBytes)
{
    if (!ctx || !outBytes || (n && (!src || !dst))) { mp_set_error("mp_bgzf_compress: bad argument"); return MP_ERR_ARG; }
    *outBytes = 0;
    if (n == 0) return 0;
    const uint64_t nPieces = (n + BG_PIECE - 1) / BG_PIECE;
    if (dstCap < nPieces * BG_SLOT) {
        mp_set_error("mp_bgzf_compress: dstCap %llu is below MP_BGZF_BOUND(%llu) = %llu", (unsigned long long)dstCap, (unsigned long long)n,
                     (unsigned long long)(nPieces * BG_SLOT));
        return MP_ERR_ARG;
    }
    if (nPieces >= (1ull << 31)) { mp_set_error("mp_bgzf_compress: input too large"); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(ctx->device));
    if (int rc = bg_reserve(ctx, n)) return rc;
    MP_CUDA(cudaFuncSetAttribute(k_bgzf_member, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BgSmem)));
    int sms = 0;
    MP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    const uint32_t grid = (uint32_t)(nPieces < (uint64_t)sms ? nPieces : (uint64_t)sms);
    cudaStream_t st = ctx->stream;
    unsigned long long *sizes = ctx->dBgzfSizes.as<unsigned long long>(), *offs = ctx->dBgzfOffs.as<unsigned long long>();
    MP_CUDA(cudaMemcpyAsync(ctx->dBgzfIn.p, src, n, cudaMemcpyHostToDevice, st));
    MP_CUDA(cudaMemsetAsync(sizes + nPieces, 0, 8, st));
    (++g_mp_launches), k_bgzf_member<<<grid, BG_THREADS, sizeof(BgSmem), st>>>(ctx->dBgzfIn.as<uint8_t>(), n, (uint32_t)nPieces, ctx->dBgzfSlots.as<uint8_t>(),
                                                                             sizes, ctx->dBgzfScratch.as<uint32_t>());
    MP_CUDA(cudaGetLastError());
    size_t tb = ctx->dScanTmp.cap;
    MP_CUDA(cub::DeviceScan::ExclusiveSum(ctx->dScanTmp.p, tb, sizes, offs, (int64_t)(nPieces + 1), st));
    (++g_mp_launches), k_bgzf_gather<<<(uint32_t)nPieces, 256, 0, st>>>(ctx->dBgzfSlots.as<uint8_t>(), offs, (uint32_t)nPieces, ctx->dBgzfOut.as<uint8_t>());
    MP_CUDA(cudaGetLastError());
    unsigned long long total = 0;
    MP_CUDA(cudaMemcpyAsync(&total, offs + nPieces, 8, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    MP_CUDA(cudaMemcpyAsync(dst, ctx->dBgzfOut.p, total, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    *outBytes = total;
    return 0;
}
