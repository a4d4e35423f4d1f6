// mp_seed.cu -- MMP seeding, SA resolution, seed merging/filtering and paired-end candidate
// generation on the device.  Replaces, for all pairs of a batch,
//   mmp<0>/mmp<2> + CHECK_AND_SET_LAST / CHECK_AND_ADD_RANGE   DV-DPfunctions.cpp:2188-2377
//   PairEndSeedingBatch::mmpSeeding post-processing             DV-DPfunctions.cpp:2474-2553
//   pairEndMerge / findRevStart / mergeAndPairPairedEnd         DV-DPfunctions.cpp:1844-2119
//
// Kernels (DESIGN.md "Seeding"):
//   k_mmp      one thread per read-strand, written as a state machine (filter probes + LKT jump | one backward-search
//              step | up to 32 text bases per trip once the range is a single suffix); a K-mer presence filter rules out
//              starts that cannot give a seed; seed slots are allocated with one atomic per warp.
//   k_expand   one thread per (seed, k) suffix-array hit that k_mmp did not resolve itself: SA lookup (dense 32-bit
//              array, or LF walk to the next sample), text position, hit record written into its read's segment.
//   k_merge    one thread per read: sort hits by (strand, position), chain within indelFuzz,
//              covered-length union, uniqueness / length filters -> SeedPos entries.
//   k_pair     one thread per pair and orientation: window join -> CandidateInfo.
#include "mp_context.h"
#include <cooperative_groups.h>
#include <cooperative_groups/scan.h>
#include <cooperative_groups/reduce.h>
namespace cg = cooperative_groups;
#include <cub/device/device_scan.cuh>
#include <algorithm>

struct MmpDev {
    int seedSAsizeThreshold, seedMinLength, uniqThreshold, indelFuzz, goodSeedLen, reseedLen, reseedAbsDiff;
    double reseedRLTratio, shortSeedRatio;
};

// ------------------------------------------------------------------------------------
// de-interleave the 32-read interleaved query buffer (QueryParser.cpp:184-203)
// ------------------------------------------------------------------------------------
__global__ void k_deinterleave(const uint32_t *__restrict__ il, uint32_t *__restrict__ out, uint32_t nReads, uint32_t wpq)
{
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t total = ((uint64_t)nReads + 31) / 32 * 32 * wpq;      // whole 32-read groups: the last one may be partial
    if (t >= total) return;
    // consecutive threads read consecutive interleaved words
    uint64_t grp = t / (32ull * wpq);
    uint32_t within = (uint32_t)(t - grp * 32ull * wpq);
    uint32_t j = within >> 5, r32 = within & 31;
    uint64_t r = grp * 32 + r32;
    if (r < nReads) out[r * wpq + j] = il[t];
}

// A lane's read lives in shared memory while the lane works on it (staged once when the lane takes the strand): word w of the
// read at rd[w * MMP_RS] -- consecutive threads hold consecutive banks -- followed by two zero words, so that the three-word window
// fetches below never leave the lane's column.  Every trip of k_mmp re-reads a few of these words; as plain global loads they were two
// thirds of the kernel's L1 traffic.
#define MMP_RS 128
__device__ __forceinline__ uint32_t read_base(const uint32_t *rd, int p)
{
    return (rd[(p >> 4) * MMP_RS] >> ((p & 15) << 1)) & 3;
}

// 13-mer key at scan position i (DV-DPfunctions.cpp:2233-2239, 2326-2332): q[i+k] at bits 2k
__device__ __forceinline__ uint32_t lkt_key(const uint32_t *rd, int len, int i, int strand)
{
    int p0 = strand ? i : len - 13 - i;                       // lowest read position of the 13-mer
    uint32_t w0 = rd[(p0 >> 4) * MMP_RS], w1 = rd[((p0 >> 4) + 1) * MMP_RS];
    uint32_t x = __funnelshift_r(w0, w1, (p0 & 15) << 1);      // base p0 in the low bits
    if (strand) return (~x) & 0x3FFFFFFu;                      // complemented, same order
    uint32_t t = __brev(x);                                    // reverse the order of the 2-bit groups
    t = ((t >> 1) & 0x55555555u) | ((t & 0x55555555u) << 1);
    return (t >> 6) & 0x3FFFFFFu;
}

// ------------------------------------------------------------------------------------
// K-mer presence filter (K = min(seedMinLength, 32)).  A backward search that starts at scan
// position i0 and empties before seedMinLength bases emits nothing and restarts at i0 + 1
// (CHECK_AND_ADD_RANGE rewinds by seed_len, DV-DPfunctions.cpp:2197-2219), so a start whose first
// K bases do not occur in the text can be skipped without touching the FM-index.  The filter is a
// word-blocked Bloom filter over all K-mers of the text (16 bits per text position, two bits per
// key inside one 64-bit word): no false negatives, ~2 % false positives which simply take the
// exact path.  The non-matching strand of every read (and every unalignable read) is rejected
// with one independent 8-byte gather per start position instead of a dependent chain of
// LKT + occ-block gathers.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ void bloom_slot(uint64_t key, uint64_t nWords, uint64_t &word, uint64_t &mask)
{
    uint64_t h = key * 0x9E3779B97F4A7C15ull;
    h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
    word = __umul64hi(h, nWords);
    mask = (1ull << (h & 63)) | (1ull << ((h >> 6) & 63));
}
// 2K bits of a 2-bit, LSB-first packed read starting at base `pos` (K <= 32)
__device__ __forceinline__ uint64_t read_window(const uint32_t *rd, int pos, int K)
{
    const int w = pos >> 4, sh = (pos & 15) << 1;
    uint32_t w0 = rd[w * MMP_RS], w1 = rd[(w + 1) * MMP_RS], w2 = rd[(w + 2) * MMP_RS];
    uint64_t v = (uint64_t)__funnelshift_r(w0, w1, sh) | ((uint64_t)__funnelshift_r(w1, w2, sh) << 32);
    return K == 32 ? v : v & ((1ull << (2 * K)) - 1);
}
// key of the K-mer the backward search would have matched after K steps from scan position i
// (text order, first base in the most significant 2-bit group)
__device__ __forceinline__ uint64_t scan_kmer(const uint32_t *rd, int len, int i, int strand, int K)
{
    if (strand) {                   // pattern = revcomp(read[i .. i+K-1]): complement, base i least significant
        uint64_t v = read_window(rd, i, K);
        return (~v) & (K == 32 ? ~0ull : ((1ull << (2 * K)) - 1));
    }
    uint64_t v = read_window(rd, len - i - K, K);     // read[q-K+1 .. q], q = len-1-i, first base least significant
    v = __brevll(v);                                   // reverse the order of the 2-bit groups
    v = ((v >> 1) & 0x5555555555555555ull) | ((v & 0x5555555555555555ull) << 1);
    return v >> (64 - 2 * K);
}
__global__ void k_bloom_build(const uint8_t *__restrict__ pac, uint64_t n, int K, unsigned long long *__restrict__ bloom, uint64_t nWords)
{
    // each thread rolls over 64 consecutive K-mer end positions
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t first = t * 64;                     // first K-mer start handled here
    if (first + K > n) return;
    const uint64_t maskK = K == 32 ? ~0ull : ((1ull << (2 * K)) - 1);
    uint64_t key = 0;
    for (int a = 0; a < K - 1; ++a) key = (key << 2) | ((pac[(first + a) >> 2] >> ((3 - ((first + a) & 3)) << 1)) & 3);
    for (int j = 0; j < 64; ++j) {
        uint64_t e = first + j + K - 1;                // last base of this K-mer
        if (e >= n) break;
        key = ((key << 2) | ((pac[e >> 2] >> ((3 - (e & 3)) << 1)) & 3)) & maskK;
        uint64_t w, m; bloom_slot(key, nWords, w, m);
        atomicOr(&bloom[w], (unsigned long long)m);
    }
}

// rank of symbol c among the first `off` symbols held in three uint4 of BWT words
__device__ __forceinline__ uint32_t words_rank(const uint4 &w0, const uint4 &w1, const uint4 &w2, uint32_t c, int off)
{
    uint32_t v = 0;
    const uint4 *w[3] = { &w0, &w1, &w2 };
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        int r = off - 64 * q;
        if (r > 0) {
            v += mp_word_count(w[q]->x, c, min(r, 16)) + mp_word_count(w[q]->y, c, min(max(r - 16, 0), 16)) +
                 mp_word_count(w[q]->z, c, min(max(r - 32, 0), 16)) + mp_word_count(w[q]->w, c, min(max(r - 48, 0), 16));
        }
    }
    return v;
}

// Occ(a, c) and Occ(b, c), a <= b.  When both positions fall into the same 64-byte block (the usual case once
// the SA range is narrower than 192) the block is fetched once.
__device__ __forceinline__ void occ_pair(const MpIndexView &ix, uint64_t a, uint64_t b, uint32_t c, uint64_t &ra, uint64_t &rb)
{
    const uint64_t ba = a / MP_BLK_SYMS, bb = b / MP_BLK_SYMS;
    const int oa = (int)(a - ba * MP_BLK_SYMS), ob = (int)(b - bb * MP_BLK_SYMS);
    const uint4 *pa = ix.blocks + ba * 4;
    uint4 h = __ldg(pa), w0 = __ldg(pa + 1), w1 = make_uint4(0, 0, 0, 0), w2 = w1;
    const int need = ba == bb ? ob : oa;
    if (need > 64) w1 = __ldg(pa + 2);
    if (need > 128) w2 = __ldg(pa + 3);
    uint32_t cnt = c == 0 ? h.x : c == 1 ? h.y : c == 2 ? h.z : h.w;
    const uint64_t base = __ldg(ix.super + (ba >> MP_SUPER_SHIFT) * 4 + c) + cnt;
    ra = base + words_rank(w0, w1, w2, c, oa);
    if (ba == bb) rb = base + words_rank(w0, w1, w2, c, ob);
    else rb = mp_occ_raw(ix, b, c);
}

// ------------------------------------------------------------------------------------
// MMP seeding (mmp<0> / mmp<2>, DV-DPfunctions.cpp:2188-2377), one thread per read-strand.
//
// Phase A: LKT jump + backward-search steps while the SA range holds more than one suffix.
// Phase B: once the range is a single suffix its text position p is looked up (one gather with
//   the dense SA) and every further backward step "extend with c" is decided by comparing c with
//   the text base at p-1: for a singleton range the step succeeds iff BWT[l] == c, and BWT[l] is
//   text[SA[l]-1] ('$' when SA[l] == 0).  The emitted seeds, the reseed bookkeeping (`last` can only
//   change while the range still shrinks, i.e. in phase A) and the rewind arithmetic are those of the
//   reference; a seed that ends in phase B already knows its text position and skips SA resolution.
//   nOcc counts the occ evaluations the reference performs for the same steps (2 per step).
// ------------------------------------------------------------------------------------
// 32 text bases ending just before position p (p >= 1), text[p-1-t] at bits 2t; positions before the text start read as 0
__device__ __forceinline__ uint64_t text_window_before(const MpIndexView &ix, uint64_t p)
{
    const int64_t first = (int64_t)p - 32;                          // base offset of the window start (may be negative)
    const uint64_t f = first < 0 ? 0 : (uint64_t)first;
    const uint64_t byte0 = (f >> 2) & ~3ull;                        // 4-byte aligned
    const uint32_t *wp = (const uint32_t *)(ix.pac + byte0);
    // big-endian: first base in the top bits; 48 bases cover any 32-base window that starts inside the first word
    const uint32_t w0 = __byte_perm(__ldg(wp), 0, 0x0123), w1 = __byte_perm(__ldg(wp + 1), 0, 0x0123), w2 = __byte_perm(__ldg(wp + 2), 0, 0x0123);
    const uint32_t sh = (uint32_t)(f - byte0 * 4) * 2;
    uint64_t t = ((uint64_t)__funnelshift_l(w1, w0, sh) << 32) | __funnelshift_l(w2, w1, sh);   // bases f .. f+31, base f in the top bits
    if (first < 0) t >>= (uint32_t)(-first) * 2;                    // keep text[p-1] in the lowest group
    return t;
}
__device__ __forceinline__ uint64_t group_reverse(uint64_t v)       // reverse the order of the thirty-two 2-bit groups
{
    v = __brevll(v);
    return ((v >> 1) & 0x5555555555555555ull) | ((v & 0x5555555555555555ull) << 1);
}

// Persistent warps over a queue of read-strands.  A lane holds one read-strand at a time and the loop below is a state machine:
// every trip performs ONE unit of work of the lane's current state (4 filter probes + LKT jump | one backward-search step | one LF
// step of a sampled-SA lookup | up to 32 text bases), so lanes that are in different phases of their reads still share every trip.
// A lane whose strand is finished takes the next one from the warp's chunk of the queue at the top of the next trip (the warp
// fetches chunks of MMP_CHUNK strands with one atomic), so no lane waits for the slowest strand of its warp: the kernel is bound by
// the latency of dependent gathers, and what counts is how many lanes have one in flight.
#define MMP_CHUNK 128u
#ifndef MMP_PROBES
#define MMP_PROBES 8       /* filter probes a lane keeps in flight per trip */
#endif
__global__ void __launch_bounds__(128, 8)
k_mmp(MpIndexView ix, const uint32_t *__restrict__ reads, const uint32_t *__restrict__ lens, uint32_t wpq,
      uint32_t nStrands, MmpDev P, MpSeed *__restrict__ seeds, uint32_t *__restrict__ stubs,
      unsigned long long *__restrict__ counters, uint32_t *__restrict__ hitsPerRead,
      uint32_t capSeeds, uint32_t capStubs, const unsigned long long *__restrict__ bloom, uint64_t bloomWords, int bloomK, int bloomStride)
{
    const uint64_t n = ix.n;
    uint32_t nOcc = 0, nLkt = 0, nSaIn = 0, nLfIn = 0, nProbe = 0, nText = 0;      // per lane: a few thousand per strand, a few dozen strands
    enum { ST_SCAN, ST_STEP, ST_TEXT, ST_SA, ST_DONE };
    // Work order: first every read on the strand that matches its mate number (mate 1 '+', mate 2 '-': the strand an FR
    // library aligns on), then every read on the other strand, so that the lanes of a warp mostly share a state.
    const uint32_t nReadsK = nStrands >> 1;
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t saMask = (1ull << ix.saShift) - 1;
    const bool saDense = mp_sa_dense(ix);
    uint32_t chunkNext = 0, chunkEnd = 0;                             // warp-uniform: the warp's current piece of the queue
    bool exhausted = false;
    uint32_t read = 0, strand = 0, skipped = 0;
    int len = 0, i = 0, seed_len = 0, last_seed_len = 0;
    extern __shared__ uint32_t shReads[];                            // [wpq + 2][blockDim.x]
    uint32_t *rd = shReads + threadIdx.x;
    uint64_t l = 0, r = n, last_l = 0, last_r = n, p = 0;
    int state = ST_DONE;
    for (;;) {
        // ---- lanes without a strand take the next ones of the warp's chunk ----
        const uint32_t idle = __ballot_sync(0xffffffffu, state == ST_DONE);
        if (idle) {
            if (chunkNext == chunkEnd && !exhausted) {
                uint32_t base = 0;
                if (lane == 0) base = (uint32_t)min(atomicAdd(&counters[6], (unsigned long long)MMP_CHUNK), (unsigned long long)nStrands);
                base = __shfl_sync(0xffffffffu, base, 0);
                if (base >= nStrands) exhausted = true;
                else { chunkNext = base; chunkEnd = base + min(MMP_CHUNK, nStrands - base); }
            }
            const uint32_t avail = chunkEnd - chunkNext;
            if (avail) {
                const uint32_t rank = __popc(idle & ((1u << lane) - 1u));
                if (state == ST_DONE && rank < avail) {
                    const uint32_t w = chunkNext + rank;
                    const uint32_t group = w >= nReadsK;
                    read = group ? w - nReadsK : w; strand = (read & 1u) ^ group;
                    len = (int)lens[read];
                    const uint32_t *src = reads + (size_t)read * wpq;
                    for (uint32_t k = 0; k < wpq; ++k) rd[k * MMP_RS] = __ldg(src + k);
                    rd[wpq * MMP_RS] = 0; rd[(wpq + 1) * MMP_RS] = 0;
                    i = 0; seed_len = 0; last_seed_len = 0; l = 0; r = n; last_l = 0; last_r = n; p = 0;
                    state = ST_SCAN;
                }
                chunkNext += min((uint32_t)__popc(idle), avail);
            } else if (exhausted && idle == 0xffffffffu) break;
        }
        if (state == ST_DONE) continue;
        bool emit = false, resolved = false, finishing = false, haveNext = false;
        uint64_t nextl = 0, nextr = 0;
        if (state == ST_SCAN) {                                   // seed_len == 0: look for the next start worth searching
            if (len - i < P.seedMinLength) { state = ST_DONE; continue; }
            bool go = true;
            if (bloom) {                                          // MMP_PROBES probes in flight
                // A match of seedMinLength bases from start i0 covers the bloomK-mer at every p in [i0, i0 + bloomStride - 1]
                // (bloomK = seedMinLength - (bloomStride - 1)), so the K-mer at p = i + bloomStride - 1 decides the bloomStride starts
                // i .. p at once, the next probe the bloomStride starts after them, and so on.  (Anchoring the probes at the
                // current start rather than on a fixed grid matters after a seed that ended on a mismatch: the scan resumes
                // seedMinLength - 1 bases before it, and the first probe already spans the mismatch.)  Only the filter words are
                // kept while the loads are in flight; the two-bit masks are hashed again when they are back.
                const int lastStart = len - P.seedMinLength;
                int m = 0;
#pragma unroll
                for (int j = 0; j < MMP_PROBES; ++j) if (i + j * bloomStride <= lastStart) m = j + 1;
                unsigned long long wv[MMP_PROBES];
#pragma unroll
                for (int j = 0; j < MMP_PROBES; ++j) {
                    wv[j] = ~0ull;
                    if (j < m) { uint64_t wi, mk; bloom_slot(scan_kmer(rd, len, i + j * bloomStride + bloomStride - 1, strand, bloomK), bloomWords, wi, mk); wv[j] = __ldg(bloom + wi); }
                }
                nProbe += m;
                int hit = m;
#pragma unroll
                for (int j = MMP_PROBES - 1; j >= 0; --j)
                    if (j < m) { uint64_t wi, mk; bloom_slot(scan_kmer(rd, len, i + j * bloomStride + bloomStride - 1, strand, bloomK), bloomWords, wi, mk); if ((wv[j] & mk) == mk) hit = j; }
                go = hit < m;
                i += hit * bloomStride;                           // first start the probes do not rule out (all dead: past the last probe)
            }
            if (go) {
                uint32_t key = lkt_key(rd, len, i, strand);
                nextl = key == 0 ? 1 : __ldg(ix.lkt + key - 1) + 1;
                nextr = __ldg(ix.lkt + key);
                i += 12; seed_len = 12; ++nLkt; haveNext = true;
            }
        } else if (state == ST_STEP) {                            // one backward-search step on a range of several suffixes
            if (i >= len) { emit = true; finishing = true; }
            else {
                uint32_t c = strand ? 3 - read_base(rd, i) : read_base(rd, len - 1 - i);
                uint64_t a = l - (l > ix.inverseSa0), b = (r + 1) - ((r + 1) > ix.inverseSa0);
                uint64_t ra, rb;
                occ_pair(ix, a, b, c, ra, rb);
                nextl = mp_cum(ix, c) + ra + 1;
                nextr = mp_cum(ix, c) + rb;
                nOcc += 2; haveNext = true;
            }
        } else if (state == ST_SA) {                              // sampled SA: one LF step per trip until a sampled index (BWTSaValue, BWT.c:968-998)
            p = mp_lf(ix, p); ++skipped; ++nLfIn;
            if ((p & saMask) == 0) { p = mp_sa_sample(ix, p) + skipped; state = ST_TEXT; }
        } else {                                                  // ST_TEXT: single suffix at text position p, up to 32 bases per trip
            if (i >= len) { emit = true; finishing = true; resolved = true; }
            else {
                const int m = min(32, len - i);
                const uint64_t tw = text_window_before(ix, p);
                uint64_t d;
                int matched;
                if (strand) {                                     // c_t = 3 - read[i+t] against text[p-1-t]
                    uint64_t rw = read_window(rd, i, 32);
                    d = ~(rw ^ tw);                               // group == 0 where the bases agree
                    d = (d | (d >> 1)) & 0x5555555555555555ull;
                    matched = d ? (__ffsll((long long)d) - 1) >> 1 : 32;
                } else {                                          // c_t = read[len-1-i-t] against text[p-1-t]
                    const int start = len - 1 - i - 31;
                    uint64_t rw = start >= 0 ? read_window(rd, start, 32) : (read_window(rd, 0, 32) << (uint32_t)(-start * 2));
                    d = rw ^ group_reverse(tw);                   // read[len-1-i-t] and text[p-1-t] both at group 31-t
                    d = (d | (d >> 1)) & 0x5555555555555555ull;
                    matched = d ? __clzll((long long)d) >> 1 : 32;
                }
                int lim = m; if ((uint64_t)lim > p) lim = (int)p;
                const bool failed = matched < lim || lim < m;     // a mismatch, or the text start reached, inside this read
                if (matched > lim) matched = lim;
                p -= matched; seed_len += matched; i += matched;
                nOcc += 2u * (uint32_t)matched; nText += matched;
                if (failed) { nOcc += 2; ++nText; emit = true; resolved = true; }
                else if (i >= len) { emit = true; finishing = true; resolved = true; }
            }
        }
        if (haveNext) {
            if (nextl <= nextr) {
                if (seed_len >= P.seedMinLength && nextr - nextl < r - l) { last_r = r; last_l = l; last_seed_len = seed_len; }
                l = nextl; r = nextr; ++seed_len; ++i;
                if (l == r) {                                     // a single suffix: look its text position up, then compare with the text
                    ++nSaIn;
                    if (saDense || (l & saMask) == 0) { p = mp_sa_sample(ix, l); state = ST_TEXT; }
                    else { p = l; skipped = 0; state = ST_SA; }
                } else state = ST_STEP;
            } else emit = true;
        }
        if (emit) {
            // CHECK_AND_ADD_RANGE (DV-DPfunctions.cpp:2197-2219); x as at DV-DPfunctions.cpp:2252-2262, 2362-2372
            int x = strand ? (finishing ? len : i) - seed_len : (finishing ? 0 : len - i);
            int diff = 0;
            if (seed_len >= P.seedMinLength) {
                if (seed_len >= P.reseedLen && last_r - last_l + 1 <= (uint64_t)P.seedSAsizeThreshold &&
                    ((uint64_t)(seed_len - last_seed_len) <= (uint64_t)P.reseedAbsDiff ||
                     seed_len * P.reseedRLTratio < (double)last_seed_len)) {
                    diff = seed_len - last_seed_len;
                    l = last_l; r = last_r; seed_len = last_seed_len;
                    resolved = false;
                }
                uint64_t d = resolved ? 0 : r - l; if (d > (uint64_t)P.seedSAsizeThreshold) d = P.seedSAsizeThreshold;
                uint32_t cnt = (uint32_t)d + 1;
                // seed slot and hit range: the lanes of the warp that emit in this trip share one pair of atomics
                uint32_t slot, hb;
                {
                    cg::coalesced_group grp = cg::coalesced_threads();
                    const uint32_t before = cg::exclusive_scan(grp, cnt), total = cg::reduce(grp, cnt, cg::plus<uint32_t>());
                    uint32_t s0 = 0, h0 = 0;
                    if (grp.thread_rank() == 0) {
                        s0 = (uint32_t)atomicAdd(&counters[0], (unsigned long long)grp.size());
                        h0 = (uint32_t)atomicAdd(&counters[1], (unsigned long long)total);
                    }
                    slot = grp.shfl(s0, 0) + grp.thread_rank();
                    hb = grp.shfl(h0, 0) + before;
                }
                atomicAdd(&hitsPerRead[read], cnt);
                if (slot < capSeeds) {
                    MpSeed sd; sd.sa_l = resolved ? p : l; sd.strandIdx = read * 2 + strand; sd.hitBase = hb;
                    sd.query_offset = (uint16_t)(x & 0x3ff); sd.seed_len = (uint16_t)(seed_len & 0xfff);
                    sd.sa_diff = (uint16_t)d; sd.pad = resolved ? 1 : 0;
                    seeds[slot] = sd;
                }
                for (uint32_t k = 0; k < cnt; ++k) if (hb + k < capStubs) stubs[hb + k] = slot;
            }
            if (finishing) state = ST_DONE;
            else {
                i -= diff;
                i -= min(seed_len, P.seedMinLength);
                ++i;
                l = 0; r = n; seed_len = 0; last_l = 0; last_r = n; last_seed_len = 0;
                state = ST_SCAN;
            }
        }
    }
    // per-warp reduction of the work counters
    unsigned long long wOcc = nOcc, wLkt = nLkt, wSa = nSaIn, wLf = nLfIn, wProbe = nProbe, wText = nText;
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        wOcc += __shfl_xor_sync(0xffffffffu, wOcc, d); wLkt += __shfl_xor_sync(0xffffffffu, wLkt, d);
        wSa += __shfl_xor_sync(0xffffffffu, wSa, d); wLf += __shfl_xor_sync(0xffffffffu, wLf, d);
        wProbe += __shfl_xor_sync(0xffffffffu, wProbe, d); wText += __shfl_xor_sync(0xffffffffu, wText, d);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&counters[2], wOcc); atomicAdd(&counters[4], wLkt); atomicAdd(&counters[7], wSa); atomicAdd(&counters[8], wLf);
        atomicAdd(&counters[9], wProbe); atomicAdd(&counters[10], wText);
    }
}

// ------------------------------------------------------------------------------------
// SA hits -> SeedAlign records (DV-DPfunctions.cpp:2477-2499)
// ------------------------------------------------------------------------------------
__global__ void k_expand(MpIndexView ix, const MpSeed *__restrict__ seeds, const uint32_t *__restrict__ stubs, uint64_t nStubs,
                         const uint32_t *__restrict__ lens, MmpDev P, const uint32_t *__restrict__ hitStart,
                         uint32_t *__restrict__ cursor, MpHit *__restrict__ hits, unsigned long long *__restrict__ counters)
{
    uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t steps = 0, done = 0;
    if (h < nStubs) {
        MpSeed sd = seeds[stubs[h]];
        uint32_t k = (uint32_t)h - sd.hitBase;
        uint64_t sa = sd.pad ? sd.sa_l : mp_sa(ix, sd.sa_l + k, &steps);     // pad = 1: text position already known (phase B of k_mmp)
        uint32_t read = sd.strandIdx >> 1, strand = sd.strandIdx & 1;
        uint32_t readLen = lens[read], off = sd.query_offset, seedlen = sd.seed_len;
        uint64_t t = strand == 0 ? sa - off : sa - (uint64_t)(uint32_t)(readLen - seedlen - off);
        MpHit hit;
        hit.offset = t;
        hit.multiplicity = ((int)seedlen >= P.goodSeedLen || seedlen >= readLen / 2) ? 1 : (uint16_t)(sd.sa_diff + 1);
        hit.length = (uint16_t)seedlen; hit.query_offset = (uint16_t)off; hit.strand = (uint16_t)strand;
        uint32_t slot = hitStart[read] + atomicAdd(&cursor[read], 1u);
        hits[slot] = hit;
        done = 1;
    }
    // work counters: one atomic per warp, not two per hit on the same two addresses
    done = __reduce_add_sync(0xffffffffu, done); steps = __reduce_add_sync(0xffffffffu, steps);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&counters[3], (unsigned long long)done);
        if (steps) atomicAdd(&counters[5], (unsigned long long)steps);
    }
}

// ------------------------------------------------------------------------------------
// per-read merge + filter (DV-DPfunctions.cpp:2501-2553).  Output SeedPos entries are
// written over the read's own hit segment: '+' entries first, then '-'.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ bool hit_less(const MpHit &a, const MpHit &b)
{
    return a.strand != b.strand ? a.strand < b.strand : a.offset < b.offset;
}
// Orders the hits of every read by (strand, offset): one warp per read, rank sort.  Lane j counts how many of the read's hits come
// before hit j (every lane reads the same record at a time: one broadcast load per comparison step) and writes hit j to that
// position of the second buffer.  NT-like indexes give dozens of hits per read (17-mers repeat by chance in 8 Gbp), where a
// per-thread insertion sort in global memory was the most expensive part of the seeding post-processing.  Hits with the same strand
// and offset are told apart by their list position; the merge below does not depend on their order.
// G = lanes per read: 32 where reads have dozens of hits, 4 where they have a handful (human-sized texts, seedMinLength 22).
template <int G>
__global__ void __launch_bounds__(128)
k_hit_sort(const uint32_t *__restrict__ hitStart, const MpHit *__restrict__ hits, uint32_t nReads, MpHit *__restrict__ sorted)
{
    const uint32_t sub = threadIdx.x % G, groupsPerGrid = gridDim.x * (blockDim.x / G);
    for (uint32_t rdx = blockIdx.x * (blockDim.x / G) + threadIdx.x / G; rdx < nReads; rdx += groupsPerGrid) {
        const uint32_t s0 = hitStart[rdx], cnt = hitStart[rdx + 1] - s0;
        const MpHit *h = hits + s0;
        for (uint32_t j = sub; j < cnt; j += G) {
            const MpHit mine = h[j];
            uint32_t rank = 0;
            for (uint32_t k = 0; k < cnt; ++k) {
                const MpHit o = h[k];
                rank += hit_less(o, mine) || (!hit_less(mine, o) && k < j);
            }
            sorted[s0 + rank] = mine;
        }
    }
}
__global__ void k_merge(const uint32_t *__restrict__ hitStart, MpHit *__restrict__ hits, uint32_t nReads, MmpDev P,
                        mp_seed_pos *__restrict__ outSeeds, uint32_t *__restrict__ nPos, uint32_t *__restrict__ nNeg)
{
    uint32_t rdx = blockIdx.x * blockDim.x + threadIdx.x;
    if (rdx >= nReads) return;
    uint32_t s0 = hitStart[rdx], s1 = hitStart[rdx + 1];
    MpHit *h = hits + s0;                           // ordered by (strand, offset) (k_hit_sort)
    int cnt = (int)(s1 - s0);
    // pass 1: chains -> (pos, total_len, keep) written to a compact list in place
    uint32_t maxLen = 0; int nOut = 0, m = 0;
    mp_seed_pos *out = outSeeds + s0;
    const uint32_t evenID = rdx & ~1u;
    while (m < cnt) {
        uint32_t strand = h[m].strand;
        uint64_t pos = h[m].offset;
        int e = m + 1;
        while (e < cnt && h[e].strand == strand && h[e].offset <= pos + (uint64_t)P.indelFuzz) ++e;
        bool uniq = false;
        for (int a = m; a < e; ++a) uniq |= (int)h[a].multiplicity <= P.uniqThreshold && (int)h[a].length >= P.seedMinLength;
        // sort the chain's read intervals by (start, end)
        for (int a = m + 1; a < e; ++a) {
            MpHit key = h[a]; int b = a - 1;
            uint32_t ks = key.query_offset, ke = key.query_offset + key.length;
            while (b >= m && (h[b].query_offset > ks || (h[b].query_offset == ks && (uint32_t)h[b].query_offset + h[b].length > ke))) { h[b + 1] = h[b]; --b; }
            h[b + 1] = key;
        }
        uint32_t total = 0, cs = 0, ce = 0;
        for (int a = m; a < e; ++a) {
            uint32_t f = h[a].query_offset, g = (uint32_t)h[a].query_offset + h[a].length;
            if (f >= ce) { total += ce - cs; cs = f; }
            ce = max(ce, g);
        }
        total += ce - cs;
        maxLen = max(maxLen, total);
        if (uniq || (int)total >= P.goodSeedLen) {
            mp_seed_pos sp; sp.pos = pos; sp.paired_seedLength = total; sp.strand_readID = evenID | (strand << 31);
            out[nOut++] = sp;      // nOut <= m < e: never overtakes unread hits (16-byte records over 16-byte records)
        }
        m = e;
    }
    // pass 2: shortSeedRatio filter, compact
    int w = 0, np = 0;
    for (int a = 0; a < nOut; ++a) {
        mp_seed_pos sp = out[a];
        if ((double)sp.paired_seedLength >= P.shortSeedRatio * (double)maxLen) {
            out[w++] = sp; np += !(sp.strand_readID >> 31);
        }
    }
    nPos[rdx] = np; nNeg[rdx] = w - np;
}

// ------------------------------------------------------------------------------------
// pairing (DV-DPfunctions.cpp:1968-2070).  write == nullptr: count only.
// ------------------------------------------------------------------------------------
#define MP_MARGIN(l) (((l) > 100) ? 30 : 25)       // DP2_MARGIN, DV-DPfunctions.cpp:1760
__device__ uint32_t pair_one(const mp_seed_pos *left, int nLeft, const mp_seed_pos *right, int nRight,
                             int negLen, int insert_low, int insert_high, uint32_t readIDLeft, mp_candidate *write)
{
    if (nLeft == 0 || nRight == 0) return 0;
    int margin = MP_MARGIN(negLen);
    int length_low = insert_low - negLen - margin; if (length_low < 0) length_low = 0;
    int length_high = insert_high - negLen + margin;
    uint32_t nc = 0;
    int preStart = 0;
    uint64_t prevLoc = 0;
    for (int a = 0; a < nLeft; ++a) {
        uint64_t readLoc = left[a].pos;
        if (a > 0 && !(prevLoc + 5 < readLoc)) continue;     // MC_Compress :2015-2026
        prevLoc = readLoc;
        for (int b = preStart; b < nRight; ++b) {
            uint64_t mateLoc = right[b].pos;
            if (readLoc + (uint64_t)(int64_t)length_high < mateLoc) break;
            else if (readLoc + (uint64_t)(int64_t)length_low <= mateLoc) {
                if (write) { mp_candidate ci; ci.readIDLeft = readIDLeft; ci.pad = 0; ci.pos[0] = readLoc; ci.pos[1] = mateLoc; write[nc] = ci; }
                ++nc; preStart = b;
            }
        }
    }
    return nc;
}
__global__ void k_pair(const uint32_t *__restrict__ hitStart, const mp_seed_pos *__restrict__ sp, const uint32_t *__restrict__ nPos,
                       const uint32_t *__restrict__ nNeg, const uint32_t *__restrict__ lens, uint32_t nPairs, int insert_low, int insert_high,
                       uint32_t *__restrict__ candCount, const uint32_t *__restrict__ candStart, mp_candidate *__restrict__ cands)
{
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nPairs) return;
    uint32_t r1 = 2 * p, r2 = 2 * p + 1;
    const mp_seed_pos *pos1 = sp + hitStart[r1], *neg1 = pos1 + nPos[r1];
    const mp_seed_pos *pos2 = sp + hitStart[r2], *neg2 = pos2 + nPos[r2];
    mp_candidate *w = cands ? cands + candStart[p] : nullptr;
    // read '+' with mate '-' (readIDLeft even), then mate '+' with read '-' (odd)
    uint32_t c0 = pair_one(pos1, nPos[r1], neg2, nNeg[r2], (int)lens[r2], insert_low, insert_high, r1, w);
    uint32_t c1 = pair_one(pos2, nPos[r2], neg1, nNeg[r1], (int)lens[r1], insert_low, insert_high, r2, w ? w + c0 : nullptr);
    if (!cands) candCount[p] = c0 + c1;
}

// ------------------------------------------------------------------------------------
static int exclusive_scan_u32(mp_context *ctx, const uint32_t *in, uint32_t *out, uint64_t n)
{
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, (int64_t)n, ctx->stream);
    if (ctx->dScanTmp.reserve(tb)) return MP_ERR_CUDA;
    cub::DeviceScan::ExclusiveSum(ctx->dScanTmp.p, tb, in, out, (int64_t)n, ctx->stream);
    return 0;
}

int mps_upload(mp_context *ctx, const uint32_t *queries, const uint32_t *readLengths, uint32_t nReads, uint32_t wpq)
{
    // a read longer than its 2-bit row would make every consumer (seeding, task extraction, the DP kernels' shared-memory rows) run
    // past its buffers: refuse the batch here, where the lengths are still on the host
    uint32_t maxLen = 0;
    for (uint32_t r = 0; r < nReads; ++r) maxLen = readLengths[r] > maxLen ? readLengths[r] : maxLen;
    if (maxLen > 16u * wpq) { mp_set_error("mp_batch_upload: a read of %u bases does not fit %u words per query", maxLen, wpq); return MP_ERR_ARG; }
    ctx->maxLenBatch = maxLen;
    uint64_t nPad = ((uint64_t)nReads + 31) / 32 * 32;
    size_t bytes = nPad * wpq * 4;
    if (ctx->dReadsIl.reserve(bytes) || ctx->dReads.reserve(bytes + 64) || ctx->dLens.reserve((size_t)nReads * 4)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpyAsync(ctx->dReadsIl.p, queries, bytes, cudaMemcpyHostToDevice, ctx->stream));
    MP_CUDA(cudaMemcpyAsync(ctx->dLens.p, readLengths, (size_t)nReads * 4, cudaMemcpyHostToDevice, ctx->stream));
    MP_CUDA(cudaMemsetAsync(ctx->dReads.p, 0, bytes + 64, ctx->stream));
    uint64_t total = nPad * wpq;
    (++g_mp_launches), k_deinterleave<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(ctx->dReadsIl.as<uint32_t>(), ctx->dReads.as<uint32_t>(), nReads, wpq);
    MP_CUDA(cudaGetLastError());
    ctx->hLens.assign(readLengths, readLengths + nReads);
    ctx->nReads = nReads; ctx->wpq = wpq; ctx->hasBatch = true; ctx->seeded = false;
    ctx->fqBatch = false; ctx->resValid = false; ctx->fmtReady = false;
    return 0;
}

// builds (once per index and K) the K-mer presence filter; MP_BLOOM=0 disables it
static int ensure_bloom(mp_context *ctx, int seedMinLength)
{
    const char *e = getenv("MP_BLOOM");
    if (e && e[0] == '0') { ctx->bloomK = 0; return 0; }
    const uint64_t n = ctx->ix.n;
    // Probe stride s: K = seedMinLength - (s - 1) must stay long enough that a random K-mer is rarely in the text
    // (4^K >= 256 n), else too many starts survive the filter and are walked.  3.1 Gbp, seedMinLength 22 -> s = 3, K = 20
    // (measured k_mmp time per 1 Mi pairs: s=1 16.3 ms, s=2 13.8, s=3 13.7, s=4 14.7, s=5 19.5).
    int kMin = 4; for (uint64_t v = 1; v < n && kMin < 40; v <<= 2) ++kMin;
    int stride = seedMinLength - kMin + 1;
    if (const char *es = getenv("MP_BLOOM_STRIDE")) stride = atoi(es);
    if (stride > 8) stride = 8;
    if (stride < 1) stride = 1;
    if (stride > seedMinLength - 12) stride = seedMinLength - 12 > 1 ? seedMinLength - 12 : 1;
    int K = seedMinLength - (stride - 1); if (K > 32) K = 32;
    if (ctx->bloomK == K && ctx->bloomStride == stride && ctx->bloomSeedMin == seedMinLength && ctx->bloomFor == (const void *)ctx->ix.blocks) return 0;
    if (n < (uint64_t)K) { ctx->bloomK = 0; return 0; }
    // a K-mer that occurs in the text more than once on average cannot be ruled out by a presence filter (60 Gbp NT with
    // seedMinLength 17: 4^17 < n): no filter then, its probes would only add gathers (and tens of GB of HBM)
    if (K < 32 && (double)n > (double)(1ull << (2 * K))) { ctx->bloomK = 0; return 0; }
    uint64_t nWords = n / 4 + 1024;                      // 16 bits per text position ...
    {                                                    // ... unless that would take more than a third of what is free (60 Gbp texts)
        size_t freeB = 0, totalB = 0; cudaMemGetInfo(&freeB, &totalB);
        const uint64_t room = (uint64_t)(freeB / 3) / 8;
        if (nWords > room) nWords = room;
        if (ctx->hbmBudget) {                            // mp_index_load_budget: what the index left of its budget, or no filter
            const uint64_t idx = mpi_index_bytes(ctx), left = ctx->hbmBudget > idx ? devbuf_fit(ctx->hbmBudget - idx) / 8 : 0;
            if (nWords > left) nWords = left;
        }
        if (nWords < 1024) { ctx->bloomK = 0; return 0; }
    }
    if (ctx->sharedIndex && ctx->dBloom.cap == 0) ctx->dBloom.p = nullptr;      // a borrowed filter with another K: build our own
    if (ctx->dBloom.reserve(nWords * 8)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemsetAsync(ctx->dBloom.p, 0, nWords * 8, ctx->stream));
    uint64_t threads = (n + 63) / 64;
    (++g_mp_launches), k_bloom_build<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(ctx->ix.pac, n, K, ctx->dBloom.as<unsigned long long>(), nWords);
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->bloomK = K; ctx->bloomStride = stride; ctx->bloomSeedMin = seedMinLength; ctx->bloomWords = nWords; ctx->bloomFor = (const void *)ctx->ix.blocks;
    ctx->hbmBytes += ctx->dBloom.cap;
    return 0;
}

extern "C" int mp_index_prepare(mp_context *ctx, const mp_align_params *params)
{
    if (!ctx || !params) { mp_set_error("mp_index_prepare: null argument"); return MP_ERR_ARG; }
    if (!ctx->hasIndex) { mp_set_error("mp_index_prepare: no index resident"); return MP_ERR_STATE; }
    MP_CUDA(cudaSetDevice(ctx->device));
    return ensure_bloom(ctx, params->mmp.seedMinLength);
}

int mps_seed_pairs(mp_context *ctx, const mp_align_params *AP)
{
    const mp_mmp_params &mp = AP->mmp;
    MmpDev P;
    P.seedSAsizeThreshold = mp.seedSAsizeThreshold; P.seedMinLength = mp.seedMinLength; P.uniqThreshold = mp.uniqThreshold;
    P.indelFuzz = mp.indelFuzz; P.goodSeedLen = mp.goodSeedLen; P.reseedLen = mp.reseedLen; P.reseedAbsDiff = mp.reseedAbsDiff;
    P.reseedRLTratio = mp.reseedRLTratio; P.shortSeedRatio = mp.shortSeedRatio;
    if (P.seedMinLength < 13 || P.seedSAsizeThreshold > 1000) { mp_set_error("mmp parameters out of range"); return MP_ERR_ARG; }
    const uint32_t nReads = ctx->nReads, nStrands = nReads * 2, nPairs = nReads / 2;
    cudaStream_t st = ctx->stream;
    if (ctx->dCounters.reserve(16 * 8) || ctx->dHitsPerRead.reserve(((size_t)nReads + 1) * 4) ||
        ctx->dHitStart.reserve(((size_t)nReads + 1) * 4) || ctx->dCursor.reserve(((size_t)nReads + 1) * 4) ||
        ctx->dNPos.reserve((size_t)nReads * 4) || ctx->dNNeg.reserve((size_t)nReads * 4)) return MP_ERR_CUDA;
    if (ctx->capSeeds < (uint64_t)nStrands * 4) ctx->capSeeds = (uint64_t)nStrands * 4;
    if (ctx->capStubs < (uint64_t)nStrands * 8) ctx->capStubs = (uint64_t)nStrands * 8;
    if (int rc = ensure_bloom(ctx, P.seedMinLength)) return rc;
    unsigned long long hc[16];
    int dev = 0, nSM = 148, mmpBlocks = 8; cudaGetDevice(&dev); cudaDeviceGetAttribute(&nSM, cudaDevAttrMultiProcessorCount, dev);
    const size_t mmpSmem = ((size_t)ctx->wpq + 2) * MMP_RS * 4;      // the reads the block's lanes are working on
    if (mmpSmem > 48 * 1024) MP_CUDA(cudaFuncSetAttribute(k_mmp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mmpSmem));
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&mmpBlocks, k_mmp, 128, mmpSmem) != cudaSuccess || mmpBlocks < 1) mmpBlocks = 8;
    MP_CUDA(cudaEventRecord(ctx->ev[0], st));
    for (int attempt = 0; attempt < 4; ++attempt) {
        if (ctx->capSeeds > 0xFFFFFFF0ull || ctx->capStubs > 0xFFFFFFF0ull) { mp_set_error("seed buffers exceed 32-bit indexing; use smaller batches"); return MP_ERR_CAPACITY; }
        if (ctx->dSeeds.reserve(ctx->capSeeds * sizeof(MpSeed)) || ctx->dStubs.reserve(ctx->capStubs * 4)) return MP_ERR_CUDA;
        MP_CUDA(cudaMemsetAsync(ctx->dCounters.p, 0, 16 * 8, st));
        MP_CUDA(cudaMemsetAsync(ctx->dHitsPerRead.p, 0, ((size_t)nReads + 1) * 4, st));
        // persistent warps: as many blocks as the device holds at once, every warp pulls chunks of read-strands from counters[6]
        (++g_mp_launches), k_mmp<<<nSM * mmpBlocks, 128, mmpSmem, st>>>(ctx->ix, ctx->dReads.as<uint32_t>(), ctx->dLens.as<uint32_t>(), ctx->wpq, nStrands, P,
                                      ctx->dSeeds.as<MpSeed>(), ctx->dStubs.as<uint32_t>(), ctx->dCounters.as<unsigned long long>(),
                                      ctx->dHitsPerRead.as<uint32_t>(), (uint32_t)ctx->capSeeds, (uint32_t)ctx->capStubs,
                                      ctx->bloomK ? ctx->dBloom.as<unsigned long long>() : nullptr, ctx->bloomWords, ctx->bloomK, ctx->bloomStride);
        MP_CUDA(cudaGetLastError());
        MP_CUDA(cudaMemcpyAsync(hc, ctx->dCounters.p, 16 * 8, cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaStreamSynchronize(st));
        if (hc[0] <= ctx->capSeeds && hc[1] <= ctx->capStubs) break;
        ctx->capSeeds = hc[0] + hc[0] / 8 + 1024; ctx->capStubs = hc[1] + hc[1] / 8 + 1024;   // rerun with exact room
        if (attempt == 3) { mp_set_error("seed buffers overflowed repeatedly"); return MP_ERR_CAPACITY; }
    }
    MP_CUDA(cudaEventRecord(ctx->ev[1], st));
    ctx->nSeeds = hc[0]; ctx->nHits = hc[1];
    if (ctx->nHits > 0xFFFFFFF0ull) { mp_set_error("too many seed hits in one batch"); return MP_ERR_CAPACITY; }
    if (exclusive_scan_u32(ctx, ctx->dHitsPerRead.as<uint32_t>(), ctx->dHitStart.as<uint32_t>(), (uint64_t)nReads + 1)) return MP_ERR_CUDA;
    // sized with a floor per read so that batch-to-batch variation does not trigger re-allocation (a cudaFree synchronises the device)
    const size_t hitSlots = std::max<size_t>(ctx->nHits + 1, (size_t)nReads * 3);
    if (ctx->dHits.reserve(hitSlots * sizeof(MpHit)) || ctx->dSeedPos.reserve(hitSlots * sizeof(mp_seed_pos))) return MP_ERR_CUDA;
    MP_CUDA(cudaMemsetAsync(ctx->dCursor.p, 0, ((size_t)nReads + 1) * 4, st));
    if (ctx->nHits)
        (++g_mp_launches), k_expand<<<(unsigned)((ctx->nHits + 127) / 128), 128, 0, st>>>(ctx->ix, ctx->dSeeds.as<MpSeed>(), ctx->dStubs.as<uint32_t>(), ctx->nHits,
            ctx->dLens.as<uint32_t>(), P, ctx->dHitStart.as<uint32_t>(), ctx->dCursor.as<uint32_t>(), ctx->dHits.as<MpHit>(),
            ctx->dCounters.as<unsigned long long>());
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaEventRecord(ctx->ev[2], st));
    if (ctx->dHits2.reserve(hitSlots * sizeof(MpHit))) return MP_ERR_CUDA;
    const char *eG = getenv("MP_HIT_SORT_G");                          // tests: 4 or 32 lanes per read whatever the hit density
    const int forceG = eG ? atoi(eG) : 0;
    if (forceG ? forceG == 32 : ctx->nHits > (uint64_t)nReads * 8)
        (++g_mp_launches), k_hit_sort<32><<<nSM * 16, 128, 0, st>>>(ctx->dHitStart.as<uint32_t>(), ctx->dHits.as<MpHit>(), nReads, ctx->dHits2.as<MpHit>());
    else
        (++g_mp_launches), k_hit_sort<4><<<nSM * 16, 128, 0, st>>>(ctx->dHitStart.as<uint32_t>(), ctx->dHits.as<MpHit>(), nReads, ctx->dHits2.as<MpHit>());
    (++g_mp_launches), k_merge<<<(nReads + 127) / 128, 128, 0, st>>>(ctx->dHitStart.as<uint32_t>(), ctx->dHits2.as<MpHit>(), nReads, P,
                                                 ctx->dSeedPos.as<mp_seed_pos>(), ctx->dNPos.as<uint32_t>(), ctx->dNNeg.as<uint32_t>());
    MP_CUDA(cudaGetLastError());
    // pairing: count, scan, write
    if (ctx->dCandCount.reserve(((size_t)nPairs + 1) * 4) || ctx->dCandStart.reserve(((size_t)nPairs + 1) * 4)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemsetAsync(ctx->dCandCount.p, 0, ((size_t)nPairs + 1) * 4, st));
    (++g_mp_launches), k_pair<<<(nPairs + 127) / 128, 128, 0, st>>>(ctx->dHitStart.as<uint32_t>(), ctx->dSeedPos.as<mp_seed_pos>(), ctx->dNPos.as<uint32_t>(),
        ctx->dNNeg.as<uint32_t>(), ctx->dLens.as<uint32_t>(), nPairs, AP->insert_low, AP->insert_high,
        ctx->dCandCount.as<uint32_t>(), nullptr, nullptr);
    if (exclusive_scan_u32(ctx, ctx->dCandCount.as<uint32_t>(), ctx->dCandStart.as<uint32_t>(), (uint64_t)nPairs + 1)) return MP_ERR_CUDA;
    uint32_t total = 0;
    MP_CUDA(cudaMemcpyAsync(&total, ctx->dCandStart.as<uint32_t>() + nPairs, 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    ctx->nCands = total;
    if (ctx->dCands.reserve(std::max<size_t>((size_t)total + 1, (size_t)nPairs * 2) * sizeof(mp_candidate))) return MP_ERR_CUDA;
    if (total)
        (++g_mp_launches), k_pair<<<(nPairs + 127) / 128, 128, 0, st>>>(ctx->dHitStart.as<uint32_t>(), ctx->dSeedPos.as<mp_seed_pos>(), ctx->dNPos.as<uint32_t>(),
            ctx->dNNeg.as<uint32_t>(), ctx->dLens.as<uint32_t>(), nPairs, AP->insert_low, AP->insert_high,
            ctx->dCandCount.as<uint32_t>(), ctx->dCandStart.as<uint32_t>(), ctx->dCands.as<mp_candidate>());
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaEventRecord(ctx->ev[3], st));
    MP_CUDA(cudaStreamSynchronize(st));
    ctx->seedParams = *AP;
    ctx->seeded = true;
    return 0;
}

// ---- downloads in the reference's array layout (DV-DPfunctions.cpp:2555-2594) ----
int mps_download_seedpos(mp_context *ctx, mp_seed_pos **readPos, uint64_t *nReadPos, mp_seed_pos **matePos, uint64_t *nMatePos)
{
    const uint32_t nReads = ctx->nReads;
    std::vector<uint32_t> hs(nReads + 1), np(nReads), nn(nReads);
    std::vector<mp_seed_pos> sp(ctx->nHits + 1);
    MP_CUDA(cudaMemcpy(hs.data(), ctx->dHitStart.p, ((size_t)nReads + 1) * 4, cudaMemcpyDeviceToHost));
    MP_CUDA(cudaMemcpy(np.data(), ctx->dNPos.p, (size_t)nReads * 4, cudaMemcpyDeviceToHost));
    MP_CUDA(cudaMemcpy(nn.data(), ctx->dNNeg.p, (size_t)nReads * 4, cudaMemcpyDeviceToHost));
    if (ctx->nHits) MP_CUDA(cudaMemcpy(sp.data(), ctx->dSeedPos.p, ctx->nHits * sizeof(mp_seed_pos), cudaMemcpyDeviceToHost));
    for (int mate = 0; mate < 2; ++mate) {
        uint64_t tot = 2;
        for (uint32_t r = mate; r < nReads; r += 2) tot += np[r] + nn[r];
        mp_seed_pos *o = (mp_seed_pos *)malloc(tot * sizeof(mp_seed_pos));
        uint64_t k = 0;
        for (uint32_t r = mate; r < nReads; r += 2) for (uint32_t a = 0; a < np[r]; ++a) o[k++] = sp[hs[r] + a];
        mp_seed_pos t; t.pos = ~0ull; t.paired_seedLength = 0xffffffffu; t.strand_readID = 0x7fffffffu; o[k++] = t;
        for (uint32_t r = mate; r < nReads; r += 2) for (uint32_t a = 0; a < nn[r]; ++a) o[k++] = sp[hs[r] + np[r] + a];
        t.strand_readID = 0xffffffffu; o[k++] = t;
        if (mate == 0) { *readPos = o; *nReadPos = tot; } else { *matePos = o; *nMatePos = tot; }
    }
    return 0;
}
