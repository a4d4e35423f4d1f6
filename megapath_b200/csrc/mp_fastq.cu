// mp_fastq.cu -- the two host loops either side of the hot path, on the device (SURVEY.md section 8 row f2):
//
//   ingest   plain four-line FASTQ text -> record index, clamped lengths, 2-bit rows (what loadPairReadsKseq + appendToQueryArrays
//            build, QueryParser.cpp:160-260 with kseq.h's name / comment split) -- mp_fastq_upload
//   egress   the annotated FASTQ soap4 -F / -P prints for a batch (pairDeepDPOutputFastqAPI, unproperlypairDPOutputFastqAPI,
//            getMappingFromHeader, decideTargetChr: BGS-IO.cpp:163-190, 1312-1446, 1966-2091; stage order of alignment.cpp:299-351)
//            -- mp_format_fastq / mp_format_fetch
//
// Both are byte work bound by HBM streaming: the text of a batch (about 700 MB for 1 Mi pairs of 150 bases) is read once by the
// newline index, once by the packer and once by the writer; the output is written once.  What the host keeps is the file read into
// page-locked memory and the write of the finished text.
//
// Layout.  The two mates' texts lie in one device buffer (mate 2 at a 16-byte aligned offset).  k_fq_count counts newlines per
// 64-byte piece, an exclusive scan turns the counts into line numbers, k_fq_lines scatters the newline offsets: line j of a mate ends
// at lineEnd[j], so record r is lines 4r .. 4r+3.  k_fq_records checks every record against the strict four-line form and stores a
// 20-byte record view; anything else makes the whole call return MP_ERR_FORMAT and the caller parses that batch itself.
// Output: one key (sequence id, score) per result and read end (k_fmt_pair_keys / k_fmt_single_keys), group bounds per pair / read,
// k_fmt_measure sizes every record, a scan over (stage, pair) gives the offsets in the reference's stage order, k_fmt_write -- one
// warp per read -- writes the records.
#include "mp_context.h"
#include <cub/cub.cuh>
#include <limits.h>

namespace {

struct FqRec {                 // one FASTQ record of a mate's text (offsets within that text)
    uint32_t hdr;              // the '@'
    uint32_t seq, qual;        // first base / first quality
    uint16_t nameLen;          // after the "/<digit>" trim
    uint16_t commentOff;       // from hdr; 0 = no comment
    uint16_t commentLen;
    uint16_t len;              // bases kept: min(length, maxReadLength - 1)
};

__device__ __forceinline__ bool fq_isspace(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13); }
__device__ __forceinline__ uint32_t fq_code(unsigned char c)          // INDEXFillCharMap (IndexHandler.cpp:26-45)
{
    switch (c) {
    case 'C': case 'c': return 1;
    case 'G': case 'g': case 'N': case 'n': return 2;
    case 'T': case 't': case 'U': case 'u': return 3;
    default: return 0;
    }
}

constexpr int FQ_PIECE = 64;
// newlines (and bytes that rule the fast path out: '\r', NUL) of a 64-byte piece
__device__ __forceinline__ uint32_t fq_piece_count(const char *text, uint64_t bytes, uint64_t t, uint32_t *bad)
{
    const uint64_t b0 = t * FQ_PIECE;
    uint32_t n = 0, odd = 0;
    if (b0 + FQ_PIECE <= bytes) {
        const uint4 *p = (const uint4 *)(text + b0);
#pragma unroll
        for (int k = 0; k < FQ_PIECE / 16; ++k) {
            const uint4 v = p[k];
            const uint32_t w[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                n += __popc(__vcmpeq4(w[j], 0x0a0a0a0au)) >> 3;
                odd |= __vcmpeq4(w[j], 0x0d0d0d0du) | __vcmpeq4(w[j], 0u);
            }
        }
    } else {
        for (uint64_t i = b0; i < bytes; ++i) { const char c = text[i]; n += c == '\n'; odd |= (c == '\r' || c == 0); }
    }
    if (odd) *bad = 1;
    return n;
}
__global__ void k_fq_count(const char *__restrict__ text, uint64_t bytes, uint32_t *__restrict__ cnt, uint32_t *__restrict__ flags)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nT = (bytes + FQ_PIECE - 1) / FQ_PIECE;
    if (t > nT) return;
    if (t == nT) { cnt[t] = 0; return; }
    uint32_t bad = 0;
    cnt[t] = fq_piece_count(text, bytes, t, &bad);
    if (bad) atomicOr(flags, 1u);
}
__global__ void k_fq_lines(const char *__restrict__ text, uint64_t bytes, const uint32_t *__restrict__ pos, uint32_t maxLines, uint32_t *__restrict__ lineEnd)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nT = (bytes + FQ_PIECE - 1) / FQ_PIECE;
    if (t >= nT) return;
    uint32_t at = pos[t];
    if (at == pos[t + 1]) return;
    const uint64_t b0 = t * FQ_PIECE, b1 = b0 + FQ_PIECE < bytes ? b0 + FQ_PIECE : bytes;
    for (uint64_t i = b0; i < b1; ++i)
        if (text[i] == '\n') { if (at < maxLines) lineEnd[at] = (uint32_t)i; ++at; }
}

// one thread per read id (mate = id & 1): the strict four-line record view (the driver's view_record), lengths, flags
__global__ void k_fq_records(const char *__restrict__ textAll, uint64_t base1, const uint32_t *__restrict__ lines0, const uint32_t *__restrict__ lines1,
                             uint32_t nReads, uint32_t maxKeep, FqRec *__restrict__ rec, uint32_t *__restrict__ lens, uint32_t *__restrict__ flags)
{
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= nReads) return;
    const uint32_t m = id & 1u, r = id >> 1;
    const char *text = textAll + (m ? base1 : 0);
    const uint32_t *L = m ? lines1 : lines0;
    const uint32_t s0 = r ? L[4 * r - 1] + 1 : 0, e0 = L[4 * r], s1 = e0 + 1, e1 = L[4 * r + 1], s2 = e1 + 1, e2 = L[4 * r + 2], s3 = e2 + 1, e3 = L[4 * r + 3];
    bool ok = text[s0] == '@' && e1 > s1 && e0 - s0 < 60000u;
    const char c0 = text[s1];
    ok = ok && c0 != '>' && c0 != '+' && c0 != '@' && text[s2] == '+' && (e3 - s3) == (e1 - s1);
    (void)e2;
    uint32_t q = s0 + 1;
    while (q < e0 && !fq_isspace((unsigned char)text[q])) ++q;
    uint32_t nameLen = q - (s0 + 1);
    FqRec R;
    R.hdr = s0; R.seq = s1; R.qual = s3;
    if (q < e0 && e0 - q - 1 > 0) { R.commentOff = (uint16_t)(q + 1 - s0); R.commentLen = (uint16_t)(e0 - q - 1); } else { R.commentOff = 0; R.commentLen = 0; }
    if (nameLen > 2 && text[s0 + 1 + nameLen - 2] == '/' && text[s0 + nameLen] >= '0' && text[s0 + nameLen] <= '9') nameLen -= 2;      // trim_readno
    R.nameLen = (uint16_t)nameLen;
    const uint32_t sl = e1 - s1, len = sl > maxKeep ? maxKeep : sl;
    R.len = (uint16_t)len;
    rec[id] = R;
    lens[id] = len;
    if (!ok) atomicOr(flags, 2u);
    atomicMax(flags + 1, len);
}

// one thread per (read, word): 16 bases LSB-first (appendToQueryArrays, QueryParser.cpp:184-203), rows as k_deinterleave leaves them
__global__ void k_fq_pack(const char *__restrict__ textAll, uint64_t base1, const FqRec *__restrict__ rec, uint32_t nReads, uint32_t wpq, uint32_t *__restrict__ out)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)nReads * wpq) return;
    const uint32_t id = (uint32_t)(t / wpq), j = (uint32_t)(t - (uint64_t)id * wpq);
    const FqRec R = rec[id];
    const char *s = textAll + ((id & 1u) ? base1 : 0) + R.seq;
    uint32_t w = 0;
    const uint32_t b0 = j * 16, b1 = b0 + 16 < R.len ? b0 + 16 : R.len;
    for (uint32_t i = b0; i < b1; ++i) w |= fq_code((unsigned char)s[i]) << ((i - b0) * 2);
    out[t] = w;
}

// ------------------------------------------------------------------------------------------------
// egress
struct AnnDev {
    const uint32_t *grid; const uint64_t *trStart; const uint32_t *trChr; const char *names; const uint64_t *nameOff;
    uint32_t gridEntries;
};
__device__ __forceinline__ int ann_chr(const AnnDev &A, uint64_t pos)          // getChrAndPos (BGS-IO.cpp:163-190)
{
    uint64_t idx = pos >> 18;
    if (idx >= A.gridEntries) idx = A.gridEntries - 1;
    uint32_t v = A.grid[idx];
    while (A.trStart[v] > pos) --v;
    return (int)A.trChr[v];
}
__device__ __forceinline__ int ann_target_chr(const AnnDev &A, uint64_t pos, uint32_t readLen)      // decideTargetChr (BGS-IO.cpp:1312-1341)
{
    const int c0 = ann_chr(A, pos), c1 = ann_chr(A, pos + readLen - 1);
    return c0 == c1 ? c0 : -1;
}
constexpr uint64_t NA = ~0ull;

// per paired result: (sequence id, score) of either end after the -F / -P rules of pairDeepDPOutputFastqAPI; group bounds per pair
__global__ void k_fmt_pair_keys(const mp_pair_result *__restrict__ res, uint32_t n, const uint32_t *__restrict__ lens, AnnDev A, int mode,
                                int2 *__restrict__ k1, int2 *__restrict__ k2, uint32_t *__restrict__ gStart, uint32_t *__restrict__ gEnd)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const mp_pair_result r = res[i];
    uint64_t a1 = r.algnmt_1, a2 = r.algnmt_2; int s1 = r.score_1, s2 = r.score_2;
    int chr1 = -1, chr2 = -1;
    if (a1 != NA) chr1 = ann_target_chr(A, a1, lens[r.readID]);
    if (a2 != NA) chr2 = ann_target_chr(A, a2, lens[r.readID + 1]);
    if (chr1 == -1) { a1 = NA; s1 = 0; }
    if (chr2 == -1) { a2 = NA; s2 = 0; }
    if (mode == 2 && (a1 == NA || a2 == NA)) { a1 = a2 = NA; s1 = s2 = 0; }
    if (chr1 == chr2 && a1 != NA && a2 != NA) { const int sum = s1 + s2; s1 = s2 = sum; }
    k1[i] = make_int2(chr1, s1); k2[i] = make_int2(chr2, s2);
    const uint32_t p = r.readID >> 1;
    if (i == 0 || res[i - 1].readID != r.readID) gStart[p] = i;
    if (i + 1 == n || res[i + 1].readID != r.readID) gEnd[p] = i + 1;
}
// per single-end result (unproperlypairDPOutputFastqAPI): group bounds per read
__global__ void k_fmt_single_keys(const mp_single_result *__restrict__ res, uint32_t n, const uint32_t *__restrict__ lens, AnnDev A,
                                  int2 *__restrict__ k, uint32_t *__restrict__ gStart, uint32_t *__restrict__ gEnd)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const mp_single_result r = res[i];
    const int chr = ann_target_chr(A, r.algnmt, lens[r.readID]);
    k[i] = make_int2(chr, chr < 0 ? 0 : r.score);
    if (i == 0 || res[i - 1].readID != r.readID) gStart[r.readID] = i;
    if (i + 1 == n || res[i + 1].readID != r.readID) gEnd[r.readID] = i + 1;
}

// atoi of a string that ends at e (glibc: (int) strtol(s, NULL, 10))
__device__ int fq_atoi(const char *s, const char *e)
{
    while (s < e && fq_isspace((unsigned char)*s)) ++s;
    bool neg = false;
    if (s < e && (*s == '-' || *s == '+')) { neg = *s == '-'; ++s; }
    unsigned long long v = 0; bool over = false;
    const unsigned long long lim = neg ? 9223372036854775808ull : 9223372036854775807ull;
    for (; s < e && *s >= '0' && *s <= '9'; ++s) {
        const unsigned d = (unsigned)(*s - '0');
        if (over || v > (lim - d) / 10) { over = true; continue; }
        v = v * 10 + d;
    }
    if (over) v = lim;
    const long long sv = neg ? (long long)(0ull - v) : (long long)v;
    return (int)sv;
}

template <bool W> struct Sink {             // counts always; stores the first `cap` bytes when W
    char *p; uint32_t n, cap;
    __device__ __forceinline__ void put(char c) { if (W && n < cap) p[n] = c; ++n; }
    __device__ void str(const char *s, uint32_t l) { if (W) for (uint32_t i = 0; i < l && n + i < cap; ++i) p[n + i] = s[i]; n += l; }
    __device__ void num(long long v) {
        char tmp[24]; int k = 0; const bool neg = v < 0; unsigned long long u = neg ? 0ull - (unsigned long long)v : (unsigned long long)v;
        do { tmp[k++] = (char)('0' + u % 10); u /= 10; } while (u);
        if (neg) put('-');
        while (k) put(tmp[--k]);
    }
};

// everything between the read name and the end of the header line (the driver's header_line: BGS-IO.cpp:1966-2091 with
// getMappingFromHeader :1348-1371).  keys: the (sequence id, score) entries of this read end; best: their maximal score (>= 0).
template <bool W> __device__ uint32_t fmt_tail(char *out, uint32_t cap, const char *comment, uint32_t commentLen, const int2 *__restrict__ keys, uint32_t G, int best,
                                               double top, const AnnDev &A)
{
    Sink<W> o = { out, 0, cap };
    if (commentLen == 6 && comment[0] == 'I' && comment[1] == 'G' && comment[2] == 'N' && comment[3] == 'O' && comment[4] == 'R' && comment[5] == 'E') {
        o.str("\tIGNORE\n", 8);
        return o.n;
    }
    const char *ce = comment + commentLen;
    int prev = 0; bool keepList = false;
    if (commentLen >= 6) {
        double scoreT = best * top;
        prev = fq_atoi(comment + 6, ce);
        if (!((double)prev < scoreT)) {
            if (scoreT < prev * top) scoreT = prev * top;
            keepList = (double)prev >= scoreT;
        }
    }
    if (prev > best) best = prev;
    const double cut = best * top;
    o.str("\tSCORE:", 7); o.num(best); o.put(';');
    if (best > 0) {
        int cur = 0;                                   // sequence ids are 1-based; -1 marks "no target sequence"
        for (;;) {
            int nxt = INT_MAX, mx = INT_MIN;
            for (uint32_t k = 0; k < G; ++k) {
                const int2 e = keys[k];
                if (e.x > cur) { if (e.x < nxt) { nxt = e.x; mx = e.y; } else if (e.x == nxt && e.y > mx) mx = e.y; }
            }
            if (nxt == INT_MAX) break;
            if (mx > 0 && (double)mx >= cut) {
                o.num(mx); o.put(',');
                const uint64_t a = A.nameOff[nxt - 1], b = A.nameOff[nxt];
                o.str(A.names + a, (uint32_t)(b - a)); o.put(';');
            }
            cur = nxt;
        }
    }
    if (commentLen >= 6 && keepList) {
        const char *p = comment + 6;
        while (p < ce && *p != ';') ++p;               // strchr(c + 6, ';')
        while (p < ce && p + 1 < ce) {
            const char *s = p + 1;
            const int ms = fq_atoi(s, ce);
            p = s; while (p < ce && *p != ';') ++p;    // strchr(p + 1, ';')
            if (p >= ce) break;
            if ((double)ms >= cut) { o.str(s, (uint32_t)(p - s)); o.put(';'); }
        }
    }
    o.put('\n');
    return o.n;
}

struct FmtView {               // everything k_fmt_measure / k_fmt_write need
    const char *text; uint64_t base1; const FqRec *rec; uint32_t nReads;
    const uint32_t *pStart, *pEnd, *rStart, *rEnd, *sStart, *sEnd;
    const int2 *kP1, *kP2, *kR1, *kR2, *kS;
    AnnDev A; double top; int mode, ignoreComments;
};
__device__ __forceinline__ int fmt_group(const FmtView &V, uint32_t id, const int2 *&keys, uint32_t &G)
{
    const uint32_t p = id >> 1, e = id & 1u;
    if (V.pEnd[p] > V.pStart[p]) { keys = (e ? V.kP2 : V.kP1) + V.pStart[p]; G = V.pEnd[p] - V.pStart[p]; return 0; }
    if (V.rEnd[p] > V.rStart[p]) { keys = (e ? V.kR2 : V.kR1) + V.rStart[p]; G = V.rEnd[p] - V.rStart[p]; return 1; }
    keys = V.kS + V.sStart[id]; G = V.mode == 2 ? 0 : V.sEnd[id] - V.sStart[id];
    return 2;
}
__device__ __forceinline__ int fmt_best(const int2 *keys, uint32_t G)
{
    int best = 0;
    for (uint32_t k = 0; k < G; ++k) { const int s = keys[k].y; if (best < s) best = s; }
    return best;
}

constexpr uint32_t FMT_SLOT = 64;          // header tails up to this size are composed once, by k_fmt_measure, and only copied by k_fmt_write
// one thread per read: size of its record (and the header tail itself when it fits its slot); the even thread of a pair stores the pair's
// size under its stage (0 deep DP, 1 rescued, 2 other)
__global__ void k_fmt_measure(FmtView V, uint32_t *__restrict__ tailLen, uint32_t *__restrict__ recLen, unsigned long long *__restrict__ lenAll,
                              char *__restrict__ tailText, uint8_t *__restrict__ segOf)
{
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = id < V.nReads;
    uint32_t mine = 0; int seg = 0;
    if (live) {
        const FqRec R = V.rec[id];
        const char *text = V.text + ((id & 1u) ? V.base1 : 0);
        const int2 *keys; uint32_t G;
        seg = fmt_group(V, id, keys, G);
        const uint32_t cl = V.ignoreComments ? 0 : R.commentLen;
        const uint32_t tail = fmt_tail<true>(tailText + (size_t)id * FMT_SLOT, FMT_SLOT, text + R.hdr + R.commentOff, cl, keys, G, fmt_best(keys, G), V.top, V.A);
        tailLen[id] = tail;
        mine = 1 + R.nameLen + tail + R.len + 3 + R.len + 1;
        recLen[id] = mine;
        segOf[id] = (uint8_t)seg;
    }
    const uint32_t other = __shfl_xor_sync(0xffffffffu, mine, 1);
    if (live && !(id & 1u)) {
        const uint32_t p = id >> 1, nPairs = V.nReads >> 1;
        for (int s = 0; s < 3; ++s) lenAll[(uint64_t)s * nPairs + p] = s == seg ? (unsigned long long)mine + other : 0ull;
    }
}

// the base soap4 prints for four input characters at once ("ACGT"[charMap[c]], IndexHandler.cpp:26-45): clearing bit 5 folds exactly the
// lower-case letters onto their upper-case ones, then C -> C, G / N -> G, T / U -> T, anything else -> A
__device__ __forceinline__ uint32_t fq_out4(uint32_t v)
{
    const uint32_t x = v & 0xDFDFDFDFu;
    const uint32_t mC = __vcmpeq4(x, 0x43434343u), mG = __vcmpeq4(x, 0x47474747u) | __vcmpeq4(x, 0x4E4E4E4Eu),
                   mT = __vcmpeq4(x, 0x54545454u) | __vcmpeq4(x, 0x55555555u);
    return 0x41414141u ^ (mC & 0x02020202u) ^ (mG & 0x06060606u) ^ (mT & 0x15151515u);
}
__device__ __forceinline__ char fq_out1(unsigned char c) { return "ACGT"[fq_code(c)]; }
// n bytes from src to dst by one warp: the bytes up to dst's next word boundary and the last few one by one, the rest as aligned 32-bit
// stores whose source word is funnel-shifted out of two aligned loads (src and dst are misaligned independently); MAP: through fq_out4
template <bool MAP> __device__ __forceinline__ void warp_copy(char *dst, const char *src, uint32_t n, uint32_t lane)
{
    uint32_t head = (4u - (uint32_t)((uintptr_t)dst & 3u)) & 3u;
    if (head > n) head = n;
    if (lane < head) dst[lane] = MAP ? fq_out1((unsigned char)src[lane]) : src[lane];
    const uint32_t nw = (n - head) >> 2;
    const char *s = src + head;
    const uint32_t mis = (uint32_t)((uintptr_t)s & 3u);
    const uint32_t *sa = (const uint32_t *)(s - mis);
    uint32_t *d = (uint32_t *)(dst + head);
    for (uint32_t w = lane; w < nw; w += 32) {
        uint32_t v = sa[w];
        if (mis) v = __funnelshift_r(v, sa[w + 1], mis * 8);
        d[w] = MAP ? fq_out4(v) : v;
    }
    const uint32_t done = head + nw * 4;
    if (lane < n - done) dst[done + lane] = MAP ? fq_out1((unsigned char)src[done + lane]) : src[done + lane];
}

// one thread per read: where its record starts in the output (its pair's offset under its stage; mate 2 behind mate 1), so that the
// writer's warps start copying after one round of independent loads instead of a chain of dependent ones
__global__ void k_fmt_offsets(uint32_t nReads, const uint8_t *__restrict__ segOf, const uint32_t *__restrict__ recLen, const unsigned long long *__restrict__ off,
                              unsigned long long *__restrict__ dstOf)
{
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= nReads) return;
    dstOf[id] = off[(uint64_t)segOf[id] * (nReads >> 1) + (id >> 1)] + ((id & 1u) ? recLen[id - 1] : 0u);
}

// one warp per read
__global__ void k_fmt_write(FmtView V, const uint32_t *__restrict__ tailLen, const unsigned long long *__restrict__ dstOf,
                            const char *__restrict__ tailText, char *__restrict__ out)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t nWarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; id < V.nReads; id += nWarps) {
        const FqRec R = V.rec[id];
        const char *text = V.text + ((id & 1u) ? V.base1 : 0);
        char *w = out + dstOf[id];
        const uint32_t tail = tailLen[id];
        if (lane == 0) w[0] = '@';
        if (tail <= FMT_SLOT) warp_copy<false>(w + 1 + R.nameLen, tailText + (size_t)id * FMT_SLOT, tail, lane);
        else if (lane == 0) {                        // a long SCORE: list: composed again, in place
            const int2 *keys; uint32_t G;
            fmt_group(V, id, keys, G);
            const uint32_t cl = V.ignoreComments ? 0 : R.commentLen;
            fmt_tail<true>(w + 1 + R.nameLen, 0xFFFFFFFFu, text + R.hdr + R.commentOff, cl, keys, G, fmt_best(keys, G), V.top, V.A);
        }
        warp_copy<false>(w + 1, text + R.hdr + 1, R.nameLen, lane);
        char *ws = w + 1 + R.nameLen + tail;
        warp_copy<true>(ws, text + R.seq, R.len, lane);
        if (lane < 3) ws[R.len + lane] = lane == 1 ? '+' : '\n';
        char *wq = ws + R.len + 3;
        warp_copy<false>(wq, text + R.qual, R.len, lane);
        if (lane == 0) wq[R.len] = '\n';
    }
}

// ------------------------------------------------------------------------------------------------
// chain: the formatted text of a batch -> the next chunk's two mate texts (the deinterleave rewrite)
// Record r of the formatted text is lines 4r .. 4r+3 of lineEnd and belongs to mate (r & 1) + 1, pair r >> 1.  Its header
// "@NAME<blanks>TAIL" becomes "@NAME'/<mate> TAIL": NAME is the first blank-delimited word after '@', NAME' is NAME without one trailing
// "/1" or "/2", TAIL is the rest of the line after the blanks that follow NAME ("@NAME'/<mate>" alone when there is none).  The other
// three lines are copied as they are (the formatter's third line is always "+").
struct ChainHdr { uint32_t name, nameLen, comm, commLen; };
__device__ __forceinline__ ChainHdr chain_header(const char *text, uint32_t s0, uint32_t e0)
{
    ChainHdr h;
    uint32_t q = s0 + 1;
    while (q < e0 && fq_isspace((unsigned char)text[q])) ++q;
    h.name = q;
    while (q < e0 && !fq_isspace((unsigned char)text[q])) ++q;
    h.nameLen = q - h.name;
    while (q < e0 && fq_isspace((unsigned char)text[q])) ++q;
    h.comm = q; h.commLen = e0 - q;
    if (h.nameLen >= 2 && text[h.name + h.nameLen - 2] == '/' && (text[h.name + h.nameLen - 1] == '1' || text[h.name + h.nameLen - 1] == '2')) h.nameLen -= 2;
    return h;
}
__device__ __forceinline__ uint32_t chain_rec_start(const uint32_t *L, uint32_t r) { return r ? L[4 * r - 1] + 1 : 0; }
// one thread per record: its rewritten size, stored mate-major (mate 1's pairs, then mate 2's) for one scan over both mates
__global__ void k_chain_measure(const char *__restrict__ text, const uint32_t *__restrict__ L, uint32_t nReads, unsigned long long *__restrict__ len)
{
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nReads) return;
    const uint32_t s0 = chain_rec_start(L, r), e0 = L[4 * r];
    const ChainHdr h = chain_header(text, s0, e0);
    len[(uint64_t)(r & 1u) * (nReads >> 1) + (r >> 1)] = 1 + h.nameLen + 2 + (h.commLen ? 1 + h.commLen : 0) + 1 + (L[4 * r + 3] - e0);
}
// one warp per record: off = the scan of k_chain_measure's sizes; mate 2's text starts at base1
__global__ void k_chain_write(const char *__restrict__ text, const uint32_t *__restrict__ L, uint32_t nReads, const unsigned long long *__restrict__ off,
                              uint64_t base1, char *__restrict__ out)
{
    const uint32_t lane = threadIdx.x & 31u, nPairs = nReads >> 1;
    const uint32_t nWarps = (gridDim.x * blockDim.x) >> 5;
    const unsigned long long off2 = off[nPairs];
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nReads; r += nWarps) {
        const uint32_t m = r & 1u, s0 = chain_rec_start(L, r), e0 = L[4 * r];
        const ChainHdr h = chain_header(text, s0, e0);
        char *w = out + (m ? base1 + off[nPairs + (r >> 1)] - off2 : off[r >> 1]);
        if (lane == 0) w[0] = '@';
        warp_copy<false>(w + 1, text + h.name, h.nameLen, lane);
        w += 1 + h.nameLen;
        if (lane == 0) { w[0] = '/'; w[1] = (char)('1' + m); if (h.commLen) w[2] = ' '; }
        w += h.commLen ? 3 : 2;
        warp_copy<false>(w, text + h.comm, h.commLen, lane);
        w += h.commLen;
        if (lane == 0) w[0] = '\n';
        warp_copy<false>(w + 1, text + e0 + 1, L[4 * r + 3] - e0, lane);
    }
}

int scan_any(mp_context *ctx, const uint32_t *in, uint32_t *out, uint64_t n)
{
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, (int64_t)n, ctx->stream);
    if (ctx->dScanTmp.reserve(tb)) return MP_ERR_CUDA;
    cub::DeviceScan::ExclusiveSum(ctx->dScanTmp.p, tb, in, out, (int64_t)n, ctx->stream);
    return 0;
}
int scan_any(mp_context *ctx, const unsigned long long *in, unsigned long long *out, uint64_t n)
{
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, (int64_t)n, ctx->stream);
    if (ctx->dScanTmp.reserve(tb)) return MP_ERR_CUDA;
    cub::DeviceScan::ExclusiveSum(ctx->dScanTmp.p, tb, in, out, (int64_t)n, ctx->stream);
    return 0;
}

}  // namespace

extern "C" void *mp_host_alloc(uint64_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { mp_set_error("cudaMallocHost(%llu) failed", (unsigned long long)bytes); return nullptr; }
    return p;
}
extern "C" void mp_host_free(void *p) { if (p) cudaFreeHost(p); }

static int fq_check_args(const char *who, uint32_t nPairs, uint32_t wpq, uint32_t maxReadLength)
{
    if (nPairs == 0 || wpq == 0 || maxReadLength < 2) { mp_set_error("%s: bad argument", who); return MP_ERR_ARG; }
    if (maxReadLength - 1 > 16u * wpq) { mp_set_error("%s: reads of up to %u bases do not fit %u words per query", who, maxReadLength - 1, wpq); return MP_ERR_ARG; }
    if (nPairs > (1u << 29)) { mp_set_error("%s: too many pairs", who); return MP_ERR_ARG; }
    return 0;
}

// Everything after the text is in dFqText (mate 1 at 0, mate 2 at base1): the record index, the checks, lengths and 2-bit rows, and the
// batch state.  mp_fastq_upload and mp_fastq_chain share it.
static int fq_ingest(mp_context *ctx, const char *who, uint64_t base1, uint64_t bytes1, uint64_t bytes2, uint32_t nPairs, uint32_t wpq,
                     uint32_t maxReadLength, const uint32_t **readLengths)
{
    // 32-bit offsets inside a mate's text; every record has at least 4 newlines + '@' + '+' + a base + a quality
    if (bytes1 >= 0xFFFFFFF0ull || bytes2 >= 0xFFFFFFF0ull || bytes1 < 8ull * nPairs || bytes2 < 8ull * nPairs) {
        mp_set_error("%s: not strict four-line FASTQ", who); return MP_ERR_FORMAT;
    }
    cudaStream_t st = ctx->stream;
    const uint32_t nReads = 2 * nPairs, maxLines = 4 * nPairs;
    const uint64_t nT[2] = { (bytes1 + FQ_PIECE - 1) / FQ_PIECE, (bytes2 + FQ_PIECE - 1) / FQ_PIECE };
    const uint64_t cntOff1 = nT[0] + 1;
    if (ctx->dFqCnt.reserve((nT[0] + nT[1] + 2) * 4) || ctx->dFqCntPos.reserve((nT[0] + nT[1] + 2) * 4) ||
        ctx->dFqLines.reserve((size_t)maxLines * 2 * 4) || ctx->dFqRec.reserve((size_t)nReads * sizeof(FqRec)) || ctx->dFqFlags.reserve(16)) return MP_ERR_CUDA;
    char *dText = ctx->dFqText.as<char>();
    uint32_t *dFlags = ctx->dFqFlags.as<uint32_t>();
    MP_CUDA(cudaMemsetAsync(dFlags, 0, 16, st));
    uint32_t totals[2] = { 0, 0 };
    for (int m = 0; m < 2; ++m) {
        const char *t = dText + (m ? base1 : 0);
        const uint64_t by = m ? bytes2 : bytes1;
        uint32_t *cnt = ctx->dFqCnt.as<uint32_t>() + (m ? cntOff1 : 0), *pos = ctx->dFqCntPos.as<uint32_t>() + (m ? cntOff1 : 0);
        (++g_mp_launches), k_fq_count<<<(unsigned)((nT[m] + 1 + 255) / 256), 256, 0, st>>>(t, by, cnt, dFlags);
        if (scan_any(ctx, cnt, pos, nT[m] + 1)) return MP_ERR_CUDA;
        (++g_mp_launches), k_fq_lines<<<(unsigned)((nT[m] + 255) / 256), 256, 0, st>>>(t, by, pos, maxLines, ctx->dFqLines.as<uint32_t>() + (size_t)m * maxLines);
        MP_CUDA(cudaMemcpyAsync(&totals[m], pos + nT[m], 4, cudaMemcpyDeviceToHost, st));
    }
    uint32_t flags[4] = { 0, 0, 0, 0 };
    MP_CUDA(cudaMemcpyAsync(flags, dFlags, 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaStreamSynchronize(st));
    if (flags[0] || totals[0] != maxLines || totals[1] != maxLines) {
        mp_set_error("%s: not strict four-line FASTQ (%u / %u lines for %u records%s)", who, totals[0], totals[1], nPairs, flags[0] ? ", CR or NUL bytes" : "");
        return MP_ERR_FORMAT;
    }
    // the record views may overwrite the previous batch's only now: nothing has been consumed before this point
    const uint64_t nPad = ((uint64_t)nReads + 31) / 32 * 32;
    const size_t rowBytes = nPad * wpq * 4;
    if (ctx->dReads.reserve(rowBytes + 64) || ctx->dLens.reserve((size_t)nReads * 4)) return MP_ERR_CUDA;
    (++g_mp_launches), k_fq_records<<<(nReads + 255) / 256, 256, 0, st>>>(dText, base1, ctx->dFqLines.as<uint32_t>(), ctx->dFqLines.as<uint32_t>() + maxLines, nReads,
                                                                       maxReadLength - 1, ctx->dFqRec.as<FqRec>(), ctx->dLens.as<uint32_t>(), dFlags);
    MP_CUDA(cudaMemcpyAsync(flags, dFlags, 8, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    if (flags[0] & 2u) {
        ctx->hasBatch = false; ctx->fqBatch = false;          // dLens was overwritten
        mp_set_error("%s: not strict four-line FASTQ (a record is not '@' / bases / '+' / qualities of the same length)", who);
        return MP_ERR_FORMAT;
    }
    MP_CUDA(cudaMemsetAsync(ctx->dReads.p, 0, rowBytes + 64, st));
    const uint64_t words = (uint64_t)nReads * wpq;
    (++g_mp_launches), k_fq_pack<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(dText, base1, ctx->dFqRec.as<FqRec>(), nReads, wpq, ctx->dReads.as<uint32_t>());
    MP_CUDA(cudaGetLastError());
    ctx->hLens.resize(nReads);
    MP_CUDA(cudaMemcpyAsync(ctx->hLens.data(), ctx->dLens.p, (size_t)nReads * 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    if (readLengths) *readLengths = ctx->hLens.data();
    ctx->maxLenBatch = flags[1];
    ctx->nReads = nReads; ctx->wpq = wpq; ctx->hasBatch = true; ctx->seeded = false;
    ctx->fqBatch = true; ctx->fqBase[0] = 0; ctx->fqBase[1] = base1; ctx->fqBytes[0] = bytes1; ctx->fqBytes[1] = bytes2;
    ctx->resValid = false; ctx->fmtReady = false;
    return 0;
}

extern "C" int mp_fastq_upload(mp_context *ctx, const char *text1, uint64_t bytes1, const char *text2, uint64_t bytes2,
                               uint32_t nPairs, uint32_t wpq, uint32_t maxReadLength, const uint32_t **readLengths)
{
    if (!ctx || !text1 || !text2) { mp_set_error("mp_fastq_upload: bad argument"); return MP_ERR_ARG; }
    if (int rc = fq_check_args("mp_fastq_upload", nPairs, wpq, maxReadLength)) return rc;
    if (bytes1 == 0 || bytes2 == 0 || text1[bytes1 - 1] != '\n' || text2[bytes2 - 1] != '\n') { mp_set_error("mp_fastq_upload: not strict four-line FASTQ"); return MP_ERR_FORMAT; }
    if (bytes1 >= 0xFFFFFFF0ull || bytes2 >= 0xFFFFFFF0ull) { mp_set_error("mp_fastq_upload: not strict four-line FASTQ"); return MP_ERR_FORMAT; }
    MP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ctx->fqBatch = false; ctx->fmtReady = false;              // the resident text of the previous batch is overwritten from here on
    const uint64_t base1 = (bytes1 + 63) & ~63ull;
    if (ctx->dFqText.reserve(base1 + bytes2 + 64)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpyAsync(ctx->dFqText.p, text1, bytes1, cudaMemcpyHostToDevice, st));
    MP_CUDA(cudaMemcpyAsync(ctx->dFqText.as<char>() + base1, text2, bytes2, cudaMemcpyHostToDevice, st));
    return fq_ingest(ctx, "mp_fastq_upload", base1, bytes1, bytes2, nPairs, wpq, maxReadLength, readLengths);
}

// The formatted text (dFmtOut) -> the deinterleave rewrite into the two mate texts of dFqText -> fq_ingest.  The formatted text is left
// as it is, so that after MP_ERR_FORMAT mp_format_fetch still returns it.
extern "C" int mp_fastq_chain(mp_context *ctx, uint32_t wpq, uint32_t maxReadLength, const uint32_t **readLengths)
{
    if (!ctx) { mp_set_error("mp_fastq_chain: bad argument"); return MP_ERR_ARG; }
    if (!ctx->fmtReady) { mp_set_error("mp_fastq_chain: no formatted batch (call mp_format_fastq first)"); return MP_ERR_STATE; }
    const uint32_t nPairs = ctx->nReads / 2, nReads = ctx->nReads, maxLines = 8 * nPairs;
    if (int rc = fq_check_args("mp_fastq_chain", nPairs, wpq, maxReadLength)) return rc;
    MP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const char *src = ctx->dFmtOut.as<char>();
    const uint64_t bytes = ctx->fmtBytes, nT = (bytes + FQ_PIECE - 1) / FQ_PIECE;
    // the formatted text's line index in the ingest's own scratch (fq_ingest rebuilds it for the mate texts afterwards)
    if (ctx->dFqCnt.reserve((nT + 1) * 4) || ctx->dFqCntPos.reserve((nT + 1) * 4) || ctx->dFqLines.reserve((size_t)maxLines * 4) || ctx->dFqFlags.reserve(16) ||
        ctx->dFmtLen.reserve(((size_t)2 * nPairs + 1) * 8) || ctx->dFmtOff.reserve(((size_t)2 * nPairs + 1) * 8)) return MP_ERR_CUDA;
    uint32_t *cnt = ctx->dFqCnt.as<uint32_t>(), *pos = ctx->dFqCntPos.as<uint32_t>(), *L = ctx->dFqLines.as<uint32_t>();
    (++g_mp_launches), k_fq_count<<<(unsigned)((nT + 1 + 255) / 256), 256, 0, st>>>(src, bytes, cnt, ctx->dFqFlags.as<uint32_t>());
    if (scan_any(ctx, cnt, pos, nT + 1)) return MP_ERR_CUDA;
    (++g_mp_launches), k_fq_lines<<<(unsigned)((nT + 255) / 256), 256, 0, st>>>(src, bytes, pos, maxLines, L);
    uint32_t lines = 0;
    MP_CUDA(cudaMemcpyAsync(&lines, pos + nT, 4, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    if (lines != maxLines) { mp_set_error("mp_fastq_chain: the formatted text has %u lines for %u pairs", lines, nPairs); return MP_ERR_FORMAT; }
    // sizes (dFmtLen, dFmtOff: the formatter's scratch, free once its text is written)
    unsigned long long *len = ctx->dFmtLen.as<unsigned long long>(), *off = ctx->dFmtOff.as<unsigned long long>();
    MP_CUDA(cudaMemsetAsync(len + 2 * (size_t)nPairs, 0, 8, st));
    (++g_mp_launches), k_chain_measure<<<(nReads + 255) / 256, 256, 0, st>>>(src, L, nReads, len);
    if (scan_any(ctx, len, off, 2ull * nPairs + 1)) return MP_ERR_CUDA;
    unsigned long long tot[2] = { 0, 0 };
    MP_CUDA(cudaMemcpyAsync(&tot[0], off + nPairs, 8, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaMemcpyAsync(&tot[1], off + 2 * (size_t)nPairs, 8, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaStreamSynchronize(st));
    const uint64_t bytes1 = tot[0], bytes2 = tot[1] - tot[0], base1 = (bytes1 + 63) & ~63ull;
    if (bytes1 >= 0xFFFFFFF0ull || bytes2 >= 0xFFFFFFF0ull) { mp_set_error("mp_fastq_chain: a mate's text exceeds 4 GB"); return MP_ERR_FORMAT; }
    ctx->fqBatch = false;                                     // the resident text of this batch is overwritten from here on
    if (ctx->dFqText.reserve(base1 + bytes2 + 64)) return MP_ERR_CUDA;
    int dev = 0, sms = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    (++g_mp_launches), k_chain_write<<<(unsigned)sms * 8, 256, 0, st>>>(src, L, nReads, off, base1, ctx->dFqText.as<char>());
    MP_CUDA(cudaGetLastError());
    return fq_ingest(ctx, "mp_fastq_chain", base1, bytes1, bytes2, nPairs, wpq, maxReadLength, readLengths);
}

// Sizes the ingest / egress buffers of a context before the batch loop, like mp_reserve does for the alignment buffers (the first
// cudaMalloc of 700 MB inside the loop stalls every context of the GPU while it runs).
extern "C" int mp_fastq_reserve(mp_context *ctx, uint64_t textBytes, uint32_t nPairs)
{
    if (!ctx || nPairs == 0) { mp_set_error("mp_fastq_reserve: bad argument"); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(ctx->device));
    const uint64_t nReads = 2ull * nPairs, nT = textBytes / FQ_PIECE + 4;
    const uint64_t outBytes = textBytes + nReads * 96;
    if (ctx->dFqText.reserve(textBytes + 256) || ctx->dFqCnt.reserve(nT * 4) || ctx->dFqCntPos.reserve(nT * 4) || ctx->dFqLines.reserve((size_t)nPairs * 8 * 4) ||
        ctx->dFqRec.reserve((size_t)nReads * sizeof(FqRec)) || ctx->dFqFlags.reserve(16) ||
        ctx->dFmtKeys.reserve((size_t)(3 * nReads) * sizeof(int2)) || ctx->dFmtGroups.reserve((size_t)(4 * (uint64_t)nPairs + 2 * nReads) * 4) ||
        ctx->dFmtRecLen.reserve((size_t)nReads * 4) || ctx->dFmtTail.reserve((size_t)nReads * 4) || ctx->dFmtLen.reserve(((size_t)3 * nPairs + 1) * 8) ||
        ctx->dFmtOff.reserve(((size_t)3 * nPairs + 1) * 8) || ctx->dFmtOut.reserve(outBytes) || ctx->dFmtTailText.reserve((size_t)nReads * FMT_SLOT) || ctx->dFmtSeg.reserve((size_t)nReads) || ctx->dFmtDst.reserve((size_t)nReads * 8) || ctx->dScanTmp.reserve((size_t)1 << 20)) return MP_ERR_CUDA;
    return 0;
}

extern "C" int mp_annotation_upload(mp_context *ctx, const mp_annotation *a)
{
    if (!ctx || !a || !a->grid || !a->trStartPos || !a->trChrID || !a->names || !a->nameOffsets || a->gridEntries == 0 || a->numTranslate == 0 || a->numSeq == 0) {
        mp_set_error("mp_annotation_upload: bad argument"); return MP_ERR_ARG;
    }
    for (uint32_t j = 0; j < a->numTranslate; ++j)
        if (a->trChrID[j] == 0 || a->trChrID[j] > a->numSeq) { mp_set_error("mp_annotation_upload: translate entry %u names sequence %u of %u", j, a->trChrID[j], a->numSeq); return MP_ERR_ARG; }
    for (uint32_t j = 0; j < a->gridEntries; ++j)
        if (a->grid[j] >= a->numTranslate) { mp_set_error("mp_annotation_upload: grid entry %u out of range", j); return MP_ERR_ARG; }
    if (a->trStartPos[0] != 0) { mp_set_error("mp_annotation_upload: the first translate segment must start at 0"); return MP_ERR_ARG; }
    MP_CUDA(cudaSetDevice(ctx->device));
    const uint64_t nameBytes = a->nameOffsets[a->numSeq];
    if (ctx->dAnnGrid.reserve((size_t)a->gridEntries * 4) || ctx->dAnnTrStart.reserve((size_t)a->numTranslate * 8) || ctx->dAnnTrChr.reserve((size_t)a->numTranslate * 4) ||
        ctx->dAnnNames.reserve(nameBytes + 1) || ctx->dAnnNameOff.reserve(((size_t)a->numSeq + 1) * 8)) return MP_ERR_CUDA;
    MP_CUDA(cudaMemcpy(ctx->dAnnGrid.p, a->grid, (size_t)a->gridEntries * 4, cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(ctx->dAnnTrStart.p, a->trStartPos, (size_t)a->numTranslate * 8, cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(ctx->dAnnTrChr.p, a->trChrID, (size_t)a->numTranslate * 4, cudaMemcpyHostToDevice));
    if (nameBytes) MP_CUDA(cudaMemcpy(ctx->dAnnNames.p, a->names, nameBytes, cudaMemcpyHostToDevice));
    MP_CUDA(cudaMemcpy(ctx->dAnnNameOff.p, a->nameOffsets, ((size_t)a->numSeq + 1) * 8, cudaMemcpyHostToDevice));
    ctx->annDnaLength = a->dnaLength; ctx->annGridEntries = a->gridEntries; ctx->annNumTr = a->numTranslate; ctx->annNumSeq = a->numSeq;
    ctx->hasAnn = true; ctx->annSrc = nullptr;
    return 0;
}

extern "C" int mp_format_fastq(mp_context *ctx, const mp_format_params *F, uint64_t *bytes)
{
    if (!ctx || !F || !bytes) { mp_set_error("mp_format_fastq: null argument"); return MP_ERR_ARG; }
    if (F->megapathMode != 1 && F->megapathMode != 2) { mp_set_error("mp_format_fastq: megapathMode must be 1 (-F) or 2 (-P)"); return MP_ERR_ARG; }
    const mp_context *an = ctx->annSrc ? ctx->annSrc : ctx;     // a bound clone reads its owner's annotation (mp_index_bind)
    if (!an->hasAnn || !ctx->fqBatch || !ctx->resValid) {
        mp_set_error("mp_format_fastq: needs mp_annotation_upload, a batch from mp_fastq_upload and its mp_align_pairs results"); return MP_ERR_STATE;
    }
    MP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint32_t nReads = ctx->nReads, nPairs = nReads / 2;
    const uint64_t nP = ctx->resCount[0], nR = ctx->resCount[1], nS = ctx->resCount[2];
    if (nP > 0xFFFFFFF0ull || nR > 0xFFFFFFF0ull || nS > 0xFFFFFFF0ull) { mp_set_error("mp_format_fastq: result arrays too large"); return MP_ERR_CAPACITY; }
    // keys: P1 | P2 | R1 | R2 | S ; groups: pStart pEnd rStart rEnd (per pair) sStart sEnd (per read)
    const size_t nKeys = 2 * nP + 2 * nR + nS + 1, nGroups = (size_t)4 * nPairs + (size_t)2 * nReads;
    if (ctx->dFmtKeys.reserve(nKeys * sizeof(int2)) || ctx->dFmtGroups.reserve(nGroups * 4) || ctx->dFmtRecLen.reserve((size_t)nReads * 4) ||
        ctx->dFmtTail.reserve((size_t)nReads * 4) || ctx->dFmtLen.reserve(((size_t)3 * nPairs + 1) * 8) || ctx->dFmtOff.reserve(((size_t)3 * nPairs + 1) * 8) ||
        ctx->dFmtTailText.reserve((size_t)nReads * FMT_SLOT) || ctx->dFmtSeg.reserve((size_t)nReads) || ctx->dFmtDst.reserve((size_t)nReads * 8)) return MP_ERR_CUDA;
    int2 *kP1 = ctx->dFmtKeys.as<int2>(), *kP2 = kP1 + nP, *kR1 = kP2 + nP, *kR2 = kR1 + nR, *kS = kR2 + nR;
    uint32_t *g = ctx->dFmtGroups.as<uint32_t>();
    uint32_t *pStart = g, *pEnd = g + nPairs, *rStart = g + 2 * (size_t)nPairs, *rEnd = g + 3 * (size_t)nPairs, *sStart = g + 4 * (size_t)nPairs, *sEnd = sStart + nReads;
    MP_CUDA(cudaMemsetAsync(g, 0, nGroups * 4, st));
    AnnDev A = { an->dAnnGrid.as<uint32_t>(), an->dAnnTrStart.as<uint64_t>(), an->dAnnTrChr.as<uint32_t>(), an->dAnnNames.as<char>(), an->dAnnNameOff.as<uint64_t>(),
                 an->annGridEntries };
    const uint32_t *lens = ctx->dLens.as<uint32_t>();
    if (nP) (++g_mp_launches), k_fmt_pair_keys<<<(unsigned)((nP + 127) / 128), 128, 0, st>>>(ctx->dRes2.as<mp_pair_result>(), (uint32_t)nP, lens, A, F->megapathMode, kP1, kP2, pStart, pEnd);
    if (nR) (++g_mp_launches), k_fmt_pair_keys<<<(unsigned)((nR + 127) / 128), 128, 0, st>>>(ctx->dRsOut.as<mp_pair_result>(), (uint32_t)nR, lens, A, F->megapathMode, kR1, kR2, rStart, rEnd);
    if (nS) (++g_mp_launches), k_fmt_single_keys<<<(unsigned)((nS + 127) / 128), 128, 0, st>>>(ctx->dS2Res.as<mp_single_result>(), (uint32_t)nS, lens, A, kS, sStart, sEnd);
    FmtView V;
    V.text = ctx->dFqText.as<char>(); V.base1 = ctx->fqBase[1]; V.rec = ctx->dFqRec.as<FqRec>(); V.nReads = nReads;
    V.pStart = pStart; V.pEnd = pEnd; V.rStart = rStart; V.rEnd = rEnd; V.sStart = sStart; V.sEnd = sEnd;
    V.kP1 = kP1; V.kP2 = kP2; V.kR1 = kR1; V.kR2 = kR2; V.kS = kS; V.A = A; V.top = F->top; V.mode = F->megapathMode; V.ignoreComments = F->ignoreComments;
    unsigned long long *lenAll = ctx->dFmtLen.as<unsigned long long>(), *off = ctx->dFmtOff.as<unsigned long long>();
    const uint64_t nLen = (uint64_t)3 * nPairs;
    MP_CUDA(cudaMemsetAsync(lenAll + nLen, 0, 8, st));
    (++g_mp_launches), k_fmt_measure<<<(nReads + 127) / 128, 128, 0, st>>>(V, ctx->dFmtTail.as<uint32_t>(), ctx->dFmtRecLen.as<uint32_t>(), lenAll, ctx->dFmtTailText.as<char>(), ctx->dFmtSeg.as<uint8_t>());
    if (scan_any(ctx, lenAll, off, nLen + 1)) return MP_ERR_CUDA;
    unsigned long long total = 0;
    MP_CUDA(cudaMemcpyAsync(&total, off + nLen, 8, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaGetLastError());
    MP_CUDA(cudaStreamSynchronize(st));
    if (ctx->dFmtOut.reserve((size_t)total + 16)) return MP_ERR_CUDA;
    int dev = 0, sms = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    (++g_mp_launches), k_fmt_offsets<<<(nReads + 255) / 256, 256, 0, st>>>(nReads, ctx->dFmtSeg.as<uint8_t>(), ctx->dFmtRecLen.as<uint32_t>(), off, ctx->dFmtDst.as<unsigned long long>());
    (++g_mp_launches), k_fmt_write<<<(unsigned)sms * 8, 256, 0, st>>>(V, ctx->dFmtTail.as<uint32_t>(), ctx->dFmtDst.as<unsigned long long>(), ctx->dFmtTailText.as<char>(), ctx->dFmtOut.as<char>());
    MP_CUDA(cudaGetLastError());
    ctx->fmtBytes = total; ctx->fmtReady = true;
    *bytes = total;
    return 0;
}

extern "C" int mp_format_fetch(mp_context *ctx, char *dst, uint64_t bytes)
{
    if (!ctx || (!dst && bytes)) { mp_set_error("mp_format_fetch: null argument"); return MP_ERR_ARG; }
    if (!ctx->fmtReady || bytes != ctx->fmtBytes) { mp_set_error("mp_format_fetch: no formatted batch of that size (call mp_format_fastq first)"); return MP_ERR_STATE; }
    MP_CUDA(cudaSetDevice(ctx->device));
    if (bytes) MP_CUDA(cudaMemcpyAsync(dst, ctx->dFmtOut.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    MP_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}
