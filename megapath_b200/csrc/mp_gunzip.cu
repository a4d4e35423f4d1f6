// mp_gunzip.cu -- gzip files inflated on the device: mp_gunzip_open / mp_gunzip_run / mp_gunzip_stats / mp_gunzip_close.
//
// A single-member gzip stream has no independent pieces, so each call splits its compressed window speculatively (the approach of
// pugz and rapidgzip):
//   find     the window is cut into chunks of MP_GUNZIP_CHUNK bytes.  k_gz_find tests, for every chunk after the first, its bit
//            offsets in order (256 at a time) and keeps the first one where a non-final dynamic-Huffman block header is valid --
//            exactly what zlib's inflate.c / inftrees.c accept (gz_dyn_header).  A true block header always passes, so a true
//            boundary is never missed when it is the first valid offset; stored and fixed blocks are never searched for.  A chunk
//            without a candidate is merged into the chunk before it.
//   decode   k_gz_decode: one thread per chunk decodes from its start (the first chunk from the state the previous call left, the
//            others from their candidates) up to the first block boundary at or after the next chunk's start, into a slot of
//            MP_GUNZIP_SLOT 16-bit symbols.  A back-reference that reaches before the chunk's first output byte is stored as a
//            marker 256 + i: byte i of the 32 KiB that precede the chunk.  The decoder can stop at any symbol boundary (slot full,
//            input exhausted) and saves a small state (GzState) from which a later launch, or the next call, resumes.
//   verify   the host walks the chunks in order: a chunk's output is used only when its start equals the verified end of the chunk
//            before it; otherwise it is decoded again from that end.  By induction every byte used was decoded from a true block
//            boundary -- false candidates cost rounds, never wrong bytes, and when every candidate is false the decode is sequential.
//   resolve  k_gz_window walks the accepted chunks in order and resolves the last 32 KiB of each (the window of the next one), then
//            k_gz_resolve replaces every other marker in parallel.  A marker that reaches before its member's first byte is zlib's
//            "invalid distance too far back".
//   check    k_gz_crc takes the CRC-32 of 32 KiB pieces of the output, cut at member ends; the host combines them per member
//            (mp_crc32.h, shared with the BGZF encoder) and checks CRC-32 and ISIZE against every trailer.
// Every read of the compressed window and every write into a slot or event list is bounds-checked: garbage decoded from a false
// start or a corrupt file ends in a refusal, never in a fault.
#include "mp_context.h"
#include "mp_crc32.h"
#include <algorithm>

namespace {

constexpr uint32_t GZ_CHUNK = MP_GUNZIP_CHUNK;
constexpr uint32_t GZ_SLOT = MP_GUNZIP_SLOT;
constexpr uint32_t GZ_EVENTS = MP_GUNZIP_EVENTS;
constexpr uint32_t GZ_WIN = 32768;
constexpr uint32_t GZ_FIND_THREADS = 256;
constexpr uint32_t GZ_CRC_PIECE = 32768;
constexpr int GZ_LB_LIT = 10, GZ_LB_DIST = 8;     // bits of the first-level decode tables

// decoder modes
enum { GZ_M_HEADER = 0, GZ_M_BLOCK = 1, GZ_M_DATA = 2, GZ_M_TRAILER = 3, GZ_M_END = 4 };
// decode results
enum { GZ_S_TARGET = 1, GZ_S_FULL = 2, GZ_S_NEED = 3, GZ_S_END = 4, GZ_S_ERROR = 5 };
// event kinds
enum { GZ_E_START = 0, GZ_E_END = 1 };

__constant__ uint16_t c_gzLenBase[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258 };
__constant__ uint8_t c_gzLenExtra[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
__constant__ uint16_t c_gzDistBase[30] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
                                           4097, 6145, 8193, 12289, 16385, 24577 };
__constant__ uint8_t c_gzDistExtra[30] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };
__constant__ uint8_t c_gzClOrder[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

// Resumable decoder state at a symbol boundary (RFC 1951 3.2.3; gzip framing RFC 1952 2.3)
struct GzState {
    uint64_t bit;               // next unread bit, counted from bit 0 of the call's first input byte
    uint32_t mode;              // GZ_M_*
    uint32_t first;             // no member header parsed yet: anything but the gzip magic is an error, not trailing bytes
    uint32_t bfinal, btype;     // current block
    uint32_t left;              // bytes left of the current stored block
    uint32_t nlen, ndist;       // code counts of the current dynamic block
    uint32_t hstage, hflags, hleft, hcrc;   // gzip header parse: stage, FLG, bytes left of FEXTRA, running CRC-32 register
    uint8_t lens[320];          // code lengths of the current dynamic block (lit/len then distance)
};
struct GzEvent { uint32_t kind, out, crc, isize; };     // member start (kind 0) or trailer (kind 1) at output offset `out`
struct GzResult {
    GzState end;
    uint32_t status, nOut, nEvents, errCode;
};
struct GzJob { uint32_t chunk, limit; uint64_t target; };  // decode chunk from states[chunk] up to `target`, at most `limit` symbols

// ---- bit reader over the call's input, LSB first; bits past the end are never buffered ----
struct GzBits {
    const uint8_t *in; uint64_t nBytes;
    uint64_t pos;               // bit position of buf's bit 0
    uint64_t buf; int cnt;
    __device__ GzBits(const uint8_t *p, uint64_t n, uint64_t bit) : in(p), nBytes(n), pos(bit), buf(0), cnt(0) {
        const uint64_t b = bit >> 3;
        if (b < nBytes) { buf = in[b] >> (bit & 7); cnt = 8 - (int)(bit & 7); }
    }
    __device__ __forceinline__ void refill() {
        uint64_t at = (pos + cnt) >> 3;
        while (cnt <= 56 && at < nBytes) { buf |= (uint64_t)in[at++] << cnt; cnt += 8; }
    }
    __device__ __forceinline__ void drop(int k) { buf >>= k; cnt -= k; pos += k; }
    __device__ __forceinline__ void skip_to_byte() { const int k = (int)((8 - (pos & 7)) & 7); if (k) { refill(); drop(k < cnt ? k : cnt); } }
};

// canonical Huffman code: first-level table (symbol | length << 9, 0 = longer code or no code) + puff-style count / symbol lists
struct GzCode {
    uint16_t count[16];
    uint16_t sym[288];
};
struct GzTables {
    uint16_t litLut[1 << GZ_LB_LIT];
    uint16_t distLut[1 << GZ_LB_DIST];
    GzCode lit, dist;
};

__device__ __forceinline__ uint32_t gz_rev(uint32_t code, int len)
{
    uint32_t r = 0;
    for (int i = 0; i < len; ++i) { r = (r << 1) | (code & 1); code >>= 1; }
    return r;
}

// inftrees.c inflate_table: 0 = usable, -1 = over-subscribed, or incomplete where zlib refuses it (always for the code-length code,
// and for lit/len and distance codes unless the only code has length 1); an all-zero code is accepted (it fails when used)
__device__ int gz_check(const uint8_t *lens, int n, bool codes)
{
    int count[16] = { 0 };
    for (int i = 0; i < n; ++i) count[lens[i]]++;
    int max = 15; while (max >= 1 && count[max] == 0) --max;
    if (max == 0) return codes ? -1 : 0;   // code-length code: every length read as 0 -> "missing end-of-block" in inflate.c
    int left = 1;
    for (int len = 1; len <= 15; ++len) { left <<= 1; left -= count[len]; if (left < 0) return -1; }
    if (left > 0 && (codes || max != 1)) return -1;
    return 0;
}

__device__ void gz_build(const uint8_t *lens, int n, GzCode &c, uint16_t *lut, int lb)
{
    uint16_t offs[16];
    for (int i = 0; i < 16; ++i) c.count[i] = 0;
    for (int i = 0; i < n; ++i) c.count[lens[i]]++;
    c.count[0] = 0;
    offs[1] = 0;
    for (int len = 1; len < 15; ++len) offs[len + 1] = offs[len] + c.count[len];
    for (int i = 0; i < (1 << lb); ++i) lut[i] = 0;
    uint32_t code = 0, codeAt[16];          // first code of every length (RFC 1951 3.2.2)
    for (int len = 1; len <= 15; ++len) { code = (code + c.count[len - 1]) << 1; codeAt[len] = code; }
    for (int s = 0; s < n; ++s) {
        const int len = lens[s];
        if (!len) continue;
        c.sym[offs[len]++] = (uint16_t)s;
        const uint32_t cd = codeAt[len]++;
        if (len <= lb) {
            const uint32_t r = gz_rev(cd, len);
            for (uint32_t k = r; k < (1u << lb); k += 1u << len) lut[k] = (uint16_t)(s | len << 9);
        }
    }
}

// decodes one symbol from the low bits of `bits` (avail of them real): >= 0 symbol (*used = its length), -1 need more input,
// -2 no such code (incomplete code)
__device__ __forceinline__ int gz_decode(const GzCode &c, const uint16_t *lut, int lb, uint64_t bits, int avail, int *used)
{
    const uint16_t e = lut[bits & ((1u << lb) - 1)];
    if (e) {
        const int len = e >> 9;
        if (len > avail) return -1;
        *used = len; return e & 511;
    }
    int code = 0, first = 0, index = 0;       // puff.c decode()
    for (int len = 1; len <= 15; ++len) {
        if (len > avail) return -1;
        code |= (int)((bits >> (len - 1)) & 1);
        const int count = c.count[len];
        if (code - count < first) { *used = len; return c.sym[index + (code - first)]; }
        index += count; first += count; first <<= 1; code <<= 1;
    }
    return -2;
}

// code-length code decode (at most 7 bits), puff style
__device__ __forceinline__ int gz_decode_small(const uint8_t *count, const uint8_t *sym, uint64_t bits, int avail, int *used)
{
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= 7; ++len) {
        if (len > avail) return -1;
        code |= (int)((bits >> (len - 1)) & 1);
        const int cnt = count[len];
        if (code - cnt < first) { *used = len; return sym[index + (code - first)]; }
        index += cnt; first += cnt; first <<= 1; code <<= 1;
    }
    return -2;
}

// The dynamic block header after BFINAL / BTYPE (RFC 1951 3.2.7) with zlib's checks (inflate.c TABLE / LENLENS / CODELENS):
// HLIT <= 286 and HDIST <= 30 codes, a complete code-length code, no repeat of a missing length or past the end, a nonzero
// end-of-block length, and lit/len and distance codes inftrees.c accepts.  The bit reader stands after BTYPE.
// 0 = valid (lens / nlen / ndist filled, reader after the header), 1 = input ends inside the header, -1 = invalid
__device__ int gz_dyn_header(GzBits &br, uint8_t *lens, uint32_t *nlenOut, uint32_t *ndistOut)
{
    br.refill();
    if (br.cnt < 14) return 1;
    const uint32_t nlen = (uint32_t)(br.buf & 31) + 257, ndist = (uint32_t)((br.buf >> 5) & 31) + 1, ncode = (uint32_t)((br.buf >> 10) & 15) + 4;
    if (nlen > 286 || ndist > 30) return -1;
    br.drop(14);
    uint8_t cl[19];
    for (int i = 0; i < 19; ++i) cl[i] = 0;
    for (uint32_t i = 0; i < ncode; ++i) {
        br.refill();
        if (br.cnt < 3) return 1;
        cl[c_gzClOrder[i]] = (uint8_t)(br.buf & 7);
        br.drop(3);
    }
    if (gz_check(cl, 19, true)) return -1;
    uint8_t ccount[8] = { 0 }, csym[19], coffs[8];
    for (int i = 0; i < 19; ++i) ccount[cl[i]]++;
    ccount[0] = 0; coffs[1] = 0;
    for (int l = 1; l < 7; ++l) coffs[l + 1] = coffs[l] + ccount[l];
    for (int i = 0; i < 19; ++i) if (cl[i]) csym[coffs[cl[i]]++] = (uint8_t)i;
    uint32_t have = 0;
    while (have < nlen + ndist) {
        br.refill();
        int used = 0;
        const int s = gz_decode_small(ccount, csym, br.buf, br.cnt, &used);
        if (s == -1) return 1;
        if (s < 0) return -1;
        if (s < 16) { br.drop(used); lens[have++] = (uint8_t)s; continue; }
        const int xb = s == 16 ? 2 : s == 17 ? 3 : 7;
        if (br.cnt < used + xb) return 1;
        const uint32_t x = (uint32_t)((br.buf >> used) & ((1u << xb) - 1));
        uint32_t rep; uint8_t v = 0;
        if (s == 16) { if (have == 0) return -1; v = lens[have - 1]; rep = 3 + x; }
        else rep = (s == 17 ? 3 : 11) + x;
        if (have + rep > nlen + ndist) return -1;
        br.drop(used + xb);
        while (rep--) lens[have++] = v;
    }
    if (lens[256] == 0) return -1;
    if (gz_check(lens, (int)nlen, false) || gz_check(lens + nlen, (int)ndist, false)) return -1;
    *nlenOut = nlen; *ndistOut = ndist;
    return 0;
}

__device__ __forceinline__ uint32_t gz_crc_byte(uint32_t c, uint32_t b)
{
    c ^= b;
    for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ 0xEDB88320u : c >> 1;
    return c;
}

__device__ void gz_fixed_lens(uint8_t *lens)
{
    for (int i = 0; i < 144; ++i) lens[i] = 8;
    for (int i = 144; i < 256; ++i) lens[i] = 9;
    for (int i = 256; i < 280; ++i) lens[i] = 7;
    for (int i = 280; i < 288; ++i) lens[i] = 8;
    for (int i = 288; i < 320; ++i) lens[i] = 5;
}

// One chunk: decode from st until the first block header at or after `target`, the slot (limit symbols) or the event list is full,
// the input ends, the file ends or an error.  Writes symbols into slot, member starts / trailers into ev.
__device__ void gz_run(const uint8_t *in, uint64_t nBytes, int fin, GzState &st, uint64_t target, uint32_t limit,
                                uint16_t *slot, GzEvent *ev, GzTables &T, GzResult &res)
{
    uint32_t o = 0, nEv = 0;
    int64_t memberAt = -1;            // output offset of the last member start inside this chunk (references may not cross it)
    GzBits br(in, nBytes, st.bit);
    uint32_t status = 0, err = 0;
    if (st.mode == GZ_M_DATA && st.btype != 0) {        // resumed inside a Huffman block: its tables again
        if (st.btype == 1) { uint8_t fl[320]; gz_fixed_lens(fl); gz_build(fl, 288, T.lit, T.litLut, GZ_LB_LIT); gz_build(fl + 288, 32, T.dist, T.distLut, GZ_LB_DIST); }
        else { gz_build(st.lens, (int)st.nlen, T.lit, T.litLut, GZ_LB_LIT); gz_build(st.lens + st.nlen, (int)st.ndist, T.dist, T.distLut, GZ_LB_DIST); }
    }
    while (!status) {
        if (st.mode == GZ_M_HEADER) {
            // gzip member header (RFC 1952 2.3.1), parsed field by field so that any length of FEXTRA / FNAME / FCOMMENT makes progress
            if (st.hstage == 0) {
                if (nEv >= GZ_EVENTS) { status = GZ_S_FULL; break; }      // before anything of the header is consumed
                br.refill();
                const uint64_t at = br.pos >> 3, rest = nBytes > at ? nBytes - at : 0;
                if (!st.first) {
                    if (rest < 2) { status = fin ? GZ_S_END : GZ_S_NEED; break; }
                    if (in[at] != 0x1f || in[at + 1] != 0x8b) { status = GZ_S_END; break; }   // trailing bytes: ignored, as gzread does
                }
                if (rest < 10) {
                    if (st.first && rest >= 1 && (in[at] != 0x1f || (rest >= 2 && in[at + 1] != 0x8b))) { status = GZ_S_ERROR; err = 1; break; }
                    status = GZ_S_NEED; break;
                }
                if (in[at] != 0x1f || in[at + 1] != 0x8b) { status = GZ_S_ERROR; err = 1; break; }
                if (in[at + 2] != 8) { status = GZ_S_ERROR; err = 2; break; }
                if (in[at + 3] & 0xe0) { status = GZ_S_ERROR; err = 3; break; }
                uint32_t c = 0xffffffffu;
                for (int i = 0; i < 10; ++i) c = gz_crc_byte(c, in[at + i]);
                st.hcrc = c; st.hflags = in[at + 3]; st.hstage = 1;
                br = GzBits(in, nBytes, (at + 10) * 8);
            }
            uint64_t at = br.pos >> 3;
            if (st.hstage == 1) {
                if (st.hflags & 4) {
                    if (at + 2 > nBytes) { status = GZ_S_NEED; break; }
                    st.hleft = in[at] | (uint32_t)in[at + 1] << 8;
                    st.hcrc = gz_crc_byte(gz_crc_byte(st.hcrc, in[at]), in[at + 1]);
                    at += 2; st.hstage = 2;
                } else st.hstage = 3;
            }
            if (st.hstage == 2) {
                while (st.hleft && at < nBytes) { st.hcrc = gz_crc_byte(st.hcrc, in[at++]); --st.hleft; }
                if (st.hleft) { br = GzBits(in, nBytes, at * 8); status = GZ_S_NEED; break; }
                st.hstage = 3;
            }
            bool stop = false;
            for (int f = 3; f <= 4 && !stop; ++f) {            // 3: FNAME, 4: FCOMMENT, zero-terminated
                if (st.hstage != (uint32_t)f) continue;
                if (st.hflags & (f == 3 ? 8 : 16)) {
                    for (;;) {
                        if (at >= nBytes) { stop = true; break; }
                        const uint8_t b = in[at++];
                        st.hcrc = gz_crc_byte(st.hcrc, b);
                        if (!b) break;
                    }
                }
                if (!stop) st.hstage = f + 1;
            }
            if (stop) { br = GzBits(in, nBytes, at * 8); status = GZ_S_NEED; break; }
            if (st.hstage == 5) {
                if (st.hflags & 2) {
                    if (at + 2 > nBytes) { br = GzBits(in, nBytes, at * 8); status = GZ_S_NEED; break; }
                    if ((in[at] | (uint32_t)in[at + 1] << 8) != (~st.hcrc & 0xffffu)) { status = GZ_S_ERROR; err = 4; break; }
                    at += 2;
                }
            }
            br = GzBits(in, nBytes, at * 8);
            ev[nEv++] = GzEvent{ GZ_E_START, o, 0, 0 };
            memberAt = o;
            st.mode = GZ_M_BLOCK; st.first = 0; st.hstage = 0;
            if (br.pos >= target) { status = GZ_S_TARGET; break; }
            continue;
        }
        if (st.mode == GZ_M_BLOCK) {
            const uint64_t at0 = br.pos;
            br.refill();
            if (br.cnt < 3) { status = GZ_S_NEED; break; }
            const uint32_t bf = (uint32_t)(br.buf & 1), bt = (uint32_t)((br.buf >> 1) & 3);
            if (bt == 3) { status = GZ_S_ERROR; err = 5; break; }
            br.drop(3);
            if (bt == 0) {
                br.skip_to_byte();
                br.refill();
                if (br.cnt < 32) { br = GzBits(in, nBytes, at0); status = GZ_S_NEED; break; }
                const uint32_t len = (uint32_t)(br.buf & 0xffff), nlen = (uint32_t)((br.buf >> 16) & 0xffff);
                if (len != (~nlen & 0xffffu)) { status = GZ_S_ERROR; err = 6; break; }
                br.drop(32);
                st.left = len;
            } else if (bt == 1) {
                uint8_t fl[320]; gz_fixed_lens(fl);
                gz_build(fl, 288, T.lit, T.litLut, GZ_LB_LIT); gz_build(fl + 288, 32, T.dist, T.distLut, GZ_LB_DIST);
            } else {
                uint32_t nl = 0, nd = 0;
                const int r = gz_dyn_header(br, st.lens, &nl, &nd);
                if (r > 0) { br = GzBits(in, nBytes, at0); status = GZ_S_NEED; break; }
                if (r < 0) { status = GZ_S_ERROR; err = 7; break; }
                st.nlen = nl; st.ndist = nd;
                gz_build(st.lens, (int)nl, T.lit, T.litLut, GZ_LB_LIT); gz_build(st.lens + nl, (int)nd, T.dist, T.distLut, GZ_LB_DIST);
            }
            st.bfinal = bf; st.btype = bt; st.mode = GZ_M_DATA;
            continue;
        }
        if (st.mode == GZ_M_DATA) {
            bool blockEnd = false;
            if (st.btype == 0) {
                // stored: the reader is byte aligned; partial data is delivered as zlib delivers it
                uint64_t at = br.pos >> 3;
                while (st.left && at < nBytes && o < limit) { slot[o++] = in[at++]; --st.left; }
                br = GzBits(in, nBytes, at * 8);
                if (st.left) { status = o >= limit ? GZ_S_FULL : GZ_S_NEED; break; }
                blockEnd = true;
            } else {
                for (;;) {
                    br.refill();
                    int used = 0;
                    const int s = gz_decode(T.lit, T.litLut, GZ_LB_LIT, br.buf, br.cnt, &used);
                    if (s == -1) { status = GZ_S_NEED; break; }
                    if (s < 0 || s > 285) { status = GZ_S_ERROR; err = 8; break; }
                    if (s < 256) {
                        if (o >= limit) { status = GZ_S_FULL; break; }
                        slot[o++] = (uint16_t)s; br.drop(used); continue;
                    }
                    if (s == 256) { br.drop(used); blockEnd = true; break; }
                    // length, distance: consumed only when every bit of the pair is present (a match is delivered whole or not at all)
                    const int li = s - 257, lx = c_gzLenExtra[li];
                    if (br.cnt < used + lx) { status = GZ_S_NEED; break; }
                    const uint32_t len = c_gzLenBase[li] + (uint32_t)((br.buf >> used) & ((1u << lx) - 1));
                    int used2 = 0;
                    const int ds = gz_decode(T.dist, T.distLut, GZ_LB_DIST, br.buf >> (used + lx), br.cnt - used - lx, &used2);
                    if (ds == -1) { status = GZ_S_NEED; break; }
                    if (ds < 0 || ds > 29) { status = GZ_S_ERROR; err = 9; break; }
                    const int dx = c_gzDistExtra[ds], tot = used + lx + used2 + dx;
                    if (br.cnt < tot) { status = GZ_S_NEED; break; }
                    const uint32_t dist = c_gzDistBase[ds] + (uint32_t)((br.buf >> (used + lx + used2)) & ((1u << dx) - 1));
                    if (memberAt >= 0 ? (int64_t)o - (int64_t)dist < memberAt : false) { status = GZ_S_ERROR; err = 10; break; }
                    if (o + len > limit) { status = GZ_S_FULL; break; }
                    br.drop(tot);
                    int64_t from = (int64_t)o - (int64_t)dist;
                    for (uint32_t k = 0; k < len; ++k, ++from) slot[o++] = from >= 0 ? slot[from] : (uint16_t)(256 + GZ_WIN + from);
                }
                if (status) break;
            }
            if (!blockEnd) continue;
            if (st.bfinal) { st.mode = GZ_M_TRAILER; continue; }
            st.mode = GZ_M_BLOCK;
            if (br.pos >= target) { status = GZ_S_TARGET; break; }
            continue;
        }
        if (st.mode == GZ_M_TRAILER) {
            const uint64_t at = (br.pos + 7) >> 3;
            if (at + 8 > nBytes) { br = GzBits(in, nBytes, at * 8); status = GZ_S_NEED; break; }
            if (nEv >= GZ_EVENTS) { status = GZ_S_FULL; break; }
            const uint32_t crc = in[at] | (uint32_t)in[at + 1] << 8 | (uint32_t)in[at + 2] << 16 | (uint32_t)in[at + 3] << 24;
            const uint32_t isz = in[at + 4] | (uint32_t)in[at + 5] << 8 | (uint32_t)in[at + 6] << 16 | (uint32_t)in[at + 7] << 24;
            ev[nEv++] = GzEvent{ GZ_E_END, o, crc, isz };
            br = GzBits(in, nBytes, (at + 8) * 8);
            st.mode = GZ_M_HEADER; st.hstage = 0;
            continue;
        }
        status = GZ_S_END;      // GZ_M_END
    }
    if (status == GZ_S_END) st.mode = GZ_M_END;
    st.bit = br.pos;
    res.end = st; res.status = status; res.nOut = o; res.nEvents = nEv; res.errCode = err;
}

// ---- kernels ----

// one CTA per chunk after the first: the first bit offset in [8 * C * chunk, 8 * C * (chunk + 1)) where a non-final dynamic block
// header is valid, or ~0
__global__ void __launch_bounds__(GZ_FIND_THREADS)
k_gz_find(const uint8_t *__restrict__ in, uint64_t nBytes, uint32_t nChunks, unsigned long long *__restrict__ cand)
{
    __shared__ unsigned long long best;
    const uint32_t chunk = blockIdx.x + 1;
    if (chunk >= nChunks) return;
    const uint64_t lo = (uint64_t)chunk * GZ_CHUNK * 8, hi = min((uint64_t)(chunk + 1) * GZ_CHUNK, nBytes) * 8;
    if (threadIdx.x == 0) best = ~0ull;
    __syncthreads();
    uint8_t lens[320];
    for (uint64_t base = lo; base < hi; base += GZ_FIND_THREADS) {
        const uint64_t bit = base + threadIdx.x;
        if (bit < hi) {
            GzBits br(in, nBytes, bit);
            br.refill();
            // BFINAL = 0, BTYPE = 2 (bits 0b100 read LSB first), then the cheap count filters inside gz_dyn_header
            if (br.cnt >= 17 && (br.buf & 7) == 4) {
                br.drop(3);
                uint32_t nl, nd;
                if (gz_dyn_header(br, lens, &nl, &nd) == 0) atomicMin(&best, (unsigned long long)bit);
            }
        }
        __syncthreads();
        if (best != ~0ull) break;
        __syncthreads();
    }
    if (threadIdx.x == 0) cand[chunk] = best;
}

__global__ void __launch_bounds__(1)
k_gz_decode(const uint8_t *__restrict__ in, uint64_t nBytes, int fin, const GzJob *__restrict__ jobs, const GzState *__restrict__ states,
            GzResult *__restrict__ res, uint16_t *__restrict__ slots, GzEvent *__restrict__ events)
{
    __shared__ GzTables T;
    const GzJob j = jobs[blockIdx.x];
    GzState st = states[j.chunk];
    gz_run(in, nBytes, fin, st, j.target, j.limit, slots + (size_t)j.chunk * GZ_SLOT, events + (size_t)j.chunk * GZ_EVENTS, T, res[j.chunk]);
}

struct GzPiece { uint32_t chunk, n, minM, pad; uint64_t at; };    // accepted output: slot `chunk`, n symbols, call output offset `at`

// out: the 32 KiB window before the call, then the call's output.  Symbol v of a piece at offset `at`: a byte (v < 256), or byte
// v - 256 of the 32 KiB before the piece, i.e. out[at + v - 256]; markers below minM reach before the member's first byte.
__device__ __forceinline__ void gz_put(const GzPiece &p, const uint16_t *slot, uint32_t i, uint8_t *out, unsigned long long *err)
{
    const uint16_t v = slot[i];
    uint8_t b;
    if (v < 256) b = (uint8_t)v;
    else if (v - 256u < p.minM) { atomicMin(err, (unsigned long long)(p.at + i)); b = 0; }
    else b = out[p.at + (v - 256u)];
    out[GZ_WIN + p.at + i] = b;
}

// the last 32 KiB of every piece, piece after piece: afterwards the window of every piece is resolved
__global__ void __launch_bounds__(1024)
k_gz_window(const GzPiece *__restrict__ pieces, uint32_t nPieces, const uint16_t *__restrict__ slots, uint8_t *__restrict__ out,
            unsigned long long *__restrict__ err)
{
    for (uint32_t k = 0; k < nPieces; ++k) {
        const GzPiece p = pieces[k];
        const uint16_t *slot = slots + (size_t)p.chunk * GZ_SLOT;
        for (uint32_t i = (p.n > GZ_WIN ? p.n - GZ_WIN : 0) + threadIdx.x; i < p.n; i += blockDim.x) gz_put(p, slot, i, out, err);
        __syncthreads();
    }
}

__global__ void k_gz_resolve(const GzPiece *__restrict__ pieces, const uint16_t *__restrict__ slots, uint8_t *__restrict__ out,
                             unsigned long long *__restrict__ err)
{
    const GzPiece p = pieces[blockIdx.y];
    const uint16_t *slot = slots + (size_t)p.chunk * GZ_SLOT;
    const uint32_t end = p.n > GZ_WIN ? p.n - GZ_WIN : 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < end; i += gridDim.x * blockDim.x) gz_put(p, slot, i, out, err);
}

// CRC-32 of each piece [off[k], off[k + 1]) of the output
__global__ void k_gz_crc(const uint8_t *__restrict__ data, const unsigned long long *__restrict__ off, uint32_t nPieces, uint32_t *__restrict__ crc)
{
    __shared__ uint32_t tab[256];
    for (uint32_t t = threadIdx.x; t < 256; t += blockDim.x) {
        uint32_t c = t;
        for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        tab[t] = c;
    }
    __syncthreads();
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nPieces) return;
    uint32_t c = 0xffffffffu;
    for (uint64_t i = off[k]; i < off[k + 1]; ++i) c = tab[(c ^ data[i]) & 0xff] ^ (c >> 8);
    crc[k] = ~c;
}

}  // namespace

struct mp_gunzip {
    mp_context *ctx = nullptr;
    uint64_t maxIn = 0; uint32_t maxChunks = 0;
    DevBuf dIn, dCand, dStates, dJobs, dRes, dSlots, dEvents, dPieces, dOut, dWin, dErr, dCrcOff, dCrc;
    PinnedBuf<GzResult> hRes; PinnedBuf<GzState> hStates; PinnedBuf<GzJob> hJobs; PinnedBuf<unsigned long long> hCand;
    PinnedBuf<GzEvent> hEv; PinnedBuf<GzPiece> hPieces; PinnedBuf<unsigned long long> hCrcOff; PinnedBuf<uint32_t> hCrc;
    GzState resume{};                 // where the next call starts (bit relative to the next call's first byte)
    uint64_t outTotal = 0;            // bytes produced by earlier calls
    uint64_t memberStart = 0;         // absolute output offset of the current member's first byte
    uint32_t memberCrc = 0;           // CRC-32 of the current member's bytes so far (earlier calls)
    bool failed = false, finished = false;
    mp_gunzip_stats_t stats{};
};

static int gz_fail(mp_gunzip *g, const char *what)
{
    g->failed = true;
    mp_set_error("mp_gunzip_run: %s", what);
    return MP_ERR_FORMAT;
}

extern "C" int mp_gunzip_open(mp_context *ctx, uint64_t maxIn, mp_gunzip **out)
{
    if (!ctx || !out || maxIn == 0 || maxIn > MP_GUNZIP_MAX_IN) { mp_set_error("mp_gunzip_open: bad argument"); return MP_ERR_ARG; }
    *out = nullptr;
    MP_CUDA(cudaSetDevice(ctx->device));
    mp_gunzip *g = new mp_gunzip;
    g->ctx = ctx; g->maxIn = maxIn;
    g->maxChunks = (uint32_t)((maxIn + GZ_CHUNK - 1) / GZ_CHUNK);
    const uint64_t nc = g->maxChunks;
    if (g->dIn.reserve(maxIn + 8) || g->dCand.reserve(nc * 8) || g->dStates.reserve(nc * sizeof(GzState)) || g->dJobs.reserve(nc * sizeof(GzJob)) ||
        g->dRes.reserve(nc * sizeof(GzResult)) || g->dSlots.reserve(nc * GZ_SLOT * 2) || g->dEvents.reserve(nc * GZ_EVENTS * sizeof(GzEvent)) ||
        g->dPieces.reserve(nc * sizeof(GzPiece)) || g->dWin.reserve(GZ_WIN) || g->dErr.reserve(8) ||
        g->hRes.resize(nc) || g->hStates.resize(nc) || g->hJobs.resize(nc) || g->hCand.resize(nc) || g->hPieces.resize(nc)) {
        delete g; return MP_ERR_CUDA;
    }
    g->resume.mode = GZ_M_HEADER; g->resume.first = 1;
    *out = g;
    return 0;
}

extern "C" void mp_gunzip_close(mp_gunzip *g)
{
    if (!g) return;
    cudaSetDevice(g->ctx->device);
    for (DevBuf *b : { &g->dIn, &g->dCand, &g->dStates, &g->dJobs, &g->dRes, &g->dSlots, &g->dEvents, &g->dPieces, &g->dOut, &g->dWin, &g->dErr,
                       &g->dCrcOff, &g->dCrc }) b->release();
    delete g;
}

extern "C" int mp_gunzip_stats(mp_gunzip *g, mp_gunzip_stats_t *s)
{
    if (!g || !s) { mp_set_error("mp_gunzip_stats: bad argument"); return MP_ERR_ARG; }
    *s = g->stats;
    return 0;
}

extern "C" int mp_gunzip_run(mp_gunzip *g, const uint8_t *src, uint64_t n, int fin, uint8_t *dst, uint64_t dstCap, uint64_t *consumed,
                             uint64_t *produced, int *done)
{
    if (!g || !consumed || !produced || !done || (n && !src) || !dst || dstCap < MP_GUNZIP_MIN_DST || n > g->maxIn) {
        mp_set_error("mp_gunzip_run: bad argument (n must be <= maxIn of mp_gunzip_open, dstCap >= MP_GUNZIP_MIN_DST)");
        return MP_ERR_ARG;
    }
    *consumed = 0; *produced = 0; *done = 0;
    if (g->failed) { mp_set_error("mp_gunzip_run: the stream already failed"); return MP_ERR_FORMAT; }
    if (g->finished) { *done = 1; return 0; }
    const double t0 = mp_now_ms();
    mp_context *ctx = g->ctx;
    MP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    mp_gunzip_stats_t S{};
    if (g->dOut.reserve(GZ_WIN + dstCap)) return MP_ERR_CUDA;
    if (n) MP_CUDA(cudaMemcpyAsync(g->dIn.p, src, n, cudaMemcpyHostToDevice, st));
    MP_CUDA(cudaMemcpyAsync(g->dOut.p, g->dWin.p, GZ_WIN, cudaMemcpyDeviceToDevice, st));
    const unsigned long long noErr = ~0ull;
    MP_CUDA(cudaMemcpyAsync(g->dErr.p, &noErr, 8, cudaMemcpyHostToDevice, st));

    // ---- chunks and their candidate starts ----
    const uint32_t nRanges = n ? (uint32_t)((n + GZ_CHUNK - 1) / GZ_CHUNK) : 1;
    S.chunks = nRanges;
    std::vector<uint32_t> chunkOf;     // chunk list: slot index = position in this list
    std::vector<uint64_t> startBit;
    chunkOf.push_back(0); startBit.push_back(g->resume.bit);
    if (nRanges > 1) {
        (++g_mp_launches), k_gz_find<<<nRanges - 1, GZ_FIND_THREADS, 0, st>>>(g->dIn.as<uint8_t>(), n, nRanges, g->dCand.as<unsigned long long>());
        MP_CUDA(cudaGetLastError());
        MP_CUDA(cudaMemcpyAsync(g->hCand.data() + 1, g->dCand.as<unsigned long long>() + 1, (nRanges - 1) * 8ull, cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaStreamSynchronize(st));
        for (uint32_t r = 1; r < nRanges; ++r) {
            const unsigned long long c = g->hCand[r];
            const uint64_t lo = (uint64_t)r * GZ_CHUNK * 8, hi = std::min((uint64_t)(r + 1) * GZ_CHUNK, n) * 8;
            S.candidates_tested += (c == ~0ull ? hi : c + 1) - lo;
            if (c == ~0ull || c <= g->resume.bit) { S.merged++; continue; }
            S.candidates++;
            chunkOf.push_back(r); startBit.push_back(c);
        }
    }
    const uint32_t m = (uint32_t)chunkOf.size();
    for (uint32_t i = 0; i < m; ++i) {
        GzState s{};
        if (i == 0) s = g->resume;
        else { s.bit = startBit[i]; s.mode = GZ_M_BLOCK; }
        g->hStates[i] = s;
    }
    MP_CUDA(cudaMemcpyAsync(g->dStates.p, g->hStates.data(), m * sizeof(GzState), cudaMemcpyHostToDevice, st));

    // ---- decode rounds and the verified walk ----
    const GzState *dStates = g->dStates.as<GzState>();
    GzResult *dRes = g->dRes.as<GzResult>();
    uint16_t *dSlots = g->dSlots.as<uint16_t>();
    GzEvent *dEv = g->dEvents.as<GzEvent>();
    std::vector<uint32_t> pending(m), limitOf(m, GZ_SLOT);
    for (uint32_t i = 0; i < m; ++i) pending[i] = i;
    uint32_t cur = 0;                   // first chunk whose output is not yet accepted; its start is verified
    uint64_t P = 0;                     // bytes accepted in this call
    uint64_t memberStart = g->memberStart;
    const uint64_t A0 = g->outTotal;
    struct Ev { uint32_t kind, crc, isize; uint64_t at; };
    std::vector<Ev> evs;                // member starts and trailers of this call in stream order (call offsets)
    int endKind = 0;                    // 0 running, GZ_S_* that ended the call
    uint64_t decErrAt = ~0ull;
    GzState endState{};
    while (!endKind) {
        const uint32_t nJobs = (uint32_t)pending.size();
        for (uint32_t k = 0; k < nJobs; ++k) {
            const uint32_t c = pending[k];
            g->hJobs[k] = GzJob{ c, limitOf[c], c + 1 < m ? startBit[c + 1] : ~0ull };
        }
        MP_CUDA(cudaMemcpyAsync(g->dJobs.p, g->hJobs.data(), nJobs * sizeof(GzJob), cudaMemcpyHostToDevice, st));
        (++g_mp_launches), k_gz_decode<<<nJobs, 1, 0, st>>>(g->dIn.as<uint8_t>(), n, fin, g->dJobs.as<GzJob>(), dStates, dRes, dSlots, dEv);
        MP_CUDA(cudaGetLastError());
        S.rounds++;
        const uint32_t lo = *std::min_element(pending.begin(), pending.end()), hi = *std::max_element(pending.begin(), pending.end());
        MP_CUDA(cudaMemcpyAsync(g->hRes.data() + lo, dRes + lo, (hi - lo + 1) * sizeof(GzResult), cudaMemcpyDeviceToHost, st));
        MP_CUDA(cudaStreamSynchronize(st));
        pending.clear();
        uint32_t nPieces = 0;
        while (!endKind && pending.empty()) {
            const GzResult &r = g->hRes[cur];
            if (P + r.nOut > dstCap) {                       // decode this chunk again, up to what dst still holds
                limitOf[cur] = (uint32_t)(dstCap - P);
                if (limitOf[cur] == 0) { endKind = GZ_S_FULL; endState = g->hStates[cur]; break; }
                pending.push_back(cur);
                break;
            }
            // accept the output: pieces are resolved in order after this round
            uint32_t minM = 0;
            if (memberStart + GZ_WIN > A0 + P) minM = (uint32_t)std::min<uint64_t>(GZ_WIN, memberStart + GZ_WIN - (A0 + P));
            if (r.nOut) g->hPieces[nPieces++] = GzPiece{ cur, r.nOut, minM, 0, P };
            if (r.nEvents) {
                if (g->hEv.resize(r.nEvents)) return MP_ERR_CUDA;
                MP_CUDA(cudaMemcpyAsync(g->hEv.data(), dEv + (size_t)cur * GZ_EVENTS, r.nEvents * sizeof(GzEvent), cudaMemcpyDeviceToHost, st));
                MP_CUDA(cudaStreamSynchronize(st));
                for (uint32_t e = 0; e < r.nEvents; ++e) {
                    const GzEvent &E = g->hEv[e];
                    if (E.kind == GZ_E_START) memberStart = A0 + P + E.out;
                    evs.push_back(Ev{ E.kind, E.crc, E.isize, P + E.out });
                }
            }
            P += r.nOut;
            switch (r.status) {
            case GZ_S_TARGET:
                if (cur + 1 < m && r.end.bit == startBit[cur + 1]) { cur++; break; }   // the next chunk started where this one ended
                // a false candidate (or none reached): decode the next chunk again from this end
                S.false_candidates++;
                cur++;
                g->hStates[cur] = r.end;
                MP_CUDA(cudaMemcpyAsync(g->dStates.as<GzState>() + cur, &g->hStates[cur], sizeof(GzState), cudaMemcpyHostToDevice, st));
                pending.push_back(cur);
                break;
            case GZ_S_FULL:
                if (P >= dstCap || limitOf[cur] < GZ_SLOT) { endKind = GZ_S_FULL; endState = r.end; break; }
                S.overflows++;
                g->hStates[cur] = r.end;
                MP_CUDA(cudaMemcpyAsync(g->dStates.as<GzState>() + cur, &g->hStates[cur], sizeof(GzState), cudaMemcpyHostToDevice, st));
                pending.push_back(cur);
                break;
            case GZ_S_ERROR: endKind = GZ_S_ERROR; decErrAt = P; endState = r.end; break;
            default: endKind = (int)r.status; endState = r.end; break;      // GZ_S_NEED, GZ_S_END
            }
        }
        if (nPieces) {
            MP_CUDA(cudaMemcpyAsync(g->dPieces.p, g->hPieces.data(), nPieces * sizeof(GzPiece), cudaMemcpyHostToDevice, st));
            (++g_mp_launches), k_gz_window<<<1, 1024, 0, st>>>(g->dPieces.as<GzPiece>(), nPieces, dSlots, g->dOut.as<uint8_t>(),
                                                                g->dErr.as<unsigned long long>());
            MP_CUDA(cudaGetLastError());
            (++g_mp_launches), k_gz_resolve<<<dim3(32, nPieces), 256, 0, st>>>(g->dPieces.as<GzPiece>(), dSlots, g->dOut.as<uint8_t>(),
                                                                               g->dErr.as<unsigned long long>());
            MP_CUDA(cudaGetLastError());
        }
    }
    // ---- CRC-32 per member: 32 KiB pieces of the output, cut at member starts and ends ----
    std::vector<uint64_t> cuts{ 0, P };
    for (const Ev &e : evs) cuts.push_back(e.at);
    std::sort(cuts.begin(), cuts.end());
    cuts.erase(std::unique(cuts.begin(), cuts.end()), cuts.end());
    std::vector<unsigned long long> off;
    for (size_t k = 0; k + 1 < cuts.size(); ++k)
        for (uint64_t a = cuts[k]; a < cuts[k + 1]; a += GZ_CRC_PIECE) off.push_back(a);
    off.push_back(P);
    const uint32_t nCrc = (uint32_t)off.size() - 1;
    unsigned long long errMarker = ~0ull;
    MP_CUDA(cudaMemcpyAsync(&errMarker, g->dErr.p, 8, cudaMemcpyDeviceToHost, st));
    if (nCrc) {
        if (g->dCrcOff.reserve(off.size() * 8) || g->dCrc.reserve(nCrc * 4ull) || g->hCrcOff.resize(off.size()) || g->hCrc.resize(nCrc)) return MP_ERR_CUDA;
        std::copy(off.begin(), off.end(), g->hCrcOff.data());
        MP_CUDA(cudaMemcpyAsync(g->dCrcOff.p, g->hCrcOff.data(), off.size() * 8, cudaMemcpyHostToDevice, st));
        (++g_mp_launches), k_gz_crc<<<(nCrc + 127) / 128, 128, 0, st>>>(g->dOut.as<uint8_t>() + GZ_WIN, g->dCrcOff.as<unsigned long long>(), nCrc,
                                                                         g->dCrc.as<uint32_t>());
        MP_CUDA(cudaGetLastError());
        MP_CUDA(cudaMemcpyAsync(g->hCrc.data(), g->dCrc.p, nCrc * 4ull, cudaMemcpyDeviceToHost, st));
    }
    MP_CUDA(cudaStreamSynchronize(st));
    // the first failure in output order: a marker reaching before its member, a decode error, or a trailer that does not match (a
    // trailer at the same offset as a marker comes first: zlib checks it before it decodes the next member)
    uint64_t errAt = errMarker;
    const char *errWhat = errMarker != ~0ull ? "invalid distance too far back" : nullptr;
    if (decErrAt < errAt) { errAt = decErrAt; errWhat = "invalid compressed data"; }
    uint32_t crc = g->memberCrc;
    uint64_t mStart = g->memberStart;               // absolute
    uint32_t k = 0;
    auto advance = [&](uint64_t to) { for (; k < nCrc && off[k + 1] <= to; ++k) crc = mp_crc32_combine(crc, g->hCrc[k], off[k + 1] - off[k]); };
    for (const Ev &e : evs) {
        if (e.at > errAt) break;
        advance(e.at);
        if (e.kind == GZ_E_START) { mStart = A0 + e.at; crc = 0; continue; }
        if (e.crc != crc || e.isize != (uint32_t)(A0 + e.at - mStart)) {
            errAt = e.at; errWhat = e.crc != crc ? "incorrect data check" : "incorrect length check";
            break;
        }
        S.members++;
    }
    advance(P);
    if (errWhat == nullptr && endKind == GZ_S_NEED && fin) { errAt = P; errWhat = "unexpected end of file"; }
    const uint64_t keep = errWhat ? std::min<uint64_t>(errAt, P) : P;
    if (keep) MP_CUDA(cudaMemcpyAsync(dst, g->dOut.as<uint8_t>() + GZ_WIN, keep, cudaMemcpyDeviceToHost, st));
    MP_CUDA(cudaStreamSynchronize(st));
    *produced = keep;
    S.out_bytes = keep;
    S.ms_total = (float)(mp_now_ms() - t0);
    if (errWhat) { S.in_bytes = 0; g->stats = S; return gz_fail(g, errWhat); }
    // ---- state for the next call: window, member, resume point ----
    MP_CUDA(cudaMemcpyAsync(g->dWin.p, g->dOut.as<uint8_t>() + P, GZ_WIN, cudaMemcpyDeviceToDevice, st));
    g->memberCrc = crc; g->memberStart = mStart; g->outTotal = A0 + P;
    *consumed = endState.bit >> 3;
    g->resume = endState;
    g->resume.bit = endState.bit & 7;
    S.in_bytes = *consumed;
    if (endKind == GZ_S_END) { g->finished = true; *done = 1; }
    MP_CUDA(cudaStreamSynchronize(st));
    g->stats = S;
    return 0;
}
