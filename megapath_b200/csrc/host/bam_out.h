// bam_out.h -- BAM output of the soap4 driver (-b): record content, MAPQ and tags as the reference writes them.
//
// Mirrors (reference file:line, relative to soap4/):
//   header                         SAMOutputHeaderConstruct             SAM.cpp:83-134
//   record layout / tags           initializeSAMAlgnmt, initializeSAMAlgnmt2, AssignCigarStrToSAMIU   BGS-IO.cpp:137-160, 434-677
//   proper pairs                   pairDeepDPOutputSAMAPI               BGS-IO.cpp:2093-2800
//   not properly paired            unproperlypairDPOutputSAMAPI         BGS-IO.cpp:1448-1915
//   boundary trimming              getChrAndPosWithBoundaryCheckDP, BoundaryCheckDP   BGS-IO.cpp:219-432
//   cigar / MD / mismatch counts   convertToCigarStr, getMisInfoForDP, readLengthWithCigar   PE.cpp:381-446, 459-625; BGS-IO.cpp:1917-1947
//   MAPQ                           bwaLikeSingleQualScore, bwaLikePairQualScore, getMapQualScoreForDP(2), getMapQualScoreForSingleDP,
//                                  getMapQualScoreForPair               BGS-IO.cpp:679-980
// The BGZF container: BgzfWriter writes the header and the EOF marker with zlib, and copies through blocks compressed elsewhere --
// by the device (mp_bgzf_compress, csrc/mp_bgzf.cu) in the driver's default -b path, or by the formatting threads with zlib
// (compress_all) under MP_HOST_IO=1 (the reference links samtools 0.1.18 for it).  Block boundaries are free, the decoded byte
// stream is what must match.
#pragma once
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <zlib.h>
#include <string>
#include <vector>

static const uint64_t NOT_ALIGNED = ~0ull;

// ------------------------------------------------------------------------------------------------ BGZF
struct BgzfWriter {
    FILE *f = nullptr; std::vector<uint8_t> buf;
    bool open(const std::string &path) { f = fopen(path.c_str(), "wb"); buf.reserve(0xff00); return f != nullptr; }
    // one BGZF block (<= 0xff00 input bytes) appended to `out`
    static void compress_block(const uint8_t *data, size_t len, std::vector<uint8_t> &out) {
        const size_t at = out.size();
        out.resize(at + 0x10000 + 64);
        uint8_t *o = out.data() + at;
        z_stream zs; memset(&zs, 0, sizeof zs);
        deflateInit2(&zs, Z_DEFAULT_COMPRESSION, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
        zs.next_in = (Bytef *)data; zs.avail_in = (uInt)len; zs.next_out = o + 18; zs.avail_out = 0x10000 + 64 - 18 - 8;
        deflate(&zs, Z_FINISH);
        size_t clen = zs.total_out; deflateEnd(&zs);
        static const uint8_t hdr[16] = { 31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0 };
        memcpy(o, hdr, 16);
        uint16_t bsize = (uint16_t)(clen + 25); o[16] = bsize & 0xff; o[17] = bsize >> 8;
        uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), data, (uInt)len), isz = (uint32_t)len;
        memcpy(o + 18 + clen, &crc, 4); memcpy(o + 22 + clen, &isz, 4);
        out.resize(at + clen + 26);
    }
    // any number of bytes -> a run of complete BGZF blocks in memory (formatting threads compress their own chunks;
    // BGZF blocks are independent, so the concatenation of the chunks' blocks is a valid stream)
    static void compress_all(const uint8_t *data, size_t len, std::vector<uint8_t> &out) {
        for (size_t at = 0; at < len; at += 0xff00) compress_block(data + at, len - at < 0xff00 ? len - at : 0xff00, out);
    }
    void flush_block(const uint8_t *data, size_t len) {
        std::vector<uint8_t> out; compress_block(data, len, out);
        fwrite(out.data(), 1, out.size(), f);
    }
    // blocks compressed elsewhere: close the block in progress, then copy them through
    void write_blocks(const std::vector<uint8_t> &blocks) {
        if (blocks.empty()) return;
        if (!buf.empty()) { flush_block(buf.data(), buf.size()); buf.clear(); }
        fwrite(blocks.data(), 1, blocks.size(), f);
    }
    void write(const void *p, size_t n) {
        const uint8_t *s = (const uint8_t *)p;
        while (n) {
            size_t room = 0xff00 - buf.size(), k = n < room ? n : room;
            buf.insert(buf.end(), s, s + k); s += k; n -= k;
            if (buf.size() >= 0xff00) { flush_block(buf.data(), buf.size()); buf.clear(); }
        }
    }
    void close() {
        if (!f) return;
        if (!buf.empty()) { flush_block(buf.data(), buf.size()); buf.clear(); }
        flush_block(nullptr, 0);                                  // EOF marker block
        fclose(f); f = nullptr;
    }
};

struct BamRecord {
    int32_t tid = -1, pos = -1, mtid = -1, mpos = -1, isize = 0;
    uint32_t flag = 0, mapq = 0, l_qseq = 0, n_cigar = 0;
    std::vector<uint8_t> data;                                    // qname, cigar, seq, qual, aux
    void put32(uint32_t v) { uint8_t b[4]; memcpy(b, &v, 4); data.insert(data.end(), b, b + 4); }
    void aux_i(const char *tag, int32_t v) { data.push_back(tag[0]); data.push_back(tag[1]); data.push_back('i'); put32((uint32_t)v); }
    void aux_z(const char *tag, const char *s, size_t len) { data.push_back(tag[0]); data.push_back(tag[1]); data.push_back('Z'); data.insert(data.end(), s, s + len); data.push_back(0); }
};

struct BamWriter {
    BgzfWriter z;
    std::vector<uint8_t> *capture = nullptr;                       // when set, encoded records are appended here instead of being compressed
    bool open(const std::string &path, const std::string &text, const std::vector<std::string> &names, const std::vector<uint32_t> &lens) {
        if (!z.open(path)) return false;
        z.write("BAM\1", 4);
        int32_t l = (int32_t)text.size(); z.write(&l, 4); z.write(text.data(), text.size());
        int32_t n = (int32_t)names.size(); z.write(&n, 4);
        for (size_t i = 0; i < names.size(); ++i) {
            int32_t ln = (int32_t)names[i].size() + 1; z.write(&ln, 4); z.write(names[i].c_str(), ln);
            int32_t lr = (int32_t)lens[i]; z.write(&lr, 4);
        }
        return true;
    }
    void write(const BamRecord &r, size_t l_qname) {
        const uint32_t bin = 0;                                   // bam_reg2bin(0, 0) == 0 (end wraps): the reference never updates it
        int32_t block = 32 + (int32_t)r.data.size();
        uint32_t x[8];
        x[0] = (uint32_t)r.tid; x[1] = (uint32_t)r.pos; x[2] = (bin << 16) | ((r.mapq & 0xff) << 8) | (uint32_t)(l_qname & 0xff);
        x[3] = (r.flag << 16) | (r.n_cigar & 0xffff); x[4] = r.l_qseq; x[5] = (uint32_t)r.mtid; x[6] = (uint32_t)r.mpos; x[7] = (uint32_t)r.isize;
        if (capture) {
            const uint8_t *b4 = (const uint8_t *)&block, *xb = (const uint8_t *)x;
            capture->insert(capture->end(), b4, b4 + 4); capture->insert(capture->end(), xb, xb + 32);
            capture->insert(capture->end(), r.data.begin(), r.data.end());
        } else { z.write(&block, 4); z.write(x, 32); z.write(r.data.data(), r.data.size()); }
    }
    void write_raw(const std::vector<uint8_t> &bytes) { if (!bytes.empty()) z.write(bytes.data(), bytes.size()); }
    void write_blocks(const std::vector<uint8_t> &blocks) { z.write_blocks(blocks); }
    void close() { z.close(); }
};

// ------------------------------------------------------------------------------------------------ helpers
static inline int write_num(long long v, char *s) { return sprintf(s, "%lld", v); }

// convertToCigarStr (PE.cpp:381-446)
static std::string convert_cigar(const char *sp, int *deletedEnd = nullptr)
{
    std::string out; int cur = 0, curM = 0; char tmp[32];
    if (deletedEnd) *deletedEnd = 0;
    const size_t n = strlen(sp);
    for (size_t i = 0; i < n; ++i) {
        char c = sp[i];
        if (c >= '0' && c <= '9') { cur = cur * 10 + (c - '0'); continue; }
        if (c == 'M' || c == 'm') { curM += cur; cur = 0; continue; }
        if (c == 'D' && ((out.empty() && curM == 0) || i == n - 1)) {       // leading / trailing deletion is ignored
            if (i == n - 1 && deletedEnd) *deletedEnd = curM;
            continue;                                                       // (currInt is NOT reset, as in the reference)
        }
        if (c == 'D' || c == 'I' || c == 'S') {
            if (curM > 0) { write_num(curM, tmp); out += tmp; out += 'M'; curM = 0; }
            write_num(cur, tmp); out += tmp; out += c; cur = 0;
        }
    }
    if (curM > 0) { write_num(curM, tmp); out += tmp; out += 'M'; }
    return out;
}
// readLengthWithCigar (BGS-IO.cpp:1917-1947)
static int ref_len_of_cigar(const char *cigar)
{
    int len = 0, x = 0; char op = 0;
    for (const char *p = cigar; *p;) {
        x = 0;
        while (*p >= '0' && *p <= '9') { x = x * 10 + (*p - '0'); p++; }
        op = *p; p++;
        if (op == 'M' || op == 'm' || op == 'D') len += x;
    }
    if (op == 'D') len -= x;
    return len;
}

struct AnnEx {                                                    // what the BAM path needs beyond Annotation
    const uint8_t *pac = nullptr;                                 // packed text (only for MD strings, -p)
    std::vector<uint64_t> seqEnd;                                 // seqOffset[i].endPos = start + length - 1 (.ann)
};

// BoundaryCheckDP (BGS-IO.cpp:219-391) -> trimmed amount (+ left, - right), corrected position, new special cigar
static long long boundary_check_dp(uint64_t pacPos, uint64_t chrEndPos, long long readLength, const char *cigar, uint64_t segmentEndPos,
                                   uint64_t &correctedPac, std::string &newCigar)
{
    newCigar.clear();
    if (pacPos + readLength * 2 <= chrEndPos + 1 && pacPos + readLength * 2 <= segmentEndPos + 1) return 0;
    segmentEndPos = chrEndPos < segmentEndPos ? chrEndPos : segmentEndPos;
    std::string leftBuf, rightBuf; char buffer[64];
    long long leftLen = 0, rightLen = 0, rightOff = 0, leftS = 0, rightS = 0;
    uint64_t refPos = pacPos;
    for (const char *p = cigar; *p;) {
        long long num = 0;
        while (*p <= '9') { num = num * 10 + (*p - '0'); p++; }
        char op = *p++;
        if (op == 'S') {
            sprintf(buffer, "%dS", (int)num);
            if (refPos <= segmentEndPos) { leftBuf += buffer; leftS += num; } else { rightBuf += buffer; rightS += num; }
        } else if (op == 'M' || op == 'm') {
            if (refPos > segmentEndPos) { rightLen += num; sprintf(buffer, "%d%c", (int)num, op); rightBuf += buffer; }
            else if (refPos + num <= segmentEndPos + 1) { leftLen += num; sprintf(buffer, "%d%c", (int)num, op); leftBuf += buffer; }
            else {
                leftLen += segmentEndPos - refPos + 1; sprintf(buffer, "%d%c", (int)(segmentEndPos - refPos + 1), op); leftBuf += buffer;
                rightLen += num - segmentEndPos + refPos - 1; sprintf(buffer, "%d%c", (int)(num - segmentEndPos + refPos - 1), op); rightBuf += buffer;
            }
            refPos += num;
        } else if (op == 'D') {
            sprintf(buffer, "%dD", (int)num);
            if (refPos > segmentEndPos) { if (rightBuf.empty()) rightOff = num; else rightBuf += buffer; }
            else if (refPos + num <= segmentEndPos + 1) leftBuf += buffer;
            else {
                sprintf(buffer, "%dD", (int)(segmentEndPos - refPos + 1)); leftBuf += buffer;
                sprintf(buffer, "%dD", (int)(num - segmentEndPos + refPos - 1));
                if (rightBuf.empty()) rightOff = num - segmentEndPos + refPos - 1; else rightBuf += buffer;
            }
            refPos += num;
        } else if (op == 'I') {
            if (refPos == chrEndPos + 1) { }
            else if (refPos <= segmentEndPos) { leftLen += num; sprintf(buffer, "%dI", (int)num); leftBuf += buffer; }
            else { rightLen += num; sprintf(buffer, "%dI", (int)num); rightBuf += buffer; }
        }
    }
    if (!leftLen || !rightLen) return 0;
    if (leftLen >= rightLen) {
        sprintf(buffer, "%dS", (int)(readLength - leftLen - leftS)); newCigar = leftBuf + buffer;
        correctedPac = pacPos;
        return -(readLength - leftLen - leftS);
    }
    sprintf(buffer, "%dS", (int)(readLength - rightLen - rightS)); newCigar = buffer + rightBuf;
    correctedPac = segmentEndPos + 1 + rightOff;
    return readLength - rightLen - rightS;
}

// getMisInfoForDP (PE.cpp:459-625): MD string + mismatch / gap counts from the special cigar
struct MisInfo { std::string md; int numMismatch = 0, gapOpen = 0, gapExt = 0, avgMismatchQual = 20; };
static MisInfo mis_info_for_dp(const AnnEx &ax, const char *qualities, unsigned queryLength, uint64_t pos, int strand, const char *sp, long long trim)
{
    MisInfo m; char tmp[32];
    // the reference advances `query` (unused below) and `pos` by the trimmed amount, never `qualities` (PE.cpp:465-487)
    if (trim > 0) pos += trim;
    (void)queryLength; (void)strand;
    auto tbase = [&](uint64_t p) -> char { return ax.pac ? "ACGT"[(ax.pac[p >> 2] >> ((3 - (p & 3)) << 1)) & 3] : 'N'; };
    int cur = 0, curMatch = 0, qPos = 0; uint64_t tPos = pos; double sumQ = 0.0;
    const int l = (int)strlen(sp);
    for (int i = 0; i < l; ++i) {
        char c = sp[i];
        if (c >= '0' && c <= '9') { cur = cur * 10 + (c - '0'); continue; }
        switch (c) {
        case 'M': curMatch += cur; qPos += cur; tPos += cur; cur = 0; break;
        case 'm':
            write_num(curMatch, tmp); m.md += tmp; m.md += tbase(tPos); sumQ += qualities[qPos];
            for (int j = 1; j < cur; ++j) { m.md += '0'; m.md += tbase(tPos + j); sumQ += qualities[qPos + j]; }
            qPos += cur; tPos += cur; m.numMismatch += cur; curMatch = 0; cur = 0; break;
        case 'I': qPos += cur; m.gapOpen++; m.gapExt += cur; cur = 0; break;
        case 'D':
            if (i == l - 1) break;
            write_num(curMatch, tmp); m.md += tmp; m.md += '^';
            for (int j = 0; j < cur; ++j) m.md += tbase(tPos + j);
            tPos += cur; m.gapOpen++; m.gapExt += cur; curMatch = 0; cur = 0; break;
        case 'S': qPos += cur; cur = 0; break;
        }
    }
    write_num(curMatch, tmp); m.md += tmp;
    if (m.numMismatch > 0) m.avgMismatchQual = (int)(sumQ / m.numMismatch);
    return m;
}

// ------------------------------------------------------------------------------------------------ MAPQ
static int g_log_n[256];
static void bwase_initialize() { g_log_n[0] = 0; for (int i = 1; i < 256; ++i) g_log_n[i] = (int)(4.343 * log((double)i) + 0.5); }
static const double mapping_score[6][2] = { {1.0, 1.0}, {0.875, 0.85}, {0.75, 0.7}, {0.625, 0.55}, {0.475, 0.4}, {0.325, 0.25} };
static const float penalty_score_avg_mis_qual[41] = { 3, 2.85, 2.71, 2.57, 2.43, 2.3, 2.17, 2.04, 1.92, 1.8, 1.69, 1.58, 1.47, 1.37, 1.27, 1.17, 1.08, 0.99, 0.91, 0.83, 0.75, 0.68, 0.61, 0.54, 0.48, 0.42, 0.37, 0.32, 0.27, 0.23, 0.19, 0.15, 0.12, 0.09, 0.07, 0.05, 0.03, 0.02, 0.01, 0, 0 };
static float penalty_ratio_x1(int x1)
{
    static const float head[66] = { 1, 0.5, 0.33, 0.25, 0.2, 0.17, 0.14, 0.13, 0.11, 0.1, 0.09, 0.08, 0.08, 0.07, 0.07, 0.06, 0.06, 0.06, 0.05, 0.05, 0.05, 0.05,
        0.04, 0.04, 0.04, 0.04, 0.04, 0.04, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.03, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02,
        0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02, 0.02 };
    if (x1 > 100) x1 = 100;
    return x1 < 66 ? head[x1] : 0.01f;
}
static int bwa_like_single(int x0, int x1)
{
    if (x0 > 1) return 0;
    if (x1 == 0) return 37;
    x1 = x1 > 255 ? 255 : x1;
    int n = g_log_n[x1];
    return 23 < n ? 0 : 23 - n;
}
static void bwa_like_pair(int x0_0, int x1_0, int x0_1, int x1_1, int op_score, int op_num, int subop_score, int subop_num, int readlen_0, int readlen_1, int *m0, int *m1)
{
    int mapq0 = bwa_like_single(x0_0, x1_0), mapq1 = bwa_like_single(x0_1, x1_1);
    op_score *= 10; subop_score *= 10;
    int mapq_p = 0;
    if (mapq0 > 0 && mapq1 > 0) { mapq_p = mapq0 + mapq1; if (mapq_p > 60) mapq_p = 60; mapq0 = mapq1 = mapq_p; }
    else {
        if (op_num == 1) {
            if (subop_num == 0) mapq_p = 29;
            else if (op_score - subop_score > (0.3 * ((readlen_0 + readlen_1) / 2))) mapq_p = 23;
            else { subop_num = subop_num > 255 ? 255 : subop_num; mapq_p = (op_score - subop_score) / 2 - g_log_n[subop_num]; if (mapq_p < 0) mapq_p = 0; }
        }
        if (mapq0 == 0) mapq0 = (mapq_p + 7 < mapq1) ? mapq_p + 7 : mapq1;
        if (mapq1 == 0) mapq1 = (mapq_p + 7 < mapq0) ? mapq_p + 7 : mapq0;
    }
    *m0 = mapq0; *m1 = mapq1;
}
static int mapq_for_dp(int n, int dpScore, int maxDPScore, int avgMismatchQual, int maxMAPQ, int minMAPQ)       // getMapQualScoreForDP
{
    if (n != 1) return minMAPQ;
    int di = 0;
    if (dpScore < maxDPScore) di = (int)((1.0 - (double)dpScore / maxDPScore) * 100.0 - 1.0) / 5 + 1;
    if (di > 5) di = 5;
    int qi = (avgMismatchQual - 1) / 20; if (qi > 1) qi = 1; else if (qi < 0) qi = 0;
    int s = (int)(maxMAPQ * mapping_score[di][qi]);
    return s < minMAPQ ? minMAPQ : s;
}
static int mapq_for_single_dp(int maxDPScore, int avgMismatchQual, int x0, int x1_t1, int x1_t2, int bestDPScore, int secondBestDPScore,
                              int maxMAPQ, int minMAPQ, int dpThres, int isBWALike)                                 // getMapQualScoreForSingleDP
{
    if (isBWALike) return bwa_like_single(x0, x1_t1 + x1_t2);
    if (x0 > 1 || x1_t1 > 0) return minMAPQ;
    float R1 = x1_t2 > 0 ? (float)(1.0 - ((float)(secondBestDPScore - dpThres)) / (0.7 * bestDPScore - dpThres)) : 1.0f;
    float R2 = penalty_ratio_x1(x1_t1 + x1_t2);
    float R3 = ((float)(bestDPScore - dpThres)) / (maxDPScore - dpThres);
    if (avgMismatchQual < 0) avgMismatchQual = 0; else if (avgMismatchQual > 40) avgMismatchQual = 40;
    int s = (int)(maxMAPQ * R1 * R2 * R3 - penalty_score_avg_mis_qual[avgMismatchQual]);
    return s < minMAPQ ? minMAPQ : s;
}

// ------------------------------------------------------------------------------------------------ record construction
// initializeSAMAlgnmt / initializeSAMAlgnmt2 (BGS-IO.cpp:434-677): qname, cigar, seq, qual, tags
struct ReadView { const std::string *name; const uint8_t *codes; const char *qual; int len; };

static void fill_seq_qual(BamRecord &r, const ReadView &rv, int strand)
{
    const int L = rv.len;
    static const uint8_t nt16[4] = { 1, 2, 4, 8 };
    std::vector<uint8_t> c(L);
    if (strand == 2) for (int i = 0; i < L; ++i) c[i] = 3 - rv.codes[L - 1 - i]; else for (int i = 0; i < L; ++i) c[i] = rv.codes[i];
    for (int i = 0; i + 1 < L; i += 2) r.data.push_back((uint8_t)((nt16[c[i]] << 4) | nt16[c[i + 1]]));
    if (L & 1) r.data.push_back((uint8_t)(nt16[c[L - 1]] << 4));
    if (strand == 2) for (int i = L - 1; i >= 0; --i) r.data.push_back((uint8_t)(rv.qual[i] - 33));
    else for (int i = 0; i < L; ++i) r.data.push_back((uint8_t)(rv.qual[i] - 33));
}
static void append_cigar_ops(BamRecord &r, const std::string &cigar)
{
    r.n_cigar = 0; int num = 0;
    for (char ch : cigar) {
        if (ch >= '0' && ch <= '9') num = num * 10 + (ch - '0');
        else if (num > 0) { uint32_t op = ch == 'M' ? 0 : ch == 'I' ? 1 : ch == 'D' ? 2 : 4; r.put32(((uint32_t)num << 4) | op); r.n_cigar++; num = 0; }
    }
}
static void init_unmapped(BamRecord &r, const ReadView &rv, int strand, const std::string &xa, const std::string &readGroup)
{
    r = BamRecord(); r.l_qseq = rv.len; r.mapq = 0;
    r.data.insert(r.data.end(), rv.name->c_str(), rv.name->c_str() + rv.name->size() + 1);
    fill_seq_qual(r, rv, strand);
    r.aux_z("RG", readGroup.c_str(), readGroup.size());
    if (!xa.empty()) r.aux_z("XA", xa.c_str(), xa.size());
}
static void init_mapped(BamRecord &r, const ReadView &rv, int strand, const std::string &xa, const std::string &cigar, int mismatchNum, int editDist,
                        int bestHitNum, int secBestHitNum, int gapOpenNum, int gapExtendNum, const std::string &md, int mapq,
                        const std::string &readGroup, bool printMDNM, int moduleId)
{
    r = BamRecord(); r.l_qseq = rv.len; r.mapq = (uint32_t)mapq;
    r.data.insert(r.data.end(), rv.name->c_str(), rv.name->c_str() + rv.name->size() + 1);
    append_cigar_ops(r, cigar);
    fill_seq_qual(r, rv, strand);
    r.aux_z("RG", readGroup.c_str(), readGroup.size());
    if (printMDNM && editDist >= 0) r.aux_i("NM", editDist);
    if (bestHitNum >= 0) r.aux_i("X0", bestHitNum);
    if (secBestHitNum >= 0) r.aux_i("X1", secBestHitNum);
    if (mismatchNum >= 0) r.aux_i("XM", mismatchNum);
    if (gapOpenNum >= 0) r.aux_i("XO", gapOpenNum);
    if (gapExtendNum >= 0) r.aux_i("XG", gapExtendNum);
    if (printMDNM && !md.empty()) r.aux_z("MD", md.c_str(), md.size());
    if (!xa.empty()) r.aux_z("XA", xa.c_str(), xa.size());
    if (moduleId != -1) r.aux_i("PH", moduleId);
}
