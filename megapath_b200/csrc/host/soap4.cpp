// soap4.cpp -- host driver with the reference soap4's command line, .ini semantics and MegaPath
// output (annotated interleaved FASTQ on stdout), calling the B200 hot path through the C-ABI of
// libmegapath_b200.so (include/megapath_b200.h).  Drop-in for the `soap4 pair ...` calls of
// runMegaPath.sh:136,199.
//
// Mirrors (reference file:line, relative to soap4/):
//   command line             parseInputArgs                     IniParam.cpp:542-942
//   .ini                     ParseIniFile                       IniParam.cpp:242-438
//   read loading             loadPairReadsKseq / appendToQueryArrays   QueryParser.cpp:160-260, kseq.h
//   batch loop, first-batch read-length detection / insert_low clamp    SOAP4.cpp:424-585
//   stage sequencing         soap3_dp_pair_align                alignment.cpp:29-355
//   per-pair best / FASTQ    outputDeepDPResult2, pairDeepDPOutputFastqAPI, unproperlypairDPOutputFastqAPI,
//                            decideTargetChr, getChrAndPos, getMappingFromHeader
//                            OutputDPResult.cpp:65-265; BGS-IO.cpp:163-190, 1312-1446, 1966-2091
//   unpaired bookkeeping     filterOutUnpairedSingleReads, DPSOutputUnpairedAlignment
//                            SeedPool.cpp:267-322; DV-DPfunctions.cpp:841-920
//   BAM output (-b)          bam_out.h
//
// Two I/O paths.  Plain FASTQ files with -F / -P (no -b): the driver only stages each batch's bytes in page-locked memory
// (stage_file / locate_records) and writes the finished text; records are indexed and packed, and the output text is composed, by
// kernels (mp_fastq_upload, mp_format_fastq; csrc/mp_fastq.cu; with -lsam host threads rewrite that text).  Everything else -- .gz, pipes, BAM, text that is not strict
// four-line FASTQ -- goes through the host parser (SeqReader, load_batch) and formatter (header_line, output_pair, output_unpaired)
// below, which are also what MP_HOST_IO=1 forces and what the device path is tested against.  With -b the formatting threads write
// raw BAM records and each worker has its own context compress them into BGZF members (mp_bgzf_compress, csrc/mp_bgzf.cu);
// MP_HOST_IO=1 keeps zlib on the formatting threads instead.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ctype.h>
#include <zlib.h>
#include <sys/stat.h>
#include <sys/mman.h>
#include <fcntl.h>
#include <unistd.h>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>
#include "megapath_b200.h"
#include "bam_out.h"

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// ------------------------------------------------------------------------------------------------
struct Options {
    std::string indexName, query1, query2, outputPrefix, iniFile;
    int maxReadLength = 120, insert_low = 1, insert_high = 500, outputBAM = 0, numCpuThreads = 4, device = 0;
    int megapathMode = 0, top = 95, ignoreComments = 0, alignmentType = 2, printMDNM = 0;
    int numGpus = 1, contextsPerGpu = 3;       // extensions: -G <n> uses GPUs device..device+n-1; MP_CONTEXTS_PER_GPU overrides 3
    int lsam = -1;                             // extension: -lsam <0|1> prints what `soap4 -F | fastq2lsam <0|1>` prints (cc/fastq2lsam.cpp)
};

static bool parse_args(int argc, char **argv, Options &o)
{
    if (argc < 2 || strcmp(argv[1], "pair") != 0) {
        fprintf(stderr, "Usage: %s pair <index prefix> <reads_1.fq[.gz]> <reads_2.fq[.gz]> [-o prefix] [-C ini] [-L len] [-T n] [-u n] [-v n] [-b] [-F|-P] [-nc] [-top n] [-c gpu]\n", argv[0]);
        if (argc >= 2) fprintf(stderr, "Only 'pair' mode is supported (the reference asserts readType == PAIR_END_READ, SOAP4.cpp:554).\n");
        return false;
    }
    if (argc < 5) { fprintf(stderr, "Invalid number of command-line arguments.\n"); return false; }
    o.indexName = argv[2]; o.query1 = argv[3]; o.query2 = argv[4]; o.outputPrefix = argv[3];
    for (int i = 5; i < argc; i++) {
        const char *a = argv[i];
        auto need = [&](const char *what) { if (i + 1 >= argc) { fprintf(stderr, "Please specify %s after '%s'\n", what, a); return false; } return true; };
        if (!strcmp(a, "-h")) { if (!need("the output option")) return false; int t = atoi(argv[++i]); if (t < 1 || t > 4) { fprintf(stderr, "The output option should be 1, 2, 3 or 4\n"); return false; } o.alignmentType = t; }
        else if (!strcmp(a, "-l") || !strcmp(a, "-L")) { if (!need("the length")) return false; o.maxReadLength = atoi(argv[++i]);
            if (o.maxReadLength < 0) { fprintf(stderr, "The length should not be less than 0\n"); return false; }
            if (o.maxReadLength > 1024) { fprintf(stderr, "The length should not be greater than %u\n", 1024u); return false; } }
        else if (!strcmp(a, "-u")) { if (!need("the maximum value of insert size")) return false; o.insert_high = atoi(argv[++i]); }
        else if (!strcmp(a, "-v")) { if (!need("the minimum value of insert size")) return false; o.insert_low = atoi(argv[++i]); }
        else if (!strcmp(a, "-b")) o.outputBAM = 1;
        else if (!strcmp(a, "-o")) { if (!need("the output file prefix")) return false; o.outputPrefix = argv[++i]; }
        else if (!strcmp(a, "-c")) { if (!need("the GPU device ID")) return false; o.device = atoi(argv[++i]); if (o.device < 0) { fprintf(stderr, "The GPU device ID should not be less than 0\n"); return false; } }
        else if (!strcmp(a, "-p")) o.printMDNM = 1;
        else if (!strcmp(a, "-G")) { if (!need("the number of GPUs")) return false; o.numGpus = atoi(argv[++i]); if (o.numGpus <= 0) { fprintf(stderr, "The number of GPUs should be positive\n"); return false; } }
        else if (!strcmp(a, "-T")) { if (!need("the number of CPU threads")) return false; o.numCpuThreads = atoi(argv[++i]); if (o.numCpuThreads <= 0) { fprintf(stderr, "Please specify a positive number of CPU threads after '-T'\n"); return false; } }
        else if (!strcmp(a, "-C")) { if (!need("ini file name")) return false; o.iniFile = argv[++i]; }
        else if (!strcmp(a, "-F")) o.megapathMode = 1;
        else if (!strcmp(a, "-P")) o.megapathMode = 2;
        else if (!strcmp(a, "-top")) { if (!need("the value of '-top'")) return false; o.top = atoi(argv[i + 1]); }   // the reference does not consume the value (IniParam.cpp:885-892)
        else if (!strcmp(a, "-nc")) o.ignoreComments = 1;
        else if (!strcmp(a, "-lsam")) { if (!need("0 or 1 (outputSeq)")) return false; o.lsam = atoi(argv[++i]) != 0; }
        else if (!strcmp(a, "-D") || !strcmp(a, "-A") || !strcmp(a, "-R") || !strcmp(a, "-e")) { if (i + 1 < argc) ++i; }
        else if (!strcmp(a, "-I")) { fprintf(stderr, "illumina quality is not supported yet\n"); return false; }
    }
    if (o.insert_low > o.insert_high) { fprintf(stderr, "The minimum value of insert size should not be greater than the maximum value of insert size.\n"); return false; }
    return true;
}

// ------------------------------------------------------------------------------------------------
// .ini (iniparser semantics: "section:key", case-insensitive keys, ';' / '#' comments)
struct Ini {
    std::map<std::string, std::string> kv;
    static std::string lower(std::string s) { for (auto &c : s) c = (char)tolower(c); return s; }
    static std::string trim(const std::string &s) { size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n"); return a == std::string::npos ? "" : s.substr(a, b - a + 1); }
    bool load(const std::string &path) {
        FILE *f = fopen(path.c_str(), "r"); if (!f) return false;
        char line[4096]; std::string sec;
        while (fgets(line, sizeof line, f)) {
            std::string s = trim(line);
            if (s.empty() || s[0] == ';' || s[0] == '#') continue;
            if (s[0] == '[') { size_t e = s.find(']'); if (e != std::string::npos) sec = lower(trim(s.substr(1, e - 1))); continue; }
            size_t eq = s.find('='); if (eq == std::string::npos) continue;
            std::string k = lower(trim(s.substr(0, eq))), v = trim(s.substr(eq + 1));
            size_t c = v.find_first_of(";#"); if (c != std::string::npos) v = trim(v.substr(0, c));
            if (v.size() >= 2 && (v[0] == '"' || v[0] == '\'') && v.back() == v[0]) v = v.substr(1, v.size() - 2);
            kv[sec + ":" + k] = v;
        }
        fclose(f); return true;
    }
    int geti(const char *k, int d) const { auto it = kv.find(lower(k)); return it == kv.end() ? d : (int)strtol(it->second.c_str(), nullptr, 0); }
    double getd(const char *k, double d) const { auto it = kv.find(lower(k)); return it == kv.end() ? d : atof(it->second.c_str()); }
    std::string gets(const char *k, const char *d) const { auto it = kv.find(lower(k)); return it == kv.end() ? d : it->second; }
};

// ------------------------------------------------------------------------------------------------
// chromosome translation (.ann names, .tra grid + translate table; HSP.c:57-330, BGS-IO.cpp:163-190)
struct Annotation {
    uint64_t dnaLength = 0; uint32_t numSeq = 0;
    std::vector<std::string> names;
    std::vector<uint64_t> seqStart, seqLen, actualLen;
    std::vector<uint32_t> grid;
    struct Tr { uint64_t startPos; uint32_t chrID; uint64_t correction; };
    std::vector<Tr> tr;
    bool load(const std::string &prefix) {
        FILE *f = fopen((prefix + ".ann").c_str(), "r"); if (!f) { fprintf(stderr, "Cannot open annotation file!\n"); return false; }
        unsigned long long n; unsigned ns, seed;
        if (fscanf(f, "%llu %u %u\n", &n, &ns, &seed) != 3) { fclose(f); return false; }
        dnaLength = n; numSeq = ns;
        char buf[4096];
        for (uint32_t i = 0; i < ns; ++i) {
            unsigned gi; if (fscanf(f, "%u ", &gi) != 1) break;
            if (!fgets(buf, sizeof buf, f)) break;
            size_t l = strlen(buf); if (l && buf[l - 1] == '\n') buf[l - 1] = 0;
            names.push_back(buf);
            unsigned long long a, b; int c; if (fscanf(f, "%llu %llu %d\n", &a, &b, &c) != 3) break;
            seqStart.push_back(a); seqLen.push_back(b);
        }
        fclose(f);
        if (names.size() != ns) { fprintf(stderr, "Annotation missing entries!\n"); return false; }
        f = fopen((prefix + ".tra").c_str(), "r"); if (!f) { fprintf(stderr, "Cannot open translate file!\n"); return false; }
        unsigned long long n2; int ns2; unsigned removed, gridEntries;
        if (fscanf(f, "%llu %d %u %u\n", &n2, &ns2, &removed, &gridEntries) != 4) { fclose(f); return false; }
        grid.resize(gridEntries);
        for (unsigned j = 0; j < gridEntries; ++j) if (fscanf(f, "%u\n", &grid[j]) != 1) { fclose(f); return false; }
        tr.resize(ns + removed);
        for (size_t j = 0; j < tr.size(); ++j) {
            unsigned long long s, c; unsigned id;
            if (fscanf(f, "%llu %u %llu\n", &s, &id, &c) != 3) { fclose(f); fprintf(stderr, "Translate missing entries!\n"); return false; }
            tr[j].startPos = s; tr[j].chrID = id; tr[j].correction = c;
        }
        for (uint32_t j = 0; j < ns; ++j) {
            unsigned long long a, l;
            if (fscanf(f, "%llu %llu\n", &a, &l) != 2) { actualLen.clear(); break; }
            actualLen.push_back(l);
        }
        if (actualLen.size() != ns) actualLen = seqLen;
        fclose(f);
        return true;
    }
    // -> end of the translate segment that holds ambPos (getChrAndPos, BGS-IO.cpp:163-190)
    uint64_t chrAndPos(uint64_t ambPos, uint64_t *tp, uint32_t *chr) const {
        uint64_t idx = ambPos >> 18;
        if (idx >= grid.size()) idx = grid.size() - 1;
        uint32_t v = grid[idx];
        while (tr[v].startPos > ambPos) v--;
        *tp = ambPos - tr[v].correction; *chr = tr[v].chrID;
        return (size_t)v + 1 < tr.size() ? tr[v + 1].startPos - 1 : dnaLength;
    }
    // getChrAndPosWithBoundaryCheckDP (BGS-IO.cpp:414-432)
    long long chrAndPosBoundaryDP(uint64_t readLength, uint64_t ambPos, const char *cigar, uint64_t *tp, uint32_t *chr, std::string &newCigar) const {
        uint64_t segEnd = chrAndPos(ambPos, tp, chr);
        uint64_t chrEnd = seqStart[*chr - 1] + seqLen[*chr - 1] - 1, corrected = 0;
        long long ret = boundary_check_dp(ambPos, chrEnd, (long long)readLength, cigar, segEnd, corrected, newCigar);
        if (ret && corrected > ambPos) chrAndPos(corrected, tp, chr);
        return ret;
    }
    // decideTargetChr (BGS-IO.cpp:1312-1341): -1 when the read window [pos, pos+readLen) crosses sequences
    int targetChr(uint64_t ambPos, uint32_t readLen) const {
        uint64_t p; uint32_t c0, c1;
        chrAndPos(ambPos, &p, &c0); chrAndPos(ambPos + readLen - 1, &p, &c1);
        return c0 == c1 ? (int)c0 : -1;
    }
};

// ------------------------------------------------------------------------------------------------
// FASTA/FASTQ reader with kseq semantics (name up to the first blank, comment = rest of the header)
static size_t count_newlines(const char *p, size_t n);
struct SeqReader {
    SeqReader() = default;
    SeqReader(const SeqReader &) = delete;
    SeqReader &operator=(const SeqReader &) = delete;
    gzFile f = nullptr; std::vector<char> own; char *base = nullptr; size_t pos = 0, end = 0; bool eof = false; int last = 0;
    // A plain regular file is memory-mapped instead: the whole file is the buffer (nothing left to fill), the record parsers below work
    // on it unchanged, and load_batch can locate a batch's records and parse them with several threads (parse_mapped).
    bool mapped = false;
    int fd = -1;                   // kept open beside the mapping: batches are staged with pread (no page faults on the source side)
    // A regular gzip file is inflated on the device (mp_gunzip_run on a context of its own, compressed bytes read with pread into a
    // page-locked buffer) into `own`, which then stands in for the mapping: [pos, end) holds the inflated text not yet consumed, and
    // ensure_lines tops it up to the next batch's records before a batch is located in it.  MP_HOST_IO=1 and pipes keep gzread.
    mp_context *gzCtx = nullptr; mp_gunzip *gz = nullptr; int gzFd = -1; uint64_t gzOff = 0, gzSize = 0; bool gzDone = false;
    char *gzIn = nullptr; double gzSeconds = 0;                     // page-locked compressed window; inflate wall time so far
    static constexpr uint64_t GZ_IN = 32ull << 20, GZ_OUT = 128ull << 20;
    ~SeqReader() {
        if (gz) mp_gunzip_close(gz);
        if (gzCtx) mp_destroy(gzCtx);
        if (gzIn) mp_host_free(gzIn);
        if (gzFd >= 0) ::close(gzFd);
    }
    // one mp_gunzip_run call appended at end (own grows as needed) -> bytes appended; 0 at the end of the file.  A stream the inflater
    // refuses delivers the bytes before the error and then ends, as gzread's reader does (unexpected end of file / data error).
    size_t gz_append() {
        if (gzDone) return 0;
        const double t = now_s();
        if (own.size() - end < GZ_OUT) { own.resize(std::max(own.size() + own.size() / 2, end + GZ_OUT)); base = own.data(); }
        const uint64_t n = std::min<uint64_t>(GZ_IN, gzSize - gzOff);
        size_t got = 0;
        while (got < n) { const ssize_t g = pread(gzFd, gzIn + got, n - got, (off_t)(gzOff + got)); if (g <= 0) break; got += (size_t)g; }
        uint64_t used = 0, produced = 0; int done = 0;
        const int rc = mp_gunzip_run(gz, (const uint8_t *)gzIn, got, gzOff + got >= gzSize, (uint8_t *)base + end, own.size() - end, &used, &produced, &done);
        gzOff += used; end += produced;
        if (rc || done || (produced == 0 && used == 0)) gzDone = true;
        eof = gzDone;
        gzSeconds += now_s() - t;
        return produced;
    }
    // device-inflated file: [pos, end) holds at least `lines` newlines or the rest of the file
    void ensure_lines(uint64_t lines) {
        if (!gz || gzDone) return;
        if (pos > 0) { memmove(base, base + pos, end - pos); end -= pos; pos = 0; }
        uint64_t have = count_newlines(base, end);
        while (have < lines && !gzDone) { const size_t e0 = end; gz_append(); have += count_newlines(base + e0, end - e0); }
    }
    bool open_gz_device(const std::string &path, int device) {
        gzFd = ::open(path.c_str(), O_RDONLY);
        struct stat sb;
        if (gzFd < 0 || fstat(gzFd, &sb) != 0) return false;
        gzSize = (uint64_t)sb.st_size;
        if (mp_init(device, &gzCtx) || mp_gunzip_open(gzCtx, GZ_IN, &gz) || !(gzIn = (char *)mp_host_alloc(GZ_IN))) return false;
        own.resize(GZ_OUT); base = own.data(); pos = end = 0;
        if (gz_append() == 0 && gzDone && gzOff == 0) return false;     // refused on the first call
        mapped = true;
        return true;
    }
    bool open(const std::string &path, int gzDevice = -1) {
        if (gzDevice >= 0 && !getenv("MP_HOST_IO")) {
            int f0 = ::open(path.c_str(), O_RDONLY);
            struct stat sb; unsigned char magic[2] = { 0, 0 };
            const bool isGz = f0 >= 0 && fstat(f0, &sb) == 0 && S_ISREG(sb.st_mode) && pread(f0, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
            if (f0 >= 0) ::close(f0);
            if (isGz) {
                if (open_gz_device(path, gzDevice)) return true;
                fprintf(stderr, "[Main] %s: device inflate refused (%s), reading it with zlib\n", path.c_str(), mp_last_error());
                if (gz) { mp_gunzip_close(gz); gz = nullptr; }
                if (gzCtx) { mp_destroy(gzCtx); gzCtx = nullptr; }
                if (gzIn) { mp_host_free(gzIn); gzIn = nullptr; }
                if (gzFd >= 0) { ::close(gzFd); gzFd = -1; }
                gzDone = false; pos = end = 0; eof = false;
            }
        }
        if (!getenv("MP_NO_MMAP")) {
            int fd = ::open(path.c_str(), O_RDONLY);
            if (fd >= 0) {
                struct stat sb; unsigned char magic[2] = { 0, 0 };
                if (fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size >= 2 && pread(fd, magic, 2, 0) == 2 && !(magic[0] == 0x1f && magic[1] == 0x8b)) {
                    void *m = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
                    if (m != MAP_FAILED) {
                        madvise(m, (size_t)sb.st_size, MADV_SEQUENTIAL);
                        base = (char *)m; pos = 0; end = (size_t)sb.st_size; eof = true; mapped = true;
                        this->fd = fd;
                        return true;
                    }
                }
                ::close(fd);
            }
        }
        f = gzopen(path.c_str(), "rb"); if (!f) return false; gzbuffer(f, 1 << 22); own.resize(1 << 22); base = own.data(); return true;
    }
    bool fill() {
        if (eof) return false;
        if (gz) { pos = end = 0; gz_append(); return end > 0; }
        int n = gzread(f, base, (unsigned)own.size()); if (n <= 0) { eof = true; return false; } pos = 0; end = (size_t)n; return true;
    }
    int getc_() { if (pos >= end && !fill()) return -1; return (unsigned char)base[pos++]; }
    // reads up to the delimiter class: 0 = blank (space/tab/newline), 2 = newline; returns delimiter or -1.  Whole buffer ranges
    // are appended at once (the per-character version of this loop was the slowest part of the driver).
    int getuntil(int mode, std::string &s, bool append) {
        if (!append) s.clear();
        for (;;) {
            if (pos >= end && !fill()) return -1;
            const char *b = base + pos, *e = base + end, *q;
            if (mode == 2) q = (const char *)memchr(b, '\n', (size_t)(e - b));
            else { q = b; while (q < e && !isspace((unsigned char)*q)) ++q; if (q == e) q = nullptr; }
            if (!q) { s.append(b, (size_t)(e - b)); pos = end; continue; }
            s.append(b, (size_t)(q - b)); pos = (size_t)(q - base) + 1;
            if (mode == 2 && !s.empty() && s.back() == '\r') s.pop_back();
            return (unsigned char)*q;
        }
    }
    struct View { const char *name, *comment, *seq, *qual; size_t nameLen, commentLen, seqLen; };
    // The usual four-line FASTQ record lying whole inside [b, e): views into the buffer, no copies.
    // -> 1: record returned, *next = first byte after it; 0: not a plain four-line record; -1: no four newlines before e
    static int view_record(const char *b, const char *e, View &v, const char **next) {
        if (b >= e || *b != '@') return 0;
        const char *n1 = (const char *)memchr(b, '\n', (size_t)(e - b));
        const char *n2 = n1 ? (const char *)memchr(n1 + 1, '\n', (size_t)(e - n1 - 1)) : nullptr;
        const char *n3 = n2 ? (const char *)memchr(n2 + 1, '\n', (size_t)(e - n2 - 1)) : nullptr;
        const char *n4 = n3 ? (const char *)memchr(n3 + 1, '\n', (size_t)(e - n3 - 1)) : nullptr;
        if (!n4) return -1;
        const char *h = b + 1, *he = n1; if (he > h && he[-1] == '\r') --he;
        const char *q = h; while (q < he && !isspace((unsigned char)*q)) ++q;
        v.name = h; v.nameLen = (size_t)(q - h);
        if (q < he) { v.comment = q + 1; v.commentLen = (size_t)(he - q - 1); } else { v.comment = he; v.commentLen = 0; }
        const char *s0 = n1 + 1, *s1 = n2; if (s1 > s0 && s1[-1] == '\r') --s1;
        if (s1 == s0 || *s0 == '>' || *s0 == '+' || *s0 == '@' || n2[1] != '+') return 0;
        const char *q0 = n3 + 1, *q1 = n4; if (q1 > q0 && q1[-1] == '\r') --q1;
        if ((size_t)(q1 - q0) != (size_t)(s1 - s0)) return 0;
        v.seq = s0; v.seqLen = (size_t)(s1 - s0); v.qual = q0;
        *next = n4 + 1;
        return 1;
    }
    // Fast path of the sequential reader.
    // -> 1: record returned; 0: not applicable here (caller falls back to read(), which gives the same answer); -1: end of file.
    int read_fast(View &v) {
        if (last != 0) return 0;
        for (int attempt = 0; attempt < 2; ++attempt) {
            if (pos >= end) { if (!fill()) return -1; }
            const char *b = base + pos, *e = base + end, *next = nullptr;
            const int st = view_record(b, e, v, &next);
            if (st == 1) { pos = (size_t)(next - base); return 1; }
            if (st == 0) return 0;
            if (attempt == 1 || eof) return 0;
            // the record crosses the end of the buffer: move the tail to the front and top the buffer up
            const size_t rest = (size_t)(e - b);
            if (rest == own.size()) return 0;                  // a record larger than the buffer: leave it to read()
            memmove(base, b, rest); pos = 0; end = rest;
            if (gz) { if (gz_append() == 0) return 0; continue; }
            int n = gzread(f, base + end, (unsigned)(own.size() - end));
            if (n <= 0) { eof = true; return 0; }
            end += (size_t)n;
        }
        return 0;
    }
    // -> length of the sequence, -1 at end of file
    int read(std::string &name, std::string &comment, std::string &seq, std::string &qual) {
        int c;
        if (last == 0) { while ((c = getc_()) >= 0 && c != '>' && c != '@') {} if (c < 0) return -1; last = c; }
        comment.clear(); seq.clear(); qual.clear();
        if ((c = getuntil(0, name, false)) < 0) return -1;
        if (c != '\n') getuntil(2, comment, false);
        while ((c = getc_()) >= 0 && c != '>' && c != '+' && c != '@') {
            if (c == '\n') continue;
            seq.push_back((char)c);
            getuntil(2, seq, true);
        }
        if (c == '>' || c == '@') last = c;
        if (c != '+') return (int)seq.size();
        std::string skip;
        getuntil(2, skip, false);                                 // rest of the '+' line
        while (qual.size() < seq.size()) { if (getuntil(2, qual, true) < 0) break; }
        last = 0;
        if (seq.size() != qual.size()) return -2;
        return (int)seq.size();
    }
};

struct ReadBatch {
    uint32_t nReads = 0, wpq = 0, maxReadLength = 0;
    std::vector<uint32_t> queries, lens;                           // what mp_batch_upload takes (read-id order, 32-read interleaved words)
    // Everything the two parser threads write is stored mate-major -- slot(id) = (id & 1) * half + id / 2 -- so that the thread
    // of mate 1 and the thread of mate 2 never write to the same cache line; the 2-bit packing into `queries` (whose layout
    // interleaves 32 consecutive reads) is done afterwards by worker threads that each own whole groups of 32 reads.
    uint32_t half = 0;
    std::vector<std::string> names_, comments_;
    std::vector<uint8_t> hasComment_;
    std::vector<uint32_t> qlen_, slen_;
    std::unique_ptr<char[]> qualBuf, seqBuf; size_t qstride = 0, qcap = 0;   // one fixed-stride row per read; qualities NUL-terminated
    size_t slot(uint32_t id) const { return (size_t)(id & 1u) * half + (id >> 1); }
    const std::string &name(uint32_t id) const { return names_[slot(id)]; }
    const std::string &comment(uint32_t id) const { return comments_[slot(id)]; }
    bool hasComment(uint32_t id) const { return hasComment_[slot(id)] != 0; }
    const char *qual(uint32_t id) const { return qualBuf.get() + slot(id) * qstride; }
    uint32_t qlen(uint32_t id) const { return qlen_[slot(id)]; }
};

static unsigned char g_charMap[256];
static char g_outChar[256];                                      // the base soap4 prints for an input character: "ACGT"[charMap[c]]
static void fill_char_map() {                                    // INDEXFillCharMap (IndexHandler.cpp:26-45)
    memset(g_charMap, 0, sizeof g_charMap);
    const char *dna = "ACGT";
    for (int i = 0; i < 4; ++i) { g_charMap[(int)dna[i]] = (unsigned char)i; g_charMap[dna[i] - 'A' + 'a'] = (unsigned char)i; }
    g_charMap['U'] = g_charMap['u'] = 3; g_charMap['N'] = g_charMap['n'] = 2;
    for (int c = 0; c < 256; ++c) g_outChar[c] = "ACGT"[g_charMap[c]];
}

static void append_read(ReadBatch &b, uint32_t id, const char *name, size_t nameLen, const char *comment, size_t commentLen,
                        const char *seq, size_t seqLen, const char *qual, size_t qualLen)
{
    const size_t sl = b.slot(id);
    uint32_t len = seqLen > b.maxReadLength - 1 ? b.maxReadLength - 1 : (uint32_t)seqLen;     // QueryParser.cpp:188
    b.slen_[sl] = len;
    memcpy(b.seqBuf.get() + sl * b.qstride, seq, len);
    if (nameLen > 2 && name[nameLen - 2] == '/' && isdigit((unsigned char)name[nameLen - 1])) nameLen -= 2;   // trim_readno
    b.names_[sl].assign(name, nameLen);
    b.hasComment_[sl] = commentLen != 0;
    if (commentLen) b.comments_[sl].assign(comment, commentLen); else b.comments_[sl].clear();
    const uint32_t ql = (uint32_t)std::min<size_t>(qualLen, len);                                 // qual.substr(0, len)
    char *qd = b.qualBuf.get() + sl * b.qstride;
    memcpy(qd, qual, ql); qd[ql] = 0; b.qlen_[sl] = ql;
}

// 2-bit packing of reads [first, last) into the 32-read interleaved words (appendToQueryArrays, QueryParser.cpp:184-203)
static void pack_reads(ReadBatch &b, uint32_t first, uint32_t last)
{
    for (uint32_t id = first; id < last; ++id) {
        const size_t sl = b.slot(id);
        const uint32_t len = b.slen_[sl];
        const char *seq = b.seqBuf.get() + sl * b.qstride;
        b.lens[id] = len;
        uint32_t *q = b.queries.data() + ((size_t)(id / 32) * 32 * b.wpq + id % 32);
        uint32_t i = 0;
        for (; i + 16 <= len; i += 16, q += 32) {
            uint32_t word = 0;
            for (int k = 0; k < 16; ++k) word |= (uint32_t)g_charMap[(unsigned char)seq[i + k]] << (k * 2);
            *q = word;
        }
        if (i < len) { uint32_t word = 0; for (int k = 0; i < len; ++i, ++k) word |= (uint32_t)g_charMap[(unsigned char)seq[i]] << (k * 2); *q = word; }
    }
}


static size_t count_newlines(const char *p, size_t n)
{
    size_t c = 0;
    for (const char *q = p, *e = p + n; (q = (const char *)memchr(q, '\n', (size_t)(e - q))) != nullptr; ++q) ++c;
    return c;
}

// A batch out of a memory-mapped FASTQ file, parsed by several threads.  Records are located, not guessed: the newlines of the
// region are counted in 256 KiB blocks (in parallel), which gives the byte offset of every 4k-th line, and every thread then parses
// its run of four-line records with the same record view as the sequential reader.  If anything is not a plain four-line record (a
// multi-line FASTA / FASTQ, a quality string of another length, a missing final newline) nothing is consumed and the caller parses the
// batch sequentially -- same records either way (tests/test_driver_host.py).
// -> records parsed, *newPos = offset behind them; -1: use the sequential parser
static long parse_mapped(const SeqReader &r, ReadBatch &b, uint32_t first, uint32_t maxRec, unsigned nThr, size_t *newPos)
{
    const char *beg = r.base + r.pos, *lim = r.base + r.end;
    *newPos = r.pos;
    if (r.last != 0) return -1;
    if (beg >= lim || maxRec == 0) return 0;
    if (lim[-1] != '\n') return -1;
    SeqReader::View v0; const char *next0 = nullptr;
    if (SeqReader::view_record(beg, lim, v0, &next0) != 1) return -1;
    const size_t B = (size_t)1 << 18, remaining = (size_t)(lim - beg), rec0 = (size_t)(next0 - beg);
    nThr = std::max(1u, nThr);
    auto par = [&](size_t n, const std::function<void(size_t)> &fn) {       // fn(k) for k in [0, n), strided over the threads
        const unsigned T = (unsigned)std::min<size_t>(nThr, std::max<size_t>(n, 1));
        std::vector<std::thread> th;
        for (unsigned t = 1; t < T; ++t) th.emplace_back([&, t] { for (size_t k = t; k < n; k += T) fn(k); });
        for (size_t k = 0; k < n; k += T) fn(k);
        for (std::thread &x : th) x.join();
    };
    // ---- newline counts per block, over a window that grows until it holds the batch (or the rest of the file) ----
    size_t window = std::min(remaining, (size_t)((double)maxRec * (double)rec0 * 1.02) + B), fullCounted = 0;
    std::vector<uint32_t> cnt;
    uint64_t lines = 0;
    for (;;) {
        const size_t nBlocks = (window + B - 1) / B;
        cnt.resize(nBlocks);
        par(nBlocks - fullCounted, [&](size_t k) { const size_t blk = fullCounted + k; cnt[blk] = (uint32_t)count_newlines(beg + blk * B, std::min(B, window - blk * B)); });
        lines = 0; for (uint32_t c : cnt) lines += c;
        if (lines >= 4ull * maxRec || window == remaining) break;
        fullCounted = window / B;                                            // the partial last block is counted again
        window = std::min(remaining, window + window / 8 + B);
    }
    if (lines < 4ull * maxRec && (lines & 3)) return -1;                      // the file ends inside the window, not after a whole record
    const uint64_t nRec = std::min<uint64_t>(maxRec, lines / 4);
    if (nRec == 0) return -1;
    std::vector<uint64_t> pre(cnt.size() + 1, 0);
    for (size_t k = 0; k < cnt.size(); ++k) pre[k + 1] = pre[k] + cnt[k];
    auto after_line = [&](uint64_t L) -> const char * {                      // first byte after the L-th newline of the region (L >= 1)
        const size_t k = (size_t)(std::lower_bound(pre.begin(), pre.end(), L) - pre.begin()) - 1;     // pre[k] < L <= pre[k+1]
        const char *q = beg + k * B;
        for (uint64_t need = L - pre[k]; need; --need) q = (const char *)memchr(q, '\n', (size_t)(lim - q)) + 1;
        return q;
    };
    const unsigned T = (unsigned)std::min<uint64_t>(nThr, std::max<uint64_t>(1, nRec / 256));
    std::vector<const char *> start(T + 1);
    std::vector<uint64_t> firstRec(T + 1);
    for (unsigned t = 0; t <= T; ++t) { firstRec[t] = nRec * t / T; start[t] = firstRec[t] == 0 ? beg : after_line(4 * firstRec[t]); }
    std::atomic<bool> bad(false);
    par(T, [&](size_t t) {
        const char *q = start[t], *e = start[t + 1];
        SeqReader::View v;
        for (uint64_t rec = firstRec[t]; rec < firstRec[t + 1]; ++rec) {
            const char *next = nullptr;
            if (SeqReader::view_record(q, e, v, &next) != 1) { bad.store(true); return; }
            append_read(b, first + 2 * (uint32_t)rec, v.name, v.nameLen, v.comment, v.commentLen, v.seq, v.seqLen, v.qual, v.seqLen);
            q = next;
        }
        if (q != e) bad.store(true);
    });
    if (bad.load()) return -1;
    *newPos = (size_t)(start[T] - r.base);
    return (long)nRec;
}

// Device ingest (mp_fastq_upload): the byte range of the next maxRec four-line records of a memory-mapped file, found by counting
// newlines in 256 KiB blocks with several threads (the same location step as parse_mapped).  Whether the range really is strict
// four-line FASTQ is checked by the kernels that index it.
// -> records in [r.pos, *newPos), 0 at the end of the file, -1: this file needs the sequential parser
static long locate_records(const SeqReader &r, uint32_t maxRec, unsigned nThr, size_t *newPos)
{
    const char *beg = r.base + r.pos, *lim = r.base + r.end;
    *newPos = r.pos;
    if (r.last != 0) return -1;
    if (beg >= lim || maxRec == 0) return 0;
    if (lim[-1] != '\n') return -1;
    SeqReader::View v0; const char *next0 = nullptr;
    if (SeqReader::view_record(beg, lim, v0, &next0) != 1) return -1;
    const size_t B = (size_t)1 << 18, remaining = (size_t)(lim - beg), rec0 = (size_t)(next0 - beg);
    nThr = std::max(1u, nThr);
    size_t window = std::min(remaining, (size_t)((double)maxRec * (double)rec0 * 1.02) + B), fullCounted = 0;
    std::vector<uint32_t> cnt;
    uint64_t lines = 0;
    for (;;) {
        const size_t nBlocks = (window + B - 1) / B;
        cnt.resize(nBlocks);
        const size_t n = nBlocks - fullCounted;
        const unsigned T = (unsigned)std::min<size_t>(nThr, std::max<size_t>(n, 1));
        auto run = [&](unsigned t) { for (size_t k = t; k < n; k += T) { const size_t blk = fullCounted + k; cnt[blk] = (uint32_t)count_newlines(beg + blk * B, std::min(B, window - blk * B)); } };
        std::vector<std::thread> th;
        for (unsigned t = 1; t < T; ++t) th.emplace_back(run, t);
        run(0);
        for (std::thread &x : th) x.join();
        lines = 0; for (uint32_t c : cnt) lines += c;
        if (lines >= 4ull * maxRec || window == remaining) break;
        fullCounted = window / B;
        window = std::min(remaining, window + window / 8 + B);
    }
    if (lines < 4ull * maxRec && (lines & 3)) return -1;
    const uint64_t nRec = std::min<uint64_t>(maxRec, lines / 4);
    if (nRec == 0) return -1;
    uint64_t need = 4 * nRec, pre = 0; size_t k = 0;
    while (pre + cnt[k] < need) pre += cnt[k++];
    const char *q = beg + k * B;
    for (need -= pre; need; --need) q = (const char *)memchr(q, '\n', (size_t)(lim - q)) + 1;
    *newPos = (size_t)(q - r.base);
    return (long)nRec;
}
static void parallel_copy(char *dst, const char *src, size_t n, unsigned nThr)
{
    const size_t piece = (size_t)4 << 20, nPieces = (n + piece - 1) / piece;
    const unsigned T = (unsigned)std::min<size_t>(std::max(1u, nThr), std::max<size_t>(nPieces, 1));
    auto run = [&](unsigned t) { for (size_t k = t; k < nPieces; k += T) memcpy(dst + k * piece, src + k * piece, std::min(piece, n - k * piece)); };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < T; ++t) th.emplace_back(run, t);
    run(0);
    for (std::thread &x : th) x.join();
}

// One mate file's next batch: every 256 KiB block is copied into the staging buffer and its newlines are counted in the copy while
// it is still in the cache -- one pass over the page cache.  -> records staged, 0 at the end of the file, -1: not for the device
// path, -2: the window estimate did not hold (the caller locates the batch exactly, locate_records, and copies it then)
static long stage_file(const SeqReader &r, double bytesPerRec, uint32_t maxRec, unsigned stageThreads, char *dst, size_t cap, size_t *bytes)
{
    const char *beg = r.base + r.pos, *lim = r.base + r.end;
    *bytes = 0;
    if (r.last != 0) return -1;
    if (beg >= lim || maxRec == 0) return 0;
    if (lim[-1] != '\n' || *beg != '@') return -1;
    const size_t B = (size_t)1 << 18, remaining = (size_t)(lim - beg);
    size_t window = std::min(remaining, (size_t)((double)maxRec * bytesPerRec * 1.02) + B), done = 0;
    std::vector<uint32_t> cnt;
    uint64_t lines = 0;
    for (;;) {
        if (window > cap) return -2;
        const size_t nBlocks = (window + B - 1) / B, n = nBlocks - done;
        cnt.resize(nBlocks);
        const unsigned T = (unsigned)std::min<size_t>(stageThreads, std::max<size_t>(n, 1));
        auto run = [&](unsigned t) {
            for (size_t k = t; k < n; k += T) {
                const size_t blk = done + k, o = blk * B, len = std::min(B, window - o);
                size_t got = 0;                                           // pread: the kernel copies from the page cache, no faults on a mapping
                while (r.fd >= 0 && got < len) { const ssize_t g = pread(r.fd, dst + o + got, len - got, (off_t)(r.pos + o + got)); if (g <= 0) break; got += (size_t)g; }
                if (got < len) memcpy(dst + o + got, beg + o + got, len - got);
                cnt[blk] = (uint32_t)count_newlines(dst + o, len);
            }
        };
        std::vector<std::thread> th;
        for (unsigned t = 1; t < T; ++t) th.emplace_back(run, t);
        run(0);
        for (std::thread &x : th) x.join();
        lines = 0; for (uint32_t c : cnt) lines += c;
        if (lines >= 4ull * maxRec || window == remaining) break;
        done = window / B;                                               // the partial last block is copied and counted again
        window = std::min(remaining, window + window / 8 + B);
    }
    if (lines < 4ull * maxRec && (lines & 3)) return -1;
    const uint64_t nRec = std::min<uint64_t>(maxRec, lines / 4);
    if (nRec == 0) return -1;
    uint64_t need = 4 * nRec, pre = 0; size_t k = 0;
    while (pre + cnt[k] < need) pre += cnt[k++];
    const char *q = dst + k * B;
    for (need -= pre; need; --need) q = (const char *)memchr(q, '\n', (size_t)(dst + window - q)) + 1;
    *bytes = (size_t)(q - dst);
    return (long)nRec;
}

static uint32_t load_batch(SeqReader &r1, SeqReader &r2, ReadBatch &b, uint32_t maxReads, unsigned packThreads = 4)
{
    const double tSetup0 = now_s();
    size_t words = ((size_t)maxReads + 31) / 32 * 32 * b.wpq;
    // batches are recycled (see BatchPool): storage that already has the right size is only cleared, so that a long run does
    // not page-fault half a gigabyte of fresh memory per batch
    b.half = (maxReads + 1) / 2;
    const size_t slots = (size_t)b.half * 2;
    b.queries.assign(words, 0); b.lens.assign(maxReads, 0);
    if (b.names_.size() != slots) { b.names_.assign(slots, ""); b.comments_.assign(slots, ""); }
    b.hasComment_.assign(slots, 0); b.qlen_.assign(slots, 0); b.slen_.assign(slots, 0);
    if (!b.qualBuf || b.qstride != (size_t)b.maxReadLength + 1 || b.qcap != slots) {
        b.qstride = (size_t)b.maxReadLength + 1; b.qcap = slots;
        b.qualBuf.reset(new char[slots * b.qstride]); b.seqBuf.reset(new char[slots * b.qstride]);
    }
    // both files memory-mapped: thread teams parse the batch's records of either file, then every thread packs whole groups of 32 reads
    if (r1.mapped && r2.mapped) {
        static const bool ltiming = getenv("MP_LOAD_TIMING") != nullptr;
        const double tl0 = now_s();
        const unsigned team = std::max(1u, packThreads);
        long n1 = -1, n2 = -1; size_t p1 = r1.pos, p2 = r2.pos;
        std::thread t2([&] { n2 = parse_mapped(r2, b, 1, maxReads / 2, team, &p2); });
        n1 = parse_mapped(r1, b, 0, (maxReads + 1) / 2, team, &p1);
        t2.join();
        if (n1 >= 0 && n2 >= 0) {
            if (n1 != n2) { fprintf(stderr, "Error: number of sequences of pair-end files not matched.\n"); exit(1); }
            r1.pos = p1; r2.pos = p2;
            b.nReads = 2 * (uint32_t)n1;
            const double tl1 = now_s();
            const uint32_t nGroups = (b.nReads + 31) / 32, T = std::min<uint32_t>(2 * team, std::max(1u, nGroups / 64));
            std::vector<std::thread> th;
            for (uint32_t t = 1; t < T; ++t) th.emplace_back([&, t] { pack_reads(b, (uint32_t)((uint64_t)nGroups * t / T) * 32, std::min(b.nReads, (uint32_t)((uint64_t)nGroups * (t + 1) / T) * 32)); });
            pack_reads(b, 0, std::min(b.nReads, (uint32_t)((uint64_t)nGroups / T) * 32));
            for (std::thread &x : th) x.join();
            if (ltiming) fprintf(stderr, "[load] setup %.3f parse %.3f pack %.3f s\n", tl0 - tSetup0, tl1 - tl0, now_s() - tl1);
            return b.nReads;
        }
        // not plain four-line FASTQ here: nothing was consumed, the sequential parsers below take the batch
    }
    // the two files are parsed by two threads: mate 1 fills the even read ids, mate 2 the odd ones.  Packing threads follow them:
    // each owns every nt-th group of 32 reads (the unit the word layout interleaves) and packs a group as soon as both parsers
    // are past it.
    std::atomic<uint32_t> prog[2]; prog[0] = 0; prog[1] = 0;        // records parsed so far, per mate
    std::atomic<int> finished(0);
    auto half = [&b, &prog, &finished, maxReads](SeqReader &r, uint32_t first) -> uint32_t {
        std::string nm, cm, sq, ql; uint32_t n = 0; SeqReader::View v;
        for (uint32_t id = first; id < maxReads; id += 2) {
            const int st = r.read_fast(v);
            if (st < 0) break;
            if (st == 1) append_read(b, id, v.name, v.nameLen, v.comment, v.commentLen, v.seq, v.seqLen, v.qual, v.seqLen);
            else {
                if (r.read(nm, cm, sq, ql) < 0) break;
                append_read(b, id, nm.data(), nm.size(), cm.data(), cm.size(), sq.data(), sq.size(), ql.data(), ql.size());
            }
            ++n;
            if ((n & 255u) == 0) prog[first].store(n, std::memory_order_release);
        }
        prog[first].store(n, std::memory_order_release);
        finished.fetch_add(1, std::memory_order_release);
        return n;
    };
    const unsigned nt = std::max(1u, packThreads);
    auto packer = [&b, &prog, &finished, nt](unsigned t) {
        for (uint32_t g = t; ; g += nt) {
            const uint32_t needPairs = (g + 1) * 16;                // the group holds reads 32g .. 32g+31 = pairs 16g .. 16g+15
            uint32_t have;
            for (;;) {
                const bool fin = finished.load(std::memory_order_acquire) == 2;
                have = std::min(prog[0].load(std::memory_order_acquire), prog[1].load(std::memory_order_acquire));
                if (have >= needPairs || fin) break;
                std::this_thread::sleep_for(std::chrono::microseconds(100));
            }
            if (have <= g * 16) break;                              // input ended before this group
            pack_reads(b, g * 32, std::min(needPairs, have) * 2);
            if (have < needPairs) break;                            // the last, partial group
        }
    };
    std::vector<std::thread> packers;
    for (unsigned t = 0; t < nt; ++t) packers.emplace_back(packer, t);
    uint32_t n2 = 0;
    std::thread t2([&] { n2 = half(r2, 1); });
    const uint32_t n1 = half(r1, 0);
    t2.join();
    for (std::thread &t : packers) t.join();
    if (n1 != n2) { fprintf(stderr, "Error: number of sequences of pair-end files not matched.\n"); exit(1); }
    b.nReads = 2 * n1;
    return b.nReads;
}

static uint32_t detect_read_length(const std::vector<uint32_t> &lens, uint32_t numQueries, uint32_t start)   // GetReadLength (QueryParser.cpp:2253-2277)
{
    if (numQueries == 0) return 100;
    uint32_t i = 0, j = 1, mx = lens[start];
    while (i < numQueries && j < 1000000) { if (mx < lens[start + i]) mx = lens[start + i]; j++; i += 2; }
    return mx;
}

// ------------------------------------------------------------------------------------------------
// FASTQ header composition
struct HeaderHit { int score; size_t s, e; };
static int mapping_from_header(const std::string *comment, std::vector<HeaderHit> &v, double top, double scoreT)   // BGS-IO.cpp:1348-1371
{
    v.clear();
    if (!comment || *comment == "IGNORE") return 0;
    const char *c = comment->c_str();
    if (comment->size() < 6) return 0;
    int score = atoi(c + 6);
    if (score < scoreT) return score;
    else if (scoreT < score * top) scoreT = score * top;
    const char *p = strchr(c + 6, ';');
    while (p && *(p + 1) != '\0') {
        HeaderHit m; m.score = atoi(p + 1); m.s = (size_t)(p + 1 - c);
        p = strchr(p + 1, ';');
        if (!p) break;
        m.e = (size_t)(p - c);
        if (score >= scoreT) v.push_back(m);
    }
    return score;
}

static void seq_and_qual(std::string &out, const ReadBatch &b, uint32_t id)
{
    // the 2-bit words hold exactly charMap[c] of the parsed characters (pack_reads), so the printed sequence is a table look-up away
    const uint32_t len = b.lens[id], ql = b.qlen(id);
    const unsigned char *sq = (const unsigned char *)b.seqBuf.get() + b.slot(id) * b.qstride;
    const size_t at = out.size();
    out.resize(at + len + 3 + ql + 1);
    char *w = &out[at];
    for (uint32_t i = 0; i < len; ++i) w[i] = g_outChar[sq[i]];
    w += len; *w++ = '\n'; *w++ = '+'; *w++ = '\n';
    memcpy(w, b.qual(id), ql); w[ql] = '\n';
}

static inline char *put_int(char *w, long long v)
{
    char tmp[24]; int n = 0; bool neg = v < 0; unsigned long long u = neg ? 0ull - (unsigned long long)v : (unsigned long long)v;
    do { tmp[n++] = (char)('0' + u % 10); u /= 10; } while (u);
    if (neg) *w++ = '-';
    while (n) *w++ = tmp[--n];
    return w;
}
// One output record: "@name\tSCORE:<best>;<score>,<chr>;...<kept entries of the previous comment>\n" (BGS-IO.cpp:1966-2091, 1348-1371),
// then sequence, "+", qualities.  Written through a raw pointer into space reserved once per record: at a million pairs per batch the
// capacity checks of a dozen small std::string appends per read were most of the formatting time.
static void header_line(std::string &ret, const ReadBatch &b, uint32_t id, const Annotation &ann, std::vector<std::pair<int, int>> &chrHits,
                        int bestScore, double top, bool ignoreComments)
{
    const std::string *comment = (!ignoreComments && b.hasComment(id)) ? &b.comment(id) : nullptr;
    const std::string &name = b.name(id);
    size_t bound = 1 + name.size() + 8 + 24 + 2 + (comment ? comment->size() + 8 : 0);
    for (size_t i = 0; i < chrHits.size(); ++i) bound += 24 + ann.names[chrHits[i].first - 1].size();
    const size_t at = ret.size();
    ret.resize(at + bound);
    char *w0 = &ret[at], *w = w0;
    *w++ = '@'; memcpy(w, name.data(), name.size()); w += name.size();
    if (comment && *comment == "IGNORE") { memcpy(w, "\tIGNORE\n", 8); w += 8; ret.resize(at + (size_t)(w - w0)); return; }
    if (chrHits.size() > 1) std::sort(chrHits.begin(), chrHits.end());
    std::vector<HeaderHit> v;
    int prev = mapping_from_header(comment, v, top, bestScore * top);
    if (prev > bestScore) bestScore = prev;
    memcpy(w, "\tSCORE:", 7); w += 7; w = put_int(w, bestScore); *w++ = ';';
    if (bestScore > 0)
        for (size_t i = 0; i < chrHits.size(); ++i) {
            if (i > 0 && chrHits[i].first == chrHits[i - 1].first) continue;
            if (-chrHits[i].second > 0 && -chrHits[i].second >= bestScore * top) {
                w = put_int(w, -(long long)chrHits[i].second); *w++ = ',';
                const std::string &cn = ann.names[chrHits[i].first - 1];
                memcpy(w, cn.data(), cn.size()); w += cn.size(); *w++ = ';';
            }
        }
    for (size_t i = 0; i < v.size(); ++i)
        if (v[i].score >= bestScore * top) { memcpy(w, comment->data() + v[i].s, v[i].e - v[i].s); w += v[i].e - v[i].s; *w++ = ';'; }
    *w++ = '\n';
    ret.resize(at + (size_t)(w - w0));
}

struct OutScratch;
struct OutCtx {
    const ReadBatch *b; const Annotation *ann; int megapathMode; double top; bool ignoreComments;
    OutScratch *scratch = nullptr;
    // BAM side
    BamWriter *bam = nullptr; std::string readGroup; bool printMDNM = false; int alignmentType = 2;
    int mismatchScore = -2, matchScore = 1, minMAPQ = 1, maxMAPQ = 60; bool bwaLike = true;
    AnnEx ax;
};
struct PairAln {       // mutable copy of one DeepDPAlignResult (the FASTQ writer edits scores / positions before the BAM writer runs)
    uint64_t a1, a2; int s1, s2, strand1, strand2, ed1, ed2, ns1, ns2, insertSize; const char *c1, *c2;
};
struct OutScratch { std::vector<PairAln> v; std::vector<std::pair<int, int>> h1, h2; };   // reused per formatting thread: no allocation per pair
struct SingleAln { uint64_t algnmt; int score, strand, editdist, num_sameScore; const char *cigar; };

static void unpack_read(const ReadBatch &b, uint32_t id, std::vector<uint8_t> &codes)
{
    const uint32_t *q = b.queries.data() + ((size_t)(id / 32) * 32 * b.wpq + id % 32);
    codes.resize(b.lens[id]);
    for (uint32_t i = 0; i < b.lens[id]; ++i) codes[i] = (q[(i >> 4) * 32] >> ((i & 15) << 1)) & 3;
}
static std::string xa_entry(const Annotation &ann, uint64_t algnmt, int strand, const char *spCigar, int editdist)
{
    uint64_t tp; uint32_t chr; ann.chrAndPos(algnmt, &tp, &chr);
    return ann.names[chr - 1] + "," + (strand == 2 ? "-" : "+") + std::to_string((unsigned long long)tp) + "," + convert_cigar(spCigar) + "," + std::to_string(editdist) + ";";
}

// one pair placed by deep DP or mate rescue: outputDeepDPResult2 (best = first maximal score sum, OutputDPResult.cpp:156-232)
// -> pairDeepDPOutputSAMAPI = pairDeepDPOutputFastqAPI (stdout) + BAM records (BGS-IO.cpp:1966-2800)
static void output_pair(OutCtx &o, std::string &fq, const mp_pair_result *first, const mp_pair_result *last, const char *cigars, int stageId)
{
    const ReadBatch &b = *o.b; const Annotation &ann = *o.ann;
    const uint32_t r1 = first->readID, r2 = r1 + 1;
    const int readlen1 = (int)b.lens[r1], readlen2 = (int)b.lens[r2];
    std::vector<PairAln> &v = o.scratch->v; v.clear();
    for (const mp_pair_result *p = first; p != last; ++p) {
        PairAln a; a.a1 = p->algnmt_1; a.a2 = p->algnmt_2; a.s1 = p->score_1; a.s2 = p->score_2; a.strand1 = p->strand_1; a.strand2 = p->strand_2;
        a.ed1 = p->editdist_1; a.ed2 = p->editdist_2; a.ns1 = p->num_sameScore_1; a.ns2 = p->num_sameScore_2; a.insertSize = p->insertSize;
        a.c1 = cigars + p->cigar_1; a.c2 = cigars + p->cigar_2;
        v.push_back(a);
    }
    // best pair = the first one with the maximal score sum (OutputDPResult.cpp:156-232): stage S1 marks it on the device (pad = 1,
    // k_pair_ready); mate-rescue groups are assembled on the host and are scanned here
    size_t best = v.size();
    for (const mp_pair_result *p = first; p != last; ++p) if (p->pad == 1) { best = (size_t)(p - first); break; }
    if (best == v.size()) {
        best = 0; int maxScore = v[0].s1 + v[0].s2;
        for (size_t i = 1; i < v.size(); ++i) if (v[i].s1 + v[i].s2 > maxScore) { best = i; maxScore = v[i].s1 + v[i].s2; }
    }
    if (o.megapathMode) {
        int best1 = 0, best2 = 0;
        std::vector<std::pair<int, int>> &h1 = o.scratch->h1, &h2 = o.scratch->h2; h1.clear(); h2.clear();
        for (PairAln &a : v) {
            int chr1 = -1, chr2 = -1;
            if (a.a1 != NOT_ALIGNED) chr1 = ann.targetChr(a.a1, readlen1);
            if (a.a2 != NOT_ALIGNED) chr2 = ann.targetChr(a.a2, readlen2);
            if (chr1 == -1) { a.a1 = NOT_ALIGNED; a.s1 = 0; }
            if (chr2 == -1) { a.a2 = NOT_ALIGNED; a.s2 = 0; }
            if (o.megapathMode == 2 && (a.a1 == NOT_ALIGNED || a.a2 == NOT_ALIGNED)) { a.a1 = a.a2 = NOT_ALIGNED; a.s1 = a.s2 = 0; }
            if (a.a1 == NOT_ALIGNED) a.s1 = 0;                                              // normalizeScore
            if (a.a2 == NOT_ALIGNED) a.s2 = 0;
            if (chr1 == chr2 && a.a1 != NOT_ALIGNED && a.a2 != NOT_ALIGNED) { int sum = a.s1 + a.s2; a.s1 = a.s2 = sum; }
            if (best1 < a.s1) best1 = a.s1;
            if (best2 < a.s2) best2 = a.s2;
            if (chr1 != -1) h1.push_back(std::make_pair(chr1, -a.s1));
            if (chr2 != -1) h2.push_back(std::make_pair(chr2, -a.s2));
        }
        header_line(fq, b, r1, ann, h1, best1, o.top, o.ignoreComments); seq_and_qual(fq, b, r1);
        header_line(fq, b, r2, ann, h2, best2, o.top, o.ignoreComments); seq_and_qual(fq, b, r2);
    }
    if (!o.bam) return;
    // ---- BAM (pairDeepDPOutputSAMAPI, BGS-IO.cpp:2112-2800) ----
    PairAln &B = v[best];
    if (B.a1 == NOT_ALIGNED && B.a2 == NOT_ALIGNED) return;
    std::vector<uint8_t> q1, q2; unpack_read(b, r1, q1); unpack_read(b, r2, q2);
    ReadView rv1 = { &b.name(r1), q1.data(), b.qual(r1), readlen1 }, rv2 = { &b.name(r2), q2.data(), b.qual(r2), readlen2 };
    const int num = (int)v.size();
    uint64_t tp_1 = 0, tp_2 = 0; uint32_t chr_1 = 0, chr_2 = 0;
    long long boundTrim1 = 0, boundTrim2 = 0; std::string newCigar1, newCigar2, cigarStr1, cigarStr2;
    MisInfo mi1, mi2; int rr1 = readlen1, rr2 = readlen2;
    int best_insert = (B.a1 != NOT_ALIGNED && B.a2 != NOT_ALIGNED) ? B.insertSize : 0;
    if (B.a1 != NOT_ALIGNED) {
        boundTrim1 = ann.chrAndPosBoundaryDP(readlen1, B.a1, B.c1, &tp_1, &chr_1, newCigar1);
        cigarStr1 = boundTrim1 ? convert_cigar(newCigar1.c_str()) : convert_cigar(B.c1);
        mi1 = mis_info_for_dp(o.ax, b.qual(r1), readlen1, B.a1, B.strand1, boundTrim1 ? newCigar1.c_str() : B.c1, boundTrim1);
        rr1 = ref_len_of_cigar(B.c1);
    }
    if (B.a2 != NOT_ALIGNED) {
        boundTrim2 = ann.chrAndPosBoundaryDP(readlen2, B.a2, B.c2, &tp_2, &chr_2, newCigar2);
        cigarStr2 = boundTrim2 ? convert_cigar(newCigar2.c_str()) : convert_cigar(B.c2);
        mi2 = mis_info_for_dp(o.ax, b.qual(r2), readlen2, B.a2, B.strand2, boundTrim2 ? newCigar2.c_str() : B.c2, boundTrim2);
        rr2 = ref_len_of_cigar(B.c2);
    }
    int bestPairNum = 0, bestPairScore = 0, secBestPairScore = 0;
    if (B.a1 != NOT_ALIGNED && B.a2 != NOT_ALIGNED) {
        bestPairNum = 1; bestPairScore = B.s1 + B.s2;
        for (int i = 0; i < num; ++i) {
            if ((size_t)i == best) continue;
            if (v[i].s1 + v[i].s2 == bestPairScore) bestPairNum++;
            else if (v[i].s1 + v[i].s2 > secBestPairScore) secBestPairScore = v[i].s1 + v[i].s2;
        }
    }
    // X0 / X1 of each end (BGS-IO.cpp:2311-2437)
    auto hit_counts = [&](bool firstEnd, int &bestHitNum, int &secBestHitNum) {
        bestHitNum = 0; secBestHitNum = 0;
        int bestScore = 0, secBestScore = 0; uint64_t bestPos = NOT_ALIGNED, secBestPos = NOT_ALIGNED;
        const uint64_t Ba = firstEnd ? B.a1 : B.a2;
        if (Ba != NOT_ALIGNED) { bestScore = firstEnd ? B.s1 : B.s2; bestPos = Ba; bestHitNum = 1; }
        if (Ba != NOT_ALIGNED && num > 1)
            for (int i = 0; i < num; ++i) {
                if ((size_t)i == best) continue;
                const int sc = firstEnd ? v[i].s1 : v[i].s2, ns = firstEnd ? v[i].ns1 : v[i].ns2; const uint64_t al = firstEnd ? v[i].a1 : v[i].a2;
                if (sc >= bestScore) {
                    if (sc == bestScore) { if (al != bestPos) bestHitNum += ns; }
                    else { secBestScore = bestScore; secBestHitNum = bestHitNum; secBestPos = bestPos; bestScore = sc; bestHitNum = ns; bestPos = al; }
                } else if (sc >= secBestScore) {
                    if (sc == secBestScore) { if (al != secBestPos) secBestHitNum += ns; }
                    else { secBestScore = sc; secBestPos = al; secBestHitNum = ns; }
                }
            }
    };
    int bestHitNum1, secBestHitNum1, bestHitNum2, secBestHitNum2;
    hit_counts(true, bestHitNum1, secBestHitNum1); hit_counts(false, bestHitNum2, secBestHitNum2);
    int mapq1 = 255, mapq2 = 255;
    if (o.alignmentType == 1 || o.alignmentType == 2) {
        bwa_like_pair(bestHitNum1, secBestHitNum1, bestHitNum2, secBestHitNum2, bestPairScore, bestPairNum, secBestPairScore, num - bestPairNum, readlen1, readlen2, &mapq1, &mapq2);
        if (boundTrim1) mapq1 = 0;
        if (boundTrim2) mapq2 = 0;
    }
    for (int end = 0; end < 2; ++end) {
        const bool e1 = end == 0;
        const uint64_t mine = e1 ? B.a1 : B.a2, mate = e1 ? B.a2 : B.a1;
        std::string xa;
        if (mine != NOT_ALIGNED && num > 1)
            for (int i = 0; i < num; ++i) {
                if ((size_t)i == best) continue;
                if (o.alignmentType == 2 && v[i].s1 + v[i].s2 < bestPairScore) continue;
                const uint64_t al = e1 ? v[i].a1 : v[i].a2;
                if (al == NOT_ALIGNED) continue;
                xa += xa_entry(ann, al, e1 ? v[i].strand1 : v[i].strand2, e1 ? v[i].c1 : v[i].c2, e1 ? v[i].ed1 : v[i].ed2);
            }
        int bh = e1 ? bestHitNum1 : bestHitNum2, sbh = e1 ? secBestHitNum1 : secBestHitNum2;
        if (o.alignmentType == 4) { bh = -1; sbh = -1; } else if (o.alignmentType != 1 && o.alignmentType != 2) sbh = -1;
        const MisInfo &mi = e1 ? mi1 : mi2; const ReadView &rv = e1 ? rv1 : rv2;
        const int strand = e1 ? B.strand1 : B.strand2, readlen = e1 ? readlen1 : readlen2;
        BamRecord rec;
        if (mine != NOT_ALIGNED) {
            int mq = e1 ? mapq1 : mapq2;
            if (mate == NOT_ALIGNED) {
                mq = mapq_for_dp(bh, e1 ? B.s1 : B.s2, readlen * o.matchScore, mi.avgMismatchQual, o.maxMAPQ, o.minMAPQ);
                if (e1 ? boundTrim1 : boundTrim2) mq = 0;
            }
            init_mapped(rec, rv, strand, xa, e1 ? cigarStr1 : cigarStr2, mi.numMismatch, mi.numMismatch + mi.gapExt, bh, sbh, mi.gapOpen, mi.gapExt, mi.md, mq,
                        o.readGroup, o.printMDNM, stageId);
        } else init_unmapped(rec, rv, e1 ? 1 : 1, "", o.readGroup);
        uint32_t flag = 1;
        if (B.a1 != NOT_ALIGNED && B.a2 != NOT_ALIGNED) flag |= 0x2;
        flag |= e1 ? 0x40 : 0x80;
        if (mine == NOT_ALIGNED) flag |= 0x4;
        if (mate == NOT_ALIGNED) flag |= 0x8;
        if (mine != NOT_ALIGNED && strand == 2) flag |= 0x10;
        if (mate != NOT_ALIGNED && (e1 ? B.strand2 : B.strand1) == 2) flag |= 0x20;
        rec.flag = flag;
        const uint32_t cm = e1 ? chr_1 : chr_2, co = e1 ? chr_2 : chr_1; const uint64_t tm = e1 ? tp_1 : tp_2, to = e1 ? tp_2 : tp_1;
        rec.tid = cm == 0 ? (co == 0 ? -1 : (int32_t)co - 1) : (int32_t)cm - 1;
        rec.pos = tm == 0 ? (to == 0 ? -1 : (int32_t)(to - 1)) : (int32_t)(tm - 1);
        rec.mtid = co == 0 ? (cm == 0 ? -1 : (int32_t)cm - 1) : (int32_t)co - 1;
        rec.mpos = to == 0 ? (tm == 0 ? -1 : (int32_t)(tm - 1)) : (int32_t)(to - 1);
        if (best_insert > 0) {
            const int rm = e1 ? rr1 : rr2, ro = e1 ? rr2 : rr1;
            if (tm > to) rec.isize = -(int32_t)(tm + rm - to); else rec.isize = (int32_t)(to + ro - tm);
        } else rec.isize = 0;
        o.bam->write(rec, rv.name->size() + 1);
    }
}

// a pair that is neither placed nor rescued: per-read single-end hits (unproperlypairDPOutputSAMAPI, BGS-IO.cpp:1448-1915)
static void output_unpaired(OutCtx &o, std::string &fq, uint32_t r1, std::vector<SingleAln> hits[2], int stageId)
{
    const ReadBatch &b = *o.b; const Annotation &ann = *o.ann;
    const uint32_t ids[2] = { r1, r1 + 1 };
    if (o.megapathMode) {
        for (int e = 0; e < 2; ++e) {
            int best = 0; std::vector<std::pair<int, int>> &h = o.scratch->h1; h.clear();
            const int hitNum = o.megapathMode == 2 ? 0 : (int)hits[e].size();
            for (int i = 0; i < hitNum; ++i) {
                SingleAln &a = hits[e][i];
                int chr = ann.targetChr(a.algnmt, b.lens[ids[e]]);
                if (chr < 0) { a.algnmt = NOT_ALIGNED; a.score = 0; } else h.push_back(std::make_pair(chr, -a.score));
                if (best < a.score) best = a.score;
            }
            header_line(fq, b, ids[e], ann, h, best, o.top, o.ignoreComments); seq_and_qual(fq, b, ids[e]);
        }
    }
    if (!o.bam) return;
    const int readlen[2] = { (int)b.lens[ids[0]], (int)b.lens[ids[1]] };
    std::vector<uint8_t> q[2]; unpack_read(b, ids[0], q[0]); unpack_read(b, ids[1], q[1]);
    ReadView rv[2] = { { &b.name(ids[0]), q[0].data(), b.qual(ids[0]), readlen[0] }, { &b.name(ids[1]), q[1].data(), b.qual(ids[1]), readlen[1] } };
    int bestIdx[2] = { -1, -1 }, bestScore[2] = { 0, 0 }, bestScoreNum[2] = { 0, 0 }, x1_t1[2] = { 0, 0 }, x1_t2[2] = { 0, 0 }, secondBestNum[2];
    uint64_t tp[2] = { 0, 0 }; uint32_t chr[2] = { 0, 0 }; long long boundTrim[2] = { 0, 0 }; int deletedEnd[2] = { 0, 0 }, mapq[2] = { 0, 0 };
    std::string newCigar[2], cigarStr[2]; MisInfo mi[2];
    for (int e = 0; e < 2; ++e) {
        const std::vector<SingleAln> &L = hits[e];
        if (!L.empty()) {
            bestIdx[e] = 0; bestScore[e] = L[0].score; bestScoreNum[e] = 1;
            for (size_t i = 1; i < L.size(); ++i) {
                if (L[i].score > bestScore[e]) { bestIdx[e] = (int)i; bestScore[e] = L[i].score; bestScoreNum[e] = 1; }
                else if (L[i].score == bestScore[e]) bestScoreNum[e]++;
            }
        }
        int secondBestScore = -9999; const int thres = (int)(0.7 * bestScore[e]);
        for (const SingleAln &a : L)
            if (a.score < bestScore[e]) { if (a.score > secondBestScore) secondBestScore = a.score; if (a.score >= thres) x1_t1[e]++; else x1_t2[e]++; }
        secondBestNum[e] = (o.alignmentType == 4 || o.alignmentType == 3) ? -1 : x1_t1[e] + x1_t2[e];
        if (bestIdx[e] >= 0 && L[bestIdx[e]].algnmt != NOT_ALIGNED && (o.alignmentType != 3 || bestScoreNum[e] == 1)) {
            const SingleAln &A = L[bestIdx[e]];
            boundTrim[e] = ann.chrAndPosBoundaryDP(readlen[e], A.algnmt, A.cigar, &tp[e], &chr[e], newCigar[e]);
            cigarStr[e] = boundTrim[e] ? convert_cigar(newCigar[e].c_str()) : convert_cigar(A.cigar, &deletedEnd[e]);
            mi[e] = mis_info_for_dp(o.ax, b.qual(ids[e]), readlen[e], A.algnmt, A.strand, boundTrim[e] ? newCigar[e].c_str() : A.cigar, boundTrim[e]);
            if (o.alignmentType == 4 || o.alignmentType == 3) mapq[e] = 255;
            else {
                double thr = 0.2 * readlen[e]; if (thr < 30.0) thr = 30.0;
                mapq[e] = mapq_for_single_dp(readlen[e] * o.matchScore, mi[e].avgMismatchQual, bestScoreNum[e], x1_t1[e], x1_t2[e], bestScore[e], secondBestScore,
                                             o.maxMAPQ, o.minMAPQ, (int)thr, o.bwaLike ? 1 : 0);
                if (!o.bwaLike) mapq[e] >>= 1;
                if (mapq[e] < o.minMAPQ) mapq[e] = o.minMAPQ;
                if (boundTrim[e]) mapq[e] = 0;        // (for the second read the reference resets it inside the same branch)
            }
            if ((o.alignmentType == 4 || o.alignmentType == 3) && e == 0 && boundTrim[e]) mapq[e] = 0;
        } else bestIdx[e] = -1;
    }
    if (!(o.alignmentType == 1 || o.alignmentType == 2)) return;       // the reference writes these records only for all-valid / all-best
    for (int e = 0; e < 2; ++e) {
        const int m = 1 - e;
        std::string xa;
        for (size_t i = 0; i < hits[e].size(); ++i) {
            if ((int)i == bestIdx[e]) continue;
            if (o.alignmentType == 2 && hits[e][i].score < bestScore[e]) continue;
            if (hits[e][i].algnmt == NOT_ALIGNED) continue;
            xa += xa_entry(ann, hits[e][i].algnmt, hits[e][i].strand, hits[e][i].cigar, hits[e][i].editdist);
        }
        BamRecord rec;
        if (bestIdx[e] >= 0)
            init_mapped(rec, rv[e], hits[e][bestIdx[e]].strand, xa, cigarStr[e], mi[e].numMismatch, mi[e].numMismatch + mi[e].gapExt, bestScoreNum[e], secondBestNum[e],
                        mi[e].gapOpen, mi[e].gapExt, mi[e].md, mapq[e], o.readGroup, o.printMDNM, stageId);
        else init_unmapped(rec, rv[e], 1, xa, o.readGroup);
        uint32_t flag = 1;
        if (bestIdx[e] < 0) flag |= 0x4;
        if (bestIdx[m] < 0) flag |= 0x8;
        flag |= e == 0 ? 0x40 : 0x80;
        if (bestIdx[e] >= 0 && hits[e][bestIdx[e]].strand == 2) flag |= 0x10;
        if (bestIdx[m] >= 0 && hits[m][bestIdx[m]].strand == 2) flag |= 0x20;
        rec.flag = flag;
        rec.tid = chr[e] == 0 ? (chr[m] == 0 ? -1 : (int32_t)chr[m] - 1) : (int32_t)chr[e] - 1;
        rec.pos = tp[e] == 0 ? (tp[m] == 0 ? -1 : (int32_t)(tp[m] - 1)) : (int32_t)(tp[e] - 1);
        rec.mtid = chr[m] == 0 ? (chr[e] == 0 ? -1 : (int32_t)chr[e] - 1) : (int32_t)chr[m] - 1;
        rec.mpos = tp[m] == 0 ? (tp[e] == 0 ? -1 : (int32_t)(tp[e] - 1)) : (int32_t)(tp[m] - 1);
        if (chr[0] > 0 && chr[0] == chr[1]) {
            // first record: tp_2 > tp_1 ? +(tp_2 - del2 + len2 - tp_1) : -(tp_1 - del1 + len1 - tp_2); second record mirrored (BGS-IO.cpp:1797-1803, 1893-1899)
            if (e == 0) rec.isize = tp[1] > tp[0] ? (int32_t)(tp[1] - deletedEnd[1] + readlen[1] - tp[0]) : -(int32_t)(tp[0] - deletedEnd[0] + readlen[0] - tp[1]);
            else rec.isize = tp[0] > tp[1] ? (int32_t)(tp[0] - deletedEnd[0] + readlen[0] - tp[1]) : -(int32_t)(tp[1] - deletedEnd[1] + readlen[1] - tp[0]);
        } else rec.isize = 0;
        o.bam->write(rec, rv[e].name->size() + 1);
    }
}

// ------------------------------------------------------------------------------------------------
// -lsam: the first consumer of the stdout contract fused into the driver.  runMegaPath.sh pipes `soap4 -F` into cc/fastq2lsam
// (:136, 162, 208, 305), which re-parses every record; here a formatted chunk (whole pairs, mate 1 then mate 2) is rewritten into the
// lines fastq2lsam prints (cc/fastq2lsam.cpp:28-77: name, 64/128/0, score, seq, qual | * *, "score,acc" list | *, [IGNORE]) before it
// leaves the process.  Records pair up by adjacent equal names after the /<digit> trim, as in fastq2lsam's main loop (:95-108).
// atoi of the characters [s, e) (glibc: (int) strtol, which saturates at the long limits)
static int atoi_range(const char *s, const char *e)
{
    while (s < e && isspace((unsigned char)*s)) ++s;
    bool neg = false;
    if (s < e && (*s == '-' || *s == '+')) { neg = *s == '-'; ++s; }
    const unsigned long long lim = neg ? 9223372036854775808ull : 9223372036854775807ull;
    unsigned long long v = 0; bool over = false;
    for (; s < e && *s >= '0' && *s <= '9'; ++s) {
        const unsigned d = (unsigned)(*s - '0');
        if (over || v > (lim - d) / 10) { over = true; continue; }
        v = v * 10 + d;
    }
    if (over) v = lim;
    return (int)(neg ? (long long)(0ull - v) : (long long)v);
}
static void fastq_chunk_to_lsam(const char *fqData, size_t fqSize, bool outputSeq, std::string &out)
{
    struct Rec { const char *name; size_t nameLen; const char *comm; size_t commLen; const char *seq; size_t seqLen; const char *qual; size_t qualLen; };
    out.clear(); out.reserve(fqSize / (outputSeq ? 1 : 4) + 4096);
    // one line through a raw pointer into space reserved for it (every "score,acc" item repeats the score: the list of a usual
    // comment is less than twice the comment, anything longer grows the space item by item)
    auto print = [&](const Rec &r, int whichEnd) {
        size_t cap = r.nameLen + 48 + (outputSeq ? r.seqLen + r.qualLen + 2 : 4) + 2 * r.commLen;
        const size_t at = out.size();
        out.resize(at + cap);
        char *w0 = &out[at], *w = w0;
        auto ensure = [&](size_t extra) {
            const size_t used = (size_t)(w - w0);
            if (used + extra + 16 > cap) { cap = (used + extra + 16) * 2; out.resize(at + cap); w0 = &out[at]; w = w0 + used; }
        };
        memcpy(w, r.name, r.nameLen); w += r.nameLen;
        *w++ = '\t';
        if (whichEnd == 1) { *w++ = '6'; *w++ = '4'; } else if (whichEnd == 2) { *w++ = '1'; *w++ = '2'; *w++ = '8'; } else *w++ = '0';
        *w++ = '\t';
        const bool ignore = r.commLen == 6 && !memcmp(r.comm, "IGNORE", 6);
        const int score = ignore ? -1 : (r.commLen > 6 ? atoi_range(r.comm + 6, r.comm + r.commLen) : 0);
        w = put_int(w, score); *w++ = '\t';
        if (outputSeq) { memcpy(w, r.seq, r.seqLen); w += r.seqLen; *w++ = '\t'; memcpy(w, r.qual, r.qualLen); w += r.qualLen; *w++ = '\t'; }
        else { memcpy(w, "*\t*\t", 4); w += 4; }
        if (score <= 0) *w++ = '*';
        else {
            // misc.h splitBy: fields between delimiters, a trailing empty field is dropped.  Every field after the first (the
            // "SCORE:n" one) is "score,acc[,acc...]" and prints as "score,acc" per accession, joined by ';'
            bool first = true;
            const char *c = r.comm, *ce = r.comm + r.commLen;
            const char *f = (const char *)memchr(c, ';', r.commLen);                 // end of field 0
            for (const char *i = f ? f + 1 : ce; i < ce;) {
                const char *j = (const char *)memchr(i, ';', (size_t)(ce - i)); if (!j) j = ce;
                const char *s0e = (const char *)memchr(i, ',', (size_t)(j - i)); if (!s0e) s0e = j;      // sub[0] = [i, s0e)
                for (const char *a = s0e < j ? s0e + 1 : j; a < j;) {
                    const char *e = (const char *)memchr(a, ',', (size_t)(j - a)); if (!e) e = j;
                    ensure((size_t)(s0e - i) + (size_t)(e - a) + 2);
                    if (!first) *w++ = ';'; else first = false;
                    memcpy(w, i, (size_t)(s0e - i)); w += s0e - i; *w++ = ','; memcpy(w, a, (size_t)(e - a)); w += e - a;
                    a = e + 1;
                }
                i = j + 1;
            }
        }
        if (score == -1) { memcpy(w, "\tIGNORE", 7); w += 7; }
        *w++ = '\n';
        out.resize(at + (size_t)(w - w0));
    };
    Rec last{}; bool hasLast = false;
    const char *p = fqData, *end = p + fqSize;
    while (p < end) {
        const char *l[4], *e[4];
        bool ok = true;
        for (int k = 0; k < 4; ++k) {
            l[k] = p; const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
            if (!nl) { ok = false; break; }
            e[k] = nl; p = nl + 1;
        }
        if (!ok) break;
        Rec r{};
        const char *h = l[0] + 1, *he = e[0];                                       // after '@'
        const char *ws = h; while (ws < he && !isspace((unsigned char)*ws)) ++ws;
        r.name = h; r.nameLen = (size_t)(ws - h);
        if (r.nameLen > 2 && h[r.nameLen - 2] == '/' && isdigit((unsigned char)h[r.nameLen - 1])) r.nameLen -= 2;      // trim_readno
        r.comm = ws < he ? ws + 1 : he; r.commLen = (size_t)(he - r.comm);
        r.seq = l[1]; r.seqLen = (size_t)(e[1] - l[1]); r.qual = l[3]; r.qualLen = (size_t)(e[3] - l[3]);
        if (hasLast) {
            if (last.nameLen == r.nameLen && !memcmp(last.name, r.name, r.nameLen)) { print(last, 1); print(r, 2); hasLast = false; }
            else { print(last, 0); last = r; }
        } else { hasLast = true; last = r; }
    }
    if (hasLast) print(last, 0);
}

int main(int argc, char **argv)
{
#ifdef MP_TEST_HOOKS
    // test-helper build only (bin/soap4_hosttest, tests/test_driver_host.py; no GPU needed): the shipped binary has none of these
    // hidden self-check used by tests/test_driver_host.py (no GPU needed): dump the records of a read file as the batch loader sees
    // them, through the zero-copy fast path (default) or through the kseq-style parser only ("generic")
    if (argc >= 5 && !strcmp(argv[1], "__load")) {           // hidden: time the batch loader alone (no GPU): __load r1 r2 maxReadLength
        fill_char_map();
        SeqReader r1, r2; if (!r1.open(argv[2]) || !r2.open(argv[3])) return 1;
        const uint32_t maxLen = (uint32_t)atoi(argv[4]);
        uint64_t total = 0, sum = 0; const double t0 = now_s();
        ReadBatch b; b.maxReadLength = maxLen; b.wpq = (maxLen + 15) / 16;
        for (;;) {
            const double t1 = now_s();
            uint32_t n = load_batch(r1, r2, b, 12 * 8192 * 128 / 6, argc >= 6 ? (unsigned)atoi(argv[5]) : 4u);
            if (n == 0) break;
            total += n; for (uint32_t i = 0; i < n; i += 1000) sum += b.lens[i] + b.queries[i] + (unsigned char)b.qual(i)[0];
            fprintf(stderr, "batch of %u reads in %.3f s\n", n, now_s() - t1);
        }
        fprintf(stderr, "%llu reads in %.3f s (checksum %llu)\n", (unsigned long long)total, now_s() - t0, (unsigned long long)sum);
        return 0;
    }
    if (argc >= 6 && !strcmp(argv[1], "__pack")) {           // hidden: batch loader output to a file (no GPU): __pack r1 r2 maxReadLength out [threads]
        fill_char_map();
        SeqReader r1, r2; if (!r1.open(argv[2]) || !r2.open(argv[3])) return 1;
        ReadBatch b; b.maxReadLength = (uint32_t)atoi(argv[4]); b.wpq = (b.maxReadLength + 15) / 16;
        const uint32_t n = load_batch(r1, r2, b, 12 * 8192 * 128 / 6, argc >= 7 ? (unsigned)atoi(argv[6]) : 3u);
        FILE *o = fopen(argv[5], "wb"); if (!o) return 1;
        const uint32_t hdr[2] = { n, b.wpq };
        fwrite(hdr, 4, 2, o); fwrite(b.lens.data(), 4, n, o);
        fwrite(b.queries.data(), 4, ((size_t)n + 31) / 32 * 32 * b.wpq, o);
        for (uint32_t id = 0; id < n; ++id) fprintf(o, "%s|%s|%.*s\n", b.name(id).c_str(), b.hasComment(id) ? b.comment(id).c_str() : "", (int)b.qlen(id), b.qual(id));
        fclose(o);
        return 0;
    }
    if (argc >= 4 && !strcmp(argv[1], "__bgzf")) {           // hidden: file -> BGZF blocks compressed in two chunks + EOF block (no GPU)
        FILE *in = fopen(argv[2], "rb"); if (!in) return 1;
        std::vector<uint8_t> data; uint8_t tmp[65536]; size_t n;
        while ((n = fread(tmp, 1, sizeof tmp, in)) > 0) data.insert(data.end(), tmp, tmp + n);
        fclose(in);
        BgzfWriter w; if (!w.open(argv[3])) return 1;
        const size_t head = std::min<size_t>(data.size(), 10);       // a few bytes through the buffered path, as the BAM header goes
        w.write(data.data(), head);
        const size_t mid = head + (data.size() - head) / 3;
        std::vector<uint8_t> a, b;
        BgzfWriter::compress_all(data.data() + head, mid - head, a);
        BgzfWriter::compress_all(data.data() + mid, data.size() - mid, b);
        w.write_blocks(a); w.write_blocks(b);
        w.close();
        return 0;
    }
    if (argc >= 4 && !strcmp(argv[1], "__lsam")) {           // hidden: annotated FASTQ file -> the -lsam lines (no GPU): __lsam file outputSeq
        FILE *in = fopen(argv[2], "rb"); if (!in) return 1;
        std::string data; char tmp[65536]; size_t n;
        while ((n = fread(tmp, 1, sizeof tmp, in)) > 0) data.append(tmp, n);
        fclose(in);
        const double tc = now_s();
        std::string out; fastq_chunk_to_lsam(data.data(), data.size(), atoi(argv[3]) != 0, out);
        fprintf(stderr, "converted %.1f MB in %.3f s\n", data.size() / 1e6, now_s() - tc);
        fwrite(out.data(), 1, out.size(), stdout);
        return 0;
    }
    if (argc >= 5 && !strcmp(argv[1], "__stage")) {          // hidden: batch boundaries of the device-ingest staging (no GPU): __stage file maxRec threads [bytesPerRec]
        SeqReader r; if (!r.open(argv[2])) { fprintf(stderr, "cannot open %s\n", argv[2]); return 1; }
        if (!r.mapped) { printf("unmapped\n"); return 0; }
        const uint32_t maxRec = (uint32_t)atoi(argv[3]); const unsigned thr = (unsigned)atoi(argv[4]);
        double bpr = argc >= 6 ? atof(argv[5]) : 0;
        for (;;) {
            // exact location, then the fused copy + count with the running estimate: both must name the same byte range
            size_t np = 0; const long n = locate_records(r, maxRec, thr, &np);
            if (bpr <= 0) { SeqReader::View v; const char *nx = nullptr; if (r.pos < r.end && SeqReader::view_record(r.base + r.pos, r.base + r.end, v, &nx) == 1) bpr = (double)(nx - (r.base + r.pos)); else bpr = 64; }
            const size_t cap = std::min<size_t>((size_t)((double)maxRec * bpr * 1.03) + ((size_t)2 << 18), r.end - r.pos + 64);
            std::vector<char> dst(cap + 64);
            size_t bytes = 0; const long m = stage_file(r, bpr, maxRec, thr, dst.data(), cap, &bytes);
            const bool same = m > 0 && bytes == np - r.pos && !memcmp(dst.data(), r.base + r.pos, bytes);
            printf("%ld %zu %ld %zu %d\n", n, np, m, bytes, same ? 1 : 0);
            if (n <= 0) break;
            bpr = (double)(np - r.pos) / (double)n;
            r.pos = np;
        }
        return 0;
    }
    if (argc >= 3 && !strcmp(argv[1], "__parse")) {
        SeqReader r; if (!r.open(argv[2])) { fprintf(stderr, "cannot open %s\n", argv[2]); return 1; }
        const bool generic = argc >= 4 && !strcmp(argv[3], "generic");
        std::string nm, cm, sq, ql; SeqReader::View v;
        for (;;) {
            int st = generic ? 0 : r.read_fast(v);
            if (st < 0) break;
            if (st == 1) { nm.assign(v.name, v.nameLen); cm.assign(v.comment, v.commentLen); sq.assign(v.seq, v.seqLen); ql.assign(v.qual, v.seqLen); }
            else { int l = r.read(nm, cm, sq, ql); if (l < 0) { if (l == -2) printf("ERR\n"); break; } }
            printf("%s|%s|%s|%s\n", nm.c_str(), cm.c_str(), sq.c_str(), ql.c_str());
        }
        return 0;
    }
#endif
    Options opt;
    if (!parse_args(argc, argv, opt)) return 1;
    const double t0 = now_s();
    {   // large inputs: every kernel is loaded with the library, not at its first launch inside the batch loop (must be set before the
        // first CUDA call); small runs keep lazy loading, which starts the process faster
        struct stat sb0;
        if (stat(opt.query1.c_str(), &sb0) == 0 && sb0.st_size > (off_t)(48 << 20)) setenv("CUDA_MODULE_LOADING", "EAGER", 0);
    }
    Ini ini;
    std::string iniPath = opt.iniFile.empty() ? std::string(argv[0]) + ".ini" : opt.iniFile;
    if (!ini.load(iniPath)) { fprintf(stderr, "Failed to open config file ... %s\n", iniPath.c_str()); return 1; }
    fprintf(stderr, "\n[Main] soap4 (megapath_b200, B200 hot path)\n");
    fprintf(stderr, "Number of CPU threads: %d\n", opt.numCpuThreads);
    fprintf(stderr, "[Main] Loading read files %s and %s\n", opt.query1.c_str(), opt.query2.c_str());
    if (ini.geti("OtherSettings:SkipSOAP3Alignment", 0) != 1) { fprintf(stderr, "SkipSOAP3Alignment=0 is not supported (the reference asserts, alignment.cpp:66)\n"); return 1; }
    const int maxLen = opt.maxReadLength;
    const int nRounds = maxLen > 120 ? ini.geti("DP:NumberOfRoundOfDeepDPForLongReads", 0) : ini.geti("DP:NumberOfRoundOfDeepDPForShortReads", 0);
    const char *schemeKey = maxLen > 120 ? "SeedingRound1ForLongReads:mmpSeedingScheme" : "SeedingRound1ForShortReads:mmpSeedingScheme";
    if (nRounds != 1 || ini.geti(schemeKey, 0) != 1) { fprintf(stderr, "only one deep-DP round with mmpSeedingScheme=1 is supported (DV-DPForBothUnalign.cpp:262-266)\n"); return 1; }
    mp_align_params P; mp_default_params(&P, 0);
    P.mmp.seedSAsizeThreshold = ini.geti("MMP:mmpSeedSAsizeThreshold", 30); P.mmp.seedMinLength = ini.geti("MMP:mmpSeedMinLength", 17);
    P.mmp.uniqThreshold = ini.geti("MMP:mmpUniqThreshold", 6); P.mmp.indelFuzz = ini.geti("MMP:mmpIndelFuzz", 5);
    P.mmp.goodSeedLen = ini.geti("MMP:mmpGoodSeedLen", 27); P.mmp.reseedLen = ini.geti("MMP:mmpReseedLen", 18);
    P.mmp.reseedRLTratio = ini.getd("MMP:mmpReseedRLTratio", 0.85); P.mmp.reseedAbsDiff = ini.geti("MMP:mmpReseedAbsDiff", 4);
    P.mmp.shortSeedRatio = ini.getd("MMP:mmpShortSeedRatio", 0.5);
    P.matchScore = ini.geti("DP:MatchScore", 1); P.mismatchScore = ini.geti("DP:MismatchScore", -2);
    P.openGapScore = ini.geti("DP:GapOpenScore", -3); P.extendGapScore = ini.geti("DP:GapExtendScore", -1);
    P.softClipLeft = ini.geti("Clipping:MaxFrontLenClipped", 3); P.softClipRight = ini.geti("Clipping:MaxEndLenClipped", 8);
    std::string arr = ini.gets("PairEnd:StrandArrangement", "+/-");
    P.peStrandLeftLeg = (arr == "-/+" || arr == "-/-") ? 2 : 1; P.peStrandRightLeg = (arr == "+/+" || arr == "-/+") ? 1 : 2;
    P.skipDefaultDP = ini.geti("OtherSettings:SkipDefaultDP", 0);
    P.maxReadLength = maxLen; P.insert_high = opt.insert_high;
    const double top = opt.top / 100.0;

    fill_char_map();
    SeqReader r1, r2;
    if (!r1.open(opt.query1, opt.device) || !r2.open(opt.query2, opt.device)) { fprintf(stderr, "Cannot open the read files\n"); return 1; }
    uint32_t maxNumQueries = 12 * 8192 * 128 / 6;                  // SOAP4.cpp:206
    if (const char *e = getenv("MP_BATCH_READS")) {                // smaller batches (multi-batch / multi-context tests on small inputs)
        const long v = atol(e); if (v >= 64 && v <= 12 * 8192 * 128 / 6) maxNumQueries = (uint32_t)v & ~63u;
    }
    if (const char *e = getenv("MP_CONTEXTS_PER_GPU")) { int v = atoi(e); if (v >= 1 && v <= 8) opt.contextsPerGpu = v; }
    const unsigned ioThreads = (unsigned)std::min(8, std::max(1, opt.numCpuThreads));
    // staging threads per mate file: four already move a batch in ~25 ms (measured: 2 -> 23.6, 4 -> 25.5, 8 -> 19, 16 -> 18 M pairs/s on 16
    // cores; more only take the cores the context threads need to keep their GPU queues full)
    unsigned stageThreads = (unsigned)std::min(4, std::max(1, opt.numCpuThreads));
    if (const char *e = getenv("MP_STAGE_THREADS")) { const int v = atoi(e); if (v >= 1 && v <= 64) stageThreads = (unsigned)v; }
    // ---- FASTQ ingest and annotated-FASTQ egress on the device (mp_fastq_upload / mp_format_fastq): plain FASTQ files in, -F / -P text
    //      out.  Everything else (.gz, pipes, -b, anything but strict four-line records) takes the host parser / formatter below.
    //      MP_HOST_IO=1 forces the host loops (tests compare the two). ----
    bool deviceIO = opt.megapathMode != 0 && !opt.outputBAM && r1.mapped && r2.mapped && !getenv("MP_HOST_IO");
    struct RawBatch { char *pin = nullptr; size_t pinCap = 0, bytes1 = 0, off2 = 0, bytes2 = 0; uint32_t nReads = 0; };
    std::mutex pinMu; std::vector<std::pair<char *, size_t>> pinPool;
    auto pin_take = [&](size_t need) -> std::pair<char *, size_t> {
        {
            std::lock_guard<std::mutex> lk(pinMu);
            for (size_t k = 0; k < pinPool.size(); ++k) if (pinPool[k].second >= need) { auto r = pinPool[k]; pinPool.erase(pinPool.begin() + (long)k); return r; }
            if (!pinPool.empty()) { mp_host_free(pinPool.back().first); pinPool.pop_back(); }          // too small: replace it
        }
        const size_t cap = need + need / 16;
        return std::make_pair((char *)mp_host_alloc(cap), cap);
    };
    auto pin_give = [&](char *p, size_t cap) { if (p) { std::lock_guard<std::mutex> lk(pinMu); pinPool.emplace_back(p, cap); } };
    // Staging buffers: one per batch in flight (a batch holds its buffer from staging until the ordered writer is through with its
    // output text).  Page-locking a gigabyte takes half a second and stalls every CUDA call of the process while it runs, so the buffers
    // are made here, by a thread that runs beside the index load, sized from the first record of either file.
    double bytesPerRec[2] = { 0, 0 };                              // running estimate per mate file (first record, then the last batch's mean)
    auto window_cap = [&](int m, const SeqReader &r) -> size_t {  // room for one batch of mate m's text: the estimate + 3 % + two count blocks
        const size_t est = (size_t)((double)(maxNumQueries / 2) * bytesPerRec[m] * 1.03) + ((size_t)2 << 18);
        return (std::min<size_t>(est, r.end - r.pos + 64) + 63) & ~(size_t)63;
    };
    // the formatted text of a batch comes back into the buffer its input came from: room for what the headers grow by (64 bytes per read to
    // begin with; batches with long SCORE: lists raise it for the buffers taken after them)
    std::atomic<size_t> growPerRead(64);
    auto batch_need = [&]() -> size_t { return window_cap(0, r1) + window_cap(1, r2) + (size_t)maxNumQueries * growPerRead.load() + ((size_t)1 << 20); };
    // device-inflated .gz inputs: [pos, end) must hold a whole batch before a batch is located in it
    auto ensure_batch = [&]() {
        std::thread e2([&] { r2.ensure_lines(4ull * (maxNumQueries / 2) + 4); });
        r1.ensure_lines(4ull * ((maxNumQueries + 1) / 2) + 4);
        e2.join();
    };
    ensure_batch();
    std::thread pinThread;
    if (deviceIO) {
        SeqReader::View v; const char *nx = nullptr;
        if (r1.end > r1.pos && r2.end > r2.pos && SeqReader::view_record(r1.base + r1.pos, r1.base + r1.end, v, &nx) == 1) bytesPerRec[0] = (double)(nx - (r1.base + r1.pos));
        if (bytesPerRec[0] > 0 && SeqReader::view_record(r2.base + r2.pos, r2.base + r2.end, v, &nx) == 1) bytesPerRec[1] = (double)(nx - (r2.base + r2.pos));
        if (bytesPerRec[0] > 0 && bytesPerRec[1] > 0) {
            const size_t need = batch_need(), cap = need + need / 16;
            const size_t batches = (size_t)((double)(r1.end - r1.pos) / (bytesPerRec[0] * (double)(maxNumQueries / 2))) + 1;
            const size_t count = std::min<size_t>((size_t)opt.numGpus * (size_t)opt.contextsPerGpu + 3, batches);
            pinThread = std::thread([&, cap, count] { for (size_t k = 0; k < count; ++k) { char *p = (char *)mp_host_alloc(cap); if (p) pin_give(p, cap); } });
        } else if (r1.end > r1.pos || r2.end > r2.pos) deviceIO = false;           // the first record is not a plain four-line one
    }

    // one index replica per GPU (loaded in parallel), contextsPerGpu contexts sharing it (mp_clone)
    fprintf(stderr, "[Main] loading index into device...\n");
    std::vector<mp_context *> owners(opt.numGpus, nullptr), contexts;
    {
        std::vector<std::thread> loaders; std::vector<std::string> errs(opt.numGpus);
        for (int g = 0; g < opt.numGpus; ++g)
            loaders.emplace_back([&, g]() {
                if (mp_init(opt.device + g, &owners[g]) || mp_index_load(owners[g], opt.indexName.c_str())) errs[g] = mp_last_error();
            });
        for (std::thread &t : loaders) t.join();
        for (int g = 0; g < opt.numGpus; ++g) if (!errs[g].empty()) { fprintf(stderr, "%s\n", errs[g].c_str()); return 1; }
        for (int g = 0; g < opt.numGpus; ++g) {
            if (mp_index_prepare(owners[g], &P)) { fprintf(stderr, "%s\n", mp_last_error()); return 1; }
            contexts.push_back(owners[g]);
            for (int k = 1; k < opt.contextsPerGpu; ++k) {
                mp_context *c = nullptr;
                if (mp_clone(owners[g], &c)) { fprintf(stderr, "%s\n", mp_last_error()); return 1; }
                contexts.push_back(c);
            }
        }
    }
    {   // large inputs: size every context's batch buffers before the batch loop (part of the set-up time, like the index load) so that
        // no batch pays for allocations; small inputs keep the lazy sizing
        struct stat sb;
        if (stat(opt.query1.c_str(), &sb) == 0 && sb.st_size > (off_t)(48 << 20)) {
            uint32_t batchReads = 12 * 8192 * 128 / 6;
            if (const char *e = getenv("MP_BATCH_READS")) { const long v = atol(e); if (v >= 64 && v <= (long)batchReads) batchReads = (uint32_t)v & ~63u; }
            for (mp_context *c : contexts) if (mp_reserve(c, &P, batchReads)) { fprintf(stderr, "%s\n", mp_last_error()); return 1; }
        }
    }
    // -b: BAM records are compressed on the device, by the worker's own context, in pieces of at most bgzfPiece bytes staged in
    // page-locked buffers of the pool (two per context, made here so that the loop allocates nothing)
    const bool deviceBgzf = opt.outputBAM && !getenv("MP_HOST_IO");
    const uint64_t bgzfPiece = 512ull * 0xff00, bgzfCap = MP_BGZF_BOUND(bgzfPiece);
    if (deviceBgzf) {
        for (mp_context *c : contexts) {
            if (mp_bgzf_reserve(c, bgzfPiece)) { fprintf(stderr, "%s\n", mp_last_error()); return 1; }
            for (int k = 0; k < 2; ++k) { char *p = (char *)mp_host_alloc(bgzfCap); if (!p) { fprintf(stderr, "%s\n", mp_last_error()); return 1; } pin_give(p, bgzfCap); }
        }
    }
    if (pinThread.joinable()) pinThread.join();
    Annotation ann;
    if (!ann.load(opt.indexName)) return 1;
    // -> 1: the next batch staged in page-locked memory (file positions advanced), 0: end of both files, -1: not for the device path
    auto stage_raw = [&](RawBatch &rb) -> int {
        static const bool ltiming = getenv("MP_DRIVER_TIMING") != nullptr;
        const double ts0 = now_s(), gz0 = r1.gzSeconds + r2.gzSeconds;
        ensure_batch();
        const double tInflate = r1.gzSeconds + r2.gzSeconds - gz0;
        const size_t cap1 = window_cap(0, r1), cap2 = window_cap(1, r2);
        auto pc = pin_take(cap1 + cap2 + (size_t)maxNumQueries * growPerRead.load() + ((size_t)1 << 20));
        if (!pc.first) { fprintf(stderr, "%s\n", mp_last_error()); exit(1); }
        rb.pin = pc.first; rb.pinCap = pc.second; rb.off2 = cap1;
        const double ts1 = now_s();
        long n1 = 0, n2 = 0;
        std::thread t2([&] { n2 = stage_file(r2, bytesPerRec[1], maxNumQueries / 2, stageThreads, rb.pin + rb.off2, cap2, &rb.bytes2); });
        n1 = stage_file(r1, bytesPerRec[0], (maxNumQueries + 1) / 2, stageThreads, rb.pin, cap1, &rb.bytes1);
        t2.join();
        const double ts2 = now_s();
        size_t p1 = r1.pos + rb.bytes1, p2 = r2.pos + rb.bytes2;
        if (n1 == -2 || n2 == -2) {
            // records much longer than the estimate: locate the batch exactly, then copy it
            std::thread l2([&] { n2 = locate_records(r2, maxNumQueries / 2, stageThreads, &p2); });
            n1 = locate_records(r1, (maxNumQueries + 1) / 2, stageThreads, &p1);
            l2.join();
            if (n1 > 0 && n2 > 0) {
                rb.bytes1 = p1 - r1.pos; rb.bytes2 = p2 - r2.pos; rb.off2 = (rb.bytes1 + 63) & ~(size_t)63;
                const size_t need = rb.off2 + rb.bytes2 + (size_t)maxNumQueries * growPerRead.load() + ((size_t)1 << 20);
                if (need > rb.pinCap) {
                    pin_give(rb.pin, rb.pinCap);
                    pc = pin_take(need);
                    if (!pc.first) { fprintf(stderr, "%s\n", mp_last_error()); exit(1); }
                    rb.pin = pc.first; rb.pinCap = pc.second;
                }
                std::thread c2([&] { parallel_copy(rb.pin + rb.off2, r2.base + r2.pos, rb.bytes2, stageThreads); });
                parallel_copy(rb.pin, r1.base + r1.pos, rb.bytes1, stageThreads);
                c2.join();
            }
        }
        if (n1 <= 0 || n2 <= 0 || rb.bytes1 >= 0xFFFFFFF0ull || rb.bytes2 >= 0xFFFFFFF0ull) {
            pin_give(rb.pin, rb.pinCap); rb.pin = nullptr;
            return n1 == 0 && n2 == 0 ? 0 : -1;
        }
        if (n1 != n2) { fprintf(stderr, "Error: number of sequences of pair-end files not matched.\n"); exit(1); }
        rb.nReads = 2 * (uint32_t)n1;
        bytesPerRec[0] = (double)rb.bytes1 / (double)n1; bytesPerRec[1] = (double)rb.bytes2 / (double)n2;
        r1.pos = p1; r2.pos = p2;
        if (ltiming) fprintf(stderr, "[timing] stage: inflate %.3f buffer %.3f copy + count %.3f rest %.3f s (%.0f MB)\n", tInflate, ts1 - ts0 - tInflate, ts2 - ts1,
                             now_s() - ts2, (rb.bytes1 + rb.bytes2) / 1e6);
        return 1;
    };
    RawBatch firstRaw; bool haveFirstRaw = false;
    if (deviceIO) {
        std::vector<uint64_t> nameOff(ann.numSeq + 1, 0); std::string nameBlob;
        for (uint32_t i = 0; i < ann.numSeq; ++i) { nameOff[i] = nameBlob.size(); nameBlob += ann.names[i]; }
        nameOff[ann.numSeq] = nameBlob.size();
        std::vector<uint64_t> trStart(ann.tr.size()); std::vector<uint32_t> trChr(ann.tr.size());
        for (size_t k = 0; k < ann.tr.size(); ++k) { trStart[k] = ann.tr[k].startPos; trChr[k] = ann.tr[k].chrID; }
        mp_annotation A; memset(&A, 0, sizeof A);
        A.dnaLength = ann.dnaLength; A.numSeq = ann.numSeq; A.gridEntries = (uint32_t)ann.grid.size(); A.numTranslate = (uint32_t)ann.tr.size();
        A.grid = ann.grid.data(); A.trStartPos = trStart.data(); A.trChrID = trChr.data(); A.names = nameBlob.data(); A.nameOffsets = nameOff.data();
        for (mp_context *c : contexts) if (mp_annotation_upload(c, &A)) { fprintf(stderr, "[Main] %s; formatting on the host\n", mp_last_error()); deviceIO = false; break; }
    }
    if (deviceIO) {
        // The first batch is staged and indexed here, as part of the set-up: its verdict decides between the device and the host loops
        // for the whole run (CRLF or multi-line files fail it), and its read lengths give the first-batch parameters (SOAP4.cpp:458-474).
        const size_t save1 = r1.pos, save2 = r2.pos;
        const int st = stage_raw(firstRaw);
        if (st == 1) {
            const uint32_t *lens = nullptr;
            const int rc = mp_fastq_upload(contexts[0], firstRaw.pin, firstRaw.bytes1, firstRaw.pin + firstRaw.off2, firstRaw.bytes2, firstRaw.nReads / 2,
                                           ((uint32_t)maxLen + 15) / 16, (uint32_t)maxLen, &lens);
            if (rc == 0) {
                std::vector<uint32_t> lv(lens, lens + firstRaw.nReads);
                const uint32_t d1 = detect_read_length(lv, firstRaw.nReads, 0), d2 = detect_read_length(lv, firstRaw.nReads, 1);
                if (opt.insert_low < (int)d2) opt.insert_low = (int)d2;
                if (opt.insert_low < (int)d1) opt.insert_low = (int)d1;
                P.insert_low = opt.insert_low;
                haveFirstRaw = true;
                // every context's ingest / egress buffers sized like the first batch (no cudaMalloc inside the batch loop)
                if (r1.pos < r1.end)
                    for (mp_context *c : contexts) if (mp_fastq_reserve(c, firstRaw.bytes1 + firstRaw.bytes2 + (firstRaw.bytes1 + firstRaw.bytes2) / 16, firstRaw.nReads / 2)) { fprintf(stderr, "%s\n", mp_last_error()); return 1; }
            } else if (rc == MP_ERR_FORMAT) {
                fprintf(stderr, "[Main] %s: host parser\n", mp_last_error());
                pin_give(firstRaw.pin, firstRaw.pinCap); r1.pos = save1; r2.pos = save2; deviceIO = false;
            } else { fprintf(stderr, "%s\n", mp_last_error()); return 1; }
        } else if (st < 0) { r1.pos = save1; r2.pos = save2; deviceIO = false; }
        // st == 0: empty input, the reader below ends at once
    }
    fprintf(stderr, "[Main] FASTQ parsing and output formatting on the %s\n", deviceIO ? "device" : "host");
    fprintf(stderr, "[Main] Finished loading index into device.\n");
    const double tIndex = now_s();
    fprintf(stderr, "[Main] Loading time : %9.4f seconds\n\n", tIndex - t0);
    fprintf(stderr, "[Main] top_percentage: %f\n", top);
    fprintf(stderr, "[Main] Reference sequence length : %llu\n\n", (unsigned long long)ann.dnaLength);
    OutCtx octx;
    octx.ann = &ann; octx.megapathMode = opt.megapathMode; octx.top = top; octx.ignoreComments = opt.ignoreComments != 0;
    octx.readGroup = opt.query1; octx.printMDNM = opt.printMDNM != 0; octx.alignmentType = opt.alignmentType;
    octx.mismatchScore = P.mismatchScore; octx.matchScore = P.matchScore; octx.minMAPQ = ini.geti("Score:MinMAPQ", 1); octx.maxMAPQ = ini.geti("Score:MaxMAPQ", 40);
    octx.bwaLike = ini.geti("Score:BWALikeScore", 0) != 0;
    BamWriter bamDP, bamGout, bamUnpair;
    std::vector<uint8_t> hostPac;
    if (opt.outputBAM) {
        if (!octx.bwaLike) { fprintf(stderr, "-b needs Score:BWALikeScore=1 (the only MAPQ scheme of the shipped .ini files)\n"); return 1; }
        bwase_initialize();
        // SAMOutputHeaderConstruct (SAM.cpp:83-134)
        std::vector<std::string> tnames; std::vector<uint32_t> tlens; std::string sq;
        for (uint32_t i = 0; i < ann.numSeq; ++i) {
            std::string nm = ann.names[i]; size_t e = nm.find_first_of(" \t\r\n"); if (e != std::string::npos) nm.resize(e);
            tnames.push_back(nm); tlens.push_back((uint32_t)ann.actualLen[i]);
            sq += "@SQ\tSN:" + nm + "\tLN:" + std::to_string(tlens.back()) + "\n";
        }
        std::string text = "@HD\tVN:1.3\tSO:unsorted\n@RG\tID:" + octx.readGroup + "\tSM:\t\n" + sq + "@PG\tID:soap4\tPN:soap4\tVN:megapath_b200\n";
        bool ok = bamDP.open(opt.outputPrefix + ".dpout.1", text, tnames, tlens) && bamUnpair.open(opt.outputPrefix + ".unpair", text, tnames, tlens) &&
                  bamGout.open(opt.outputPrefix + ".gout.1", text, tnames, tlens);
        for (int t = 2; ok && t <= opt.numCpuThreads; ++t) {       // the reference opens one .gout file per CPU thread; the pipeline globs them
            BamWriter extra; ok = extra.open(opt.outputPrefix + ".gout." + std::to_string(t), text, tnames, tlens); extra.close();
        }
        if (!ok) { fprintf(stderr, "cannot create the BAM output files with prefix %s\n", opt.outputPrefix.c_str()); return 1; }
        if (opt.printMDNM) {                                        // MD strings need the text
            FILE *pf = fopen((opt.indexName + ".pac").c_str(), "rb");
            if (!pf) { fprintf(stderr, "cannot open %s.pac\n", opt.indexName.c_str()); return 1; }
            hostPac.resize((ann.dnaLength + 3) / 4 + 8);
            if (fread(hostPac.data(), 1, (ann.dnaLength + 3) / 4, pf) != (ann.dnaLength + 3) / 4) { fprintf(stderr, "short .pac\n"); return 1; }
            fclose(pf); octx.ax.pac = hostPac.data();
        }
    }

    // ---- pipeline: reader thread -> GPU workers (one per context; each formats its own batch) -> ordered writer (this thread).
    //      The reference overlaps read loading with alignment the same way (aio_thread.cpp:804, SOAP4.cpp:424-441, 576-585). ----
    struct Job {
        uint64_t seq = 0; ReadBatch *b = nullptr; uint32_t nReads = 0; std::vector<std::string> fqParts; std::string log; std::vector<uint8_t> bam[3];
        uint64_t pairsAligned = 0; double loadSeconds = 0, alignSeconds = 0; bool failed = false;
        // device ingest / egress: the batch's FASTQ text staged in page-locked memory; the formatted text comes back into the same buffer
        bool dev = false, uploaded = false; RawBatch raw; uint64_t outBytes = 0;
    };
    std::mutex mu; std::condition_variable cvIn, cvOut, cvRoom;
    std::vector<ReadBatch *> batchPool;                            // recycled read batches (guarded by mu)
    std::deque<Job *> inq; std::map<uint64_t, Job *> doneq; bool readerDone = false; size_t inflight = 0;
    Job *firstJob = nullptr;                                       // the batch already uploaded to contexts[0] (device ingest)
    const size_t maxInflight = contexts.size() + 2;
    const int stageUnpaired = P.skipDefaultDP ? 2 : 3;

    std::thread reader([&]() {
        uint64_t seq = 0; bool detected = false; double last = now_s();
        bool devIO = deviceIO;
        if (haveFirstRaw) {                                         // staged and uploaded to the first context during set-up
            Job *j = new Job; j->dev = true; j->uploaded = true; j->raw = firstRaw; j->nReads = firstRaw.nReads; j->seq = seq++;
            detected = true;
            std::unique_lock<std::mutex> lk(mu);
            ++inflight; firstJob = j; cvIn.notify_all();
        }
        for (;;) {
            Job *j = new Job;
            if (devIO) {
                const int st = stage_raw(j->raw);
                if (st == 0) { delete j; break; }
                if (st == 1) { j->dev = true; j->nReads = j->raw.nReads; }
                else devIO = false;                                 // the rest of the input goes through the sequential parser
            }
            if (!j->dev) {
            { std::lock_guard<std::mutex> lk(mu); if (!batchPool.empty()) { j->b = batchPool.back(); batchPool.pop_back(); } }
            if (!j->b) j->b = new ReadBatch;
            j->b->maxReadLength = (uint32_t)maxLen; j->b->wpq = ((uint32_t)maxLen + 15) / 16;
            const double gz0 = r1.gzSeconds + r2.gzSeconds;
            ensure_batch();
            if (getenv("MP_DRIVER_TIMING") && (r1.gz || r2.gz)) fprintf(stderr, "[timing] load: inflate %.3f s\n", r1.gzSeconds + r2.gzSeconds - gz0);
            if (load_batch(r1, r2, *j->b, maxNumQueries, ioThreads) == 0) { delete j->b; delete j; break; }
            j->nReads = j->b->nReads;
            }
            j->seq = seq++;
            double t = now_s(); j->loadSeconds = t - last;
            if (!detected) {                                       // first batch: read-length detection and insert_low clamp (SOAP4.cpp:458-474)
                uint32_t d1 = detect_read_length(j->b->lens, j->b->nReads, 0), d2 = detect_read_length(j->b->lens, j->b->nReads, 1);
                if (opt.insert_low < (int)d2) opt.insert_low = (int)d2;
                if (opt.insert_low < (int)d1) opt.insert_low = (int)d1;
                P.insert_low = opt.insert_low;
                detected = true;
            }
            std::unique_lock<std::mutex> lk(mu);
            cvRoom.wait(lk, [&] { return inflight < maxInflight; });
            ++inflight; inq.push_back(j);
            cvIn.notify_one();
            lk.unlock();
            last = now_s();
        }
        std::lock_guard<std::mutex> lk(mu); readerDone = true; cvIn.notify_all(); cvOut.notify_all();
    });

    auto worker = [&](mp_context *gpu) {
        OutCtx oc = octx;                                           // per-worker copy: own batch pointer
        for (;;) {
            Job *j = nullptr;
            {
                std::unique_lock<std::mutex> lk(mu);
                const bool mayFirst = gpu == contexts[0];
                cvIn.wait(lk, [&] { return (mayFirst && firstJob) || !inq.empty() || readerDone; });
                if (mayFirst && firstJob) { j = firstJob; firstJob = nullptr; }
                else { if (inq.empty()) return; j = inq.front(); inq.pop_front(); }
            }
            const double ts = now_s();
            const uint32_t numQueries = j->nReads, nPairs = numQueries / 2;
            mp_results R;
            static const bool timing = getenv("MP_DRIVER_TIMING") != nullptr;      // per-batch host breakdown on stderr
            double tUp = 0, tAl = 0, tFmt = 0, libWallMs = 0, tCmp = 0;
            int rcUp = 0;
            if (j->dev && !j->uploaded) {
                rcUp = mp_fastq_upload(gpu, j->raw.pin, j->raw.bytes1, j->raw.pin + j->raw.off2, j->raw.bytes2, nPairs, ((uint32_t)maxLen + 15) / 16, (uint32_t)maxLen, nullptr);
                if (rcUp == MP_ERR_FORMAT) {
                    // the input stops being strict four-line FASTQ in mid-file: this batch goes through the host parser, from the staged
                    // bytes.  Its records must be the ones the newline count promised, else the batch boundaries are not the reference's.
                    fprintf(stderr, "[Main] batch %llu is not strict four-line FASTQ: host parser and formatter for this batch (if the run stops here, the records do not "
                                    "lie where the line count put them: rerun with MP_HOST_IO=1)\n", (unsigned long long)j->seq);
                    SeqReader m1, m2;
                    m1.base = j->raw.pin; m1.end = j->raw.bytes1; m1.eof = true; m1.mapped = true;
                    m2.base = j->raw.pin + j->raw.off2; m2.end = j->raw.bytes2; m2.eof = true; m2.mapped = true;
                    j->b = new ReadBatch; j->b->maxReadLength = (uint32_t)maxLen; j->b->wpq = ((uint32_t)maxLen + 15) / 16;
                    const uint32_t got = load_batch(m1, m2, *j->b, numQueries, ioThreads);
                    if (got != numQueries || m1.pos != m1.end || m2.pos != m2.end) {
                        fprintf(stderr, "Error: the read files are not four-line FASTQ throughout; run with MP_HOST_IO=1\n"); exit(1);
                    }
                    j->dev = false; rcUp = 0;
                }
            }
            if (!j->dev && !rcUp) rcUp = mp_batch_upload(gpu, j->b->queries.data(), j->b->lens.data(), numQueries, j->b->wpq);
            mp_results_on_device(gpu, j->dev ? 1 : 0);               // the host formatter needs the result arrays, the device formatter does not
            tUp = now_s();
            if (rcUp || mp_align_pairs(gpu, &P, &R)) {
                j->log = std::string(mp_last_error()) + "\n"; j->failed = true;
            } else {
                char line[512];
                snprintf(line, sizeof line, "[Main] %u pairs of reads are proceeded to deep DP Round 1.\n[Main] Number of pairs aligned by DP: %llu\n[Main] Number of alignments aligned by DP: %llu\n"
                         "[Main] Number of reads aligned by single-end DP: %llu\n[Main] Number of alignments aligned by DP: %llu\n[Main] Number of pairs aligned by DP: %llu\n[Main] Number of alignments aligned by DP: %llu\n",
                         nPairs, (unsigned long long)R.numDPAlignedPair, (unsigned long long)R.numDPAlignment, (unsigned long long)R.numSingleDPAligned,
                         (unsigned long long)R.numSingleDPAlignment, (unsigned long long)R.numRescuedPair, (unsigned long long)R.numRescuedAlignment);
                j->log = line;
                j->pairsAligned = R.numDPAlignedPair + R.numRescuedPair;
                tAl = now_s();
                if (timing) { mp_stats st; if (mp_last_stats(gpu, &st) == 0) libWallMs = st.ms_wall; }
                // ---- output: stage order of the reference (deep DP pairs, rescued pairs, then everything else) ----
                if (j->dev) {
                    // the batch's whole stdout text is composed on the device and DMA'd into the staging buffer the input came from
                    mp_format_params F; F.top = top; F.megapathMode = opt.megapathMode; F.ignoreComments = opt.ignoreComments;
                    uint64_t ob = 0;
                    const double tf0 = now_s();
                    int rc = mp_format_fastq(gpu, &F, &ob);
                    const double tf1 = now_s();
                    if (!rc && ob > j->raw.bytes1 + j->raw.bytes2) {       // later buffers are sized for this growth (+ 25 %)
                        const size_t g = (size_t)((ob - j->raw.bytes1 - j->raw.bytes2) / std::max<uint32_t>(numQueries, 1u)), want = g + g / 4 + 16;
                        size_t cur = growPerRead.load();
                        while (want > cur && !growPerRead.compare_exchange_weak(cur, want)) {}
                    }
                    if (!rc && ob > j->raw.pinCap) {
                        pin_give(j->raw.pin, j->raw.pinCap); j->raw.pin = nullptr;
                        auto pc = pin_take(ob + (ob >> 4));
                        if (!pc.first) rc = -1; else { j->raw.pin = pc.first; j->raw.pinCap = pc.second; }
                    }
                    if (!rc) rc = mp_format_fetch(gpu, j->raw.pin, ob);
                    if (timing) fprintf(stderr, "[timing]  batch %llu: format (device) %.3f fetch %.3f s (%.0f MB)\n", (unsigned long long)j->seq, tf1 - tf0, now_s() - tf1, ob / 1e6);
                    if (rc) { j->log += std::string(mp_last_error()) + "\n"; j->failed = true; }
                    else if (opt.lsam < 0) j->outBytes = ob;
                    else {
                        // -lsam: the device-made text is cut at pair boundaries (every eighth line, found by counting newlines in blocks) and
                        // each piece rewritten into fastq2lsam's lines by one of the -T threads
                        const char *txt = j->raw.pin;
                        const size_t B = (size_t)1 << 18, nBlocks = ((size_t)ob + B - 1) / B;
                        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
                        const unsigned nThr = std::min<unsigned>((unsigned)std::max(1, opt.numCpuThreads), std::max<unsigned>(1u, hw / (unsigned)contexts.size()));
                        std::vector<uint32_t> cnt(nBlocks);
                        auto par = [&](size_t n, const std::function<void(size_t)> &fn) {
                            const unsigned T = (unsigned)std::min<size_t>(nThr, std::max<size_t>(n, 1));
                            std::vector<std::thread> th;
                            for (unsigned t = 1; t < T; ++t) th.emplace_back([&, t] { for (size_t k = t; k < n; k += T) fn(k); });
                            for (size_t k = 0; k < n; k += T) fn(k);
                            for (std::thread &x : th) x.join();
                        };
                        par(nBlocks, [&](size_t k) { cnt[k] = (uint32_t)count_newlines(txt + k * B, std::min(B, (size_t)ob - k * B)); });
                        std::vector<uint64_t> pre(nBlocks + 1, 0);
                        for (size_t k = 0; k < nBlocks; ++k) pre[k + 1] = pre[k] + cnt[k];
                        const uint64_t nPairsOut = pre[nBlocks] / 8;
                        const unsigned nc = (unsigned)std::min<uint64_t>(nThr, std::max<uint64_t>(1, nPairsOut / 4096));
                        std::vector<size_t> cut(nc + 1, (size_t)ob);
                        cut[0] = 0;
                        for (unsigned c = 1; c < nc; ++c) {
                            const uint64_t L = 8 * (nPairsOut * c / nc);            // the piece starts behind the L-th newline
                            if (L == 0) { cut[c] = 0; continue; }
                            const size_t k = (size_t)(std::lower_bound(pre.begin(), pre.end(), L) - pre.begin()) - 1;
                            const char *q = txt + k * B;
                            for (uint64_t need = L - pre[k]; need; --need) q = (const char *)memchr(q, '\n', (size_t)(txt + ob - q)) + 1;
                            cut[c] = (size_t)(q - txt);
                        }
                        j->fqParts.assign(nc, std::string());
                        par(nc, [&](size_t c) { if (cut[c + 1] > cut[c]) fastq_chunk_to_lsam(txt + cut[c], cut[c + 1] - cut[c], opt.lsam != 0, j->fqParts[c]); });
                    }
                } else if (opt.megapathMode || opt.outputBAM) {
                    ReadBatch &b = *j->b;
                    oc.b = &b;
                    // Formatting is spread over the -T host threads: every chunk of pairs writes its own text / BAM records, and the
                    // chunks are concatenated in order, so the stream is the one a single thread would have produced.
                    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
                    const unsigned nThr = std::min<unsigned>((unsigned)std::max(1, opt.numCpuThreads), std::max<unsigned>(1u, hw / (unsigned)contexts.size()));
                    struct Chunk { std::string fq; std::vector<uint8_t> bam, bamz; };   // bamz: the chunk's BAM records as BGZF blocks
                    auto run_chunks = [&](uint64_t nItems, int bamSlot, const std::function<uint64_t(uint64_t)> &alignStart,
                                          const std::function<void(OutCtx &, std::string &, uint64_t, uint64_t)> &body) {
                        if (nItems == 0) return;
                        const unsigned nc = (unsigned)std::min<uint64_t>(nThr, (nItems + 4095) / 4096);
                        std::vector<uint64_t> cut(nc + 1, nItems);
                        cut[0] = 0;
                        for (unsigned c = 1; c < nc; ++c) cut[c] = std::max(cut[c - 1], alignStart(nItems * c / nc));
                        std::vector<Chunk> chunks(nc);
                        auto one = [&](unsigned c) {
                            OutCtx occ = oc; BamWriter capw; capw.capture = &chunks[c].bam;
                            OutScratch scr; occ.scratch = &scr;
                            occ.bam = opt.outputBAM ? &capw : nullptr;
                            chunks[c].fq.reserve((size_t)(cut[c + 1] - cut[c]) * (size_t)(4 * maxLen + 160));
                            body(occ, chunks[c].fq, cut[c], cut[c + 1]);
                            if (opt.lsam >= 0 && !chunks[c].fq.empty()) { std::string ls; fastq_chunk_to_lsam(chunks[c].fq.data(), chunks[c].fq.size(), opt.lsam != 0, ls); chunks[c].fq.swap(ls); }
                            if (!deviceBgzf && !chunks[c].bam.empty()) { BgzfWriter::compress_all(chunks[c].bam.data(), chunks[c].bam.size(), chunks[c].bamz); std::vector<uint8_t>().swap(chunks[c].bam); }
                        };
                        std::vector<std::thread> ths;
                        for (unsigned c = 1; c < nc; ++c) ths.emplace_back(one, c);
                        one(0);
                        for (std::thread &t : ths) t.join();
                        if (deviceBgzf) {
                            // the chunks' records, in order, through one staging buffer: every full piece is compressed as it fills
                            const double tc0 = now_s();
                            auto sp = pin_take(bgzfCap), dp = pin_take(bgzfCap);
                            int rc = (!sp.first || !dp.first) ? MP_ERR_CUDA : 0;
                            size_t fill = 0;
                            auto flush = [&]() {
                                uint64_t ob = 0;
                                rc = mp_bgzf_compress(gpu, (const uint8_t *)sp.first, fill, (uint8_t *)dp.first, dp.second, &ob);
                                if (!rc) j->bam[bamSlot].insert(j->bam[bamSlot].end(), (const uint8_t *)dp.first, (const uint8_t *)dp.first + ob);
                                fill = 0;
                            };
                            for (Chunk &c : chunks)
                                for (size_t at = 0; at < c.bam.size() && !rc;) {
                                    const size_t k = std::min<size_t>(c.bam.size() - at, bgzfPiece - fill);
                                    memcpy(sp.first + fill, c.bam.data() + at, k); fill += k; at += k;
                                    if (fill == bgzfPiece) flush();
                                }
                            if (fill && !rc) flush();
                            pin_give(sp.first, sp.second); pin_give(dp.first, dp.second);
                            if (rc) { j->log += std::string(mp_last_error()) + "\n"; j->failed = true; }
                            tCmp += now_s() - tc0;
                        }
                        // the chunks stay separate strings (no 700 MB concatenation): the writer emits them in this order
                        for (Chunk &c : chunks) { j->fqParts.emplace_back(std::move(c.fq)); j->bam[bamSlot].insert(j->bam[bamSlot].end(), c.bamz.begin(), c.bamz.end()); }
                    };
                    std::vector<uint8_t> done(nPairs, 0);
                    for (int which = 0; which < 2; ++which) {
                        const mp_pair_result *arrp = which == 0 ? R.pairs : R.rescued; const uint64_t n = which == 0 ? R.n_pairs : R.n_rescued;
                        run_chunks(n, which,
                                   [&](uint64_t i) { while (i > 0 && i < n && arrp[i].readID == arrp[i - 1].readID) ++i; return i; },   // keep the hits of one pair together
                                   [&](OutCtx &occ, std::string &fq, uint64_t lo, uint64_t hi) {
                                       for (uint64_t i = lo, e; i < hi; i = e) {
                                           e = i + 1;
                                           while (e < n && arrp[e].readID == arrp[i].readID) ++e;
                                           output_pair(occ, fq, arrp + i, arrp + e, R.cigars, which == 0 ? 1 : 2);      // PH: hspaux->dpStageId
                                           done[arrp[i].readID >> 1] = 1;
                                       }
                                   });
                    }
                    // pairs neither placed by deep DP nor rescued: per-read single-end hits (alignment.cpp:299-351)
                    run_chunks(nPairs, 2, [](uint64_t p) { return p; },
                               [&](OutCtx &occ, std::string &fq, uint64_t lo, uint64_t hi) {
                                   // singles are ordered by readID: find where this chunk starts
                                   uint64_t si = 0;
                                   { uint64_t a = 0, z = R.n_singles; while (a < z) { uint64_t m = (a + z) / 2; if (R.singles[m].readID < 2 * lo) a = m + 1; else z = m; } si = a; }
                                   for (uint64_t p = lo; p < hi; ++p) {
                                       if (done[p]) continue;
                                       std::vector<SingleAln> hits[2];
                                       for (uint32_t e = 0; e < 2; ++e) {
                                           const uint32_t id = (uint32_t)(2 * p + e);
                                           while (si < R.n_singles && R.singles[si].readID < id) ++si;
                                           uint64_t en = si;
                                           while (en < R.n_singles && R.singles[en].readID == id) {
                                               const mp_single_result &sr = R.singles[en];
                                               SingleAln a = { sr.algnmt, sr.score, (int)sr.strand, sr.editdist, sr.num_sameScore, R.cigars + sr.cigar };
                                               hits[e].push_back(a); ++en;
                                           }
                                           // OutputBuffer::ready: sort by (algnmt, score), drop duplicates (DV-DPfunctions.h:167-196, .cpp:248-251)
                                           std::sort(hits[e].begin(), hits[e].end(), [](const SingleAln &x, const SingleAln &y) { return std::make_pair(x.algnmt, x.score) < std::make_pair(y.algnmt, y.score); });
                                           hits[e].erase(std::unique(hits[e].begin(), hits[e].end(), [](const SingleAln &x, const SingleAln &y) { return x.algnmt == y.algnmt && x.score == y.score; }), hits[e].end());
                                       }
                                       output_unpaired(occ, fq, (uint32_t)(2 * p), hits, stageUnpaired);
                                   }
                               });
                }
                tFmt = now_s();
                mp_results_release(gpu, &R);
            }
            if (timing) fprintf(stderr, "[timing] batch %llu: upload %.3f align %.3f (lib wall %.3f) format %.3f (bgzf compress %.3f) release %.3f s; started at %.3f\n",
                                (unsigned long long)j->seq, tUp - ts, tAl - tUp, libWallMs / 1e3, tFmt - tAl, tCmp, now_s() - tFmt, ts - t0);
            j->alignSeconds = now_s() - ts;
            std::lock_guard<std::mutex> lk(mu);
            if (j->b) { batchPool.push_back(j->b); j->b = nullptr; }   // the text output no longer refers to the batch
            doneq[j->seq] = j; cvOut.notify_all();
        }
    };
    std::vector<std::thread> workers;
    for (mp_context *c : contexts) workers.emplace_back(worker, c);

    // ---- ordered writer ----
    double totalLoad = 0, totalAlign = 0; const double tLoop0 = now_s();
    uint64_t totalPairsAligned = 0, next = 0; bool failed = false, announced = false;
    double writeSeconds = 0; uint64_t writtenBytes = 0;
    for (;;) {
        Job *j = nullptr;
        {
            std::unique_lock<std::mutex> lk(mu);
            cvOut.wait(lk, [&] { return doneq.count(next) || (readerDone && inflight == 0); });
            auto it = doneq.find(next);
            if (it == doneq.end()) break;
            j = it->second; doneq.erase(it); --inflight; cvRoom.notify_one();
        }
        fprintf(stderr, "[Main] Loaded %u short reads from the query file.\n[Main] Elapsed time on host : %9.4f seconds\n\n", j->nReads, j->loadSeconds);
        if (!announced) { fprintf(stderr, "All reads are directly processed by DP\n"); announced = true; }
        fputs(j->log.c_str(), stderr);
        if (j->failed) failed = true;
        const double tw0 = now_s();
        if (j->outBytes) { fwrite(j->raw.pin, 1, (size_t)j->outBytes, stdout); writtenBytes += j->outBytes; }
        for (const std::string &part : j->fqParts) if (!part.empty()) { fwrite(part.data(), 1, part.size(), stdout); writtenBytes += part.size(); }
        pin_give(j->raw.pin, j->raw.pinCap); j->raw.pin = nullptr;
        writeSeconds += now_s() - tw0;
        if (opt.outputBAM) { bamDP.write_blocks(j->bam[0]); bamGout.write_blocks(j->bam[1]); bamUnpair.write_blocks(j->bam[2]); }
        fprintf(stderr, "[Main] Elapsed time : %9.4f seconds\n\n", j->alignSeconds);
        if (getenv("MP_DRIVER_TIMING")) fprintf(stderr, "[timing] batch %llu written at %.3f\n", (unsigned long long)j->seq, now_s() - t0);
        totalLoad += j->loadSeconds; totalAlign += j->alignSeconds; totalPairsAligned += j->pairsAligned;
        delete j; ++next;
    }
    reader.join();
    for (std::thread &t : workers) t.join();
    fflush(stdout);
    if (opt.outputBAM) { bamDP.close(); bamGout.close(); bamUnpair.close(); }
    const double tLoop1 = now_s();                                  // every batch aligned and written: the end of the batch loop
    for (ReadBatch *rb : batchPool) delete rb;
    // (the staging buffers are left to the end of the process: unlocking gigabytes page by page here would only delay the exit)
    if (failed) return 1;
    if (getenv("MP_DRIVER_TIMING")) fprintf(stderr, "[timing] writer: %.3f s in stdout writes, %.1f MB; batch loop from %.3f to %.3f\n", writeSeconds, writtenBytes / 1e6, tLoop0 - t0, tLoop1 - t0);
    fprintf(stderr, "[Main] Overall number of pairs of reads aligned: %llu\n", (unsigned long long)totalPairsAligned);
    fprintf(stderr, "[Main] Overall read load time : %9.4f seconds\n", totalLoad);
    fprintf(stderr, "[Main] Overall alignment time (excl. read loading) : %9.4f seconds\n", tLoop1 - tLoop0);
    for (size_t k = contexts.size(); k-- > 0;) mp_destroy(contexts[k]);
    fprintf(stderr, "[Main] Overall running time: %f\n", now_s() - t0);
    return 0;
}
