// mp_cigar.h -- pattern -> "special" CIGAR (M match, m mismatch, I, D, S), shared by device and host code.
#pragma once
#include <stdint.h>

#define MP_MARGIN(l) (((l) > 100) ? 30 : 25)       // DP2_MARGIN / DPS_MARGIN, DV-DPfunctions.cpp:1760, 267

__host__ __device__ inline int dp_cutoff(uint32_t readLen)           // definitions.h:166-167
{
    double v = 0.2 * readLen; if (v < 30.0) v = 30.0; return (int)v;
}

// ---- pattern -> special CIGAR (CigarStringEncoder, DV-DPfunctions.h:344-427; use at .cpp:3447-3471) ----
struct CigStats { int nI, nD, nS, gapPenalty, textLen; };
__host__ __device__ inline int ndigits(int v) { return v >= 100 ? 3 : v >= 10 ? 2 : 1; }
// The encoder merges consecutive equal types while scanning the (end -> start) pattern and prints the
// runs in reverse.  `out` == nullptr: measure only.  Text is written backwards from out + textLen.
__host__ __device__ inline CigStats cigar_encode(const uint8_t *__restrict__ pat, int open, int ext, char *out, int textLen)
{
    CigStats st; st.nI = st.nD = st.nS = st.gapPenalty = st.textLen = 0;
    char *w = out ? out + textLen : nullptr;
    int curType = 'N', curCnt = 0, lastType = 'N';
    const uint8_t *p = pat;
    while (true) {
        int type, cnt; bool end = false;
        if (*p == 0) { type = 0; cnt = 0; end = true; }
        else if (*p == 'V') { type = lastType; cnt = (int)p[1] - 1; p += 2; }
        else { type = *p; cnt = 1; lastType = type; ++p; }
        if (!end && type == curType) { curCnt += cnt; continue; }
        // flush the finished run
        if (curCnt > 0 && curType != 'N') {
            int nd = ndigits(curCnt);
            st.textLen += nd + 1;
            if (curType == 'I') st.nI += curCnt; else if (curType == 'D') st.nD += curCnt; else if (curType == 'S') st.nS += curCnt;
            if (curType == 'I' || curType == 'D') st.gapPenalty += open + (curCnt - 1) * ext;
            if (w) {
                *--w = (char)curType;
                int v = curCnt;
                for (int d = 0; d < nd; ++d) { *--w = (char)('0' + v % 10); v /= 10; }
            }
        }
        if (end) break;
        curType = type; curCnt = cnt;
    }
    return st;
}

#ifdef __CUDACC__
#include "mp_context.h"
// The special CIGAR of a leg and the encoder's statistics.  The traceback (k_dp_tb) and the exact-occurrence test (k_dp_prepare) build
// both while they emit the pattern and leave the text at the end of the task's pattern row; only when pattern and text would not both
// fit the row (hundreds of one-base runs) is the text encoded here from the pattern.
__device__ __forceinline__ CigStats leg_stats(const MpDpOut &o)
{
    CigStats st; st.nI = o.nI; st.nD = o.nD; st.nS = o.nS; st.gapPenalty = o.gapPenalty; st.textLen = o.cigLen;
    return st;
}
__device__ __forceinline__ void leg_text(const MpDpOut &o, const uint8_t *pat, uint32_t patStride, int open, int ext, char *out)
{
    if (o.cigStored) { const uint8_t *src = pat + patStride - o.cigLen; for (int k = 0; k < (int)o.cigLen; ++k) out[k] = (char)src[k]; }
    else cigar_encode(pat, open, ext, out, o.cigLen);
}
#endif
