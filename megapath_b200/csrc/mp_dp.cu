// mp_dp.cu -- semi-global affine-gap DP with traceback on the device.
// Replaces SemiGlobalAligner::performAlignment -> callDP -> SemiGlobalAlignment ->
// GenerateDPTable + GPUBacktrack (CPU_DPfunctions.cpp:270-312; CPU_DP.cpp:881-978, 788-871,
// 122-619, 622-786) and the task packing of PairEndAlgnBatch::packRead/repackDNA
// (DV-DPfunctions.cpp:3009-3073).
//
// The reference encodes the recurrence as 8-bit saturating deltas with "score trimming";
// observable results equal the plain recurrence below (SURVEY.md 9.4; oracle/mp_oracle_dp.cpp,
// checked against the reference's own callDP).  Integer ALU / DPX work, no tensor cores.
//
// k_dp_fill<K>: one warp per PAIR of tasks.  The two tasks travel in the low and high 16-bit halves of
// every register, so each recurrence step is one packed DPX instruction for both (VIADDMNMX.U16x2,
// VIMNMX3.U16x2, VIMNMX.U16x2); scores carry a +16384 bias so that unsigned halves never borrow.
// Lane l owns read columns l*K+1 .. l*K+K and walks the reference rows with a one-row skew per lane
// (anti-diagonal wavefront); the right-most H / I of a lane's strip travel to lane l+1 by shuffle, the
// reference rows come from shared memory.  Every cell leaves one traceback byte
//    (H-Hdiag-mm)*42 + (H-Hleft-open)*3 + g          g 0 = D==H, 1 = neither, 2 = raised by the clip floor
// (the information the reference keeps, CPU_DP.cpp:183, 529-533) in a step-major table in HBM (layout at cell_offset):
// a warp's stores of one step are one full 128-byte line per task.
// The answer cell (first strict maximum in row-major order, tie count, CPU_DP.cpp:545-590) is kept per
// column in packed registers and reduced across the warp at the end.
// k_dp_tb<K>: one thread per task walks its own table (GPUBacktrack, CPU_DP.cpp:622-786) -- thousands of
// independent walks in flight hide the dependent-load latency that a single walking lane cannot.
// k_dp_prepare: runs first; writes the tasks' packed sequence rows, and tasks whose read occurs unchanged in its window get their
// (provably identical) answer without the DP, the others are compacted for the two kernels above.
#include "mp_context.h"
#include "mp_cigar.h"
#include <cub/device/device_scan.cuh>
#include <algorithm>
#include <type_traits>

#ifndef MP_FILL_MINBLOCKS
#define MP_FILL_MINBLOCKS 6      /* blocks per SM the K = 5 fill kernel is compiled for (register budget 80) */
#endif
#define DP_BIAS   0x4000
#define DP_BIAS2  0x40004000u
#define DP_NEG2   0x20C020C0u      /* (bias - 8000) in both halves: "minus infinity" that never underflows */
#define DP_C      0x5000           /* flag arithmetic: C - hf stays positive, 2C = 0 mod 256 */
#define DP_C2     0x50005000u
#define DP_CM1_2  0x4FFF4FFFu

__device__ __forceinline__ int h0_value(int j, int clipLt, int open)       // row 0 (CPU_DP.cpp:397-429)
{
    return j <= clipLt ? 0 : open - (j - clipLt - 1);
}
// base x of a packed row: 16 bases per word, first base in the low bits (the read order of the batch's dReads rows)
__device__ __forceinline__ uint32_t packed_base(const uint32_t *row, int x) { return (row[x >> 4] >> ((x & 15) * 2)) & 3u; }
__device__ __forceinline__ uint32_t pack2(int v) { return ((uint32_t)v & 0xffffu) * 0x00010001u; }
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel)); return d;
}
// x * m + y with a multiplier the compiler cannot see through: keeps the add on the FMA pipe (IMAD) instead of the ALU pipe,
// which carries every min/max/permute of the recurrence and is the pipe that limits the kernel
__device__ __forceinline__ uint32_t fma_add(uint32_t x, uint32_t m, uint32_t y)
{
    uint32_t d; asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(x), "r"(m), "r"(y)); return d;
}

struct FillOut { int32_t score; uint32_t row, col, cnt; };

// Trace table of one task PAIR (S steps, S a multiple of 4; 2*S*32*K bytes).  Step t = row + lane.
//   word region  : step-major blocks of WORDS*256 bytes: [word w][task half h][lane] u32; byte c holds column 4w+c of the lane's
//                  strip for the row it had 3-c steps earlier, i.e. four cells of one DIAGONAL: the traceback's usual move stays
//                  inside one 32-byte sector
//   remainder    : the K%4 left-over columns of four consecutive steps share u32 words: group g = (t-1)/4 holds REM*256 bytes
//                  [word][half][lane] u32, byte position ((t-1)%4)*REM + (k-4*WORDS)
// so that every store of a warp is a full 128-byte line per task and one running pointer serves both tasks.
// cell_offset is relative to (pair table + half*128).
template <int K>
__device__ __forceinline__ size_t cell_offset(int r, int c, int S)
{
    const int lane = (c - 1) / K, k = (c - 1) - lane * K, t = r + lane;
    constexpr int WORDS = K / 4, REM = K % 4, WB = WORDS * 256;
    if (k < 4 * WORDS) return (size_t)(t + 3 - (k & 3)) * WB + (size_t)(k >> 2) * 256 + lane * 4 + (k & 3);
    const int b = ((t - 1) & 3) * REM + (k - 4 * WORDS);
    return (size_t)S * WB + (size_t)((t - 1) >> 2) * (REM * 256) + (size_t)(b >> 2) * 256 + lane * 4 + (b & 3);
}
// Trace byte of a cell: (4*H - zd - zr) mod 256 with zd = 1 unless D == H, zr = 1 where the clip floor raised the cell (then zd = 1 too).
//   bits 7..2 (after rounding up): H mod 64 -- neighbouring cells differ by less than 8, so every difference GPUBacktrack looks at
//                                  (H - Hdiag, H - Hleft, H - Hup; CPU_DP.cpp:183, 529-533 keeps the first two as 4-bit deltas) is exact
//   bits 1..0 = (-(zd + zr)) & 3 : 0 = D == H, 3 = neither, 2 = raised by the clip floor
__device__ __forceinline__ int trace_h(uint32_t cell) { return (int)(((cell + 3u) >> 2) & 63u); }
// -> the reference's flag (0 = raised by the clip floor, 1 = D == H, 2 = otherwise; CPU_DP.cpp:529-533)
__device__ __forceinline__ int trace_flag(uint32_t cell) { const uint32_t g = cell & 3u; return g == 0 ? 1 : g == 3 ? 2 : 0; }
__device__ __forceinline__ int trace_diff(int a, int b) { return ((a - b + 32) & 63) - 32; }      // a - b for values known mod 64

// Answer bookkeeping of one lane (see k_dp_fill), per task of the pair: the best value its eligible cells have reached (biased x4 units),
// and the first and the last ROW in which a cell reached it.  Which column, and how many cells tie, is read back from the lane's own
// trace bytes when the table is complete (dp_resolve_lane): a step that sets a new best therefore costs a handful of instructions, which
// matters for divergent reads -- every cell of the optimal path is a new best of its lane, so the tracker runs on most steps there.
// Kept out of line and in local memory: it must not cost the hot loop registers.
struct DpTrack { int lb[2], rfirst[2], rlast[2], thrT[2], thr[2], N[2]; uint32_t elig[2]; };
__device__ __forceinline__ uint32_t dp_track_t2(const DpTrack *tr, int o4)
{
    // from now on only cells that at least tie with this lane's best matter: (H + open) + T2 has bit 15 set <=> H >= threshold
    const int a = max(tr->thrT[0], tr->lb[0]), b = max(tr->thrT[1], tr->lb[1]);
    return (uint32_t)(0x8000 + o4 - a) | ((uint32_t)(0x8000 + o4 - b) << 16);
}
// every column of the lane may hold the answer (all lanes but the one or two at the ends of the eligible column range): cm = packed
// maximum of the lane's K cells of this row (H + open), q = cm + T2
__device__ __noinline__ uint32_t dp_track_row(DpTrack *tr, uint32_t cm, uint32_t q, int i, int o4)
{
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        if (!((q >> (16 * half)) & 0x8000u) || i > tr->N[half] || !tr->elig[half]) continue;      // (padding columns hold anything)
        const int v = (int)((cm >> (16 * half)) & 0xffffu) + o4;
        if (v > tr->lb[half]) { tr->lb[half] = v; tr->rfirst[half] = i; tr->rlast[half] = i; }
        else if (v == tr->lb[half]) tr->rlast[half] = i;
    }
    return dp_track_t2(tr, o4);
}
// a lane whose columns are only partly eligible (j < L - clipRt, or j > L): the row maximum is taken over the eligible columns
template <int K>
__device__ __noinline__ uint32_t dp_track_row_masked(DpTrack *tr, const uint32_t *ho, uint32_t q, int i, int o4)
{
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        if (!((q >> (16 * half)) & 0x8000u) || i > tr->N[half]) continue;
        int v = -(1 << 20);
#pragma unroll
        for (int k = 0; k < K; ++k)
            if ((tr->elig[half] >> k) & 1u) v = max(v, (int)((ho[k] >> (16 * half)) & 0xffffu) + o4);
        if (v < max(tr->thrT[half], tr->lb[half])) continue;
        if (v > tr->lb[half]) { tr->lb[half] = v; tr->rfirst[half] = i; tr->rlast[half] = i; }
        else tr->rlast[half] = i;
    }
    return dp_track_t2(tr, o4);
}

// The cells of one lane that equal the task's best score Ms, looked up in the trace bytes the lane wrote itself: first (row, column) in
// row-major order and their number, over rows r0..r1 (the first and last row in which the lane's row maximum reached Ms).  A trace byte
// holds H mod 64.  In row r0 some cell of the lane equals Ms and neighbours in a row differ by at most 1 - open <= 7, so all K <= 10
// cells lie within 63 of Ms and H is exact; below r0 every cell follows from the one above it (vertical neighbours differ by < 32).
template <int K>
__device__ __noinline__ void dp_resolve_lane(const uint8_t *tab, int S, int j0, uint32_t elig, int r0, int r1, int Ms, uint32_t &key, uint32_t &cnt)
{
    int H[K], ph[K];
    uint32_t kfirst = 0xffffffffu, c = 0u;
    for (int r = r0; r <= r1; ++r) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (!((elig >> k) & 1u)) continue;
            const int h = trace_h(__ldcg(tab + cell_offset<K>(r, j0 + k, S)));      // written by this lane in this kernel: never the read-only path
            if (r == r0) H[k] = Ms - ((Ms - h) & 63); else H[k] += trace_diff(h, ph[k]);
            ph[k] = h;
            if (H[k] == Ms) { if (kfirst == 0xffffffffu) kfirst = ((uint32_t)r << 12) | (uint32_t)(j0 + k); ++c; }
        }
    }
    key = kfirst; cnt = c;
}

// k_dp_fill<K, MM, OPEN>: MM / OPEN = mismatch and gap-open score as compile-time constants (0 = take them from P at run time).
//
// Scores are carried times four with a +0x4000 bias in unsigned 16-bit halves (task A low, task B high): the two free low bits of
// every H take the cell's two flags, so a trace byte is one add away from H.  Per cell pair the ALU pipe sees
//   PRMT (substitution penalty of both tasks from the row's 8-byte table, selector = the column's two read bases),
//   VIADDMNMX x2 (D, I), VIMNMX3 (H), VIMNMX (clip floor), VIADDMNMX x2 (the two flags), PRMT (byte packing, one per cell)
// and the FMA pipe the plain adds (IMAD).  The answer cell (first strict maximum in row-major order + tie count, CPU_DP.cpp:545-590)
// is NOT tracked per cell: a lane compares the maximum of its K cells of a step with a threshold and only cells that reach it
// take the exact (scalar, per-lane) bookkeeping path.  The threshold starts at max(cutoff, LB) where LB is the score of the ungapped
// path along the task's hinted diagonal -- a true lower bound of the best score, so no cell that can be the answer or tie with
// it is skipped -- and follows the lane's own best.
template <int K, int MM, int OPEN, bool MASKED>
__global__ void __launch_bounds__(128, K <= 5 ? MP_FILL_MINBLOCKS : K <= 8 ? 5 : 4)
k_dp_fill(const uint32_t *__restrict__ refSeq, const uint32_t *__restrict__ refLens, uint32_t refStride,
          const uint32_t *__restrict__ readSeq, const uint32_t *__restrict__ readLens, uint32_t readStride,
          const int32_t *__restrict__ cutoffs, const int16_t *__restrict__ hints, uint32_t taskBase, uint32_t nTasks, MpDpParams P,
          uint8_t *__restrict__ tables, size_t tableStride, int S, FillOut *__restrict__ fill,
          const uint32_t *__restrict__ active, const uint32_t *__restrict__ nActive, uint32_t one)
{
    extern __shared__ uint2 refShared[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t pairId = blockIdx.x * 4 + wib;
    const uint32_t lA = pairId * 2, lB = lA + 1;             // slots inside this launch: tables are indexed by slot
    if (active) nTasks = *nActive;                           // only the tasks the exact-occurrence test left over (k_dp_prepare)
    if (lA >= nTasks) return;
    const bool hasB = lB < nTasks;
    const uint32_t tA = taskBase + (active ? active[lA] : lA), tB = hasB ? taskBase + (active ? active[lB] : lB) : tA;
    const int mm = MM ? MM : P.mismatch, open = OPEN ? OPEN : P.open, clipLt = P.clipLt;
    int NA = (int)refLens[tA], LA = (int)readLens[tA], cutA = cutoffs[tA];
    int NB = hasB ? (int)refLens[tB] : 0, LB = hasB ? (int)readLens[tB] : 0, cutB = hasB ? cutoffs[tB] : 0;
    // CPU_DP.cpp:296-324: outside these bounds the reference aborts the SIMD group
    const bool okA = !(cutA > LA || cutA <= 0 || LA >= 255 + open - 1 + cutA || LA > 32 * K);
    const bool okB = hasB && !(cutB > LB || cutB <= 0 || LB >= 255 + open - 1 + cutB || LB > 32 * K);
    if (!okA) { NA = 0; LA = 0; }
    if (!okB) { NB = 0; LB = 0; }
    const int maxN = max(NA, NB), maxL = max(LA, LB);
    const uint32_t PEN = (uint32_t)(4 * (1 - mm));              // 4 * (match - mismatch) < 0x80
    // FOLD (compile-time scores with |open| >= |mismatch|): the row tables hold the non-negative ADDEND (open-form diagonal + addend =
    // diagonal + substitution score), so one H form per column serves the diagonal, D and I.  Otherwise they hold the penalty.
    constexpr bool FOLD = MM != 0 && OPEN != 0 && (-4 * OPEN + 4 >= 4 * (1 - MM));
    const uint32_t O4v = (uint32_t)(-4 * open);
    const uint32_t TMATCH = FOLD ? O4v + 4u : 0u, TMIS = FOLD ? O4v + 4u - PEN : PEN;
    // ---- reference rows -> substitution tables: bytes 0..3 = penalty of task A's row against read base 0..3, bytes 4..7 task B;
    //      rows a task does not have mismatch everything ----
    uint2 *refS = refShared + (size_t)wib * S;
    {
        const uint32_t *fa = refSeq + (size_t)tA * refStride, *fb = refSeq + (size_t)tB * refStride;
        const uint32_t all = TMIS * 0x01010101u;
        for (int r = lane; r < maxN; r += 32) {
            const uint32_t a = r < NA ? packed_base(fa, r) : 4u, b = r < NB ? packed_base(fb, r) : 4u;
            refS[r] = make_uint2(a < 4u ? (all & ~(0xFFu << (8 * a))) | (TMATCH << (8 * a)) : all,
                                 b < 4u ? (all & ~(0xFFu << (8 * b))) | (TMATCH << (8 * b)) : all);
        }
    }
    __syncwarp();
    const uint32_t *ra = readSeq + (size_t)tA * readStride, *rbp = readSeq + (size_t)tB * readStride;
    const int j0 = lane * K + 1;
    // per column: PRMT selector (nibble 0 = A's base, nibble 2 = 4 + B's base, nibbles 1 / 3 replicate the sign bit of the same
    // byte = 0), H of the row above in open form (H + open: what D and I consume, and with FOLD the diagonal too), D, clip floor
    uint32_t sel[K], HO[K], Dp[K], fl[K];
    const uint32_t O4 = pack2(-4 * open), FOUR2 = 0x00040004u, NEG_E4 = 0xFFFCFFFCu;
    const uint32_t negOne = 0u - one;                           // 0xFFFFFFFF the compiler cannot fold (fma_add)
    uint32_t basesA = 0, basesB = 0;                            // this lane's read bases, 2 bits each (lower-bound prologue)
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int j = j0 + k;
        const uint32_t a = j <= LA ? packed_base(ra, j - 1) : 0u, b = j <= LB ? packed_base(rbp, j - 1) : 0u;
        basesA |= a << (2 * k); basesB |= b << (2 * k);
        sel[k] = a | ((8u | a) << 4) | ((4u + b) << 8) | ((12u + b) << 12);
        // !MASKED (see the tracker below): a column beyond the read takes addend 0 -- a substitution score of `open`, below any real one
        // -- by selecting the sign replica (0x00) of a table byte, so that its cells stay below the real cells they derive from
        if (!MASKED && j > LA) sel[k] = (sel[k] & ~0xFu) | 8u;
        if (!MASKED && j > LB) sel[k] = (sel[k] & ~0xF00u) | 0xC00u;
        const uint32_t h0 = pack2(4 * h0_value(j, clipLt, open) + DP_BIAS);
        HO[k] = h0 - O4;
        Dp[k] = DP_NEG2;
        fl[k] = j <= clipLt ? DP_BIAS2 : 0u;
        asm volatile("" : "+r"(fl[k]));                         // keep it in a register: recomputing it costs two ALU-pipe slots per cell
    }
    // lane 0 takes its left neighbour (column 0: H = 0, no I) from constants; as multiply-adds so the selection stays off the ALU pipe
    const uint32_t keepLeft = lane == 0 ? 0u : one, leftH0 = lane == 0 ? DP_BIAS2 - O4 : 0u, leftI0 = lane == 0 ? DP_NEG2 : 0u;
    // ---- threshold: max(cutoff, lower bound from the hinted diagonal), per task ----
    int thrA = 0x7FF0, thrB = 0x7FF0;                           // biased x4 units; 0x7FF0: nothing can reach it (task absent)
    {
        const int minColA = max(LA - P.clipRt, 1), minColB = max(LB - P.clipRt, 1);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const bool live = half ? okB : okA;
            const int Lh = half ? LB : LA, Nh = half ? NB : NA, cut = half ? cutB : cutA, minCol = half ? minColB : minColA;
            const int dg = live && hints ? (int)hints[half ? tB : tA] : -1;
            const uint32_t bases = half ? basesB : basesA;
            int best = -(1 << 20);
            if (live) {
                // ungapped path: column j in row j + dg, starting from H[dg][0] = 0; valid while the row exists
                int loc[K], tot = 0;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int j = j0 + k, r = j + dg;
                    int s = 0;
                    if (dg >= 0 && j <= Lh && r <= Nh) {
                        const uint2 tb = refS[r - 1];
                        const uint32_t e = ((half ? tb.y : tb.x) >> (8 * ((bases >> (2 * k)) & 3u))) & 0xFFu;
                        s = FOLD ? (int)e - (int)O4v : 4 - (int)e;
                    }
                    tot += s; loc[k] = tot;
                }
                int incl = tot;
#pragma unroll
                for (int dlt = 1; dlt < 32; dlt <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, dlt); if (lane >= dlt) incl += v; }
                const int before = incl - tot;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int j = j0 + k;
                    if (dg >= 0 && j >= minCol && j <= Lh && j + dg <= Nh) best = max(best, before + loc[k]);
                }
            }
#pragma unroll
            for (int dlt = 16; dlt; dlt >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, dlt));
            const int thr = DP_BIAS + max(4 * cut, best);
            if (live) { if (half) thrB = thr; else thrA = thr; }
        }
    }
    // lane-level answer bookkeeping (dp_track_row): thr - 1 = nothing yet.  elig: which of the lane's columns may hold the answer
    // (L - clipRt <= j <= L, CPU_DP.cpp:545-590); a half without eligible columns (or without a task) gets a threshold nothing reaches.
    DpTrack tr;
    uint32_t eligA = 0, eligB = 0;
    {
        const int minColA = max(LA - P.clipRt, 1), minColB = max(LB - P.clipRt, 1);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int j = j0 + k;
            eligA |= (uint32_t)(j >= minColA && j <= LA) << k;
            eligB |= (uint32_t)(j >= minColB && j <= LB) << k;
        }
    }
    tr.lb[0] = thrA - 1; tr.lb[1] = thrB - 1; tr.rfirst[0] = tr.rfirst[1] = 0; tr.rlast[0] = tr.rlast[1] = 0;
    tr.thr[0] = thrA; tr.thr[1] = thrB;           // read back after the loop: nothing the loop does not need stays in a register
    tr.thrT[0] = eligA ? thrA : 0x7FF0; tr.thrT[1] = eligB ? thrB : 0x7FF0; tr.N[0] = NA; tr.N[1] = NB; tr.elig[0] = eligA; tr.elig[1] = eligB;
    const int lastLane = maxL > 0 ? (maxL - 1) / K : 0;
    const int steps = maxN + lastLane;
    const bool mine = lane <= lastLane;                         // lanes that own read columns (every lane runs the loop: full-mask shuffles)
    // lanes without read columns run the steady groups like everyone else (straight-line code, full 128-byte trace lines) on
    // padding cells; nothing there reaches their threshold.  (H + open) + T2 has bit 15 set <=> H >= threshold
    uint32_t T2 = dp_track_t2(&tr, (int)O4v);
    uint32_t prevLeftO = pack2(4 * h0_value(j0 - 1, clipLt, open) + DP_BIAS) - O4;            // H[i-1][j0-1] in open form
    const uint2 *rowP = refS - lane;                            // row of step t = 1 is 1 - lane: table index t - 1 - lane
    constexpr int WORDS = K / 4, REM = K % 4, WB = WORDS * 256;
    uint8_t *tabP = tables + (size_t)lA * tableStride;          // pair table: 2 * tableStride bytes
    uint8_t *pw = tabP + WB + lane * 4;                         // word block of step 1
    uint8_t *pr = tabP + (size_t)S * WB + lane * 4;             // remainder group 0
    // what a lane hands to its right neighbour before it has computed anything: the column-0 boundary (H = 0, no I).  Lanes beyond the
    // read never get real input; with this start their padding cells stay ordinary small scores (never near 0x8000, where the
    // threshold test of a half without eligible columns would fire)
    uint32_t sendH = DP_BIAS2 - O4, sendI = DP_NEG2;
    uint32_t accA[REM ? REM : 1] = {0}, accB[REM ? REM : 1] = {0};
    uint32_t hist[WORDS][3][4];                                 // codes of the last steps, slot = step % 4 (see cell_offset)
#pragma unroll
    for (int w = 0; w < WORDS; ++w)
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int q = 0; q < 4; ++q) hist[w][c][q] = 0;
    // One wavefront step of this lane; u = (t-1) % 4 is a compile-time constant in every caller.
    // CHECKED = false in the steady phase, where every owning lane has a row that exists in BOTH tasks: no range test,
    // and the four unrolled steps need no register shuffling between them.
    auto step = [&](const int t, auto uTag, auto checked) {
        constexpr int u = decltype(uTag)::value;
        constexpr bool CHECKED = decltype(checked)::value;
        const uint32_t rH = __shfl_up_sync(0xffffffffu, sendH, 1);                // open form: H + open of the left lane's last column
        const uint32_t rI = __shfl_up_sync(0xffffffffu, sendI, 1);
        const int i = t - lane;
        const uint2 *rowQ = rowP++;
        uint32_t code[K] = {};
        const bool compute = !CHECKED || (mine && i >= 1 && i <= maxN);
        if (compute) {
            uint32_t t2 = fma_add(rH, keepLeft, leftH0);                          // H left + open
            uint32_t Il = fma_add(rI, keepLeft, leftI0);
            const uint2 tb = *rowQ;
            uint32_t Hd = prevLeftO;                                              // H diag, open form
            prevLeftO = t2;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint32_t e = prmt(tb.x, tb.y, sel[k]);                      // FOLD: substitution score - open (>= 0); else 0 / penalty
                const uint32_t hs = FOLD ? fma_add(e, one, Hd) : fma_add(e, negOne, Hd + (O4 + FOUR2));     // Hdiag + s(i,j)
                const uint32_t d = __viaddmax_u16x2(Dp[k], NEG_E4, HO[k]);         // max(D + ext, Hup + open)
                Il = __viaddmax_u16x2(Il, NEG_E4, t2);                             // max(I + ext, Hleft + open)
                const uint32_t h = __vimax3_u16x2(hs, d, Il);
                const uint32_t hf = __vmaxu2(h, fl[k]);                            // clip floor for j <= clipLt (CPU_DP.cpp:505-510)
                const uint32_t nhf = fma_add(hf, negOne, DP_C2);                   // C - H
                const uint32_t zdc = __viaddmax_u16x2(d, nhf, DP_CM1_2);           // C - (D == H ? 0 : 1)
                const uint32_t zrc = __viaddmax_u16x2(h, nhf, DP_CM1_2);           // C - (raised by the floor ? 1 : 0)
                code[k] = fma_add(zdc, one, fma_add(zrc, one, hf));                // low byte: 4H - zd - zr  (2C = 0 mod 256)
                Hd = HO[k];
                t2 = HO[k] = fma_add(O4, negOne, hf);
                Dp[k] = d;
            }
            sendH = t2; sendI = Il;
            // any cell of this step at or above the threshold?  (HO = H + open; T2 carries the offset)
            {
                uint32_t cm = HO[0];
#pragma unroll
                for (int k = 1; k + 1 < K; k += 2) cm = __vimax3_u16x2(cm, HO[k], HO[k + 1]);
                if (K % 2 == 0) cm = __vmaxu2(cm, HO[K - 1]);
                const uint32_t q = cm + T2;
                if (q & 0x80008000u) {
                    if (MASKED) {
                        uint32_t ho[K], z;                                         // a copy: HO itself must stay in registers, and the
                        asm volatile("mov.u32 %0, 0;" : "=r"(z));                  // copy must not be hoisted out of this rare branch
#pragma unroll
                        for (int k = 0; k < K; ++k) ho[k] = HO[k] + z;
                        T2 = dp_track_row_masked<K>(&tr, ho, q, i, (int)O4v);
                    } else T2 = dp_track_row(&tr, cm, q, i, (int)O4v);
                }
            }
#pragma unroll
            for (int kk = 0; kk < REM; ++kk) {
                const int bpos = u * REM + kk, pos = bpos & 3;                     // byte position inside the group's remainder words
                const uint32_t selA = 0x3210u ^ ((uint32_t)(4 ^ pos) << (4 * pos)), selB = 0x3210u ^ ((uint32_t)(6 ^ pos) << (4 * pos));
#pragma unroll
                for (int q = 0; q < REM; ++q)
                    if (q == (bpos >> 2)) {
                        accA[q] = __byte_perm(accA[q], code[4 * WORDS + kk], selA);
                        accB[q] = __byte_perm(accB[q], code[4 * WORDS + kk], selB);
                    }
            }
#pragma unroll
            for (int w = 0; w < WORDS; ++w)
#pragma unroll
                for (int c = 0; c < 3; ++c) hist[w][c][u] = code[4 * w + c];
        }
        // trace words: byte c of word w holds column 4w+c of row i-(3-c), so that a diagonal run of four cells shares one word.
        // Low halves -> task A, high halves -> task B.  Rows maxN+1..maxN+3 only flush the older bytes.
        if (!CHECKED || (mine && i >= 1 && i <= maxN + 3)) {
#pragma unroll
            for (int w = 0; w < WORDS; ++w) {
                const uint32_t c0 = hist[w][0][(u + 1) & 3], c1 = hist[w][1][(u + 2) & 3], c2 = hist[w][2][(u + 3) & 3], c3 = code[4 * w + 3];
                const uint32_t p01 = __byte_perm(c0, c1, 0x6240), p23 = __byte_perm(c2, c3, 0x6240);
                // p01 bytes: [c0.lo, c1.lo, c0.hi, c1.hi]
                const uint32_t wa = __byte_perm(p01, p23, 0x5410), wb = __byte_perm(p01, p23, 0x7632);
                *(uint32_t *)(pw + u * WB + w * 256) = wa;
                if (hasB) *(uint32_t *)(pw + u * WB + w * 256 + 128) = wb;
            }
        }
    };
    // remainder words of the four-step group that ends at step t
    auto flush = [&](const int t) {
        if (REM && mine && t - lane >= 1 && t - 3 - lane <= maxN) {
#pragma unroll
            for (int q = 0; q < REM; ++q) {
                *(uint32_t *)(pr + q * 256) = accA[q];
                if (hasB) *(uint32_t *)(pr + q * 256 + 128) = accB[q];
            }
        }
        pr += REM * 256;
    };
    auto group = [&](const int t, auto checked) {
        step(t, std::integral_constant<int, 0>(), checked);
        step(t + 1, std::integral_constant<int, 1>(), checked);
        step(t + 2, std::integral_constant<int, 2>(), checked);
        step(t + 3, std::integral_constant<int, 3>(), checked);
        flush(t + 3);
        pw += 4 * WB;

    };
    if (maxL > 0) {
        const int steadyN = (NA > 0 && NB > 0) ? min(NA, NB) : maxN;    // rows present in every live task of the pair
        const int stepsR = (steps + 3 + 3) & ~3;                        // + 3 flush steps, whole groups
        const int rampEnd = min(32, stepsR);                            // from here on every lane (owning or not) has a row >= 1
        const int steadyEnd = max(steadyN & ~3, rampEnd);               // up to here no owning lane has run out of rows
        // ramp-up and ramp-down share the CHECKED code, the steady groups in between run the straight-line variant
#pragma unroll 1
        for (int t = 1; t <= stepsR; ) {
            if (t > rampEnd && t <= steadyEnd) {
#pragma unroll 1
                for (; t <= steadyEnd; t += 4) group(t, std::false_type());
            } else { group(t, std::true_type()); t += 4; }
        }
    }
    __syncwarp();
    // ---- winner per task: best value over the lanes; the lanes that hold it read the position of its first cell (row-major) and the
    //      number of cells that tie back from their own trace bytes ----
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int lb = tr.lb[half], thr = tr.thr[half];
        int gbest = lb;
#pragma unroll
        for (int dlt = 16; dlt; dlt >>= 1) gbest = max(gbest, __shfl_xor_sync(0xffffffffu, gbest, dlt));
        uint32_t key = 0xffffffffu, c2 = 0u;
        if (lb == gbest && gbest >= thr && tr.elig[half])
            dp_resolve_lane<K>(tables + (size_t)(blockIdx.x * 8 + (threadIdx.x >> 5) * 2) * tableStride + half * 128, S, (int)(threadIdx.x & 31) * K + 1, tr.elig[half], tr.rfirst[half], tr.rlast[half], (gbest - DP_BIAS) >> 2, key, c2);
#ifdef MP_DEBUG_TRACK
        if (pairId == 0 && half == 0) printf("dbg lane %d lb %d gbest %d thr %d thrT %d elig %x r0 %d r1 %d T2 %x N %d L %d partial %d key %x\n", lane, lb, gbest, thr, tr.thrT[0], tr.elig[0], tr.rfirst[0], tr.rlast[0], T2, NA, LA, (int)partial, key);
        if (lb == gbest && gbest >= thr && tr.elig[half] && (key == 0xffffffffu || tr.rfirst[half] < 1 || tr.rlast[half] > (half ? NB : NA)))
            printf("track: pair %u half %d lane %d gbest %d thr %d lb %d r0 %d r1 %d N %d L %d elig %x key %x cnt %u partial %d\n", pairId, half, lane, gbest, thr, lb,
                   tr.rfirst[half], tr.rlast[half], half ? NB : NA, half ? LB : LA, tr.elig[half], key, c2, (int)partial);
#endif
#pragma unroll
        for (int dlt = 16; dlt; dlt >>= 1) { key = min(key, __shfl_xor_sync(0xffffffffu, key, dlt)); c2 += __shfl_xor_sync(0xffffffffu, c2, dlt); }
        if (lane == 0 && (half == 0 || hasB)) {
            FillOut f; f.score = (gbest - DP_BIAS) >> 2; f.row = key >> 12; f.col = key & 0xfffu; f.cnt = c2;
            if (gbest < thr || !(half ? okB : okA) || key == 0xffffffffu) { f.score = 0; f.row = 0; f.col = 0; f.cnt = 0; }
            fill[half == 0 ? tA : tB] = f;
        }
    }
}

// ---- GPUBacktrack (CPU_DP.cpp:622-786), literal; one thread per task ----
// The walk is bound by memory TRANSACTIONS (every lane of a warp touches its own sector), so all three streams go through
// one-word register caches: the trace table (a diagonal run of four cells shares a word, see cell_offset), the two sequences
// (packed words of 16 bases) and the pattern (four bytes per store; WORDPAT needs patStride % 4 == 0).
template <int K, bool WORDPAT>
__global__ void __launch_bounds__(128)
k_dp_tb(const uint32_t *__restrict__ refSeq, const uint32_t *__restrict__ refLens, uint32_t refStride,
        const uint32_t *__restrict__ readSeq, const uint32_t *__restrict__ readLens, uint32_t readStride,
        const int32_t *__restrict__ cutoffs, uint32_t taskBase, uint32_t nTasks, MpDpParams P,
        const uint8_t *__restrict__ tables, size_t tableStride, int S, const FillOut *__restrict__ fill,
        MpDpOut *__restrict__ outs, uint8_t *__restrict__ patterns, uint32_t patStride,
        const uint32_t *__restrict__ active, const uint32_t *__restrict__ nActive)
{
    const uint32_t lt = blockIdx.x * blockDim.x + threadIdx.x;
    if (active) nTasks = *nActive;
    if (lt >= nTasks) return;
    const uint32_t task = taskBase + (active ? active[lt] : lt);
    const int L = (int)readLens[task], cutoff = cutoffs[task];
    const int mm = P.mismatch, open = P.open, ext = -1, clipLt = P.clipLt;
    MpDpOut o; memset(&o, 0, sizeof o);
    const FillOut f = fill[task];
    if (cutoff > L || cutoff <= 0 || L >= 255 + open - 1 + cutoff || L > 32 * K || f.score < cutoff) { outs[task] = o; return; }
    const uint8_t *tab = tables + (size_t)(lt & ~1u) * tableStride + (lt & 1u) * 128;   // pair table + this task's half
    uint8_t *pat = patterns + (size_t)task * patStride;
    // ---- cached accessors ----
    uint32_t tabW = 0; size_t tabIdx = ~(size_t)0;
    auto cellAt = [&](int r, int c) -> uint32_t {           // trace byte of (row r >= 1, column c >= 1)
        const size_t off = cell_offset<K>(r, c, S);
        if ((off >> 2) != tabIdx) { tabIdx = off >> 2; tabW = __ldcs((const uint32_t *)tab + tabIdx); }   // read once or twice: keep it out of L1
        return (tabW >> ((off & 3) * 8)) & 0xffu;
    };
    auto flagAt = [&](int r, int c) -> int {                // flag of any cell including the virtual row 0 / column 0
        if (c == 0) return 0;                               // column 0 cells are stored as 0 (CPU_DP.cpp:447-450)
        if (r == 0) return c <= clipLt ? 0 : 1;             // row 0 (CPU_DP.cpp:405-427)
        return trace_flag(cellAt(r, c));
    };
    auto hmodAt = [&](int r, int c) -> int {                // H[r][c] mod 64 for any cell including row 0 / column 0
        if (r == 0) return h0_value(c, clipLt, open) & 63;
        if (c == 0) return 0;
        return trace_h(cellAt(r, c));
    };
    const uint32_t *rsRow = readSeq + (size_t)task * readStride, *fsRow = refSeq + (size_t)task * refStride;
    uint32_t rsW = 0, fsW = 0; int rsIdx = -1, fsIdx = -1;
    auto readBase = [&](int x) -> uint32_t {
        if ((x >> 4) != rsIdx) { rsIdx = x >> 4; rsW = __ldg(rsRow + rsIdx); }
        return (rsW >> ((x & 15) * 2)) & 3u;
    };
    auto refBase = [&](int x) -> uint32_t {
        if ((x >> 4) != fsIdx) { fsIdx = x >> 4; fsW = __ldg(fsRow + fsIdx); }
        return (fsW >> ((x & 15) * 2)) & 3u;
    };
    uint32_t p = 0, pacc = 0;
    auto emit = [&](uint32_t byte) {
        if (WORDPAT) {
            pacc |= byte << ((p & 3) * 8);
            if ((p & 3) == 3) { ((uint32_t *)pat)[p >> 2] = pacc; pacc = 0; }
        } else pat[p] = (uint8_t)byte;
        ++p;
    };
    // The special CIGAR is built while the pattern is emitted (same run merging as cigar_encode, which scans the finished pattern): a
    // finished run is written backwards from the end of the task's pattern row, so the text ends up in read order.  If pattern and
    // text would meet (hundreds of one-base runs), only the statistics are kept and the assembly pass encodes from the pattern.
    int cgType = 'N', cgCnt = 0, cgLast = 'N', cgLen = 0, cgI = 0, cgD = 0, cgS = 0, cgGap = 0;
    bool cgStored = P.cigText != 0;
    uint8_t *cw = pat + patStride;
    auto cgFlush = [&]() {
        if (cgCnt > 0 && cgType != 'N') {
            const int nd = ndigits(cgCnt);
            cgLen += nd + 1;
            if (cgType == 'I') cgI += cgCnt; else if (cgType == 'D') cgD += cgCnt; else if (cgType == 'S') cgS += cgCnt;
            if (cgType == 'I' || cgType == 'D') cgGap += open + (cgCnt - 1) * ext;
            if (cgStored) {
                if (cw - (nd + 1) < pat + p + 8) cgStored = false;
                else { *--cw = (uint8_t)cgType; int v = cgCnt; for (int d = 0; d < nd; ++d) { *--cw = (uint8_t)('0' + v % 10); v /= 10; } }
            }
        }
    };
    auto cgEvent = [&](int type, int cnt) { if (type == cgType) cgCnt += cnt; else { cgFlush(); cgType = type; cgCnt = cnt; } };
    auto sym = [&](uint32_t ch) { emit(ch); cgEvent((int)ch, 1); cgLast = (int)ch; };                                   // one pattern symbol
    auto rep = [&](uint32_t c) { emit('V'); emit(c & 0xffu); cgEvent(cgLast, (int)(c & 0xffu) - 1); };                   // 'V' <count>: the symbol before it, count times in all
    const int hitRow = (int)f.row, hitCol = (int)f.col;
    o.score = f.score; o.count = min(f.cnt, 255u);
    int clipR = L - hitCol;
    if (clipR > 0) { sym('S'); rep((uint32_t)clipR); }
    int i = L - clipR, j = hitRow;
    enum { NORMAL, I_EXT, D_EXT, SM_EXIT, SI_EXIT, SD_EXIT };
    int state = NORMAL;
    int accum = 0;
    // Every difference the reference reads from its table is rebuilt from H mod 64 of the two cells (trace byte layout above):
    // dd = H - Hdiag, hd = H - Hleft, vd = H - Hup.  `hcur` is H mod 64 of the current cell; a diagonal move hands the
    // predecessor's byte over, so the usual step costs one table access (and stays inside one cached word).
    uint32_t cell = cellAt(j, i);
    while (i > 0 && j > 0) {
        const int flag = trace_flag(cell), hcur = trace_h(cell);
        if (state == NORMAL) {
            // diagonal predecessor, including the virtual row 0 / column 0 (CPU_DP.cpp:405-450)
            uint32_t diagCell = 0; int dflag, hdiag;
            if (i - 1 == 0) { dflag = 0; hdiag = 0; }
            else if (j - 1 == 0) { dflag = (i - 1) <= clipLt ? 0 : 1; hdiag = h0_value(i - 1, clipLt, open) & 63; }
            else { diagCell = cellAt(j - 1, i - 1); dflag = trace_flag(diagCell); hdiag = trace_h(diagCell); }
            const int dd = trace_diff(hcur, hdiag);
            bool eq = refBase(j - 1) == readBase(i - 1);
            int ms = eq ? 1 : mm;
            if (dd == ms) {
                if (i != 1 && dflag == 0) { state = SM_EXIT; break; }
                sym(eq ? 'M' : 'm'); --j; --i;
                cell = diagCell;                                     // valid whenever the loop continues (i > 0 && j > 0)
                continue;
            } else if (flag == 1) {
                int vd = trace_diff(hcur, hmodAt(j - 1, i));
                sym('D'); --j;
                if (vd != open) { accum = (int8_t)(vd - ext); state = D_EXT; }
            } else {
                int hd = trace_diff(hcur, hmodAt(j, i - 1));
                sym('I'); --i;
                if (hd != open) { accum = (int8_t)(hd - ext); state = I_EXT; }
            }
        } else if (state == D_EXT) {
            int vd = trace_diff(hcur, hmodAt(j - 1, i));
            if (vd + accum == open && flagAt(j - 1, i) == 0) { state = SD_EXIT; break; }
            sym('D'); --j;
            if (vd + accum == open) state = NORMAL; else accum = (int8_t)(accum + vd - ext);
        } else {
            int hd = trace_diff(hcur, hmodAt(j, i - 1));
            if (hd + accum == open && flagAt(j, i - 1) == 0) { state = SI_EXIT; break; }
            sym('I'); --i;
            if (hd + accum == open) state = NORMAL; else accum = (int8_t)(accum + hd - ext);
        }
        if (i > 0 && j > 0) cell = cellAt(j, i);
    }
    bool discard = false;
    if (j == 0) {
        int sc = min(clipLt & 0xff, i);
        if (sc < i) { sym('I'); rep((uint32_t)(i - sc)); }
        sym('S'); rep((uint32_t)sc);
    } else if (state == SI_EXIT) {
        sym('I'); sym('S'); rep((uint32_t)(i - 1));
    } else if (state == SD_EXIT) {
        sym('D'); sym('S'); rep((uint32_t)(i - 1));
        discard = true;                                   // CPU_DP.cpp:842-857
    } else if (state == SM_EXIT) {
        sym((refBase(j - 1) == readBase(i - 1)) ? 'M' : 'm');
        sym('S'); rep((uint32_t)(i - 1));
        j -= 1;
    }
    o.patLen = p;
    emit(0);                                              // terminator
    if (WORDPAT && (p & 3)) ((uint32_t *)pat)[p >> 2] = pacc;
    cgFlush();
    if (cw < pat + p + 8) cgStored = false;               // the pattern grew into the text written earlier: the pattern is intact, the text is not
    o.cigLen = (uint16_t)cgLen; o.nI = (uint16_t)cgI; o.nD = (uint16_t)cgD; o.nS = (uint16_t)cgS; o.gapPenalty = (int16_t)cgGap; o.cigStored = cgStored ? 1 : 0;
    if (discard) { o.score = 0; o.hitLoc = 0; } else o.hitLoc = (uint32_t)j;
    outs[task] = o;
}

// ------------------------------------------------------------------------------------
// k_dp_prepare: one warp per task of a sub-batch, ahead of the DP kernels.
//  * tasks != nullptr (mpd_run_tasks; replaces packRead / repackDNA): gathers the task's reference window from the packed text and its
//    read from the batch, oriented (strand 2 reverse-complemented), into the task's two packed rows, and writes its scalars.  A task
//    that does not fit its rows is dropped (refLen = readLen = 0, hint -1), never written past them.
//  * tasks == nullptr (mpd_run_explicit): rows and scalars are already in place.
//  * needDp != nullptr: runs the exact-occurrence test on the packed words and sets needDp for every slot of the sub-batch.
//
// Exact-occurrence test.  If the read occurs in its reference window without a single difference, the DP answer is known:
//  * no cell can exceed its column index (a column adds at most the match score 1; clips, gaps and mismatches add <= 0), so the
//    maximum over the eligible columns is L, reached only in column L, exactly at the rows where an occurrence ends;
//  * the answer cell is the first such row (row-major order), the tie count the number of occurrences (CPU_DP.cpp:545-590);
//  * on the diagonal of an occurrence H = column index, so every traceback step sees H - Hdiag = 1 with equal bases, no cell of the
//    diagonal was raised by the clip floor (H >= 1 there), and GPUBacktrack emits L times 'M'; it stops at column 0, and when that
//    is also row 0 it appends the zero-length left clip "SV\0" (CPU_DP.cpp:788-871).
// Such tasks skip k_dp_fill / k_dp_tb; the others are compacted into `active`.  Every lane screens window offsets o, o + 32, ...: one
// XOR of a funnel-shifted pair of window words against a read word compares 16 bases.
// ------------------------------------------------------------------------------------
// 16 bases of the packed text (4 bases per byte, first base in the top bits) as one little-endian word -> first base in the low bits
__device__ __forceinline__ uint32_t pac_word(uint32_t x)
{
    x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
    return ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
}
__device__ __forceinline__ uint32_t reverse_bases(uint32_t x)          // base k -> base 15 - k
{
    x = __brev(x);
    return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}
__device__ __forceinline__ uint32_t base_mask(int n) { return n >= 16 ? 0xffffffffu : (1u << (2 * n)) - 1u; }   // the first n > 0 bases

__global__ void __launch_bounds__(128)
k_dp_prepare(MpIndexView ix, const uint32_t *__restrict__ reads, uint32_t wpq, const MpDpTask *__restrict__ tasks,
             uint32_t maxRefLen, uint32_t maxReadLen, uint32_t *__restrict__ refSeq, uint32_t refStride,
             uint32_t *__restrict__ readSeq, uint32_t readStride, uint32_t *__restrict__ refLens, uint32_t *__restrict__ readLens,
             int32_t *__restrict__ cutoffs, int16_t *__restrict__ hints, uint32_t taskBase, uint32_t nTasks, int maxL, MpDpParams P,
             MpDpOut *__restrict__ outs, uint8_t *__restrict__ patterns, uint32_t patStride, uint32_t *__restrict__ needDp)
{
    extern __shared__ uint32_t prepShared[];            // per warp: the window row + one zero word, the read row
    const int lane = threadIdx.x & 31;
    const uint32_t lt = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (lt == 0 && lane == 0 && needDp) needDp[nTasks] = 0;      // the scan runs over nTasks + 1 flags: the last sum is the total
    if (lt >= nTasks) return;
    const uint32_t task = taskBase + lt;
    uint32_t *win = prepShared + (threadIdx.x >> 5) * (refStride + 1 + readStride), *rw = win + refStride + 1;
    uint32_t *fo = refSeq + (size_t)task * refStride, *ro = readSeq + (size_t)task * readStride;
    int N, L, cutoff;
    if (tasks) {
        MpDpTask tk = tasks[task];
        if (!tk.valid || tk.refLen > maxRefLen || tk.readLen > maxReadLen) { tk.refLen = 0; tk.valid = 0; }
        N = (int)tk.refLen; L = tk.valid ? (int)tk.readLen : 0; cutoff = tk.cutoff;
        // window word w = text bases refStart + 16w .. + 15, from two aligned words of the text (the text buffer is allocation-aligned and
        // padded behind its last byte)
        const uint32_t *pac32 = (const uint32_t *)ix.pac;
        for (int w = lane; w < (int)refStride; w += 32) {
            uint32_t v = 0;
            if (16 * w < N) {
                const uint64_t p = tk.refStart + 16 * (uint32_t)w;
                const uint32_t sh = (uint32_t)(p & 15) * 2;
                const uint32_t lo = pac_word(__ldg(pac32 + (p >> 4))), hi = sh ? pac_word(__ldg(pac32 + (p >> 4) + 1)) : 0u;
                v = __funnelshift_r(lo, hi, sh) & base_mask(N - 16 * w);
            }
            fo[w] = v; win[w] = v;
        }
        const uint32_t *rd = reads + (size_t)tk.readID * wpq;
        for (int w = lane; w < (int)readStride; w += 32) {
            uint32_t v = 0;
            if (16 * w < L) {
                if (tk.strand == 1) v = rd[w];
                else {
                    // reverse complement: base 16w + k = 3 - read[L-1-16w-k], the complement of read[s .. s+15] reversed, s = L-16-16w >= -15
                    const int s = L - 16 - 16 * w, s0 = s < 0 ? 0 : s;
                    uint32_t x = __funnelshift_r(rd[s0 >> 4], (s0 & 15) ? rd[(s0 >> 4) + 1] : 0u, (uint32_t)(s0 & 15) * 2);
                    if (s < 0) x <<= 2 * (uint32_t)(-s);                      // base k = read[s + k]
                    v = ~reverse_bases(x);
                }
                v &= base_mask(L - 16 * w);
            }
            ro[w] = v; rw[w] = v;
        }
        if (lane == 0) { refLens[task] = (uint32_t)N; readLens[task] = (uint32_t)L; cutoffs[task] = cutoff; hints[task] = tk.valid ? tk.diag : (int16_t)-1; }
    } else {
        N = (int)refLens[task]; L = (int)readLens[task]; cutoff = cutoffs[task];
        for (int w = lane; w < (int)refStride; w += 32) win[w] = fo[w];
        for (int w = lane; w < (int)readStride; w += 32) rw[w] = ro[w];
    }
    if (!needDp) return;
    if (lane == 0) win[refStride] = 0u;                  // the funnel shift of the window's last word reads one word further
    __syncwarp();
    // same admission test as the DP kernels; scores must be the usual kind (match 1, everything else <= 0)
    const bool ok = !(cutoff > L || cutoff <= 0 || L >= 255 + P.open - 1 + cutoff || L > maxL) && L > 0 && N >= L &&
                    P.mismatch <= 0 && P.open <= 0;
    uint32_t occ = 0, first = 0xffffffffu;
    if (ok) {
        const int nw = (L + 15) >> 4;
        const uint32_t m0 = nw == 1 ? base_mask(L) : 0xffffffffu;
        for (int o = lane; o <= N - L; o += 32) {
            const uint32_t *wq = win + (o >> 4), sh = (uint32_t)(o & 15) * 2;
            bool same = ((__funnelshift_r(wq[0], wq[1], sh) ^ rw[0]) & m0) == 0;
            for (int k = 1; same && k < nw; ++k)
                same = ((__funnelshift_r(wq[k], wq[k + 1], sh) ^ rw[k]) & (k + 1 == nw ? base_mask(L - 16 * k) : 0xffffffffu)) == 0;
            if (same) { first = min(first, (uint32_t)o); ++occ; }
        }
        occ = __reduce_add_sync(0xffffffffu, occ);
        first = __reduce_min_sync(0xffffffffu, first);
    }
    if (occ == 0) { if (lane == 0) needDp[lt] = 1; return; }
    uint8_t *pat = patterns + (size_t)task * patStride;
    for (int k = lane; k < L; k += 32) pat[k] = 'M';
    if (lane == 0) {
        uint32_t p = (uint32_t)L;
        if (first == 0) { pat[p++] = 'S'; pat[p++] = 'V'; pat[p++] = 0; }      // j == 0: min(clipLt, i = 0) = 0 clipped bases
        pat[p] = 0;
        MpDpOut o; memset(&o, 0, sizeof o);
        o.score = L; o.hitLoc = first; o.count = min(occ, 255u); o.patLen = p;
        // its CIGAR is "<L>M" (a zero-length clip prints nothing), kept at the end of the pattern row like k_dp_tb does
        const int nd = ndigits(L);
        if (P.cigText && p + 8 + nd + 1 <= patStride) {
            uint8_t *cw = pat + patStride; *--cw = 'M';
            int v = L; for (int d = 0; d < nd; ++d) { *--cw = (uint8_t)('0' + v % 10); v /= 10; }
            o.cigStored = 1;
        }
        o.cigLen = (uint16_t)(nd + 1);
        outs[task] = o;
        needDp[lt] = 0;
    }
}
// slots of the tasks that still need the DP, in order; also adds up what the fill kernel is about to do (work accounting)
__global__ void k_dp_compact(const uint32_t *__restrict__ needDp, const uint32_t *__restrict__ pos, uint32_t nTasks, uint32_t taskBase,
                             const uint32_t *__restrict__ refLens, const uint32_t *__restrict__ readLens,
                             uint32_t *__restrict__ active, unsigned long long *__restrict__ counters)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long cells = 0; uint32_t exact = 0;
    if (t < nTasks) {
        if (needDp[t]) { active[pos[t]] = t; cells = (unsigned long long)refLens[taskBase + t] * readLens[taskBase + t]; }
        else exact = 1;
    }
    cells = __reduce_add_sync(0xffffffffu, (uint32_t)cells);        // refLen * readLen < 2^24 per task: 32 of them fit 32 bits
    exact = __reduce_add_sync(0xffffffffu, exact);
    if ((threadIdx.x & 31) == 0 && counters) { if (cells) atomicAdd(&counters[15], cells); if (exact) atomicAdd(&counters[14], (unsigned long long)exact); }
}

// Packed rows (k_dp_prepare, k_dp_fill, k_dp_tb): per task a window row of ceil(maxRefLen / 16) and a read row of ceil(maxReadLen / 16)
// words, 16 bases per word, first base in the low bits; the read already oriented.  Bases beyond a row's length are zero.
// dTasks != nullptr: k_dp_prepare fills rows, lengths, cutoffs and hints from the tasks; otherwise they are in place (dHints may be null).
static int launch_dp(mp_context *ctx, const MpDpTask *dTasks, uint32_t *dRef, uint32_t *dRefLens, uint32_t *dRead, uint32_t *dReadLens,
                     int32_t *dCutoffs, int16_t *dHints, uint32_t nTasks, uint32_t maxRefLen, uint32_t maxReadLen, const MpDpParams &Pin,
                     MpDpOut *dOuts, uint8_t *dPatterns, uint32_t patStride)
{
    if (nTasks == 0) return 0;
    const uint32_t refStride = (maxRefLen + 15) >> 4, readStride = (maxReadLen + 15) >> 4;
    MpDpParams P = Pin;
    if (const char *e = getenv("MP_CIG_TEXT")) if (e[0] == '0') P.cigText = 0;       // tests: the assembly pass encodes every CIGAR from its pattern
    const int K = maxReadLen <= 160 ? 5 : maxReadLen <= 256 ? 8 : 10;
    if (maxReadLen > 320) { mp_set_error("read length %u exceeds the DP kernel bound 320", maxReadLen); return MP_ERR_ARG; }
    if ((size_t)4 * (((size_t)maxRefLen + 44) & ~(size_t)3) * sizeof(uint2) > 200 * 1024) {
        mp_set_error("DP window of %u reference bases exceeds the shared-memory staging of the fill kernel (max ~6300)", maxRefLen); return MP_ERR_CAPACITY;
    }
    const int S = ((int)maxRefLen + 44) & ~3;                 // steps 1 .. maxRefLen + 31 + 3 flush steps, rounded up to groups of four, plus slack
    const size_t tableStride = (size_t)S * 32 * K;
    if (ctx->dFill.reserve((size_t)nTasks * sizeof(FillOut))) return MP_ERR_CUDA;
    // the traceback tables of one sub-batch stay in HBM between the two kernels.  A chunk of stage S1 has up to 2^18 tasks:
    // size for that even when this launch is smaller, and only talk to the allocator when the buffer really is too small
    const size_t typical = nTasks >= (1u << 15) ? (size_t)(1u << 18) * tableStride : (size_t)(nTasks + 1) * tableStride;
    const size_t ideal = std::max<size_t>((size_t)(nTasks + 1) * tableStride, typical);
    if (ctx->dTable.cap < ideal) {
        size_t freeB = 0, totalB = 0; cudaMemGetInfo(&freeB, &totalB);
        const size_t maxBytes = std::min<size_t>((size_t)24 << 30, (freeB + ctx->dTable.cap) / 2);
        const size_t want = std::min<size_t>(ideal, maxBytes);
        if (ctx->dTable.cap < want && ctx->dTable.reserve(want)) return MP_ERR_CUDA;
    }
    // tables are laid out per task PAIR: an odd final task still needs a whole pair table
    const uint32_t per = (uint32_t)std::min<size_t>(nTasks, (ctx->dTable.cap / tableStride) & ~(size_t)1);
    if (per == 0) { mp_set_error("not enough device memory for the DP traceback tables"); return MP_ERR_CUDA; }
    uint8_t *tab = ctx->dTable.as<uint8_t>();
    FillOut *fill = ctx->dFill.as<FillOut>();
    const size_t smem = (size_t)4 * S * sizeof(uint2);          // one 8-byte substitution table per reference row and warp
    // exact-occurrence shortcut (k_dp_prepare): MP_DP_EXACT=0 sends every task through the DP kernels
    static const bool useExact = !(getenv("MP_DP_EXACT") && getenv("MP_DP_EXACT")[0] == '0');
    // the lean tracker of k_dp_fill takes a lane's row maximum over all of its columns: legal when no column left of the eligible range
    // (j < L - clipRt) can reach a cutoff, i.e. L - clipRt - 1 < 30 <= cutoff for every read length of the batch (definitions.h:166-167)
    const bool rowMaxOk = (int)maxReadLen - P.clipRt - 1 < 30;
    const uint32_t perMax = std::min<uint32_t>(per, nTasks);
    if (useExact && (ctx->dExFlag.reserve(((size_t)perMax + 1) * 4) || ctx->dExPos.reserve(((size_t)perMax + 1) * 4) ||
                     ctx->dExIdx.reserve(((size_t)perMax + 1) * 4) || ctx->dCounters.reserve(16 * 8))) return MP_ERR_CUDA;
    const size_t prepSmem = (size_t)4 * (refStride + 1 + readStride) * 4;
    for (uint32_t base = 0; base < nTasks; base += per) {
        const uint32_t n = std::min<uint32_t>(per, nTasks - base);
        dim3 gridF((n + 7) / 8), gridT((n + 127) / 128), block(128);
        const uint32_t *active = nullptr, *nActive = nullptr;
        if (dTasks || useExact) {
            cudaEvent_t stop_ = ctx->ev_begin(2);
            uint32_t *needDp = useExact ? ctx->dExFlag.as<uint32_t>() : nullptr;
            (++g_mp_launches), k_dp_prepare<<<(n + 3) / 4, block, prepSmem, ctx->stream>>>(ctx->ix, ctx->dReads.as<uint32_t>(), ctx->wpq, dTasks,
                maxRefLen, maxReadLen, dRef, refStride, dRead, readStride, dRefLens, dReadLens, dCutoffs, dHints, base, n, 32 * K, P,
                dOuts, dPatterns, patStride, needDp);
            if (useExact) {
                size_t tb = 0;
                cub::DeviceScan::ExclusiveSum(nullptr, tb, needDp, ctx->dExPos.as<uint32_t>(), (int64_t)n + 1, ctx->stream);
                if (ctx->dScanTmp.reserve(tb)) return MP_ERR_CUDA;
                cub::DeviceScan::ExclusiveSum(ctx->dScanTmp.p, tb, needDp, ctx->dExPos.as<uint32_t>(), (int64_t)n + 1, ctx->stream);
                (++g_mp_launches), k_dp_compact<<<(n + 255) / 256, 256, 0, ctx->stream>>>(needDp, ctx->dExPos.as<uint32_t>(), n, base,
                    dRefLens, dReadLens, ctx->dExIdx.as<uint32_t>(), ctx->dCounters.as<unsigned long long>());
                active = ctx->dExIdx.as<uint32_t>(); nActive = ctx->dExPos.as<uint32_t>() + n;
            }
            ctx->ev_end(stop_);
        }
#define LAUNCH(KK) do { \
        cudaEvent_t stop_ = ctx->ev_begin(0); \
        if (P.mismatch == -2 && P.open == -3 && rowMaxOk) { \
            if (smem > 48 * 1024) MP_CUDA(cudaFuncSetAttribute(k_dp_fill<KK, -2, -3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            (++g_mp_launches), k_dp_fill<KK, -2, -3, false><<<gridF, block, smem, ctx->stream>>>(dRef, dRefLens, refStride, dRead, dReadLens, readStride, dCutoffs, dHints, \
                base, n, P, tab, tableStride, S, fill, active, nActive, 1u); \
        } else if (P.mismatch == -2 && P.open == -3) { \
            if (smem > 48 * 1024) MP_CUDA(cudaFuncSetAttribute(k_dp_fill<KK, -2, -3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            (++g_mp_launches), k_dp_fill<KK, -2, -3, true><<<gridF, block, smem, ctx->stream>>>(dRef, dRefLens, refStride, dRead, dReadLens, readStride, dCutoffs, dHints, \
                base, n, P, tab, tableStride, S, fill, active, nActive, 1u); \
        } else { \
            if (smem > 48 * 1024) MP_CUDA(cudaFuncSetAttribute(k_dp_fill<KK, 0, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            (++g_mp_launches), k_dp_fill<KK, 0, 0, true><<<gridF, block, smem, ctx->stream>>>(dRef, dRefLens, refStride, dRead, dReadLens, readStride, dCutoffs, dHints, \
                base, n, P, tab, tableStride, S, fill, active, nActive, 1u); \
        } \
        ctx->ev_end(stop_); stop_ = ctx->ev_begin(1); \
        if ((patStride & 3) == 0 && ((uintptr_t)dPatterns & 3) == 0) \
            (++g_mp_launches), k_dp_tb<KK, true><<<gridT, block, 0, ctx->stream>>>(dRef, dRefLens, refStride, dRead, dReadLens, readStride, dCutoffs, \
                base, n, P, tab, tableStride, S, fill, dOuts, dPatterns, patStride, active, nActive); \
        else \
            (++g_mp_launches), k_dp_tb<KK, false><<<gridT, block, 0, ctx->stream>>>(dRef, dRefLens, refStride, dRead, dReadLens, readStride, dCutoffs, \
                base, n, P, tab, tableStride, S, fill, dOuts, dPatterns, patStride, active, nActive); \
        ctx->ev_end(stop_); } while (0)
        if (K == 5) LAUNCH(5); else if (K == 8) LAUNCH(8); else LAUNCH(10);
#undef LAUNCH
        MP_CUDA(cudaGetLastError());
    }
    return 0;
}

int mpd_run_explicit(mp_context *ctx, uint32_t *dRef, uint32_t *dRefLens, uint32_t maxRefLen, uint32_t *dRead, uint32_t *dReadLens,
                     uint32_t maxReadLen, int32_t *dCutoffs, uint32_t nTasks, const MpDpParams &P, MpDpOut *dOuts, uint8_t *dPatterns,
                     uint32_t patStride)
{
    // The SemiGlobalAligner seam carries no seed diagonal: the fill kernel's threshold starts at the cutoff.  MP_DP_TEST_HINT=<d> (parity
    // tests) hands every task the same diagonal hint instead, right or wrong -- results must not depend on it.
    int16_t *dHints = nullptr;
    if (const char *e = getenv("MP_DP_TEST_HINT")) {
        std::vector<int16_t> h(nTasks, (int16_t)atoi(e));
        if (ctx->dHintTest.reserve((size_t)nTasks * 2)) return MP_ERR_CUDA;
        MP_CUDA(cudaMemcpyAsync(ctx->dHintTest.p, h.data(), (size_t)nTasks * 2, cudaMemcpyHostToDevice, ctx->stream));
        MP_CUDA(cudaStreamSynchronize(ctx->stream));
        dHints = ctx->dHintTest.as<int16_t>();
    }
    return launch_dp(ctx, nullptr, dRef, dRefLens, dRead, dReadLens, dCutoffs, dHints, nTasks, maxRefLen, maxReadLen, P,
                     dOuts, dPatterns, patStride);
}

int mpd_run_tasks(mp_context *ctx, const MpDpTask *dTasks, uint32_t nTasks, uint32_t maxRefLen, uint32_t maxReadLen,
                  const MpDpParams &P, MpDpOut *dOuts, uint8_t *dPatterns, uint32_t patStride)
{
    if (nTasks == 0) return 0;
    // packed rows (launch_dp), then lengths, cutoffs and hints of every task
    const size_t refW = (size_t)nTasks * ((maxRefLen + 15) >> 4), readW = (size_t)nTasks * ((maxReadLen + 15) >> 4);
    if (ctx->dRefSeq.reserve(refW * 4 + (size_t)nTasks * 14 + 16) || ctx->dReadSeq.reserve(readW * 4)) return MP_ERR_CUDA;
    uint32_t *dRef = ctx->dRefSeq.as<uint32_t>();
    uint32_t *dRefLens = dRef + refW;
    uint32_t *dReadLens = dRefLens + nTasks;
    int32_t *dCutoffs = (int32_t *)(dReadLens + nTasks);
    int16_t *dHints = (int16_t *)(dCutoffs + nTasks);
    return launch_dp(ctx, dTasks, dRef, dRefLens, ctx->dReadSeq.as<uint32_t>(), dReadLens, dCutoffs, dHints, nTasks, maxRefLen, maxReadLen, P,
                     dOuts, dPatterns, patStride);
}
