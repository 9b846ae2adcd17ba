// pbsc_dp_thread.cuh — Overlapper::extendMatch (Thirdparty/overlapper.cpp:421-701) as ONE ALIGNMENT PER THREAD.
//
// The warp-per-row kernel (dp_align_kernel) spends its instructions on lanes the matrix does not use: a query of the DP
// fallback is ~140 bases, the read retrieved for it ~1.1x that, so the 201-cell band is wider than the whole matrix, a band
// column holds ~150 computed cells of 224 lane slots, and every cell pays for the band-clipping predicates and the column
// max-scan.  Here a thread walks its own matrix column by column exactly like the reference's loop (no idle lanes, no
// predicates, no scan: the "up" dependency is a register), a warp holds 32 rows of (nearly) equal query length, and the
// previous column lives in shared memory as a 256-entry circular array of 16-bit scores indexed by the matrix row.
//
// The code below is plain scalar C++ over four small accessor types, so that tests/cpp/test_dp_thread.cpp can compile the
// very same fill/traceback with g++ and compare it with the oracle; the kernel instantiates it with shared-memory and
// interleaved-global accessors (pbsc_dp.cu).  Where two neighbouring columns allow it, the fill sweeps both at once with two
// 16-bit scores per register (fill_pair); tests/cpp/test_dp_pair.cpp and test_dp_pair_masked.cpp check that against the
// one-column fill (fill_col).
//
// Rules reproduced (all relative to the reference's band table, band row r = j - (origin + i), 0 <= r <= 200):
//   * the table is zero-initialised and column 0 / row 0 are never written: they read as 0;
//   * first computed cell of a column: "up" is not consulted; "left" only if it is inside the band (r < 200);
//   * last computed cell (when it is not also the first): "left" is ignored, even if the band was clipped by the matrix
//     and the cell exists;
//   * the traceback compares the cell with ALL in-band neighbours (also the ones the fill ignored), a neighbour outside the
//     band never compares equal; its three tie-break orders are the reference's (:620-680).
// A computed cell only ever reads cells computed in the previous column, row 0, or (first computed column) cells nothing has
// written yet, so an in-place array indexed by the matrix row reproduces the zero-initialised table.  Queries longer than
// QMAX stay with the warp-per-row kernel.
#ifndef PBSC_DP_THREAD_CUH
#define PBSC_DP_THREAD_CUH

#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#if defined(__CUDACC__)
#define PBSC_DPT_HD __host__ __device__ __forceinline__
#else
#define PBSC_DPT_HD inline
#endif

namespace pbsc { namespace dpt {

constexpr int HALF = 100;              // bandwidth 200 (LongReadOverlap.cpp:629)
constexpr int BW = 2 * HALF + 1;       // cells per band column
constexpr int CPW = 10;                // cells per 32-bit word of traceback flags (3 bits each)
constexpr int WMAX = (BW + CPW - 1) / CPW;
constexpr int NEVER = -(1 << 28);      // a neighbour that is not there: never the maximum, never equal
constexpr int OP_M = 0, OP_I = 1, OP_D = 2;
constexpr int HSLOTS = 256;            // circular previous-column array: the live rows are [jb - 1, jb + 200]

// append "v != x" to a word of flags, for v >= x: x - v is negative exactly when they differ, and its sign bit is shifted in
// by one funnel shift (the caller inverts the finished word)
PBSC_DPT_HD uint32_t push_ne(uint32_t w, int v, int x)
{
#if defined(__CUDA_ARCH__)
    return __funnelshift_l((uint32_t)(x - v), w, 1);
#else
    return (w << 1) | ((uint32_t)(x - v) >> 31);
#endif
}
PBSC_DPT_HD int imax(int a, int b) { return a > b ? a : b; }
PBSC_DPT_HD int imin(int a, int b) { return a < b ? a : b; }

// longest read retrieved for a query of qmax bases: query.length()*1.1+20 (LongReadOverlap.cpp:611), rounded up
PBSC_DPT_HD constexpr int max_len_bound(int qmax) { return qmax + qmax / 10 + 21; }

// the scores fit 16 bits (|score| <= 8 * qlen) and the read fits its shared-memory slot.  Columns whose band misses the
// matrix (the reference's `continue`, overlapper.cpp:470-471) can only be the first ones (band above the matrix) or the
// last ones (band below it); the fill skips them like the reference: the first computed column then reads a column array
// that is still all zero, like the reference's zero-initialised table, and nothing reads the trailing ones (the traceback
// starts in a computed cell and leaves the matrix before it could enter a skipped column).
PBSC_DPT_HD bool eligible(int qlen, int mlen, int /*origin*/, int qmax) { return qlen >= 1 && qlen <= qmax && mlen >= 1 && mlen <= max_len_bound(qmax); }
// flag words per column: ordinals count from the even row at or below the first computed one, the widest column has
// min(201, mlen) cells
PBSC_DPT_HD int words_per_col(int mlen) { return (imin(BW, mlen) + 1 + CPW - 1) / CPW; }

// ---- two 16-bit scores in one 32-bit word: the low half belongs to column i, the high half to column i + 1 ----------------
// Device: the sm_100 SIMD instructions (VIADD.16x2, VIMNMX3.S16x2, VIADDMNMX.S16x2, PRMT).  Host: the same lane arithmetic,
// which aborts if a lane leaves the int16 range, so the host tests catch a packed score that would wrap.
PBSC_DPT_HD int lo16(uint32_t x) { return (int)(int16_t)(x & 0xFFFFu); }
PBSC_DPT_HD int hi16(uint32_t x) { return (int)(int16_t)(x >> 16); }
#if !defined(__CUDA_ARCH__)
PBSC_DPT_HD uint32_t pk16(int lo, int hi)
{
    if (lo < -32768 || lo > 32767 || hi < -32768 || hi > 32767) { printf("packed 16-bit lane overflow\n"); abort(); }
    return (uint32_t)(uint16_t)lo | ((uint32_t)(uint16_t)hi << 16);
}
#endif
PBSC_DPT_HD uint32_t v2add(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vadd2(a, b);
#else
    return pk16(lo16(a) + lo16(b), hi16(a) + hi16(b));
#endif
}
PBSC_DPT_HD uint32_t v2sub(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vsub2(a, b);
#else
    return pk16(lo16(a) - lo16(b), hi16(a) - hi16(b));
#endif
}
PBSC_DPT_HD uint32_t v2max3(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __vimax3_s16x2(a, b, c);
#else
    return pk16(imax(imax(lo16(a), lo16(b)), lo16(c)), imax(imax(hi16(a), hi16(b)), hi16(c)));
#endif
}
// max(a + b, c) per half
PBSC_DPT_HD uint32_t v2addmax(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __viaddmax_s16x2(a, b, c);
#else
    return pk16(imax(lo16(a) + lo16(b), lo16(c)), imax(hi16(a) + hi16(b), hi16(c)));
#endif
}
// min(a + b, c) per half
PBSC_DPT_HD uint32_t v2addmin(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __viaddmin_s16x2(a, b, c);
#else
    return pk16(imin(lo16(a) + lo16(b), lo16(c)), imin(hi16(a) + hi16(b), hi16(c)));
#endif
}
PBSC_DPT_HD uint32_t v2max(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vmaxs2(a, b);
#else
    return pk16(imax(lo16(a), lo16(b)), imax(hi16(a), hi16(b)));
#endif
}
// bytes of (b:a) picked by the four nibbles of sel (__byte_perm without the sign-replicate mode)
PBSC_DPT_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    const uint64_t ab = (uint64_t)a | ((uint64_t)b << 32);
    uint32_t r = 0;
    for (int k = 0; k < 4; k++) r |= (uint32_t)((ab >> (8 * ((sel >> (4 * k)) & 7u))) & 0xFFu) << (8 * k);
    return r;
#endif
}

// the bits of b where m is set, those of a elsewhere (one LOP3); m selects whole 16-bit halves here
PBSC_DPT_HD uint32_t sel16(uint32_t a, uint32_t b, uint32_t m) { return (a & ~m) | (b & m); }
PBSC_DPT_HD int popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// Phase hooks of the fill: clk_mark(H, p) charges the time since the previous mark to phase p, clk_cells(H, p, n) counts n
// computed cells for the path p.  No-ops for every accessor except the one of the kernel's -DPBSC_STAGE_CLOCKS measurement
// build (pbsc_dp.cu), which overloads them.
constexpr int CLK_COLS = 0, CLK_MASKED = 1, CLK_BLOCKS = 2;   // one-column fills; masked paired blocks; unmasked paired blocks
template <class HS> PBSC_DPT_HD void clk_mark(HS&, int) {}
template <class HS> PBSC_DPT_HD void clk_cells(HS&, int, int) {}
// Hook of the paired fill: pair_sweep(H, fB, lB) before a sweep of fill_pair, whose second column computes rows fB .. lB, and
// pair_sweep(H, 1, 0) after it.  A no-op except for the accessor of the host test tests/cpp/test_dp_pair_masked.cpp, which
// checks the sweep's stores against those rows.
template <class HS> PBSC_DPT_HD void pair_sweep(HS&, int, int) {}

// running state of the fill across columns
struct FillBest { int rowVal = 0, rowI = 0; bool anyRow = false; };
PBSC_DPT_HD void note_last_row(FillBest& b, int v, int i)
{
    // best cell of the last row: first column with the strictly largest score (:553-561)
    if (!b.anyRow || v > b.rowVal) { b.rowVal = v; b.rowI = i; b.anyRow = true; }
}

// Fill.  H: previous/current column, zero on entry: get(j) / set(j, v) one score; pairs_ok(j) / get2(j, u) / set2(j, u, w)
// the packed scores of rows j + 2u, j + 2u + 1 (j even, u = 0..4) when those ten rows do not wrap around the circular array.
// S: the read, S.base(x) = code of s2[x], S.bits(x) = 2-bit codes of s2[x .. x + 9] in bits 0..19.  F: flag words
// (put(n, w)).  q(x) = code of s1[x].
// Flags of cell (i, j): ordinal k = j - (first & ~1), word (i - 1) * W + k / 10, bits 3 * (9 - k % 10) ..+2 =
// {equals diagonal, equals up - 1, equals left - 1}.  Ordinals start at an even row so that whole flag words are five
// aligned pairs of rows: one 32-bit shared-memory load and store per two cells.
//
// fill_col: one column i (wbase = its first flag word), one cell at a time.
template <class HS, class SS, class FS, class QF>
PBSC_DPT_HD void fill_col(int i, int mlen, int origin, int wbase, HS& H, const SS& S, FS& F, const QF& q, FillBest& best)
{
    const int nRows = mlen + 1;
    {
        const int jb = origin + i;
        const int first = imax(jb, 1);
        const int last = imin(jb + BW, nRows) - 1;
        if (last < first) return;   // the band misses the matrix
        const int c1 = q(i - 1);
        const uint32_t c1rep = (uint32_t)c1 * 0x55555u;
        int j = first;
        int diagOld = H.get(j - 1);
        int widx = wbase, kin = (first & 1) + 1;
        int up, v;
        uint32_t w;
        {
            // first cell of the column (overlapper.cpp:497-509)
            const int leftOld = H.get(j);
            const int d = diagOld + (S.base(j - 1) == c1 ? 1 : -8);
            const int l1 = (j == jb + BW - 1) ? NEVER : leftOld - 1;
            const int u1 = first > jb ? -1 : NEVER;   // row 0 of the matrix reads 0; above band row 0 there is nothing
            v = imax(d, l1);
            w = (v == d ? 1u : 0u) | (v == u1 ? 2u : 0u) | (v == l1 ? 4u : 0u);
            H.set(j, v);
            up = v; diagOld = leftOld;
            j++;
        }
        // middle cells [first + 1, last): all three neighbours
        auto rolled = [&](int jend)
        {
#if defined(__CUDA_ARCH__)
            #pragma unroll 1
#endif
            for (; j < jend; j++)
            {
                const int leftOld = H.get(j);
                const int d = diagOld + (S.base(j - 1) == c1 ? 1 : -8);
                const int l1 = leftOld - 1, u1 = up - 1;
                const int vv = imax(imax(d, l1), u1);
                w = (w << 3) | (vv == d ? 1u : 0u) | (vv == u1 ? 2u : 0u) | (vv == l1 ? 4u : 0u);
                H.set(j, vv);
                up = vv; diagOld = leftOld;
                if (++kin == CPW) { F.put(widx++, w); w = 0; kin = 0; }
            }
        };
        rolled(imin(last, (first & ~1) + CPW));   // up to the end of the first flag word
#if defined(__CUDA_ARCH__)
        #pragma unroll 1
#endif
        while (j + CPW <= last)                   // whole flag words: kin == 0 and j is even here
        {
            if (!H.pairs_ok(j)) { rolled(j + CPW); continue; }
            const uint32_t x = S.bits(j - 1) ^ c1rep;
            uint32_t ww = 0;
#if defined(__CUDA_ARCH__)
            #pragma unroll
#endif
            for (int u = 0; u < CPW / 2; u++)
            {
                const uint32_t old2 = H.get2(j, u);
                const int leftA = (int)(int16_t)(old2 & 0xFFFFu), leftB = (int)old2 >> 16;
                // max(d, left - 1, up - 1) = max(d + 1, left, up) - 1: the three candidates without their own decrements
                const int eA = diagOld + ((x & (3u << (4 * u))) == 0u ? 2 : -7);
                const int xA = imax(imax(eA, leftA), up);
                const int vA = xA - 1;
                const int eB = leftA + ((x & (12u << (4 * u))) == 0u ? 2 : -7);
                const int xB = imax(imax(eB, leftB), vA);
                const int vB = xB - 1;
                ww = push_ne(push_ne(push_ne(ww, xA, leftA), xA, up), xA, eA);   // bit 2 left, bit 1 up, bit 0 diagonal
                ww = push_ne(push_ne(push_ne(ww, xB, leftB), xB, vA), xB, eB);
                H.set2(j, u, ((uint32_t)vA & 0xFFFFu) | ((uint32_t)vB << 16));
                up = vB; diagOld = leftB;
            }
            F.put(widx++, ww ^ 0x3FFFFFFFu);   // "differs" bits -> "equals" bits
            j += CPW;
        }
        rolled(last);
        if (last > first)
        {
            // last cell of the column (:510-516): no left in the fill; the traceback still sees it when it is in the band
            const int d = diagOld + (S.base(last - 1) == c1 ? 1 : -8);
            const int u1 = up - 1;
            const int l1 = (last == jb + BW - 1) ? NEVER : H.get(last) - 1;
            v = imax(d, u1);
            w = (w << 3) | (v == d ? 1u : 0u) | (v == u1 ? 2u : 0u) | (v == l1 ? 4u : 0u);
            H.set(last, v);
            if (++kin == CPW) { F.put(widx++, w); w = 0; kin = 0; }
        }
        if (kin) F.put(widx, w << (3 * (CPW - kin)));
        if (last == nRows - 1) note_last_row(best, v, i);
        clk_cells(H, CLK_COLS, last - first + 1);
        clk_mark(H, CLK_COLS);
    }
}

// Can fill_pair take columns i and i + 1 (i < qlen)?  Both bands start at row 1 (the band top is above the matrix in both),
// or both start inside the matrix at band row 0 with column i's first row even.  Then column i + 1's ordinals count from the
// same even row as column i's, and its cell in row j - 1 is one ordinal behind column i's cell in row j.  Both columns must
// meet the matrix.  Any other column (the one or two where the band top crosses row 1, every other column when the band
// top is at an odd row, the ones whose band misses the matrix, the last one of an odd count) goes through fill_col.
PBSC_DPT_HD bool pairable(int i, int mlen, int origin)
{
    const int jb = origin + i;
    return jb <= 0 ? jb + BW - 1 >= 1 : (jb >= 2 && (jb & 1) == 0 && jb + 1 <= mlen);
}

// fill_pair: columns A = i and B = i + 1 in one sweep.  Step j computes A(j) and B(j - 1), which are independent: A(j) reads
// A(j - 1) and column i - 1 (rows j - 1, j), B(j - 1) reads B(j - 2), A(j - 2) and A(j - 1).  B(j - 1) replaces row j - 1
// of column i - 1 in H, which A read last at step j - 1, so after the sweep H holds column i + 1 (rows of column i are
// never stored: nothing reads them).  Each column keeps its own flag words, exactly as fill_col writes them.
//
// The sweep is a run of ten-step blocks from A's row j0 = fA & ~1, where the flag ordinals of both columns start, until B's
// last row lB is computed.  A block from row j writes A's flag word of rows j .. j + 9 and completes B's of rows j - 10 ..
// j - 1.  One 32-bit register per quantity, A in the low half and B in the high half:
//   up = the result of the step before; left = (column i - 1 at row j, A(j - 1)), one PRMT from H's pair word; diagonal =
//   the left of the step before; x = max(d + 1, left, up) with d + 1 = diagonal + (2 or -7), and the "equals" flags from
//   max(candidate + 2 - x, 1), which is 2 or 1 per half.  Five pair stores of B per block (rows j - 2 .. j + 7; B(j + 8) is
//   stored after the last block).  Every pair is addressed on its own, so a block may wrap around H's circular array: rows of
//   a warp's alignments reach the wrap at different blocks, and a branch there would make the warp run both paths.
// A block whose twenty cells are all middle cells of their columns runs as just described.  The first block and the last one
// or two (the masked blocks) apply fill_col's rules per half with selects, from bit masks of the block's steps computed once
// per block:
//   * first cell (row fA, fB): "up" is the sentinel in the max; the flags compare it with row 0 (0) when the band top is
//     above the matrix, else never;
//   * last cell (row lA, lB) when it is not also the first, or when it is band row 200: "left" is the sentinel in the max;
//     the flags still compare it unless the row is band row 200 (only the last row of a column can be);
//   * steps whose row lies outside the column: no flags, and the pair stores keep H's old half; A's row 0 (band top above
//     the matrix) is set to 0, which B's first cell reads as its diagonal;
//   * the first block completes no word of B, a block past lA writes no word of A.
// 16 bits suffice for the packed differences: every cell of column i is >= -2 i - 209 (the band's top cell reads its left
// neighbour, which reads its up neighbour; down a column each cell reads its up neighbour) and <= i + 1, so for
// qlen <= 4000 a difference of two candidates is > -12300, and the sentinel plus 2 - x lies in [-24000, -11789].
constexpr uint32_t SENT2 = 0xB1E0B1E0u;   // -20000 per half: below every cell, so never the maximum and never equal to it

template <bool M> struct Masked { static constexpr bool value = M; };

template <class HS, class SS, class FS, class QF>
PBSC_DPT_HD void fill_pair(int i, int mlen, int origin, int wbase, HS& H, const SS& S, FS& F, const QF& q, FillBest& best)
{
    const int nRows = mlen + 1;
    const int W = words_per_col(mlen);
    const int jbA = origin + i, jbB = jbA + 1;
    const int fA = imax(jbA, 1), fB = imax(jbB, 1);
    const int lA = imin(jbA + BW, nRows) - 1, lB = imin(jbB + BW, nRows) - 1;
    const int j0 = fA & ~1;
    const int cA = q(i - 1), cB = q(i);
    const uint32_t cArep = (uint32_t)cA * 0x55555u, cBrep = (uint32_t)cB * 0x55555u;
    pair_sweep(H, fB, lB);
    // per half, for the masked blocks: "up" of the first cell as its flags see it; the last cell leaves "left" out of the max;
    // the last cell is band row 200
    const bool a200 = lA == jbA + BW - 1, b200 = lB == jbB + BW - 1;
    const uint32_t upF = (jbA <= 0 ? 0u : 0xB1E0u) | (jbB <= 0 ? 0u : 0xB1E00000u);
    const uint32_t exL = (lA > fA || a200 ? 0xFFFFu : 0u) | (lB > fB || b200 ? 0xFFFF0000u : 0u);
    const uint32_t row200 = (a200 ? 0xFFFFu : 0u) | (b200 ? 0xFFFF0000u : 0u);
    // D = (column i - 1 at row j - 1, A(j - 2)): the diagonals; V = (A(j - 1), B(j - 2)): the ups (before j0: no cells)
#if defined(__CUDA_ARCH__)
    uint32_t D = (uint32_t)H.get(j0 - 1) & 0xFFFFu, V = 0u;
#else
    uint32_t D = pk16(H.get(j0 - 1), 0), V = 0u;
#endif
    // the read windows of a block (bases j - 1 .. j + 8 for A, j - 2 .. j + 7 for B), loaded one block ahead; the first one
    // from the sweep's first base, origin + i - 1 (or 0), shifted: the steps before it compute no cell
    uint32_t na, nb;
    {
        const uint32_t w = S.bits(imax(j0 - 1, 0));
        na = j0 ? w : w << 2;
        nb = na << 2;
    }
    uint32_t wB = 0, vl = 0;   // B's pending flags (rows j - 10 .. j - 2); (A(lA), B(lB)) once computed
    int xA = wbase, xB = wbase + W;
    int j = j0;
    auto block = [&](auto masked)
    {
        constexpr bool M = decltype(masked)::value;
        // bit s: step s computes a cell of A (row j + s), bit 16 + s: of B (row j + s - 1); the first and the last cells
        uint32_t inM = 0x03FF03FFu, firstM = 0u, lastM = 0u;
        bool head = false;
        if constexpr (M)
        {
            auto below = [](int n) { return (1u << imin(imax(n, 0), CPW)) - 1u; };   // steps 0 .. n - 1
            auto at = [&](int n) { return below(n + 1) & ~below(n); };               // step n
            inM = (below(lA - j + 1) & ~below(fA - j)) | ((below(lB - j + 2) & ~below(fB - j + 1)) << 16);
            firstM = at(fA - j) | (at(fB - j + 1) << 16);
            lastM = at(lA - j) | (at(lB - j + 1) << 16);
            head = j == j0;
        }
        const uint32_t xa = na ^ cArep, xb = nb ^ cBrep;
        if (!M || j + CPW <= lA) na = S.bits(j + CPW - 1);       // the next block's, when it has cells of A
        if (!M || j + CPW - 1 <= lB) nb = S.bits(j + CPW - 2);   // ... of B
        const uint32_t ma = (xa | (xa >> 1)) & 0x55555u, mb = (xb | (xb >> 1)) & 0x55555u;   // bit 2s: step s mismatches
        const uint32_t m1 = (ma & 0xFFFFu) | (mb << 16);                                       // steps 0..7, both halves
        const uint32_t m2 = (ma >> 16) | (mb & 0xF0000u);                                      // steps 8, 9
        uint32_t hw[CPW / 2];
#if defined(__CUDA_ARCH__)
        #pragma unroll
#endif
        for (int u = 0; u < CPW / 2; u++) hw[u] = H.get2(j + 2 * u, 0);   // each pair on its own: the block may wrap
        // flags of steps 0..4 and 5..9, per half sum over the steps s of (7 + f_s) * 8^(4 - s mod 5) = 0x7FFF + the three-bit
        // "equals" flags f_s; at most 14 * 4681 < 2^16, so the halves never carry into each other
        uint32_t Wa = 0, Wb = 0;
#if defined(__CUDA_ARCH__)
        #pragma unroll
#endif
        for (int s = 0; s < CPW; s++)
        {
            const uint32_t p = (s < 8 ? m1 >> (2 * s) : m2 >> (2 * (s - 8))) & 0x00010001u;
            const uint32_t e = v2add(D, p * 0xFFF7u + 0x00020002u);   // diagonal + 2 (match) or - 7 per half, no carry across
            const uint32_t L = prmt(hw[s >> 1], V, (s & 1) ? 0x5432u : 0x5410u);
            // per half: the step computes its column's first cell, its last cell, a cell at all (constants when unmasked)
            const uint32_t mf = ((firstM >> s) & 0x00010001u) * 0xFFFFu, ml = ((lastM >> s) & 0x00010001u) * 0xFFFFu;
            const uint32_t mi = ((inM >> s) & 0x00010001u) * 0xFFFFu;
            const uint32_t X = v2max3(e, sel16(L, SENT2, ml & exL), sel16(V, SENT2, mf));
            const uint32_t K = v2add(~X, 0x00030003u);   // 2 - X: max(candidate + K, 1) is 2 where the candidate equals X, else 1
            uint32_t fU, fL;
            if constexpr (M)
            {
                // the flags' "up" of a first cell and "left" of a last cell are not in the max and may exceed X:
                // max(min(c + K, X + 2 - c), 1) is 2 where c equals X, else 1
                const uint32_t X2 = v2add(X, 0x00020002u), U = sel16(V, upF, mf), Lf = sel16(L, SENT2, ml & row200);
                fU = v2max(v2addmin(U, K, v2sub(X2, U)), 0x00010001u);
                fL = v2max(v2addmin(Lf, K, v2sub(X2, Lf)), 0x00010001u);
            }
            else { fU = v2addmax(V, K, 0x00010001u); fL = v2addmax(L, K, 0x00010001u); }
            uint32_t f = v2addmax(e, K, 0x00010001u) + (fU << 1) + (fL << 2);
            f = sel16(0x00070007u, f, mi);   // no flags outside the column
            if (s < CPW / 2) Wa = (Wa << 3) + f; else Wb = (Wb << 3) + f;
            uint32_t Vn = v2add(X, 0xFFFFFFFFu);   // X - 1 per half
            if (M && s == 0 && j == 0) Vn &= 0xFFFF0000u;   // A(0): row 0 reads 0
            if ((s & 1) == 0)
            {
                const uint32_t b2 = prmt(V, Vn, 0x7632u);   // B(j + s - 2), B(j + s - 1)
                if (s == 0) { if (!head) H.set2(j - 2, 0, b2); }   // inside B's rows in every block but the first
                else
                {
                    const uint32_t t = inM >> (16 + s - 1);   // which of the two rows are B's cells
                    H.set2(j + s - 2, 0, sel16(hw[s / 2 - 1], b2, ((t & 1u) * 0xFFFFu) | ((t & 2u) * 0x7FFF8000u)));
                }
            }
            vl = sel16(vl, Vn, ml);
            D = L; V = Vn;
        }
        Wa -= 0x7FFF7FFFu; Wb -= 0x7FFF7FFFu;
        if (!M || j <= lA) F.put(xA++, ((Wa & 0x7FFFu) << 15) | (Wb & 0x7FFFu));
        if (!head) F.put(xB++, (wB << 3) | (Wa >> 28));
        wB = ((Wa >> 1) & 0x7FF8000u) | (Wb >> 16);
        clk_cells(H, M ? CLK_MASKED : CLK_BLOCKS, popc(inM));
        j += CPW;
    };
#if defined(__CUDA_ARCH__)
    #pragma unroll 1
#endif
    do
    {
        block(Masked<true>{});   // the first block, then the last one or two
        clk_mark(H, CLK_MASKED);
#if defined(__CUDA_ARCH__)
        #pragma unroll 1
#endif
        while (j + CPW <= lA) block(Masked<false>{});
        clk_mark(H, CLK_BLOCKS);
    } while (j - 1 <= lB);
    if (j - 2 <= lB) H.set(j - 2, hi16(V));   // the last block left B(j - 2) for the next one
    if (j - CPW <= lB) F.put(xB, wB << 3);    // B's last word: rows j - 10 .. j - 2 and no cell in row j - 1
    if (lA == nRows - 1) note_last_row(best, lo16(vl), i);
    if (lB == nRows - 1) note_last_row(best, hi16(vl), i + 1);
    pair_sweep(H, 1, 0);
}

// Read window.  A sweep from column i (fill_col, or fill_pair of i and i + 1) reads the read from base origin + i - 1 on, and
// S.bits at origin + i + 200 at most, which takes that base's word and the next one; with 16 bases per word, those are words
// win_lo(i) .. win_hi(i), at most 15, clipped to the read and the zero word after it.  win_hi grows by at most one word from
// a sweep to the next (two columns on), and win_hi(i + 2) <= win_lo(i) + 14: the ring slot of the word it adds holds a word at
// least two below win_lo(i), which the sweep before does not read.  So an accessor that keeps only a ring of 16 words of the
// read (the kernel's global-read passes, pbsc_dp.cu) needs one load per sweep: fill() calls win_fetch(S, mlen, origin, i, inext) before the sweep from i and win_store(S, what it returned) after
// it, and the next sweep from inext finds its words in the ring.  For an accessor that holds the whole read both do nothing.
PBSC_DPT_HD int win_lo(int i, int origin) { return imax(origin + i - 1, 0) >> 4; }
PBSC_DPT_HD int win_hi(int i, int mlen, int origin) { return imin(((origin + i + BW - 1) >> 4) + 1, (mlen + 15) >> 4); }
template <class SS> PBSC_DPT_HD int win_fetch(const SS&, int /*mlen*/, int /*origin*/, int /*i*/, int /*inext*/) { return 0; }
template <class SS, class T> PBSC_DPT_HD void win_store(const SS&, const T&) {}

// the two query bases a sweep from column i reads, q(i - 1) and q(i), loaded before it
struct QCols
{
    int i0, c0, c1;
    PBSC_DPT_HD int operator()(int x) const { return x == i0 ? c0 : c1; }
};

// Whole fill: columns 1..qlen, in pairs where pairable() allows (pair = false: one column at a time throughout); (bi, bj) =
// start of the traceback, bi = 0 when there is none.
template <class HS, class SS, class FS, class QF>
PBSC_DPT_HD void fill(int qlen, int mlen, int origin, HS& H, const SS& S, FS& F, const QF& q, int& bi, int& bj, bool pair = true)
{
    const int nRows = mlen + 1;
    const int W = words_per_col(mlen);
    FillBest best;
    int i = 1, wbase = 0;
    // the query bases of a sweep (columns i, i + 1) and the read word the next sweep adds to a window accessor are loaded one
    // sweep ahead, so that no sweep starts on a load
    int c0 = q(0), c1 = qlen > 1 ? q(1) : 0;
    bool pr = pair && 1 < qlen && pairable(1, mlen, origin);
#if defined(__CUDA_ARCH__)
    #pragma unroll 1
#endif
    while (i <= qlen)
    {
        const int inext = i + (pr ? 2 : 1);
        const auto wn = win_fetch(S, mlen, origin, i, inext);
        const int n0 = inext <= qlen ? q(inext - 1) : 0, n1 = inext < qlen ? q(inext) : 0;
        const QCols qc{i - 1, c0, c1};
        if (pr) fill_pair(i, mlen, origin, wbase, H, S, F, qc, best);
        else fill_col(i, mlen, origin, wbase, H, S, F, qc, best);
        win_store(S, wn);
        wbase += (inext - i) * W;
        i = inext; c0 = n0; c1 = n1;
        pr = pair && i < qlen && pairable(i, mlen, origin);
    }
    const int bestRowVal = best.rowVal, bestRowI = best.rowI;
    const bool anyRow = best.anyRow;
    // best cell of the last column: first row with the strictly largest score (:564-570); H holds that column now
    int bestColVal = 0, bestColJ = 0;
    bool anyCol = false;
    {
        const int jb = origin + qlen;
        const int first = imax(jb, 1), last = imin(jb + BW, nRows) - 1;
        for (int j = first; j <= last; j++)
        {
            const int v = H.get(j);
            if (!anyCol || v > bestColVal) { bestColVal = v; bestColJ = j; anyCol = true; }
        }
    }
    // start of the traceback (:577-586)
    if (anyCol && (!anyRow || bestColVal > bestRowVal)) { bi = qlen; bj = bestColJ; }
    else { bi = anyRow ? bestRowI : 0; bj = nRows - 1; }
    if (!(anyRow || anyCol) || bi <= 0 || bj <= 0) bi = 0;
}

// Traceback from (bi, bj), bi > 0.  ops.put(n, op) receives the alignment columns last column first.
template <class SS, class FS, class QF, class OS>
PBSC_DPT_HD void traceback(int qlen, int mlen, int origin, const SS& S, const FS& F, const QF& q, int bi, int bj, OS& ops,
                           int& n_out, int& ed_out, int& i_out, int& j_out)
{
    const int W = words_per_col(mlen);
    int i = bi, j = bj, n = 0, ed = 0;
    int ckey = -1;
    uint32_t cword = 0;
#if defined(__CUDA_ARCH__)
    #pragma unroll 1
#endif
    while (i > 0 && j > 0)
    {
        const int k = j - (imax(origin + i, 1) & ~1);
        const int kw = k / CPW;
        const int key = (i - 1) * W + kw;
        if (key != ckey) { cword = F.get(key); ckey = key; }
        const uint32_t f = (cword >> (3 * (CPW - 1 - (k - kw * CPW)))) & 7u;
        const int s2p = S.base(j - 1), s2n = j < mlen ? S.base(j) : -1;
        const int s1p = q(i - 1), s1n = i < qlen ? q(i) : -2;
        const bool eqD = (f & 1u) != 0, eqU = (f & 2u) != 0, eqL = (f & 4u) != 0;
        int op;
        if (s2p == s2n) op = eqU ? OP_I : (eqL ? OP_D : OP_M);        // s2 homopolymer: prefer consuming s2 (:620-640)
        else if (s1p == s1n) op = eqL ? OP_D : (eqU ? OP_I : OP_M);   // s1 homopolymer: prefer consuming s1 (:642-661)
        else op = eqD ? OP_M : (eqL ? OP_D : OP_I);                   // (:663-680)
        if (op == OP_M) { if (s1p != s2p) ed++; i--; j--; }
        else if (op == OP_I) { ed++; j--; }
        else { ed++; i--; }
        ops.put(n, op);
        n++;
    }
    n_out = n; ed_out = ed; i_out = i; j_out = j;
}

}}  // namespace pbsc::dpt

#endif
