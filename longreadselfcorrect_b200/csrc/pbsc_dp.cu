// pbsc_dp.cu — DP / multiple-alignment fallback for seed pairs the FM-index walk could not bridge
// (PacBioSelfCorrectionProcess::correctByMSAlignment, PacBio/PacBioSelfCorrectionProcess.cpp:208-245).
//
// Per failed seed pair (a "job"), with query = beginningkmer + raw read between the seeds + target seed:
//   dp_collect_kernel   SA intervals of the query's first k-mer and of its last k-mer on both strands; up to `coverage`
//                       suffix-array rows are taken from each (LongReadOverlap::retrieveStr, PacBio/LongReadOverlap.cpp:667-756)
//   dp_retrieve_kernel  thread per row: spell the read onwards from the k-mer by LF-mapping, one 32-byte sector per step
//                       (the same block holds the BWT symbol, RLBWT::getChar, and its rank, RLBWT::getOcc)
//   dp_align_kernel     warp per row: Overlapper::extendMatch (Thirdparty/overlapper.cpp:421-701): 201-cell band, +1/-1/-8;
//                       a band column lives in registers (7 cells per lane), the dependency along the column is a max-scan,
//                       only three "equals predecessor" bits per cell go to memory for the traceback, whose homopolymer-aware
//                       tie-breaks are replayed exactly; then the overlap-length / identity filters of
//                       LongReadOverlap::retrieveMatches (PacBio/LongReadOverlap.cpp:593-662)
//   dp_msa_kernel       thread per job: MultipleAlignment::_addSequence + calculateBaseConsensus
//                       (Thirdparty/multiple_alignment.cpp:240-393, 517-594) on per-column symbol counts instead of padded
//                       rows (see "column model" below)
// Jobs are processed in chunks that fit a scratch budget (20 GB, or half of what is free).
#include <cub/cub.cuh>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <vector>
#include <type_traits>
#include "pbsc_batch.cuh"
#include "pbsc_task.cuh"
#include <chrono>
#include "pbsc_dp.cuh"
#include "pbsc_dp_thread.cuh"
#include "pbsc_dp_msa.cuh"

namespace pbsc {

constexpr int DP_HALF = 100;              // bandwidth 200 (LongReadOverlap.cpp:629)
constexpr int DP_BW = 2 * DP_HALF + 1;    // cells per band column
constexpr int DP_CPL = 7;                 // cells per lane: 32 x 7 = 224 >= 201
constexpr int DP_NEG = -(1 << 28);
constexpr int DP_WARPS = 8;               // warps per block of the alignment kernel

struct __align__(16) DpJob
{
    uint64_t lo[4];    // first suffix-array row of: source k-mer fwd (RBWT), rvc (BWT), target k-mer fwd (RBWT), rvc (BWT)
    uint32_t cnt[4];   // rows taken from each: min(interval size, coverage)
    uint32_t task;     // index into the task array
    uint32_t qlen, k, maxLen;
    uint64_t row0;     // first row, numbered over the whole DP stage
    uint64_t mem;      // byte offset of the job's scratch, over the whole DP stage
};

__host__ __device__ inline uint32_t dp_max_len(uint32_t qlen)
{
    // size_t maxLength = query.length()*1.1+20 (LongReadOverlap.cpp:611); product and sum are exact IEEE operations
#ifdef __CUDA_ARCH__
    return (uint32_t)(uint64_t)__dadd_rn(__dmul_rn((double)qlen, 1.1), 20.0);
#else
    volatile double m = (double)qlen * 1.1;
    return (uint32_t)(uint64_t)(m + 20.0);
#endif
}
__host__ __device__ inline uint64_t dp_seq_bytes(uint32_t maxLen) { return align_up((size_t)maxLen, 16); }
__host__ __device__ inline uint64_t dp_row_bytes(uint32_t qlen, uint32_t maxLen) { return dp_seq_bytes(maxLen) + align_up((size_t)qlen + maxLen, 16); }
__host__ __device__ inline uint64_t dp_msa_bytes(uint32_t qlen)
{
    const uint64_t np = (uint64_t)qlen + 1;
    return align_up(np * 5 * 2, 16) + align_up(np * 2, 16) + 2 * align_up(np * 4, 16) + (uint64_t)dp_gap_cap(qlen) * sizeof(GapCol);
}
__host__ __device__ inline uint64_t dp_job_bytes(uint32_t qlen, uint32_t maxLen, uint32_t rows)
{
    return align_up(align_up((size_t)qlen, 16) + (uint64_t)rows * dp_row_bytes(qlen, maxLen) + dp_msa_bytes(qlen), 128);
}

// ---- stage 0: which failed walks get the fallback, and how many rows each one retrieves --------------------------------
__global__ void __launch_bounds__(128)
dp_collect_kernel(const __grid_constant__ FmIndexDev idx, uint64_t n_items, const uint32_t* __restrict__ list, WalkTask* tasks,
                  const uint8_t* __restrict__ codes, const uint64_t* __restrict__ offsets, uint32_t coverage, DpJob* jobs,
                  uint64_t* job_rows, uint64_t* job_bytes, unsigned int* n_jobs)
{
    const uint64_t it = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (it >= n_items) return;
    const uint64_t ti = list ? list[it] : it;
    WalkTask& tk = tasks[ti];
    if (!tk.valid) return;
    if (tk.dp_wanted != 1) return;   // 0: not asked for, 2: already collected by an earlier DP stage of this round
    tk.dp_status = PBSC_DP_NONE;
    if (!(tk.status == -1 || tk.status == -2 || tk.status == -3)) return;
    tk.dp_wanted = 2;
    const uint8_t* read = codes + offsets[tk.read];
    const uint32_t k = (uint32_t)tk.k;
    const uint32_t qlen = k + (uint32_t)(tk.trg_start - tk.src_end - 1) + (uint32_t)tk.trg_len;
    DpJob J;
    Interval f, r;
    tw::both_strands(idx, [&](int j) { return (int)task_query_base(tk, read, (uint32_t)j); }, (int)k, f, r);
    J.lo[0] = f.lo; J.cnt[0] = (uint32_t)min(f.size(), (uint64_t)coverage);
    J.lo[1] = r.lo; J.cnt[1] = (uint32_t)min(r.size(), (uint64_t)coverage);
    // initKmer = reverseComplement(last k bases of the query) (LongReadOverlap.cpp:680)
    tw::both_strands(idx, [&](int j) { return 3 - (int)task_query_base(tk, read, qlen - 1 - (uint32_t)j); }, (int)k, f, r);
    J.lo[2] = f.lo; J.cnt[2] = (uint32_t)min(f.size(), (uint64_t)coverage);
    J.lo[3] = r.lo; J.cnt[3] = (uint32_t)min(r.size(), (uint64_t)coverage);
    const uint32_t rows = J.cnt[0] + J.cnt[1] + J.cnt[2] + J.cnt[3];
    // maquery.getNumRows() <= 3 (PacBioSelfCorrectionProcess.cpp:238): fewer than three rows can never pass
    if (rows < 3) { tk.dp_status = PBSC_DP_FEW_ROWS; return; }
    J.task = (uint32_t)ti; J.qlen = qlen; J.k = k; J.maxLen = dp_max_len(qlen);
    J.row0 = 0; J.mem = 0;
    const unsigned int j = atomicAdd(n_jobs, 1u);
    atomicMax(n_jobs + 3, qlen);   // longest query of this stage (sizes the alignment passes)
    jobs[j] = J;
    job_rows[j] = rows;
    job_bytes[j] = dp_job_bytes(qlen, J.maxLen, rows);
}

__global__ void dp_offsets_kernel(uint64_t n_jobs, DpJob* jobs, const uint64_t* __restrict__ row_off, const uint64_t* __restrict__ mem_off)
{
    const uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j < n_jobs) { jobs[j].row0 = row_off[j]; jobs[j].mem = mem_off[j]; }
}

__device__ __forceinline__ void job_view(uint8_t* mem, const DpJob& J, uint32_t rows, JobView& v)
{
    uint8_t* p = mem;
    v.q = p; p += align_up((size_t)J.qlen, 16);
    v.rows = p;
    v.seqBytes = dp_seq_bytes(J.maxLen);
    v.rowBytes = dp_row_bytes(J.qlen, J.maxLen);
    p += (uint64_t)rows * v.rowBytes;
    const uint64_t np = (uint64_t)J.qlen + 1;
    v.baseCnt = (uint16_t*)p; p += align_up(np * 5 * 2, 16);
    v.startAt = (uint16_t*)p; p += align_up(np * 2, 16);
    v.head = (uint32_t*)p; p += align_up(np * 4, 16);
    v.tail = (uint32_t*)p; p += align_up(np * 4, 16);
    v.pool = (GapCol*)p;
}
__device__ __forceinline__ uint32_t job_rows_of(const DpJob& J) { return J.cnt[0] + J.cnt[1] + J.cnt[2] + J.cnt[3]; }

// ---- stage 1a: thread per job of the chunk: the query, and one descriptor per row -------------------------------------
__global__ void __launch_bounds__(128)
dp_rows_kernel(uint64_t j0, uint64_t j1, const DpJob* __restrict__ jobs, const WalkTask* __restrict__ tasks, const uint8_t* __restrict__ codes,
               const uint64_t* __restrict__ offsets, uint8_t* mem, uint64_t mem0, DpRow* rows, uint64_t row_base)
{
    const uint64_t j = j0 + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= j1) return;
    const DpJob J = jobs[j];
    const WalkTask tk = tasks[J.task];
    const uint8_t* read = codes + offsets[tk.read];
    const uint32_t nr = job_rows_of(J);
    JobView v;
    job_view(mem + (J.mem - mem0), J, nr, v);
    for (uint32_t x = 0; x < J.qlen; x++) v.q[x] = task_query_base(tk, read, x);
    for (uint32_t r = 0; r < nr; r++)
    {
        DpRow R;
        R.job = (uint32_t)j; R.local = r; R.len = 0; R.seq_start = 0; R.nops = 0; R.start0 = R.start1 = 0; R.pass = 0;
        rows[J.row0 - row_base + r] = R;
    }
}

// ---- stage 1b: thread per row: LongReadOverlap::retrieveStr ------------------------------------------------------------
__global__ void __launch_bounds__(128)
dp_retrieve_kernel(const __grid_constant__ FmIndexDev idx, uint64_t n_rows, DpRow* rows, const DpJob* __restrict__ jobs, uint8_t* mem, uint64_t mem0)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    DpRow R = rows[i];
    const DpJob J = jobs[R.job];
    JobView v;
    job_view(mem + (J.mem - mem0), J, job_rows_of(J), v);
    uint8_t* buf = v.rows + (uint64_t)R.local * v.rowBytes;
    // which of the four suffix-array ranges this row comes from, in the order the reference pushes them
    uint32_t l = R.local;
    int kind = 0;
    while (l >= J.cnt[kind]) { l -= J.cnt[kind]; kind++; }
    uint64_t sa = J.lo[kind] + l;
    const FmTable& t = idx.t[(kind == 0 || kind == 2) ? PBSC_RBWT : PBSC_BWT];
    const bool compl_ = (kind == 1 || kind == 2);   // the string is the reverse complement of what LF-mapping spells
    const uint32_t k = J.k, qlen = J.qlen, maxLen = J.maxLen;
    const uint8_t* q = v.q;
    uint32_t len, start;
    if (kind < 2)
    {
        // seeded by the query's first k-mer: query[0,k) followed by the read's continuation
        for (uint32_t x = 0; x < k; x++) buf[x] = q[x];
        uint32_t pos = k;
        #pragma unroll 1
        for (uint32_t n = k; n < maxLen; n++)
        {
            const int c = lf_step(t, sa);
            if (c < 0) break;
            buf[pos++] = (uint8_t)(compl_ ? 3 - c : c);
        }
        len = pos; start = 0;
    }
    else
    {
        // seeded by the query's last k-mer: the read's preceding bases followed by query[qlen-k, qlen)
        for (uint32_t x = 0; x < k; x++) buf[maxLen - k + x] = q[qlen - k + x];
        uint32_t pos = maxLen - k;
        #pragma unroll 1
        for (uint32_t n = k; n < maxLen; n++)
        {
            const int c = lf_step(t, sa);
            if (c < 0) break;
            buf[--pos] = (uint8_t)(compl_ ? 3 - c : c);
        }
        start = pos; len = maxLen - pos;
    }
    // a read that spells the query itself is ignored (LongReadOverlap.cpp:622-624)
    bool same = len >= qlen;
    if (same)
    {
        const uint8_t* s = buf + start + (kind < 2 ? 0 : len - qlen);
        for (uint32_t x = 0; x < qlen && same; x++) same = s[x] == q[x];
    }
    R.len = len; R.seq_start = start; R.pass = same ? 0 : 2;
    rows[i] = R;
}

// ---- stage 2: banded alignment (warp per row), traceback and filters (lane per row) -------------------------------------
// A warp takes 32 consecutive rows.  It fills them one after the other, all lanes on one band column at a time, and keeps
// each row's traceback bits in its own piece of the warp's arena; then every lane walks back through ITS row.  The traceback
// is a serial chain of ~(query + read) steps: done by the whole warp it was a third of the kernel's instructions
// (ncu, profiles/r1_dp_align_v0.txt), done lane-parallel it is 1/32 of that.
struct RowGeom
{
    const uint8_t* s2; const uint8_t* q; uint8_t* ops;
    int qlen, mlen, origin;
};
__device__ __forceinline__ void row_geometry(const DpRow& R, const DpJob& J, uint8_t* mem, uint64_t mem0, RowGeom& g)
{
    JobView v;
    job_view(mem + (J.mem - mem0), J, job_rows_of(J), v);
    uint8_t* buf = v.rows + (uint64_t)R.local * v.rowBytes;
    g.s2 = buf + R.seq_start;
    g.ops = buf + v.seqBytes;
    g.q = v.q;
    g.qlen = (int)J.qlen; g.mlen = (int)R.len;
    const int k = (int)J.k;
    const bool isRC = R.local >= J.cnt[0] + J.cnt[1];
    const int start_1 = isRC ? g.qlen - k : 0, start_2 = isRC ? g.mlen - k : 0;
    g.origin = (start_2 - start_1 + 1) - (DP_HALF + 1);
}

// fill one row's band, column by column, all 32 lanes; returns the traceback start cell (bi, bj), bi == 0 when there is none
__device__ __forceinline__ void dp_fill_row(const RowGeom& g, uint32_t* __restrict__ flags, int& bi, int& bj)
{
    const int lane = threadIdx.x & 31;
    const uint8_t* __restrict__ s2 = g.s2;
    const uint8_t* __restrict__ q = g.q;
    const int qlen = g.qlen, mlen = g.mlen, origin = g.origin;
    const int nRows = mlen + 1;
    const int rbase = lane * DP_CPL;
    int prev[DP_CPL];
    int sw[DP_CPL];   // s2[j-1] of this lane's rows in the current column; -1 outside the string
    int idle[DP_CPL]; // what a cell the fill does not visit reads as: 0 inside the band (the zero-initialised table), never-equal outside
    #pragma unroll
    for (int t = 0; t < DP_CPL; t++)
    {
        idle[t] = (rbase + t < DP_BW) ? 0 : DP_NEG;
        prev[t] = idle[t];
        const int j = origin + 1 + rbase + t;
        sw[t] = (j >= 1 && j <= mlen) ? (int)s2[j - 1] : -1;
    }
    int bestRowVal = 0, bestRowI = 0, bestColVal = 0, bestColJ = 0;
    bool anyRow = false, anyCol = false;
    #pragma unroll 1
    for (int i = 1; i <= qlen; i++)
    {
        const int jb = origin + i;
        const int first = max(jb, 1);
        const int last = min(jb + DP_BW, nRows) - 1;
        const bool skipCol = (last + 1 <= 0) || first >= nRows || first > last;
        // band rows [rlo, rhi] of this column are computed; rowNoLeft is the band row that ignores its left neighbour
        const int rlo = skipCol ? (1 << 20) : first - jb, rhi = skipCol ? (1 << 20) : last - jb;
        const unsigned span = skipCol ? 0u : (unsigned)(rhi - rlo);   // (unsigned)(r - rlo) <= span  <=>  rlo <= r <= rhi
        const int rowNoLeft = (rhi != rlo) ? rhi : -1;
        const int c1 = (int)q[i - 1];
        const int pn0 = __shfl_down_sync(FULL, prev[0], 1);
        int a[DP_CPL], cur[DP_CPL];
        int run = DP_NEG;
        #pragma unroll
        for (int t = 0; t < DP_CPL; t++)
        {
            const int r = rbase + t;
            const bool comp = (unsigned)(r - rlo) <= span;
            const int sub = sw[t] == c1 ? 1 : -8;
            const int pl = (t < DP_CPL - 1) ? prev[t + 1] : pn0;
            // first row of the band: left if it is in the band; last row (when not also the first): no left
            // (band row 200's left neighbour is outside the band: DP_NEG, never the maximum)
            const int left1 = (r != rowNoLeft) ? pl - 1 : DP_NEG;
            const int v0 = __viaddmax_s32(prev[t], sub, left1);          // max(diag, left - 1), one DPX instruction
            run = comp ? __viaddmax_s32(v0, r, run) : run;               // prefix maximum of v0 + r
            a[t] = run;
        }
        int incl = run;
        #pragma unroll
        for (int off = 1; off < 32; off <<= 1)
        {
            const int o = __shfl_up_sync(FULL, incl, off);
            if (lane >= off) incl = max(incl, o);
        }
        int excl = __shfl_up_sync(FULL, incl, 1);
        if (lane == 0) excl = DP_NEG;
        #pragma unroll
        for (int t = 0; t < DP_CPL; t++)
        {
            const int r = rbase + t;
            const bool comp = (unsigned)(r - rlo) <= span;
            cur[t] = comp ? max(a[t], excl) - r : idle[t];
        }
        // traceback bits: does the cell equal each in-band neighbour plus its step (overlapper.cpp:607-610)
        int upPrev = __shfl_up_sync(FULL, cur[DP_CPL - 1], 1);
        if (lane == 0) upPrev = DP_NEG;   // band row 0 has no cell above it in the band: never equal
        uint32_t w = 0;
        #pragma unroll
        for (int t = 0; t < DP_CPL; t++)
        {
            const int r = rbase + t;
            const bool comp = (unsigned)(r - rlo) <= span;
            const int diag = prev[t] + (sw[t] == c1 ? 1 : -8);
            const int pl = (t < DP_CPL - 1) ? prev[t + 1] : pn0;
            const int upv = t > 0 ? cur[t - 1] : upPrev;
            uint32_t f = (cur[t] == diag) ? 1u : 0u;
            f |= (cur[t] == upv - 1) ? 2u : 0u;
            f |= (cur[t] == pl - 1) ? 4u : 0u;
            w |= (comp ? f : 0u) << (3 * t);
        }
        flags[(size_t)i * 32 + lane] = w;
        // best cell of the last row: first column with the strictly largest score (overlapper.cpp:553-561)
        if (!skipCol && last == nRows - 1)
        {
            // the last row is the last computed cell of the column, band row rhi; its score is the end of the column's prefix
            // maximum: c[rhi] = (max over computed r of a[r] + r) - rhi
            const int vv = __shfl_sync(FULL, incl, 31) - rhi;
            if (!anyRow || vv > bestRowVal) { bestRowVal = vv; bestRowI = i; anyRow = true; }
        }
        // best cell of the last column: first row with the strictly largest score (:564-570)
        if (i == qlen && !skipCol)
        {
            int lv = DP_NEG, lr = 0x7fffffff;
            #pragma unroll
            for (int t = 0; t < DP_CPL; t++)
            {
                const int r = rbase + t;
                const bool comp = (unsigned)(r - rlo) <= span;
                if (comp && cur[t] > lv) { lv = cur[t]; lr = r; }
            }
            #pragma unroll
            for (int off = 16; off > 0; off >>= 1)
            {
                const int ov = __shfl_xor_sync(FULL, lv, off), orr = __shfl_xor_sync(FULL, lr, off);
                if (ov > lv || (ov == lv && orr < lr)) { lv = ov; lr = orr; }
            }
            if (lr != 0x7fffffff) { anyCol = true; bestColVal = lv; bestColJ = jb + lr; }
        }
        // next column: the band slides down by one row
        const int nx = __shfl_down_sync(FULL, sw[0], 1);
        #pragma unroll
        for (int t = 0; t < DP_CPL; t++) { prev[t] = cur[t]; if (t < DP_CPL - 1) sw[t] = sw[t + 1]; }
        if (lane == 31)
        {
            const int j = jb + 1 + rbase + (DP_CPL - 1);
            sw[DP_CPL - 1] = (j >= 1 && j <= mlen) ? (int)s2[j - 1] : -1;
        }
        else sw[DP_CPL - 1] = nx;
    }
    // start of the traceback (:577-586)
    if (anyCol && (!anyRow || bestColVal > bestRowVal)) { bi = qlen; bj = bestColJ; }
    else { bi = anyRow ? bestRowI : 0; bj = nRows - 1; }
    if (!(anyRow || anyCol) || bi <= 0 || bj <= 0) bi = 0;
}

#ifndef PBSC_DP_MINB
#define PBSC_DP_MINB 2   // measured on config 2: DP stage 709 ms at 3 resident blocks (80 registers, spills), 681 ms at 2 (109 registers)
#endif
__global__ void __launch_bounds__(DP_WARPS * 32, PBSC_DP_MINB)
dp_align_kernel(uint64_t n_rows, DpRow* rows, const DpJob* __restrict__ jobs, const WalkTask* __restrict__ tasks, uint8_t* mem, uint64_t mem0,
                uint32_t* arenas, uint64_t arena_words, unsigned long long* counter, unsigned int* n_bad)
{
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    uint32_t* arena = arenas + ((size_t)blockIdx.x * DP_WARPS + wib) * arena_words;
    for (;;)
    {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(counter, 32ull);
        base = __shfl_sync(FULL, base, 0);
        if (base >= n_rows) break;
        const int nb = (int)min((unsigned long long)32, n_rows - base);
        int g0 = 0;
        uint64_t used = 0;
        // this lane's row of the current group: where its bits are and where its traceback starts
        uint64_t my_off = 0; int my_bi = 0, my_bj = 0; bool my_todo = false;
        for (int kk = 0; kk <= nb; kk++)
        {
            // fill row kk (if any), after making room by tracing back the rows filled so far when the arena is full
            uint64_t need = 0;
            DpRow R; DpJob J; RowGeom g;
            bool fill = false;
            if (kk < nb)
            {
                R = rows[base + kk];
                if (R.pass == 2)
                {
                    J = jobs[R.job];
                    row_geometry(R, J, mem, mem0, g);
                    need = ((uint64_t)g.qlen + 1) * 32;
                    fill = true;
                }
            }
            if (kk == nb || (fill && used + need > arena_words))
            {
                // lane-parallel traceback of rows [g0, kk)
                __syncwarp();
                if (lane >= g0 && lane < kk && my_todo)
                {
                    DpRow Rm = rows[base + lane];
                    const DpJob Jm = jobs[Rm.job];
                    RowGeom gm;
                    row_geometry(Rm, Jm, mem, mem0, gm);
                    const uint32_t* fl = arena + my_off;
                    const uint8_t* __restrict__ s2 = gm.s2;
                    const uint8_t* __restrict__ q = gm.q;
                    const int qlen = gm.qlen, mlen = gm.mlen, origin = gm.origin;
                    int i = my_bi, j = my_bj, n = 0, ed = 0;
                    if (i <= 0) { atomicAdd(n_bad, 1u); Rm.pass = 0; }   // the reference would abort on its empty-cigar assert
                    else
                    {
                        // one word ahead: the next step is usually one column to the left in the same word
                        int r = j - (origin + i);
                        uint32_t word = fl[(size_t)i * 32 + r / DP_CPL];
                        int wcol = i, widx = r / DP_CPL;
                        #pragma unroll 1
                        while (i > 0 && j > 0)
                        {
                            r = j - (origin + i);
                            const int wi = r / DP_CPL;
                            if (wcol != i || widx != wi) { word = fl[(size_t)i * 32 + wi]; wcol = i; widx = wi; }
                            const uint32_t nextWord = i > 1 ? fl[(size_t)(i - 1) * 32 + wi] : 0u;
                            const uint32_t f = (word >> (3 * (r - wi * DP_CPL))) & 7u;
                            const int s2p = (int)s2[j - 1], s2n = j < mlen ? (int)s2[j] : -1;
                            const int s1p = (int)q[i - 1], s1n = i < qlen ? (int)q[i] : -2;
                            const bool eqD = f & 1u, eqU = (f & 2u) != 0, eqL = (f & 4u) != 0;
                            int op;
                            if (s2p == s2n) op = eqU ? OP_I : (eqL ? OP_D : OP_M);        // s2 homopolymer: prefer consuming s2 (:620-640)
                            else if (s1p == s1n) op = eqL ? OP_D : (eqU ? OP_I : OP_M);   // s1 homopolymer: prefer consuming s1 (:642-661)
                            else op = eqD ? OP_M : (eqL ? OP_D : OP_I);                   // (:663-680)
                            if (op == OP_M) { if (s1p != s2p) ed++; i--; j--; }
                            else if (op == OP_I) { ed++; j--; }
                            else { ed++; i--; }
                            if (op != OP_I) { word = nextWord; wcol = i; }
                            gm.ops[n] = (uint8_t)op;
                            n++;
                        }
                        const WalkTask& tk = tasks[Jm.task];
                        // identity = 0.65 (+0.05 above 50, +0.05 above 100), min_overlap = path.length()/10
                        // (PacBioSelfCorrectionProcess.cpp:225-235)
                        const uint64_t fsum = (uint64_t)(int64_t)tk.freq_sum;
                        double identity = 0.65;
                        identity = __dadd_rn(identity, fsum > 50 ? 0.05 : 0.0);
                        identity = __dadd_rn(identity, fsum > 100 ? 0.05 : 0.0);
                        const double pct = __ddiv_rn(__dmul_rn((double)(n - ed), 100.0), (double)n);   // getPercentIdentity (overlapper.cpp:71-74)
                        const bool passOverlap = (uint64_t)n >= (uint64_t)(qlen / 10);
                        const bool passIdentity = __ddiv_rn(pct, 100.0) >= identity;
                        Rm.nops = (uint32_t)n; Rm.start0 = i; Rm.start1 = j;
                        Rm.pass = (passOverlap && passIdentity) ? 1u : 0u;
                    }
                    rows[base + lane] = Rm;
                    my_todo = false;
                }
                __syncwarp();
                g0 = kk; used = 0;
            }
            if (fill)
            {
                int bi, bj;
                dp_fill_row(g, arena + used, bi, bj);
                if (lane == kk) { my_off = used; my_bi = bi; my_bj = bj; my_todo = true; }
                used += need;
            }
        }
    }
}

// ---- stage 2t: banded alignment, one alignment per thread (pbsc_dp_thread.cuh) -------------------------------------------
// Rows whose every query column meets the matrix are sorted by query length and aligned here, 32 rows of one length per
// warp, in up to three passes of the same kernel: queries of at most 256 bases (80 % of the rows on config 2) with 128
// threads per block, three blocks per SM; longer ones up to 1024 bases with 64 threads per block (the 2-bit read in shared
// memory is longer), four blocks per SM; up to 4000 bases (the 16-bit score limit) with one warp per block.  What is left
// stays `pass == 2` for dp_align_kernel.
template <int QMAX_, int NT_, bool GREAD_>
struct DptCfg
{
    static constexpr int QMAX = QMAX_;                                          // longest query
    static constexpr int NT = NT_;                                              // threads per block
    static constexpr bool GREAD = GREAD_;                                       // the 2-bit read in global memory instead of shared
    static constexpr int HWORDS = dpt::HSLOTS / 2;                              // 16-bit scores, two per word
    static constexpr int SWORDS = (dpt::max_len_bound(QMAX_) + 15) / 16 + 1;    // 2-bit read + one word of slack for bits()
    static constexpr int SMEM = (HWORDS + (GREAD_ ? 0 : SWORDS)) * NT_ * 4;
};
// The previous column (512 B per alignment) has to be in shared memory; the read does not: for the longer queries it is kept in
// global memory, word n of the 32 lanes of a warp side by side (coalesced, L1/L2 resident), which takes the resident warps per
// SM from 8 to 12 (queries up to 1024 bases) and from 4 to 13 (up to 4000).
using DptShort = DptCfg<256, 128, false>;   // 75 776 B per block: three blocks (12 warps) per SM
using DptLong = DptCfg<1024, 64, true>;     // 32 768 B per block: six blocks (12 warps) per SM (51 456 B and 8 warps with the read in shared memory)
using DptHuge = DptCfg<4000, 32, true>;     // 16 384 B per block: 13 blocks (13 warps) per SM; 8 * 4000 still fits 16 bits
constexpr uint32_t DPT_KEY_NONE = 0x3FFFu;
constexpr int DPT_KEY_BITS = 14;

__device__ __forceinline__ int dp_row_origin(const DpRow& R, const DpJob& J)
{
    const int k = (int)J.k, qlen = (int)J.qlen, mlen = (int)R.len;
    const bool isRC = R.local >= J.cnt[0] + J.cnt[1];
    const int start_1 = isRC ? qlen - k : 0, start_2 = isRC ? mlen - k : 0;
    return (start_2 - start_1 + 1) - (DP_HALF + 1);
}

// sort key of a row: longest queries first, forward rows before reverse-complement rows; DPT_KEY_NONE = not for this pass
__global__ void __launch_bounds__(256)
dp_keys_kernel(uint64_t n_rows, const DpRow* __restrict__ rows, const DpJob* __restrict__ jobs, uint32_t* keys, uint32_t* order, int qmax,
               unsigned long long* n_eligible)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const DpRow R = rows[i];
    uint32_t key = DPT_KEY_NONE;
    if (R.pass == 2)
    {
        const DpJob J = jobs[R.job];
        if (dpt::eligible((int)J.qlen, (int)R.len, dp_row_origin(R, J), qmax))
            key = ((uint32_t)(qmax - (int)J.qlen) << 1) | (R.local >= J.cnt[0] + J.cnt[1] ? 1u : 0u);
    }
    keys[i] = key;
    order[i] = (uint32_t)i;
    // how many rows this pass could take; one atomic per warp
    const unsigned m = __ballot_sync(__activemask(), key != DPT_KEY_NONE);
    if (key != DPT_KEY_NONE && (threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(n_eligible, (unsigned long long)__popc(m));
}

template <class C>
struct DptH   // previous column: 16-bit scores, slot j & 255, word (slot >> 1) of this thread's column of shared memory
{
    uint32_t* p;
    __device__ __forceinline__ int get(int j) const
    {
        const int s = j & (dpt::HSLOTS - 1);
        return (int)reinterpret_cast<const short*>(p + (s >> 1) * C::NT)[s & 1];
    }
    __device__ __forceinline__ void set(int j, int v)
    {
        const int s = j & (dpt::HSLOTS - 1);
        reinterpret_cast<short*>(p + (s >> 1) * C::NT)[s & 1] = (short)v;
    }
    // five aligned pairs from the even row j on: one base address, constant offsets
    __device__ __forceinline__ bool pairs_ok(int j) const { return ((j >> 1) & (C::HWORDS - 1)) <= C::HWORDS - 5; }
    __device__ __forceinline__ uint32_t get2(int j, int u) const { return p[((j >> 1) & (C::HWORDS - 1)) * C::NT + u * C::NT]; }
    __device__ __forceinline__ void set2(int j, int u, uint32_t w) { p[((j >> 1) & (C::HWORDS - 1)) * C::NT + u * C::NT] = w; }
};
template <class C>
struct DptS   // the retrieved read at 2 bits per base, 16 bases per word, in this thread's column of shared memory
{
    const uint32_t* p;
    __device__ __forceinline__ int base(int x) const { return (int)((p[(x >> 4) * C::NT] >> (2 * (x & 15))) & 3u); }
    __device__ __forceinline__ uint32_t bits(int x) const
    {
        const uint32_t* w = p + (x >> 4) * C::NT;
        return __funnelshift_r(w[0], w[C::NT], 2 * (x & 15));   // shift < 32; bits 20.. are ignored by the caller
    }
};
struct DptSG   // the same read in global memory: word n of this lane at p[n * 32] (the 32 lanes of a warp side by side)
{
    const uint32_t* p;
    __device__ __forceinline__ int base(int x) const { return (int)((p[(size_t)(x >> 4) * 32] >> (2 * (x & 15))) & 3u); }
    __device__ __forceinline__ uint32_t bits(int x) const
    {
        const uint32_t* w = p + (size_t)(x >> 4) * 32;
        return __funnelshift_r(w[0], w[32], 2 * (x & 15));
    }
};
struct DptF   // flag words of this lane: word n of the lane at arena[n * 32 + lane] (a warp's stores coalesce)
{
    uint32_t* p;
    __device__ __forceinline__ void put(int n, uint32_t w) { p[(size_t)n * 32] = w; }
    __device__ __forceinline__ uint32_t get(int n) const { return p[(size_t)n * 32]; }
};
struct DptQ { const uint8_t* q; __device__ __forceinline__ int operator()(int x) const { return (int)q[x]; } };
struct DptOps { uint8_t* ops; __device__ __forceinline__ void put(int n, int op) { ops[n] = (uint8_t)op; } };

// arena_words: flag words of one warp's 32 rows = 32 * (longest query of this pass) * WMAX
template <class C>
__global__ void __launch_bounds__(C::NT, 227 * 1024 / (C::SMEM + 1024))
dp_align_thread_kernel(uint64_t n_rows, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ order, DpRow* rows,
                       const DpJob* __restrict__ jobs, const WalkTask* __restrict__ tasks, uint8_t* mem, uint64_t mem0, uint32_t* arenas,
                       uint64_t arena_words, unsigned long long* counter, unsigned int* n_bad, const unsigned long long* __restrict__ n_eligible,
                       unsigned long long min_rows, unsigned int* n_thread_rows, uint32_t* rarena, int pair)
{
    extern __shared__ uint32_t dpt_smem[];
    // One alignment per thread pays when there are enough of them to fill the machine: an alignment of L query bases is a
    // serial chain of ~L x 201 cells, a few milliseconds for L in the thousands.  A pass with only a few rows leaves them
    // (`pass == 2`) to the warp-per-row kernel, which works inside one alignment.
    const unsigned long long n_el = *n_eligible;
    if (n_el < min_rows) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(n_thread_rows, (unsigned int)n_el);   // reported in pbsc_timing
    const int lane = threadIdx.x & 31;
    uint32_t* Hs = dpt_smem + threadIdx.x;
    const uint64_t warp = (uint64_t)blockIdx.x * (C::NT / 32) + (threadIdx.x >> 5);
    // the read's words: this thread's column of shared memory, or this lane's column of the warp's slab in global memory
    uint32_t* Ss = C::GREAD ? rarena + warp * (uint64_t)(C::SWORDS * 32) + lane : dpt_smem + C::HWORDS * C::NT + threadIdx.x;
    constexpr int SSTRIDE = C::GREAD ? 32 : C::NT;
    DptF F{arenas + warp * arena_words + lane};
    for (;;)
    {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(counter, 32ull);
        base = __shfl_sync(FULL, base, 0);
        if (base >= n_rows) break;
        const uint64_t t = base + lane;
        const uint32_t key = t < n_rows ? keys[t] : DPT_KEY_NONE;
        if (__shfl_sync(FULL, key, 0) == DPT_KEY_NONE) break;   // sorted: nothing but other rows from here on
        if (key == DPT_KEY_NONE) continue;
        const uint64_t ri = order[t];
        DpRow R = rows[ri];
        const DpJob J = jobs[R.job];
        RowGeom g;
        row_geometry(R, J, mem, mem0, g);
        // the read at 2 bits per base, the column at zero
        for (int x = 0; x < g.mlen; x += 16)
        {
            uint32_t w = 0;
            const int m = min(16, g.mlen - x);
            for (int y = 0; y < m; y++) w |= (uint32_t)g.s2[x + y] << (2 * y);
            Ss[(x >> 4) * SSTRIDE] = w;
        }
        Ss[((g.mlen + 15) >> 4) * SSTRIDE] = 0u;
        #pragma unroll 8
        for (int x = 0; x < C::HWORDS; x++) Hs[x * C::NT] = 0u;
        DptH<C> H{Hs};
        const typename std::conditional<C::GREAD, DptSG, DptS<C>>::type S{Ss};
        const DptQ q{g.q};
        int bi, bj;
        dpt::fill(g.qlen, g.mlen, g.origin, H, S, F, q, bi, bj, pair != 0);
        if (bi <= 0) { atomicAdd(n_bad, 1u); R.pass = 0; }   // the reference would abort on its empty-cigar assert
        else
        {
            DptOps ops{g.ops};
            int n, ed, i0, j0;
            dpt::traceback(g.qlen, g.mlen, g.origin, S, F, q, bi, bj, ops, n, ed, i0, j0);
            const WalkTask& tk = tasks[J.task];
            // identity = 0.65 (+0.05 above 50, +0.05 above 100), min_overlap = path.length()/10
            // (PacBioSelfCorrectionProcess.cpp:225-235)
            const uint64_t fsum = (uint64_t)(int64_t)tk.freq_sum;
            double identity = 0.65;
            identity = __dadd_rn(identity, fsum > 50 ? 0.05 : 0.0);
            identity = __dadd_rn(identity, fsum > 100 ? 0.05 : 0.0);
            const double pct = __ddiv_rn(__dmul_rn((double)(n - ed), 100.0), (double)n);   // getPercentIdentity (overlapper.cpp:71-74)
            const bool passOverlap = (uint64_t)n >= (uint64_t)(g.qlen / 10);
            const bool passIdentity = __ddiv_rn(pct, 100.0) >= identity;
            R.nops = (uint32_t)n; R.start0 = i0; R.start1 = j0;
            R.pass = (passOverlap && passIdentity) ? 1u : 0u;
        }
        rows[ri] = R;
    }
}

// ---- stage 3: thread per job: multiple alignment on per-column counts, consensus ---------------------------------------
// (the column model and the per-job code are in pbsc_dp_msa.cuh, shared with the host check tests/cpp/test_dp_msa.cpp)
// what msa::consensus asks the task for, when it needs it (pbsc_dp_msa.cuh)
struct MsaCtx
{
    WalkTask& tk; uint8_t* outpool;
    __device__ __forceinline__ int min_call() const
    {
        // min_call_coverage = totalFreq > 50 ? totalFreq * 0.4 : 15 (PacBioSelfCorrectionProcess.cpp:236-240)
        const uint64_t fsum = (uint64_t)(int64_t)tk.freq_sum;
        return (int)(fsum > 50 ? (uint64_t)__dmul_rn((double)fsum, 0.4) : 15);
    }
    __device__ __forceinline__ uint8_t* out() const { return outpool + tk.out_off; }
    __device__ __forceinline__ uint32_t cap() const { return tk.out_cap; }
};

// EXPERIMENT (PBSC_DP_SORT_JOBS, off by default): jobs of a chunk in order of decreasing work (alignment columns of the rows
// that passed the filters), optionally dealt out across warps (warp w, lane l takes rank l * n_warps + w) so that every warp
// holds one job of each weight class.  Measured on config 2: natural order 78 ms, dealt out 134 ms, plainly sorted 189 ms —
// the thread-per-job kernel is bound by the locality of its scattered scratch accesses, not by its longest job.
__global__ void __launch_bounds__(128)
dp_job_keys_kernel(uint64_t j0, uint64_t j1, const DpJob* __restrict__ jobs, const DpRow* __restrict__ rows, uint64_t row_base, uint32_t* keys,
                   uint32_t* order)
{
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j0 + t >= j1) return;
    const DpJob J = jobs[j0 + t];
    const uint32_t nr = job_rows_of(J);
    const DpRow* R = rows + (J.row0 - row_base);
    uint32_t passing = 0, cost = 0;
    for (uint32_t r = 0; r < nr; r++)
    {
        const DpRow x = R[r];
        if (x.pass == 1) { passing++; cost += x.nops; }
    }
    if (passing < 3) cost = 0;
    keys[t] = 0xFFFFu - min(0xFFFFu, cost >> 3);
    order[t] = (uint32_t)t;
}

__global__ void __launch_bounds__(64)
dp_msa_kernel(uint64_t j0, uint64_t j1, const uint32_t* __restrict__ order, int deal, const DpJob* __restrict__ jobs, WalkTask* tasks,
              const DpRow* __restrict__ rows, uint64_t row_base, uint8_t* mem, uint64_t mem0, uint8_t* outpool, unsigned int* n_bad,
              uint32_t big_thr, uint32_t* big_list, unsigned int* n_big)
{
    const uint64_t tx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t njc = j1 - j0;
    uint64_t rank = tx;
    if (order && deal)
    {
        const uint64_t n_warps = (njc + 31) / 32;
        rank = (tx & 31) * n_warps + (tx >> 5);
        if (tx >= n_warps * 32) return;
    }
    if (rank >= njc) return;
    const uint64_t jx = j0 + (order ? order[rank] : rank);
    const DpJob J = jobs[jx];
    WalkTask& tk = tasks[J.task];
    const uint32_t nr = job_rows_of(J);
    const DpRow* R = rows + (J.row0 - row_base);
    if (big_list)
    {
        // a pile-up of more than big_thr alignment columns goes to the warp-per-job kernel: this launch would wait for it
        uint32_t cost = 0, passing = 0;
        for (uint32_t r = 0; r < nr; r++) { const DpRow x = R[r]; if (x.pass == 1) { passing++; cost += x.nops; } }
        if (passing >= 3 && cost >= big_thr) { big_list[atomicAdd(n_big, 1u)] = (uint32_t)(jx - j0); return; }
    }
    JobView v;
    job_view(mem + (J.mem - mem0), J, nr, v);
    const MsaCtx ctx{tk, outpool};
    uint32_t n = 0;
    const int rc = msa::consensus(v, J.qlen, J.k, R, nr, ctx, n);
    if (rc == 1) { tk.dp_status = PBSC_DP_FEW_ROWS; return; }
    if (rc == 2) { atomicAdd(n_bad, 1u); tk.dp_status = PBSC_OVF_DP; return; }
    tk.out_len = n;
    tk.dp_status = PBSC_DP_OK;
}

// the large pile-ups dp_msa_kernel set aside: one warp per job, the alignment columns of every row cut into 32 segments
// (msa::consensus_warp, pbsc_dp_msa.cuh); warps take jobs from a queue
constexpr int MSA_WARPS = 4;
__global__ void __launch_bounds__(MSA_WARPS * 32)
dp_msa_warp_kernel(uint64_t j0, const uint32_t* __restrict__ big_list, const unsigned int* __restrict__ n_big, unsigned long long* counter,
                   const DpJob* __restrict__ jobs, WalkTask* tasks, const DpRow* __restrict__ rows, uint64_t row_base, uint8_t* mem, uint64_t mem0,
                   uint8_t* outpool, unsigned int* n_bad)
{
    __shared__ unsigned int gap_counter[MSA_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long n = *n_big;
    for (;;)
    {
        unsigned long long it = 0;
        if (lane == 0) it = atomicAdd(counter, 1ull);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it >= n) break;
        const uint64_t jx = j0 + big_list[it];
        const DpJob J = jobs[jx];
        WalkTask& tk = tasks[J.task];
        const uint32_t nr = job_rows_of(J);
        const DpRow* R = rows + (J.row0 - row_base);
        JobView v;
        job_view(mem + (J.mem - mem0), J, nr, v);
        const MsaCtx ctx{tk, outpool};
        uint32_t nout = 0;
        const int rc = msa::consensus_warp(v, J.qlen, J.k, R, nr, ctx, nout, &gap_counter[warp]);
        __syncwarp();
        if (lane == 0)
        {
            if (rc == 1) tk.dp_status = PBSC_DP_FEW_ROWS;
            else if (rc == 2) { atomicAdd(n_bad, 1u); tk.dp_status = PBSC_OVF_DP; }
            else { tk.out_len = nout; tk.dp_status = PBSC_DP_OK; }
        }
        __syncwarp();
    }
}

template <class T>
static cudaError_t arena(pbsc_index* idx, const char* name, size_t count, T** out) { return arena_get(idx, name, (count ? count : 1) * sizeof(T), (void**)out); }

DpStats& last_dp_stats() { static thread_local DpStats s; return s; }

// one pass of dp_align_thread_kernel<C>: queries of at most min(C::QMAX, longest query of the stage) bases
struct DptPass
{
    bool on = false; uint64_t qmax = 0, arena_words = 0, min_rows = 0, read_words = 0; int blocks = 0;
    int pair = 1;   // dpt::fill sweeps two columns at once where it can (PBSC_DPT_PAIR=0: one at a time)
    uint64_t flag_words() const { return on ? arena_words * (uint64_t)blocks : 0; }
};
template <class C>
static cudaError_t dpt_pass_setup(pbsc_index* idx, uint64_t q_longest, uint64_t q_prev_max, int cap_per_sm, DptPass& g)
{
    g.on = q_longest > q_prev_max;   // something is left for this pass
    if (!g.on) return cudaSuccess;
    g.qmax = std::min<uint64_t>((uint64_t)C::QMAX, q_longest);
    g.arena_words = 32ull * g.qmax * dpt::WMAX;
    cudaError_t e = cudaFuncSetAttribute(dp_align_thread_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM);
    if (e != cudaSuccess) return e;
    int per = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, dp_align_thread_kernel<C>, C::NT, C::SMEM);
    if (e != cudaSuccess) return e;
    if (cap_per_sm > 0) per = std::min(per, cap_per_sm);
    g.blocks = idx->sm_count * std::max(per, 1);
    g.arena_words *= (uint64_t)(C::NT / 32);   // per block
    g.read_words = C::GREAD ? (uint64_t)g.blocks * (C::NT / 32) * (uint64_t)(C::SWORDS * 32) : 0;
    return cudaSuccess;
}
template <class C>
static void dpt_pass_launch(const DptPass& g, cudaStream_t st, uint64_t nrows, DpRow* rows, const DpJob* jobs, const WalkTask* tasks, uint8_t* mem,
                            uint64_t mem0, uint32_t* keys, uint32_t* keys2, uint32_t* order, uint32_t* order2, uint8_t* sort_tmp, size_t sort_bytes,
                            uint32_t* slabs, unsigned long long* counter, unsigned int* cnt, uint32_t* rarena)
{
    cudaMemsetAsync(counter, 0, 16, st);   // counter[0]: work queue, counter[1]: rows eligible for this pass
    dp_keys_kernel<<<(unsigned)((nrows + 255) / 256), 256, 0, st>>>(nrows, rows, jobs, keys, order, (int)g.qmax, counter + 1);
    cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, keys, keys2, order, order2, (int)nrows, 0, DPT_KEY_BITS, st);
    const int tb = (int)std::min<uint64_t>((uint64_t)g.blocks, (nrows + C::NT - 1) / C::NT);
    dp_align_thread_kernel<C><<<tb, C::NT, C::SMEM, st>>>(nrows, keys2, order2, rows, jobs, tasks, mem, mem0, slabs, g.arena_words / (C::NT / 32), counter,
                                                          cnt + 1, counter + 1, g.min_rows, cnt + 2, rarena, g.pair);
}

int run_dp_fallback(pbsc_index* idx, const pbsc_params* p, DeviceBatch& b, void* tasks_v, uint64_t n_items, const uint32_t* list, uint8_t* outpool,
                    uint32_t q_cap, uint64_t* launches)
{
    WalkTask* tasks = (WalkTask*)tasks_v;
    cudaStream_t st = idx->stream;
    if (n_items == 0) return PBSC_OK;
    // PBSC_ROUND_TRACE=1: host wall clock between the steps of this stage (diagnostics)
    const bool htrace = getenv("PBSC_ROUND_TRACE") != nullptr;
    auto h0 = std::chrono::steady_clock::now();
    auto hmark = [&](const char* what) {
        if (!htrace) return;
        const auto now = std::chrono::steady_clock::now();
        const double ms = std::chrono::duration<double, std::milli>(now - h0).count();
        if (ms > 2.0) fprintf(stderr, "[pbsc round trace]     dp host: %-22s %8.2f ms\n", what, ms);
        h0 = now;
    };
    DpJob* jobs; uint64_t *job_rows, *job_bytes, *row_off, *mem_off; unsigned int* cnt; unsigned long long* qctr;
    PBSC_CUDA(arena(idx, "dp.jobs", n_items, &jobs));
    PBSC_CUDA(arena(idx, "dp.job_rows", n_items + 1, &job_rows));
    PBSC_CUDA(arena(idx, "dp.job_bytes", n_items + 1, &job_bytes));
    PBSC_CUDA(arena(idx, "dp.row_off", n_items + 1, &row_off));
    PBSC_CUDA(arena(idx, "dp.mem_off", n_items + 1, &mem_off));
    PBSC_CUDA(arena(idx, "dp.cnt", 4, &cnt));
    PBSC_CUDA(arena(idx, "dp.qctr", 4, &qctr));
    PBSC_CUDA(cudaMemsetAsync(cnt, 0, 16, st));
    cudaEvent_t ev[2];
    PBSC_CUDA(cudaEventCreate(&ev[0])); PBSC_CUDA(cudaEventCreate(&ev[1]));
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } guard{ev};
    PBSC_CUDA(cudaEventRecord(ev[0], st));
    dp_collect_kernel<<<(unsigned)((n_items + 127) / 128), 128, 0, st>>>(idx->dev, n_items, list, tasks, b.codes.p, b.offsets.p, (uint32_t)p->pb_coverage,
                                                                        jobs, job_rows, job_bytes, cnt);
    unsigned int hcnt[4] = {0, 0, 0, 0};
    PBSC_CUDA(cudaMemcpyAsync(hcnt, cnt, 16, cudaMemcpyDeviceToHost, st));
    PBSC_CUDA(cudaStreamSynchronize(st));
    if (launches) *launches += 1;
    const uint64_t nj = hcnt[0];
    DpStats& S = last_dp_stats();
    hmark("collect + sync");
    if (nj == 0) return PBSC_OK;
    // offsets of every job's rows and scratch
    {
        size_t tb = 0, tb2 = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tb, job_rows, row_off, (int)(nj + 1), st);
        cub::DeviceScan::ExclusiveSum(nullptr, tb2, job_bytes, mem_off, (int)(nj + 1), st);
        tb = std::max(tb, tb2);
        uint8_t* tmp;
        PBSC_CUDA(arena(idx, "dp.cubtmp", tb, &tmp));
        PBSC_CUDA(cudaMemsetAsync(job_rows + nj, 0, 8, st));
        PBSC_CUDA(cudaMemsetAsync(job_bytes + nj, 0, 8, st));
        cub::DeviceScan::ExclusiveSum(tmp, tb, job_rows, row_off, (int)(nj + 1), st);
        cub::DeviceScan::ExclusiveSum(tmp, tb, job_bytes, mem_off, (int)(nj + 1), st);
        dp_offsets_kernel<<<(unsigned)((nj + 255) / 256), 256, 0, st>>>(nj, jobs, row_off, mem_off);
    }
    std::vector<uint64_t> h_row(nj + 1), h_mem(nj + 1);
    PBSC_CUDA(cudaMemcpyAsync(h_row.data(), row_off, (nj + 1) * 8, cudaMemcpyDeviceToHost, st));
    PBSC_CUDA(cudaMemcpyAsync(h_mem.data(), mem_off, (nj + 1) * 8, cudaMemcpyDeviceToHost, st));
    PBSC_CUDA(cudaStreamSynchronize(st));
    if (launches) *launches += 3;
    hmark("scans + sync");
    S.jobs += nj; S.rows += h_row[nj];
    // scratch budget of one chunk
    // Large chunks matter: the multiple-alignment kernel is one thread per job and a launch lasts as long as its longest job,
    // so few, full launches beat many small ones (repeat-rich 100x workload: DP stage 2.9 s with 6 GB chunks, 2.4 s with 20 GB).
    uint64_t budget = 20ull << 30;
    {
        // what is free now plus what the grow-only arena already holds for this purpose; cudaMemGetInfo costs 5-60 ms with tens
        // of gigabytes allocated (PBSC_ROUND_TRACE), so it is asked only when this stage needs more than the arena has
        const auto it = idx->arena.find("dp.mem");
        const uint64_t have = it != idx->arena.end() ? (uint64_t)it->second.cap : 0;
        if (h_mem[nj] > have)
        {
            size_t free_b = 0, total_b = 0;
            if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) budget = std::min<uint64_t>(budget, std::max<uint64_t>(2ull << 30, (free_b + have) / 2));
        }
        else budget = std::max<uint64_t>(have, 1);
    }
    if (const char* e = getenv("PBSC_DP_CHUNK_MB")) { if (atoll(e) > 0) budget = (uint64_t)atoll(e) << 20; }
    uint64_t max_job = 0;
    for (uint64_t j = 0; j < nj; j++) max_job = std::max(max_job, h_mem[j + 1] - h_mem[j]);
    if (max_job > budget) budget = max_job;
    const uint64_t pool_bytes = std::min(budget, h_mem[nj]);
    uint8_t* mem;
    hmark("budget");
    PBSC_CUDA(arena(idx, "dp.mem", pool_bytes, &mem));
    hmark("arena dp.mem");
    // alignment kernel geometry: one flag slab per resident warp, sized for the longest query of this stage
    int per_sm = 0;
    PBSC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dp_align_kernel, DP_WARPS * 32, 0));
    if (per_sm < 1) per_sm = 1;
    if (const char* e = getenv("PBSC_DP_BLOCKS_PER_SM")) { if (atoi(e) > 0) per_sm = std::min(per_sm, atoi(e)); }
    const int ablocks = idx->sm_count * per_sm;
    // per-warp arena of traceback bits: 32 rows of a typical query, and at least one row of the longest
    uint64_t arena_words = std::max<uint64_t>(((uint64_t)q_cap + 2) * 32, 1ull << 18);
    if (const char* e = getenv("PBSC_DP_ARENA_KB")) { if (atoll(e) > 0) arena_words = std::max<uint64_t>(((uint64_t)q_cap + 2) * 32, (uint64_t)atoll(e) * 256); }
    uint32_t* slabs;
    PBSC_CUDA(arena(idx, "dp.flags", arena_words * (uint64_t)ablocks * DP_WARPS, &slabs));
    uint64_t max_rows = 0;
    for (uint64_t j0 = 0; j0 < nj;)
    {
        uint64_t j1 = j0 + 1;
        while (j1 < nj && h_mem[j1 + 1] - h_mem[j0] <= pool_bytes) j1++;
        max_rows = std::max(max_rows, h_row[j1] - h_row[j0]);
        j0 = j1;
    }
    DpRow* rows;
    hmark("flags arena + chunking");
    PBSC_CUDA(arena(idx, "dp.rows", max_rows, &rows));
    // thread-per-alignment kernel (stage 2t): sort keys, the sorted order, one flag arena per resident warp
    bool use_thread = true;
    if (const char* e = getenv("PBSC_DP_THREAD")) use_thread = atoi(e) != 0;
    uint32_t *tkeys = nullptr, *tkeys2 = nullptr, *torder = nullptr, *torder2 = nullptr, *tslabs = nullptr, *treads = nullptr;
    uint8_t* sort_tmp = nullptr;
    size_t sort_bytes = 0;
    // the longest query of this stage decides which passes run and how large their flag arenas are
    const uint64_t q_longest = std::min<uint64_t>(q_cap, hcnt[3]);
    DptPass pass_s, pass_l, pass_h;
    if (use_thread)
    {
        int cap = 0;
        if (const char* e = getenv("PBSC_DPT_BLOCKS_PER_SM")) cap = atoi(e);
        const bool longer = !(getenv("PBSC_DPT_LONG") && atoi(getenv("PBSC_DPT_LONG")) == 0);
        PBSC_CUDA(dpt_pass_setup<DptShort>(idx, q_longest, 0, cap, pass_s));
        if (longer) PBSC_CUDA(dpt_pass_setup<DptLong>(idx, q_longest, DptShort::QMAX, 0, pass_l));
        if (longer) PBSC_CUDA(dpt_pass_setup<DptHuge>(idx, q_longest, DptLong::QMAX, 0, pass_h));
        // fewest rows worth a pass (PBSC_DPT_MIN_ROWS overrides all three; the tests run with 1 to force every pass)
        // (config 2, first DP stage of a step: the few thousand rows of the 4000-base pass take 22 ms here and 35 ms in the
        // warp-per-row kernel, which also serialises: a warp there fills 32 rows one after the other)
        pass_s.min_rows = 512; pass_l.min_rows = 2048; pass_h.min_rows = 2048;
        if (const char* e = getenv("PBSC_DPT_MIN_ROWS")) pass_s.min_rows = pass_l.min_rows = pass_h.min_rows = (uint64_t)std::max(0ll, atoll(e));
        // PBSC_DPT_PAIR=0: the scalar fill, one column per sweep (for comparing the two; both give the same flags and scores)
        if (const char* e = getenv("PBSC_DPT_PAIR")) pass_s.pair = pass_l.pair = pass_h.pair = atoi(e) != 0 ? 1 : 0;
        PBSC_CUDA(arena(idx, "dp.tkeys", max_rows, &tkeys));
        PBSC_CUDA(arena(idx, "dp.tkeys2", max_rows, &tkeys2));
        PBSC_CUDA(arena(idx, "dp.torder", max_rows, &torder));
        PBSC_CUDA(arena(idx, "dp.torder2", max_rows, &torder2));
        cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, tkeys, tkeys2, torder, torder2, (int)max_rows, 0, DPT_KEY_BITS, st);
        PBSC_CUDA(arena(idx, "dp.sorttmp", sort_bytes, &sort_tmp));
        PBSC_CUDA(arena(idx, "dp.tflags", std::max(pass_s.flag_words(), std::max(pass_l.flag_words(), pass_h.flag_words())), &tslabs));
        PBSC_CUDA(arena(idx, "dp.treads", std::max<uint64_t>(1, std::max(pass_l.on ? pass_l.read_words : 0, pass_h.on ? pass_h.read_words : 0)), &treads));
    }
    // job order of the multiple-alignment kernel
    // 0: natural order (default: neighbouring threads work on neighbouring scratch, which is what this memory-bound kernel
    // wants: 78 ms on config 2), 1: sorted by work and dealt out across warps (134 ms), 2: sorted (189 ms)
    int sort_jobs = 0;
    if (const char* e = getenv("PBSC_DP_SORT_JOBS")) sort_jobs = atoi(e);
    uint32_t *jkeys = nullptr, *jkeys2 = nullptr, *jord = nullptr, *jord2 = nullptr;
    uint8_t* jsort_tmp = nullptr;
    size_t jsort_bytes = 0;
    if (sort_jobs)
    {
        PBSC_CUDA(arena(idx, "dp.jkeys", nj, &jkeys));
        PBSC_CUDA(arena(idx, "dp.jkeys2", nj, &jkeys2));
        PBSC_CUDA(arena(idx, "dp.jord", nj, &jord));
        PBSC_CUDA(arena(idx, "dp.jord2", nj, &jord2));
        cub::DeviceRadixSort::SortPairs(nullptr, jsort_bytes, jkeys, jkeys2, jord, jord2, (int)nj, 0, 16, st);
        PBSC_CUDA(arena(idx, "dp.jsorttmp", jsort_bytes, &jsort_tmp));
    }
    // pile-ups of at least this many alignment columns are left to the warp-per-job kernel (PBSC_MSA_WARP_MIN: 0 = every job,
    // -1 = none)
    uint32_t msa_big_thr = 8192;
    if (const char* e = getenv("PBSC_MSA_WARP_MIN")) msa_big_thr = atoll(e) < 0 ? 0xffffffffu : (uint32_t)atoll(e);
    uint32_t* msa_big = nullptr;
    unsigned long long* msa_q = nullptr;
    PBSC_CUDA(arena(idx, "dp.msa_big", nj, &msa_big));
    PBSC_CUDA(arena(idx, "dp.msa_q", 2, &msa_q));
    // PBSC_DP_PROFILE=1: per-kernel CUDA-event times of this stage on stderr (diagnostics, off by default)
    struct Prof
    {
        bool on = false; cudaStream_t st; std::vector<std::pair<const char*, cudaEvent_t>> ev;
        void mark(const char* name) { if (!on) return; cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); ev.emplace_back(name, e); }
        void report()
        {
            if (!on || ev.size() < 2) return;
            cudaEventSynchronize(ev.back().second);
            std::vector<std::pair<const char*, float>> acc;
            for (size_t x = 1; x < ev.size(); x++)
            {
                float ms = 0; cudaEventElapsedTime(&ms, ev[x - 1].second, ev[x].second);
                bool found = false;
                for (auto& a : acc) if (!strcmp(a.first, ev[x].first)) { a.second += ms; found = true; }
                if (!found) acc.emplace_back(ev[x].first, ms);
            }
            fprintf(stderr, "[pbsc dp profile]");
            for (auto& a : acc) fprintf(stderr, " %s %.1f ms;", a.first, a.second);
            fprintf(stderr, "\n");
            for (auto& e : ev) cudaEventDestroy(e.second);
        }
    } prof;
    prof.st = st;
    if (const char* e = getenv("PBSC_DP_PROFILE")) prof.on = atoi(e) != 0;
    hmark("pass setup + arenas");
    prof.mark("start");
    for (uint64_t j0 = 0; j0 < nj;)
    {
        uint64_t j1 = j0 + 1;
        while (j1 < nj && h_mem[j1 + 1] - h_mem[j0] <= pool_bytes) j1++;
        const uint64_t nrows = h_row[j1] - h_row[j0], njc = j1 - j0;
        dp_rows_kernel<<<(unsigned)((njc + 127) / 128), 128, 0, st>>>(j0, j1, jobs, tasks, b.codes.p, b.offsets.p, mem, h_mem[j0], rows, h_row[j0]);
        dp_retrieve_kernel<<<(unsigned)((nrows + 127) / 128), 128, 0, st>>>(idx->dev, nrows, rows, jobs, mem, h_mem[j0]);
        prof.mark("rows+retrieve");
        PBSC_CUDA(cudaMemsetAsync(qctr, 0, 32, st));
        if (pass_s.on)
        {
            dpt_pass_launch<DptShort>(pass_s, st, nrows, rows, jobs, tasks, mem, h_mem[j0], tkeys, tkeys2, torder, torder2, sort_tmp, sort_bytes, tslabs,
                                      qctr + 1, cnt, treads);
            prof.mark("align_thread_256");
            if (launches) *launches += 4;   // keys, the sort's kernels counted as two, alignment
        }
        if (pass_l.on)
        {
            // the rows the first pass left: longer queries
            dpt_pass_launch<DptLong>(pass_l, st, nrows, rows, jobs, tasks, mem, h_mem[j0], tkeys, tkeys2, torder, torder2, sort_tmp, sort_bytes, tslabs,
                                     qctr + 1, cnt, treads);
            prof.mark("align_thread_1024");
            if (launches) *launches += 4;
        }
        if (pass_h.on)
        {
            dpt_pass_launch<DptHuge>(pass_h, st, nrows, rows, jobs, tasks, mem, h_mem[j0], tkeys, tkeys2, torder, torder2, sort_tmp, sort_bytes, tslabs,
                                     qctr + 1, cnt, treads);
            prof.mark("align_thread_4000");
            if (launches) *launches += 4;
        }
        const int nb = (int)std::min<uint64_t>((uint64_t)ablocks, (nrows + DP_WARPS * 32 - 1) / (DP_WARPS * 32));
        dp_align_kernel<<<nb, DP_WARPS * 32, 0, st>>>(nrows, rows, jobs, tasks, mem, h_mem[j0], slabs, arena_words, qctr, cnt + 1);
        prof.mark("align_warp");
        const uint32_t* jorder = nullptr;
        if (sort_jobs)
        {
            dp_job_keys_kernel<<<(unsigned)((njc + 127) / 128), 128, 0, st>>>(j0, j1, jobs, rows, h_row[j0], jkeys, jord);
            size_t sb = jsort_bytes;
            cub::DeviceRadixSort::SortPairs(jsort_tmp, sb, jkeys, jkeys2, jord, jord2, (int)njc, 0, 16, st);
            jorder = jord2;
            if (launches) *launches += 3;
        }
        PBSC_CUDA(cudaMemsetAsync(msa_q, 0, 16, st));
        dp_msa_kernel<<<(unsigned)((((njc + 31) / 32) * 32 + 63) / 64), 64, 0, st>>>(j0, j1, jorder, sort_jobs == 1, jobs, tasks, rows, h_row[j0], mem,
                                                                                         h_mem[j0], outpool, cnt + 1, msa_big_thr,
                                                                                         msa_big_thr != 0xffffffffu ? msa_big : nullptr, (unsigned int*)(msa_q + 1));
        prof.mark("msa");
        if (msa_big_thr != 0xffffffffu)
        {
            const int wb = (int)std::min<uint64_t>((uint64_t)idx->sm_count * 4, (njc + MSA_WARPS - 1) / MSA_WARPS);
            dp_msa_warp_kernel<<<wb, MSA_WARPS * 32, 0, st>>>(j0, msa_big, (const unsigned int*)(msa_q + 1), msa_q, jobs, tasks, rows, h_row[j0], mem, h_mem[j0],
                                                              outpool, cnt + 1);
            prof.mark("msa_warp");
            if (launches) *launches += 1;
        }
        PBSC_CUDA(cudaGetLastError());
        if (launches) *launches += 4;
        S.chunks++;
        j0 = j1;
    }
    PBSC_CUDA(cudaEventRecord(ev[1], st));
    hmark("chunk loop (launches)");
    prof.report();
    PBSC_CUDA(cudaMemcpyAsync(hcnt, cnt, 12, cudaMemcpyDeviceToHost, st));
    PBSC_CUDA(cudaStreamSynchronize(st));
    S.bad += hcnt[1];
    S.thread_rows += hcnt[2];
    PBSC_OCC_TAKE(3, st);
    float ms = 0;
    cudaEventElapsedTime(&ms, ev[0], ev[1]);
    S.ms += ms;
    return PBSC_OK;
}

}  // namespace pbsc
