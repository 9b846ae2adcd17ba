// Host check of the masked blocks of the paired-column fill (fill_pair in longreadselfcorrect_b200/csrc/pbsc_dp_thread.cuh): a
// paired sweep runs as ten-step blocks from row fA & ~1 until column i + 1's last row, the first block and the last one or two
// with the first-cell, last-cell and outside-the-column rules applied per half.  dpt::fill with pairing on is compared with
// the same fill one column at a time (every flag word and which words were written, the traceback start, the final column)
// over placements aimed at those blocks: first row odd and even, first or last row at band row 200, columns of 1 to 28 rows
// from the first block's row, last rows of the two columns equal or one apart, first and last blocks across the wrap of the
// 256-slot circular array.  The accessor of the previous column also checks, through the fill's pair_sweep hook, that a
// paired sweep changes no slot of a row outside [fB, lB] (the rows of column i + 1) and stores at most one score on its own
// (the one the last block leaves) besides its pair stores.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>
#include "../../longreadselfcorrect_b200/csrc/pbsc_dp_thread.cuh"

using namespace pbsc::dpt;

static long n_sweeps = 0, n_bad_stores = 0, n_many_sets = 0, max_sets = 0;

struct HHost
{
    int16_t a[HSLOTS];
    bool sweep = false;
    int fB = 1, lB = 0, sets = 0;
    HHost() { for (int i = 0; i < HSLOTS; i++) a[i] = 0; }
    int get(int j) const { return a[j & (HSLOTS - 1)]; }
    bool pairs_ok(int j) const { return ((j >> 1) & (HSLOTS / 2 - 1)) <= HSLOTS / 2 - 5; }
    uint32_t get2(int j, int u) const
    {
        const int s = (j & (HSLOTS - 1)) + 2 * u;
        if ((j & 1) || s + 1 >= HSLOTS) { printf("bad pair access\n"); exit(2); }
        return (uint32_t)(uint16_t)a[s] | ((uint32_t)(uint16_t)a[s + 1] << 16);
    }
    // during a paired sweep, a store may change only the slots of rows fB .. lB
    void store(int row, int16_t v)
    {
        int16_t& slot = a[row & (HSLOTS - 1)];
        if (sweep && (row < fB || row > lB) && slot != v)
        {
            if (++n_bad_stores <= 10) printf("paired sweep over rows %d..%d changes the slot of row %d\n", fB, lB, row);
        }
        slot = v;
    }
    void set2(int j, int u, uint32_t w)
    {
        const int s = (j & (HSLOTS - 1)) + 2 * u;
        if ((j & 1) || s + 1 >= HSLOTS) { printf("bad pair access\n"); exit(2); }
        store(j + 2 * u, (int16_t)(w & 0xFFFFu)); store(j + 2 * u + 1, (int16_t)(w >> 16));
    }
    void set(int j, int v)
    {
        if (v < -32768 || v > 32767) { printf("16-bit overflow\n"); exit(2); }
        if (sweep) sets++;
        store(j, (int16_t)v);
    }
};
// the fill's hook: (fB, lB) before a paired sweep, (1, 0) after it
void pair_sweep(HHost& H, int fB, int lB)
{
    if (fB <= lB) { H.sweep = true; H.fB = fB; H.lB = lB; H.sets = 0; return; }
    n_sweeps++;
    if (H.sets > max_sets) max_sets = H.sets;
    if (H.sets > 1) n_many_sets++;
    H.sweep = false;
}
struct SHost   // aborts on an access that starts outside the read: the device's read slot ends one word after it
{
    std::vector<uint32_t> w; int n;
    explicit SHost(const std::vector<uint8_t>& s) : w(s.size() / 16 + 2, 0u), n((int)s.size()) { for (size_t x = 0; x < s.size(); x++) w[x >> 4] |= (uint32_t)s[x] << (2 * (x & 15)); }
    void check(int x) const { if (x < 0 || x >= n) { printf("read access at %d outside the read (%d bases)\n", x, n); exit(2); } }
    int base(int x) const { check(x); return (int)((w[x >> 4] >> (2 * (x & 15))) & 3u); }
    uint32_t bits(int x) const
    {
        check(x);
        const uint64_t both = (uint64_t)w[x >> 4] | ((uint64_t)w[(x >> 4) + 1] << 32);
        return (uint32_t)(both >> (2 * (x & 15))) & 0xFFFFFu;
    }
};
struct FHost
{
    std::vector<uint32_t> w; std::vector<char> written;
    explicit FHost(size_t n) : w(n, 0xDEADBEEFu), written(n, 0) {}
    void put(int n, uint32_t v) { if (n < 0 || (size_t)n >= w.size()) { printf("flag word %d out of range\n", n); exit(2); } w[n] = v; written[n] = 1; }
    uint32_t get(int n) const { if (n < 0 || (size_t)n >= w.size() || !written[n]) { printf("flag word %d read before written\n", n); exit(2); } return w[n]; }
};

static std::mt19937_64 rng(20261022);
static int rnd(int lo, int hi) { return lo + (int)(rng() % (uint64_t)(hi - lo + 1)); }
static std::vector<uint8_t> random_seq(int n, int alphabet, int homop)
{
    std::vector<uint8_t> s;
    while ((int)s.size() < n)
    {
        const uint8_t c = (uint8_t)rnd(0, alphabet - 1);
        const int run = homop ? rnd(1, homop) : 1;
        for (int r = 0; r < run && (int)s.size() < n; r++) s.push_back(c);
    }
    return s;
}

static long n_cases = 0, n_failed = 0;
// which placements the cases reached: [first row odd][first row at band row 200], last row at band row 200, lB == lA,
// lB == lA + 1, lA - j0 = 1 .. 25 (a pair has at least one row after j0), first block across the wrap, last block across it
static long seen_first[2][2], seen_last200, seen_eq, seen_plus1, seen_len[26], seen_wrap_first, seen_wrap_last;

static void note_placements(int qlen, int mlen, int origin)
{
    for (int i = 1; i < qlen; i++)
    {
        if (!pairable(i, mlen, origin)) continue;
        const int jbA = origin + i, fA = imax(jbA, 1), lA = imin(jbA + BW, mlen + 1) - 1, lB = imin(jbA + 1 + BW, mlen + 1) - 1;
        const int j0 = fA & ~1;
        seen_first[fA & 1][fA == jbA + BW - 1]++;
        seen_last200 += lA == jbA + BW - 1;
        seen_eq += lB == lA;
        seen_plus1 += lB == lA + 1;
        if (lA - j0 <= 25) seen_len[lA - j0]++;
        seen_wrap_first += (j0 & (HSLOTS - 1)) + 10 > HSLOTS;   // rows j0 .. j0 + 9
        int jl = j0;
        while (jl + 10 - 1 <= lB) jl += 10;                     // the last block: rows jl .. jl + 9
        seen_wrap_last += (jl & (HSLOTS - 1)) + 10 > HSLOTS;
    }
}

static void compare(const std::vector<uint8_t>& q, const std::vector<uint8_t>& r, int origin, const char* what)
{
    const int qlen = (int)q.size(), mlen = (int)r.size();
    if (!eligible(qlen, mlen, origin, 4000)) return;
    n_cases++;
    note_placements(qlen, mlen, origin);
    const SHost S(r);
    auto qf = [&](int x) { return (int)q[x]; };
    const size_t nw = (size_t)qlen * words_per_col(mlen);
    HHost H0, H1; FHost F0(nw), F1(nw);
    int bi0 = 0, bj0 = 0, bi1 = 0, bj1 = 0;
    fill(qlen, mlen, origin, H0, S, F0, qf, bi0, bj0, false);
    fill(qlen, mlen, origin, H1, S, F1, qf, bi1, bj1, true);
    bool ok = bi0 == bi1 && bj0 == bj1;
    size_t bad = nw;
    for (size_t n = 0; n < nw && ok; n++)
        if (F0.written[n] != F1.written[n] || (F0.written[n] && F0.w[n] != F1.w[n])) { ok = false; bad = n; }
    const int jb = origin + qlen, first = imax(jb, 1), last = imin(jb + BW, mlen + 1) - 1;
    int badrow = -1;
    for (int j = first; j <= last && ok; j++)
        if (H0.get(j) != H1.get(j)) { ok = false; badrow = j; }
    if (!ok && ++n_failed <= 10)
        printf("%s MISMATCH qlen=%d mlen=%d origin=%d: start (%d,%d)/(%d,%d) word %zd row %d\n", what, qlen, mlen, origin, bi0, bj0, bi1, bj1,
               bad == nw ? (ssize_t)-1 : (ssize_t)bad, badrow);
}

int main()
{
    // band tops (jb = origin + i) above the matrix, at rows 1 .. 30, on both sides of the 256-row wrap and of its second
    // turn; columns from one row to 28 rows past the first block's row (matrix-limited: lB == lA) and band-limited ones
    // (lB == lA + 1, last row at band row 200)
    std::vector<int> tops;
    for (int t = -BW - 1; t <= -BW + 30; t++) tops.push_back(t);
    for (int t = -30; t <= 30; t++) tops.push_back(t);
    for (int t = HSLOTS - 30; t <= HSLOTS + 12; t++) tops.push_back(t);
    for (int t = 2 * HSLOTS - 16; t <= 2 * HSLOTS + 4; t++) tops.push_back(t);
    for (int qlen : {2, 3, 6, 13})
        for (int top : tops)
        {
            const int origin = top - 1;
            std::vector<int> lens;
            for (int d = -2; d <= 28; d++) lens.push_back(imax(top, 1) + d);   // last row of the first column near its first
            for (int d = -3; d <= 14; d++) lens.push_back(top + BW - 1 + d);   // ... near band row 200
            for (int mlen : lens)
            {
                if (mlen < 1) continue;
                const int alphabet = rnd(0, 2) ? 4 : 2;
                const std::vector<uint8_t> qs = random_seq(qlen, alphabet, rnd(0, 1) * 3);
                std::vector<uint8_t> rs = random_seq(mlen, alphabet, rnd(0, 1) * 3);
                // a copy of the query at the band's diagonal now and then, so that the paths run through matches
                if (rnd(0, 1)) for (int x = 0; x < qlen; x++) if (top + x >= 1 && top + x <= mlen) rs[top + x - 1] = qs[x];
                compare(qs, rs, origin, "placement");
            }
        }
    // longer queries with random placements: blocks of every phase against the wrap, many columns per matrix
    for (int it = 0; it < 400; it++)
    {
        const int qlen = rnd(14, 700), alphabet = it % 3 ? 4 : 2;
        const std::vector<uint8_t> qs = random_seq(qlen, alphabet, it % 4 == 0 ? 4 : 0);
        const int mlen = rnd(1, max_len_bound(qlen) - 1);
        const std::vector<uint8_t> rs = random_seq(mlen, alphabet, it % 4 == 0 ? 4 : 0);
        compare(qs, rs, rnd(-BW - 2, mlen + 1), "random");
    }
    bool covered = seen_first[0][0] && seen_first[1][0] && seen_first[1][1] && seen_last200 && seen_eq && seen_plus1 && seen_wrap_first && seen_wrap_last;
    for (int d = 1; d <= 25; d++) covered = covered && seen_len[d];
    printf("cases %ld paired-sweeps %ld failed %ld bad-stores %ld sweeps-with-scalar-stores %ld max-scalar-stores %ld covered %d\n", n_cases, n_sweeps,
           n_failed, n_bad_stores, n_many_sets, max_sets, covered ? 1 : 0);
    if (!covered)
    {
        printf("first row even %ld, odd %ld, odd at band row 200 %ld; last row at band row 200 %ld; lB == lA %ld, lB == lA + 1 %ld; wrap first %ld, last %ld; lA - j0:",
               seen_first[0][0], seen_first[1][0], seen_first[1][1], seen_last200, seen_eq, seen_plus1, seen_wrap_first, seen_wrap_last);
        for (int d = 1; d <= 25; d++) printf(" %ld", seen_len[d]);
        printf("\n");
    }
    return (n_failed || n_bad_stores || n_many_sets || !covered || n_sweeps < 1000) ? 1 : 0;
}
