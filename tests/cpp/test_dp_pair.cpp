// Host check of the paired-column fill of longreadselfcorrect_b200/csrc/pbsc_dp_thread.cuh: dpt::fill with pairing on (two
// columns per sweep, packed 16-bit halves) against the same fill one column at a time.  Every flag word (and which words were
// written), the traceback start and the final column's scores must be identical.  The host accessors abort on a misaligned
// pair access, a score outside 16 bits or a flag word read before it was written; the packed host operations abort on a lane
// overflow.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>
#include "../../longreadselfcorrect_b200/csrc/pbsc_dp_thread.cuh"

using namespace pbsc::dpt;

struct HHost
{
    int16_t a[HSLOTS];
    HHost() { for (int i = 0; i < HSLOTS; i++) a[i] = 0; }
    int get(int j) const { return a[j & (HSLOTS - 1)]; }
    bool pairs_ok(int j) const { return ((j >> 1) & (HSLOTS / 2 - 1)) <= HSLOTS / 2 - 5; }
    uint32_t get2(int j, int u) const
    {
        const int s = (j & (HSLOTS - 1)) + 2 * u;
        if ((j & 1) || s + 1 >= HSLOTS) { printf("bad pair access\n"); exit(2); }
        return (uint32_t)(uint16_t)a[s] | ((uint32_t)(uint16_t)a[s + 1] << 16);
    }
    void set2(int j, int u, uint32_t w)
    {
        const int s = (j & (HSLOTS - 1)) + 2 * u;
        if ((j & 1) || s + 1 >= HSLOTS) { printf("bad pair access\n"); exit(2); }
        a[s] = (int16_t)(w & 0xFFFFu); a[s + 1] = (int16_t)(w >> 16);
    }
    void set(int j, int v) { if (v < -32768 || v > 32767) { printf("16-bit overflow\n"); exit(2); } a[j & (HSLOTS - 1)] = (int16_t)v; }
};
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

static std::mt19937_64 rng(20261021);
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
static std::vector<uint8_t> mutate(const std::vector<uint8_t>& s, double err, int alphabet)
{
    std::vector<uint8_t> o;
    for (size_t x = 0; x < s.size(); x++)
    {
        const double u = (double)(rng() % 1000000) / 1e6;
        if (u < err * 0.5) { o.push_back((uint8_t)rnd(0, alphabet - 1)); o.push_back(s[x]); }
        else if (u < err * 0.8) { }
        else if (u < err) o.push_back((uint8_t)rnd(0, alphabet - 1));
        else o.push_back(s[x]);
    }
    return o;
}

static long n_cases = 0, n_failed = 0, n_paired_cols = 0;

// true when both fills agree
static bool compare(const std::vector<uint8_t>& q, const std::vector<uint8_t>& r, int origin, const char* what)
{
    const int qlen = (int)q.size(), mlen = (int)r.size();
    if (!eligible(qlen, mlen, origin, 4000)) return true;
    n_cases++;
    for (int i = 1; i < qlen; i++) n_paired_cols += pairable(i, mlen, origin) ? 1 : 0;
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
    // the last column, which the traceback start was taken from
    const int jb = origin + qlen, first = imax(jb, 1), last = imin(jb + BW, mlen + 1) - 1;
    int badrow = -1;
    for (int j = first; j <= last && ok; j++)
        if (H0.get(j) != H1.get(j)) { ok = false; badrow = j; }
    if (!ok)
    {
        n_failed++;
        if (n_failed <= 10)
            printf("%s MISMATCH qlen=%d mlen=%d origin=%d: start (%d,%d)/(%d,%d) word %zd row %d\n", what, qlen, mlen, origin, bi0, bj0, bi1, bj1,
                   bad == nw ? (ssize_t)-1 : (ssize_t)bad, badrow);
    }
    return ok;
}

int main(int argc, char** argv)
{
    const int cases = argc > 1 ? atoi(argv[1]) : 3000;
    // every band origin, from above the matrix to below it, on small matrices: odd and even qlen, first row odd and even,
    // bands clipped in one column of a pair only, computed columns next to skipped ones
    for (int qlen = 1; qlen <= 24; qlen += 1)
        for (int extra : {-qlen / 2, 0, 7, 230})
        {
            const int mlen = imax(1, qlen + extra);
            const std::vector<uint8_t> q = random_seq(qlen, 4, 0);
            const std::vector<uint8_t> r = mutate(q, 0.2, 4);
            std::vector<uint8_t> rr = r;
            rr.resize(mlen, 1);
            for (int origin = -BW - 3; origin <= mlen + 2; origin++) compare(q, rr, origin, "sweep");
        }
    // medium lengths over many origins (bands crossing the matrix top and bottom in the middle of the query)
    for (int it = 0; it < 60; it++)
    {
        const int qlen = rnd(190, 420), alphabet = it % 3 == 0 ? 2 : 4, homop = it % 4 == 0 ? 5 : 0;
        const std::vector<uint8_t> q = random_seq(qlen, alphabet, homop);
        std::vector<uint8_t> r = mutate(q, it % 2 ? 0.1 : 0.3, alphabet);
        r.resize(imin((int)r.size(), max_len_bound(qlen)));
        const int mlen = (int)r.size();
        for (int origin = -BW - 2; origin <= mlen + 1; origin += rnd(1, 9)) compare(q, r, origin, "medium");
    }
    // random cases like the kernel's: forward / reverse placements, errors, two-letter and homopolymer strings, lengths past the
    // 256-row circular array
    for (int it = 0; it < cases; it++)
    {
        const int qmax = (it % 23 == 5) ? 4000 : (it % 5 == 2) ? 1024 : 256;
        const int alphabet = (it % 5 == 0) ? 2 : 4, homop = (it % 4 == 0) ? 4 : 0;
        const int qlen = rnd(1, qmax);
        const std::vector<uint8_t> q = random_seq(qlen, alphabet, homop);
        std::vector<uint8_t> r = (it % 11 == 10) ? random_seq(rnd(1, max_len_bound(qlen) - 1), alphabet, homop) : mutate(q, (it % 3) * 0.12 + 0.02, alphabet);
        if (r.empty()) r.push_back(0);
        const bool isRC = it & 1;
        const std::vector<uint8_t> flank = random_seq(rnd(0, 40), alphabet, homop);
        if (isRC) r.insert(r.begin(), flank.begin(), flank.end()); else r.insert(r.end(), flank.begin(), flank.end());
        if ((int)r.size() > max_len_bound(qlen) - 1) r.resize(max_len_bound(qlen) - 1);
        const int mlen = (int)r.size();
        const int k = imin(qlen, imin(mlen, rnd(13, 19)));
        int origin = ((isRC ? mlen - k : 0) - (isRC ? qlen - k : 0) + 1) - (HALF + 1);
        if (it % 7 == 3) origin = rnd(-BW - 2, mlen + 1);
        compare(q, r, origin, "random");
    }
    // 4000 bases at the 16-bit bounds: all mismatches (the diagonal falls by 8 per column), all gaps, one letter against
    // another, a homopolymer against itself, for the placements the caller uses and a few others
    {
        const int qlen = 4000, mlen = max_len_bound(qlen) - 1;
        const std::vector<uint8_t> qa(qlen, 0), rc(mlen, 1), ra(mlen, 0), rshort(qlen / 2, 2);
        std::vector<uint8_t> alt(qlen), alt2(mlen);
        for (int x = 0; x < qlen; x++) alt[x] = (uint8_t)(x & 1);
        for (int x = 0; x < mlen; x++) alt2[x] = (uint8_t)(2 + (x & 1));
        for (int origin : {-HALF, -HALF - 1, 0, 1, mlen - qlen - HALF, -BW + 1, 57})
        {
            compare(qa, rc, origin, "allmismatch");
            compare(qa, ra, origin, "homopolymer");
            compare(qa, rshort, origin, "short-read");
            compare(alt, alt2, origin, "twoletter-mismatch");
        }
    }
    printf("cases %ld paired-columns %ld failed %ld\n", n_cases, n_paired_cols, n_failed);
    return n_failed ? 1 : (n_cases < 1000 ? 3 : 0);
}
