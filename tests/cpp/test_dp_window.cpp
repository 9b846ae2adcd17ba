// Host check of the read window of longreadselfcorrect_b200/csrc/pbsc_dp_thread.cuh: dpt::fill with a read accessor that keeps
// only a ring of 16 words of the 2-bit read, refilled through the fill's win_fetch / win_store hooks the way the kernel's
// global-read passes do it (pbsc_dp.cu, DptSR), against the same fill over the whole read, paired and one column at a time.
// The ring aborts on a read of a word outside the window of the current sweep (dpt::win_lo .. win_hi), on a read of a slot
// that does not hold the word asked for, on a window of more than 15 words and on a refill that overwrites a word the sweep
// just done read.  Every flag word, the traceback start, the final column, and the traceback from that start (ops, n, ed,
// end cell) must be identical.
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
struct SHost   // the whole read: word n at w[n], the zero word after the read included (the kernel's slab)
{
    std::vector<uint32_t> w; int n;
    explicit SHost(const std::vector<uint8_t>& s) : w((s.size() + 15) / 16 + 1, 0u), n((int)s.size()) { for (size_t x = 0; x < s.size(); x++) w[x >> 4] |= (uint32_t)s[x] << (2 * (x & 15)); }
    void check(int x) const { if (x < 0 || x >= n) { printf("read access at %d outside the read (%d bases)\n", x, n); exit(2); } }
    int base(int x) const { check(x); return (int)((w[x >> 4] >> (2 * (x & 15))) & 3u); }
    uint32_t bits(int x) const
    {
        check(x);
        const uint64_t both = (uint64_t)w[x >> 4] | ((uint64_t)w[(x >> 4) + 1] << 32);
        return (uint32_t)(both >> (2 * (x & 15))) & 0xFFFFFu;
    }
};
static long n_refills = 0, max_live = 0;
struct SRing   // the kernel's ring (DptSR): word n in slot n & 15, tagged here with the word it holds
{
    const SHost& full;
    mutable uint32_t slot[16];
    mutable int tag[16];
    mutable int lo = 0, hi = -1;       // window of the sweep in progress
    mutable bool sweep = false;
    SRing(const SHost& f, int mlen, int origin) : full(f)
    {
        for (int s = 0; s < 16; s++) { slot[s] = 0xDEADBEEFu; tag[s] = -1; }
        // what the kernel's row setup stores: the window of the first sweep
        for (int n = win_lo(1, origin); n <= win_hi(1, mlen, origin); n++) { slot[n & 15] = full.w.at(n); tag[n & 15] = n; }
    }
    uint32_t word(int n) const
    {
        if (!sweep || n < lo || n > hi) { printf("ring read of word %d outside the window %d..%d of the sweep\n", n, lo, hi); exit(2); }
        if (tag[n & 15] != n) { printf("ring slot %d holds word %d, not %d\n", n & 15, tag[n & 15], n); exit(2); }
        return slot[n & 15];
    }
    int base(int x) const { full.check(x); return (int)((word(x >> 4) >> (2 * (x & 15))) & 3u); }
    uint32_t bits(int x) const
    {
        full.check(x);
        const uint64_t both = (uint64_t)word(x >> 4) | ((uint64_t)word((x >> 4) + 1) << 32);
        return (uint32_t)(both >> (2 * (x & 15))) & 0xFFFFFu;
    }
};
struct RingWord { uint32_t w; int n; };
RingWord win_fetch(const SRing& S, int mlen, int origin, int i, int inext)
{
    S.lo = win_lo(i, origin); S.hi = win_hi(i, mlen, origin); S.sweep = true;
    if (S.hi - S.lo + 1 > max_live) max_live = S.hi - S.lo + 1;
    if (S.hi - S.lo + 1 > 15) { printf("window of %d words\n", S.hi - S.lo + 1); exit(2); }
    const int n = win_hi(inext, mlen, origin);
    if (n > S.hi + 1) { printf("window grows by %d words\n", n - S.hi); exit(2); }
    RingWord x{0u, -1};
    if (n >= 0 && n > S.hi) { x.w = S.full.w.at(n); x.n = n; }
    return x;
}
void win_store(const SRing& S, const RingWord& x)
{
    S.sweep = false;
    if (x.n < 0) return;
    const int old = S.tag[x.n & 15];
    if (old >= S.lo && old <= S.hi) { printf("refill of word %d overwrites word %d of the sweep's window\n", x.n, old); exit(2); }
    S.slot[x.n & 15] = x.w; S.tag[x.n & 15] = x.n;
    n_refills++;
}
struct FHost
{
    std::vector<uint32_t> w; std::vector<char> written;
    explicit FHost(size_t n) : w(n, 0xDEADBEEFu), written(n, 0) {}
    void put(int n, uint32_t v) { if (n < 0 || (size_t)n >= w.size()) { printf("flag word %d out of range\n", n); exit(2); } w[n] = v; written[n] = 1; }
    uint32_t get(int n) const { if (n < 0 || (size_t)n >= w.size() || !written[n]) { printf("flag word %d read before written\n", n); exit(2); } return w[n]; }
};
struct OpsHost { std::vector<uint8_t> v; void put(int n, int op) { if ((int)v.size() <= n) v.resize(n + 1); v[n] = (uint8_t)op; } };

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

static long n_cases = 0, n_failed = 0, n_tracebacks = 0;

struct Run
{
    FHost F; HHost H; int bi = 0, bj = 0; OpsHost ops; int n = 0, ed = 0, i0 = 0, j0 = 0;
    explicit Run(size_t nw) : F(nw) {}
};
template <class SS>
static void run(Run& R, const std::vector<uint8_t>& q, int mlen, int origin, const SS& S, const SHost& full, bool pair)
{
    const int qlen = (int)q.size();
    auto qf = [&](int x) { if (x < 0 || x >= qlen) { printf("query access at %d outside the query (%d bases)\n", x, qlen); exit(2); } return (int)q[x]; };
    fill(qlen, mlen, origin, R.H, S, R.F, qf, R.bi, R.bj, pair);
    if (R.bi > 0) traceback(qlen, mlen, origin, full, R.F, qf, R.bi, R.bj, R.ops, R.n, R.ed, R.i0, R.j0);
}

// true when the fills over the ring agree with the fills over the whole read
static bool compare(const std::vector<uint8_t>& q, const std::vector<uint8_t>& r, int origin, const char* what)
{
    const int qlen = (int)q.size(), mlen = (int)r.size();
    if (!eligible(qlen, mlen, origin, 4000)) return true;
    n_cases++;
    const SHost S(r);
    const size_t nw = (size_t)qlen * words_per_col(mlen);
    bool ok = true;
    Run ref(nw);
    run(ref, q, mlen, origin, S, S, false);   // the whole read, one column at a time
    if (ref.bi > 0) n_tracebacks++;
    for (int v = 0; v < 3 && ok; v++)
    {
        Run x(nw);
        const SRing ring(S, mlen, origin);
        if (v == 0) run(x, q, mlen, origin, S, S, true);            // the whole read, paired
        else run(x, q, mlen, origin, ring, S, v == 1);               // the ring, paired and one column at a time
        ok = ref.bi == x.bi && ref.bj == x.bj;
        for (size_t n = 0; n < nw && ok; n++)
            if (ref.F.written[n] != x.F.written[n] || (ref.F.written[n] && ref.F.w[n] != x.F.w[n])) ok = false;
        const int jb = origin + qlen, first = imax(jb, 1), last = imin(jb + BW, mlen + 1) - 1;
        for (int j = first; j <= last && ok; j++)
            if (ref.H.get(j) != x.H.get(j)) ok = false;
        if (ok && ref.bi > 0)
            ok = ref.n == x.n && ref.ed == x.ed && ref.i0 == x.i0 && ref.j0 == x.j0 && ref.ops.v == x.ops.v;
        if (!ok)
        {
            n_failed++;
            if (n_failed <= 10)
                printf("%s MISMATCH (variant %d) qlen=%d mlen=%d origin=%d: start (%d,%d)/(%d,%d) n %d/%d ed %d/%d\n", what, v, qlen, mlen, origin,
                       ref.bi, ref.bj, x.bi, x.bj, ref.n, x.n, ref.ed, x.ed);
        }
    }
    return ok;
}

int main(int argc, char** argv)
{
    const int cases = argc > 1 ? atoi(argv[1]) : 1500;
    // every band origin, from above the matrix to below it, on small matrices
    for (int qlen = 1; qlen <= 20; qlen += 1)
        for (int extra : {-qlen / 2, 0, 7, 230})
        {
            const int mlen = imax(1, qlen + extra);
            const std::vector<uint8_t> q = random_seq(qlen, 4, 0);
            std::vector<uint8_t> r = mutate(q, 0.2, 4);
            r.resize(mlen, 1);
            for (int origin = -BW - 3; origin <= mlen + 2; origin++) compare(q, r, origin, "sweep");
        }
    // the query lengths at the ends of the passes, both strands, homopolymer and two-letter strings, reads at the length bound
    for (int qlen : {1, 2, 255, 256, 257, 1024, 4000})
        for (int it = 0; it < (qlen >= 1024 ? 6 : 12); it++)
        {
            const int alphabet = (it % 3 == 0) ? 2 : 4, homop = (it % 4 == 1) ? 6 : 0;
            const std::vector<uint8_t> q = (it % 6 == 5) ? std::vector<uint8_t>(qlen, 2) : random_seq(qlen, alphabet, homop);
            std::vector<uint8_t> r = mutate(q, (it % 3) * 0.1 + 0.03, alphabet);
            const bool isRC = it & 1;
            const std::vector<uint8_t> flank = random_seq(rnd(0, 40) + (it % 4 == 2 ? max_len_bound(qlen) : 0), alphabet, homop);
            if (isRC) r.insert(r.begin(), flank.begin(), flank.end()); else r.insert(r.end(), flank.begin(), flank.end());
            if (r.empty()) r.push_back(0);
            if ((int)r.size() > max_len_bound(qlen) - 1) r.resize(max_len_bound(qlen) - 1);   // it % 4 == 2: at the bound
            const int mlen = (int)r.size();
            const int k = imin(qlen, imin(mlen, rnd(13, 19)));
            const int origin = ((isRC ? mlen - k : 0) - (isRC ? qlen - k : 0) + 1) - (HALF + 1);
            compare(q, r, origin, "lengths");
            compare(q, r, origin - rnd(1, 150), "lengths-above");
            compare(q, r, origin + rnd(1, 150), "lengths-below");
        }
    // random cases like the kernel's, past the 256-row circular array and the 16-word ring
    for (int it = 0; it < cases; it++)
    {
        const int qmax = (it % 23 == 5) ? 4000 : (it % 3 == 2) ? 1024 : 256;
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
    printf("cases %ld tracebacks %ld refills %ld widest-window %ld failed %ld\n", n_cases, n_tracebacks, n_refills, max_live, n_failed);
    return n_failed ? 1 : (n_cases < 1000 || n_tracebacks < 500 ? 3 : 0);
}
