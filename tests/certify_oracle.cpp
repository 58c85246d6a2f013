// CPU restatement of the c21 key certificates of include/azb.h (azb_certify_keys): the interval inertia count JT, the
// greedy mu, the enclosure of lambda_1, the bound points and the verdict, with the IEEE operations of the kernels in
// azdopt_b200/csrc/azb_certify.cuh, so the results are bit-identical.  TEST INFRASTRUCTURE ONLY.
//
// Every operation runs with the rounding mode set to downward (compiled with -frounding-math, so the compiler neither
// folds nor moves floating point across fesetround).  A rounding up is written through a negation, which is exact:
// ru(1/l) = -rd(-1/l), ru(a - b) = -rd(b - a), ru(a + b) = -rd(-a - b).  (Not two sqrt calls in two modes: the
// compiler may merge calls of the same pure function despite -frounding-math.)
#include <cfenv>
#include <cmath>
#include <cstdint>
#include <cstring>

namespace {

constexpr int STEPS = 12;

struct Down {  // the downward rounding mode for the lifetime of the object
    int old;
    Down() : old(std::fegetround()) { std::fesetround(FE_DOWNWARD); }
    ~Down() { std::fesetround(old); }
};

// JT(T, x): count or -1 (undecided); the rounding mode must be downward
int jt(const uint8_t *par, uint32_t n, double x) {
    double lo[64], hi[64];
    for (uint32_t v = 0; v < n; ++v) lo[v] = hi[v] = -x;
    int count = 0;
    for (uint32_t v = n - 1; v >= 1; --v) {
        const double l = lo[v], u = hi[v];
        if (!(l > 0.0 || u < 0.0)) return -1;
        count += l > 0.0;
        const double r_lo = 1.0 / u, r_hi = -(-1.0 / l);
        const uint32_t p = par[v];
        lo[p] = lo[p] - r_hi;
        hi[p] = -(r_lo - hi[p]);
    }
    if (!(lo[0] > 0.0 || hi[0] < 0.0)) return -1;
    return count + (lo[0] > 0.0);
}

double delta(double c, int j) {  // 4^j ulp(c), 1 <= c < 2^1000
    uint64_t bits;
    std::memcpy(&bits, &c, 8);
    const uint64_t e = (bits >> 52) & 0x7ff, d = (e - 52 + 2 * (uint64_t)j) << 52;
    double out;
    std::memcpy(&out, &d, 8);
    return out;
}

bool c_ok(double c) { return c >= 1.0 && c < 0x1p1000; }

uint32_t greedy_mu(const uint8_t *par, uint32_t n) {
    uint64_t used = 0;
    uint32_t mu = 0;
    for (uint32_t v = n - 1; v >= 1; --v) {
        const uint32_t p = par[v];
        if (!(((used >> v) | (used >> p)) & 1u)) {
            used |= (1ull << v) | (1ull << p);
            ++mu;
        }
    }
    return mu;
}

// [t_lo, t_hi] around bound - mu; the rounding mode must be downward
void points(uint32_t N, uint32_t mu, double bound, double *t_lo, double *t_hi) {
    double b_lo = bound, b_hi = bound;
    if (bound < 0.0) {
        // ru(sqrt(x)) is rd(sqrt(x)) when that is exact (the remainder x - s^2 is exact in the fma), else the next double
        const double x = (double)(N - 1);
        const double s_lo = std::sqrt(x);
        const double s_hi = std::fma(s_lo, s_lo, -x) == 0.0 ? s_lo : std::nextafter(s_lo, INFINITY);
        b_lo = s_lo + 1.0;
        b_hi = -(-s_hi - 1.0);
    }
    *t_lo = b_lo - (double)mu;
    *t_hi = -((double)mu - b_hi);
}

bool star_tie(uint32_t N, double bound) {
    uint32_t s = 0;
    while ((s + 1) * (s + 1) <= N - 1) ++s;
    return bound < 0.0 || (s * s == N - 1 && bound == (double)(s + 1));
}

}  // namespace

extern "C" {

int orc_cert_jt(const uint8_t *par, uint32_t n, double x) {
    Down d;
    return jt(par, n, x);
}

uint32_t orc_cert_mu(const uint8_t *par, uint32_t n) { return greedy_mu(par, n); }

void orc_cert_points(uint32_t N, uint32_t mu, double bound, double *t_lo, double *t_hi) {
    Down d;
    points(N, mu, bound, t_lo, t_hi);
}

// azb_certify_pruned_kernel's decision for one class on n vertices with the cost kernel's c and mu_cost: 1 when the keep
// test drops it (not (double)mu_cost + c <= thr, rounded to nearest) and key > bound is not proven, else 0.  N is the
// search's vertex count, which the default bound (< 0) is taken at.
int orc_cert_unproven(const uint8_t *par, uint32_t n, uint32_t N, double c, uint32_t mu_cost, double thr, double bound) {
    std::fesetround(FE_TONEAREST);
    const double key = (double)mu_cost + c;
    if (key <= thr) return 0;
    Down d;
    double t_lo, t_hi;
    points(N, greedy_mu(par, n), bound, &t_lo, &t_hi);
    if (jt(par, n, t_hi) >= 1) return 0;
    if (!c_ok(c)) return 1;
    for (int j = 0; j < STEPS; ++j) {
        const double x = c - delta(c, j);
        if (!(x > t_hi)) break;
        if (jt(par, n, x) >= 1) return 0;
    }
    return 1;
}

// azb_certify_keys on m trees of n vertices, c = l1[i]
void orc_certify(const uint8_t *par, uint32_t m, uint32_t n, const double *l1, double bound, double *lo_out, double *hi_out,
                 uint32_t *mu_out, int8_t *verdict_out) {
    Down d;
    const double nan = std::nan("");
    const bool tie = star_tie(n, bound);
    for (uint32_t t = 0; t < m; ++t) {
        const uint8_t *p = par + (size_t)t * n;
        const uint32_t mu = greedy_mu(p, n);
        const double c = l1[t];
        double t_lo, t_hi;
        points(n, mu, bound, &t_lo, &t_hi);
        double l1_lo = nan, l1_hi = nan;
        if (c_ok(c)) {
            double a = nan, z = nan;
            for (int j = 0; j < STEPS; ++j) {
                const double x = c - delta(c, j);
                if (jt(p, n, x) >= 1) {
                    a = x;
                    break;
                }
            }
            for (int j = 0; a == a && j < STEPS; ++j) {
                const double x = -(-c - delta(c, j));
                if (jt(p, n, x) == 0) {
                    z = x;
                    break;
                }
            }
            if (a == a && z == z) l1_lo = a, l1_hi = z;
        }
        int v;
        if (tie && mu == 1) v = 0;
        else if (l1_hi <= t_lo || jt(p, n, t_lo) == 0) v = -1;
        else if (l1_lo >= t_hi || jt(p, n, t_hi) >= 1) v = 1;
        else v = 2;
        lo_out[t] = l1_lo;
        hi_out[t] = l1_hi;
        mu_out[t] = mu;
        verdict_out[t] = (int8_t)v;
    }
}

}  // extern "C"
