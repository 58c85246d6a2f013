// azb_certify.cuh — certificates for c21 keys against a bound (azb_certify_keys, azb_trees_within_proof).  The
// definitions (interval inertia count JT, greedy mu, the enclosure of lambda_1, the bound points and the verdict) are in
// include/azb.h; DESIGN.md §4.12 has the argument.  Every rounding is one IEEE binary64 operation rounded down (_rd) or
// up (_ru), in exactly the order of the definition: tests/certify_oracle.cpp restates it bit for bit on the CPU.
//
// One thread per tree.  Its parent array and its vertex intervals live in a column of [n][AZB_CERT_THREADS] shared
// arrays (dynamic shared memory, azb_certify_smem bytes), so indexing by vertex needs no local memory.
#pragma once
#include "azb_common.cuh"

#define AZB_CERT_THREADS 64  // trees per block
#define AZB_CERT_STEPS 12    // enclosure steps j = 0 .. 11: c -+ 4^j ulp(c)

struct AzbCertBound {   // the bound as a real number (include/azb.h)
    double bound;       // used when dflt == 0
    uint32_t N;         // dflt: the bound is sqrt(N - 1) + 1
    int dflt;
    int tie;            // a star (mu = 1) has key = bound exactly
};

static inline size_t azb_certify_smem(uint32_t n) { return (size_t)n * AZB_CERT_THREADS * 17; }

// JT(T, x): the number of eigenvalues of A above x, or -1 when some interval holds 0 (undecided).  par, lo and hi point
// at this thread's column (stride AZB_CERT_THREADS); parents[v] < v, so an interval is final when the loop reaches it.
// An interval with a NaN end counts as holding 0.
__device__ __forceinline__ int azb_cert_jt(const uint8_t *par, double *lo, double *hi, uint32_t n, double x) {
    constexpr uint32_t T = AZB_CERT_THREADS;
    const double mx = -x;
#pragma unroll 1
    for (uint32_t v = 0; v < n; ++v) lo[v * T] = hi[v * T] = mx;
    int count = 0;
#pragma unroll 1
    for (uint32_t v = n - 1; v >= 1; --v) {
        const double l = lo[v * T], u = hi[v * T];
        if (!(l > 0.0 || u < 0.0)) return -1;
        count += l > 0.0;
        const double r_lo = __ddiv_rd(1.0, u), r_hi = __ddiv_ru(1.0, l);
        const uint32_t p = par[v * T];
        lo[p * T] = __dsub_rd(lo[p * T], r_hi);
        hi[p * T] = __dsub_ru(hi[p * T], r_lo);
    }
    if (!(lo[0] > 0.0 || hi[0] < 0.0)) return -1;
    return count + (lo[0] > 0.0);
}

// 4^j ulp(c) for 1 <= c < 2^1000, exactly
__device__ __forceinline__ double azb_cert_delta(double c, int j) {
    const long long e = (__double_as_longlong(c) >> 52) & 0x7ff;
    return __longlong_as_double((e - 52 + 2 * j) << 52);
}

__device__ __forceinline__ bool azb_cert_c_ok(double c) { return c >= 1.0 && c < 0x1p1000; }

// greedy leaf matching: v = n-1 .. 1 is matched to parents[v] when both are free
__device__ __forceinline__ uint32_t azb_cert_mu(const uint8_t *par, uint32_t n) {
    constexpr uint32_t T = AZB_CERT_THREADS;
    unsigned long long used = 0;
    uint32_t mu = 0;
#pragma unroll 1
    for (uint32_t v = n - 1; v >= 1; --v) {
        const uint32_t p = par[v * T];
        if (!(((used >> v) | (used >> p)) & 1ull)) {
            used |= (1ull << v) | (1ull << p);
            ++mu;
        }
    }
    return mu;
}

// t_lo <= bound - mu <= t_hi
__device__ __forceinline__ void azb_cert_t(const AzbCertBound &b, uint32_t mu, double &t_lo, double &t_hi) {
    double b_lo = b.bound, b_hi = b.bound;
    if (b.dflt) {
        b_lo = __dadd_rd(__dsqrt_rd((double)(b.N - 1)), 1.0);
        b_hi = __dadd_ru(__dsqrt_ru((double)(b.N - 1)), 1.0);
    }
    t_lo = __dsub_rd(b_lo, (double)mu);
    t_hi = __dsub_ru(b_hi, (double)mu);
}

// this thread's tree t (when t < m) into its column of the shared parents
__device__ __forceinline__ void azb_cert_load(const uint8_t *__restrict__ par, uint32_t t, uint32_t n, uint8_t *s_par) {
#pragma unroll 1
    for (uint32_t v = 0; v < n; ++v) s_par[v * AZB_CERT_THREADS] = par[(size_t)t * n + v];
}

// Every output may be null.  tally (azb_trees_within_proof's result classes): tally[0..3] += the trees with verdict
// -1, 0, +1, 2.  Dynamic shared memory: azb_certify_smem(n).
__global__ void __launch_bounds__(AZB_CERT_THREADS) azb_certify_kernel(const uint8_t *__restrict__ par, uint32_t m, uint32_t n,
                                                                       const double *__restrict__ l1, AzbCertBound b,
                                                                       double *__restrict__ out_lo, double *__restrict__ out_hi,
                                                                       uint32_t *__restrict__ out_mu, int8_t *__restrict__ out_v,
                                                                       unsigned long long *__restrict__ tally) {
    extern __shared__ double s_cert[];
    constexpr uint32_t T = AZB_CERT_THREADS;
    double *lo = s_cert + threadIdx.x, *hi = s_cert + (size_t)n * T + threadIdx.x;
    uint8_t *sp = reinterpret_cast<uint8_t *>(s_cert + (size_t)2 * n * T) + threadIdx.x;
    const uint32_t t = blockIdx.x * T + threadIdx.x;
    int verdict = 3;  // no tree
    if (t < m) {
        azb_cert_load(par, t, n, sp);
        const uint32_t mu = azb_cert_mu(sp, n);
        const double c = l1[t], nan = __longlong_as_double(0x7ff8000000000000ll);
        double t_lo, t_hi;
        azb_cert_t(b, mu, t_lo, t_hi);
        // One JT call site (inlined once, so the kernel keeps no stack).  Points i: 0 .. S-1 rd(c - d_i), S .. 2S-1
        // ru(c + d_{i-S}), 2S t_lo, 2S+1 t_hi; the verdict's shortcuts come first at 2S and 2S+1.
        constexpr int S = AZB_CERT_STEPS;
        double a = nan, z = nan, l1_lo = nan, l1_hi = nan;
        verdict = 2;
#pragma unroll 1
        for (int i = azb_cert_c_ok(c) ? 0 : 2 * S; i < 2 * S + 2;) {
            if (i == 2 * S) {
                if (a == a && z == z) l1_lo = a, l1_hi = z;
                if (b.tie && mu == 1) {
                    verdict = 0;
                    break;
                }
                if (l1_hi <= t_lo) {
                    verdict = -1;
                    break;
                }
            }
            if (i == 2 * S + 1 && l1_lo >= t_hi) {
                verdict = 1;
                break;
            }
            const double x = i < S ? __dsub_rd(c, azb_cert_delta(c, i))
                                   : (i < 2 * S ? __dadd_ru(c, azb_cert_delta(c, i - S)) : (i == 2 * S ? t_lo : t_hi));
            const int k = azb_cert_jt(sp, lo, hi, n, x);
            if (i < S) {
                if (k >= 1) a = x, i = S;
                else if (++i == S) i = 2 * S;  // no lower end: both ends stay NaN
            } else if (i < 2 * S) {
                if (k == 0) z = x, i = 2 * S;
                else ++i;
            } else if (i == 2 * S) {
                if (k == 0) {
                    verdict = -1;
                    break;
                }
                ++i;
            } else {
                if (k >= 1) verdict = 1;
                break;
            }
        }
        if (out_lo) out_lo[t] = l1_lo;
        if (out_hi) out_hi[t] = l1_hi;
        if (out_mu) out_mu[t] = mu;
        if (out_v) out_v[t] = (int8_t)verdict;
    }
    if (tally) {
        const int c0 = __syncthreads_count(verdict == -1), c1 = __syncthreads_count(verdict == 0);
        const int c2 = __syncthreads_count(verdict == 1), c3 = __syncthreads_count(verdict == 2);
        if (threadIdx.x == 0) {
            if (c0) atomicAdd(&tally[0], (unsigned long long)c0);
            if (c1) atomicAdd(&tally[1], (unsigned long long)c1);
            if (c2) atomicAdd(&tally[2], (unsigned long long)c2);
            if (c3) atomicAdd(&tally[3], (unsigned long long)c3);
        }
    }
}

// The grow side of azb_trees_within_proof, on one chunk's decoded canonical arrays right after azb_grow_keep_kernel:
// every class the keep kernel dropped (key (double)mu + lambda_1 not <= thr) must have key > bound.  That is proven when
// JT at t_hi (from the greedy mu) counts >= 1, or else JT counts >= 1 at one of the points rd(c - 4^j ulp(c)),
// j = 0 .. 11, that lie above t_hi (c = the cost kernel's lambda_1).  *unproven += the dropped classes for which
// neither holds.  Dynamic shared memory: azb_certify_smem(n).
__global__ void __launch_bounds__(AZB_CERT_THREADS) azb_certify_pruned_kernel(const uint8_t *__restrict__ par, uint32_t m,
                                                                              uint32_t n, const double *__restrict__ l1,
                                                                              const uint32_t *__restrict__ mu_cost, double thr,
                                                                              AzbCertBound b,
                                                                              unsigned long long *__restrict__ unproven) {
    extern __shared__ double s_cert[];
    constexpr uint32_t T = AZB_CERT_THREADS;
    double *lo = s_cert + threadIdx.x, *hi = s_cert + (size_t)n * T + threadIdx.x;
    uint8_t *sp = reinterpret_cast<uint8_t *>(s_cert + (size_t)2 * n * T) + threadIdx.x;
    const uint32_t t = blockIdx.x * T + threadIdx.x;
    bool open = false;
    if (t < m && !(__dadd_rn((double)mu_cost[t], l1[t]) <= thr)) {
        azb_cert_load(par, t, n, sp);
        double t_lo, t_hi;
        azb_cert_t(b, azb_cert_mu(sp, n), t_lo, t_hi);
        open = azb_cert_jt(sp, lo, hi, n, t_hi) < 1;
        const double c = l1[t];
        if (open && azb_cert_c_ok(c)) {
#pragma unroll 1
            for (int j = 0; j < AZB_CERT_STEPS; ++j) {
                const double x = __dsub_rd(c, azb_cert_delta(c, j));
                if (!(x > t_hi)) break;
                if (azb_cert_jt(sp, lo, hi, n, x) >= 1) {
                    open = false;
                    break;
                }
            }
        }
    }
    const int cnt = __syncthreads_count(open);
    if (threadIdx.x == 0 && cnt) atomicAdd(unproven, (unsigned long long)cnt);
}
