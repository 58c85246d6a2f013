// Runs azb_certify_pruned_kernel (azdopt_b200/csrc/azb_certify.cuh) on classes given one by one, with any lambda_1, mu and
// threshold, so tests can compare its decision for each class with the CPU restatement (certify_oracle.cpp) and with
// exact arithmetic, including inputs the cost kernel never produces.  TEST INFRASTRUCTURE ONLY.
#include <cstdint>

#include "../azdopt_b200/csrc/azb_certify.cuh"

// out[i] = 1 when the kernel counts class i (m classes of n vertices) as dropped and not proven above the bound, else 0.
// bound < 0: sqrt(N - 1) + 1.  Returns a cudaError_t.
extern "C" int harness_unproven(const uint8_t *par, uint32_t m, uint32_t n, const double *l1, const uint32_t *mu,
                                const double *thr, double bound, uint32_t N, uint8_t *out) {
    uint8_t *d_par = nullptr;
    double *d_l1 = nullptr;
    uint32_t *d_mu = nullptr;
    unsigned long long *d_cnt = nullptr;
    cudaError_t e = cudaMalloc(&d_par, (size_t)m * n);
    if (!e) e = cudaMalloc(&d_l1, (size_t)m * 8);
    if (!e) e = cudaMalloc(&d_mu, (size_t)m * 4);
    if (!e) e = cudaMalloc(&d_cnt, (size_t)m * 8);
    if (!e) e = cudaMemcpy(d_par, par, (size_t)m * n, cudaMemcpyHostToDevice);
    if (!e) e = cudaMemcpy(d_l1, l1, (size_t)m * 8, cudaMemcpyHostToDevice);
    if (!e) e = cudaMemcpy(d_mu, mu, (size_t)m * 4, cudaMemcpyHostToDevice);
    if (!e) e = cudaMemset(d_cnt, 0, (size_t)m * 8);
    const size_t smem = azb_certify_smem(n);
    if (!e) e = cudaFuncSetAttribute(azb_certify_pruned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const AzbCertBound b{bound, N, bound < 0.0 ? 1 : 0, 0};
    for (uint32_t i = 0; !e && i < m; ++i) {
        azb_certify_pruned_kernel<<<1, AZB_CERT_THREADS, smem>>>(d_par + (size_t)i * n, 1, n, d_l1 + i, d_mu + i, thr[i], b,
                                                                 d_cnt + i);
        e = cudaGetLastError();
    }
    unsigned long long *cnt = new unsigned long long[m];
    if (!e) e = cudaMemcpy(cnt, d_cnt, (size_t)m * 8, cudaMemcpyDeviceToHost);
    for (uint32_t i = 0; !e && i < m; ++i) out[i] = (uint8_t)cnt[i];
    delete[] cnt;
    cudaFree(d_par);
    cudaFree(d_l1);
    cudaFree(d_mu);
    cudaFree(d_cnt);
    return (int)e;
}
