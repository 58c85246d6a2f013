// azb_mlp_tc.cuh — the prior model on the 5th-generation tensor cores (AZB_MLP_TC).
// Replaces ActionModel::write_predictions (az-discrete-opt/src/nabla/model/dfdx.rs:69-84; module stack
// graph-state/examples/04-c21-tree.rs:46-52), which runs four cuBLAS sgemm + elementwise launches through dfdx.
//
// One kernel per Linear layer, Y = act(X W^T + b), bf16 operands, fp32 accumulation in TMEM:
//   * X [rows x Kpad] and W [Npad x Kpad] are both K-major (row-major with K contiguous) bf16, so A and B tiles are
//     fetched by TMA (cp.async.bulk.tensor.2d, SWIZZLE_128B, 64-element = 128-byte inner box) into a 4-stage
//     shared-memory ring guarded by full/empty mbarriers;
//   * one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M = 128, N = BN, K = 16 per instruction) on
//     shared-memory matrix descriptors; the accumulator [128 x BN] fp32 lives in TMEM;
//   * tcgen05.commit releases ring slots and finally signals the epilogue warps, which read TMEM with
//     tcgen05.ld.32x32b (warp w%4 <-> TMEM lanes 32(w%4)..), add the bias, apply ReLU (or the Sigmoid head) and store
//     bf16 activations for the next layer (or the f32 h_theta rows).
// The input rows are exactly {0,1} (write_vec), so layer 1 loses nothing to bf16; weights and hidden activations are
// rounded to bf16 (tests compare with the f32 forward at 2e-2 absolute on the sigmoid outputs).
//
// AZB_MLP_TC3 ("bf16x3"): the reference's forward is f32 (dfdx sgemm).  Every operand is split into two bf16 halves,
// x = hi + lo with hi = bf16(x), lo = bf16(x - hi), and a dot product becomes three tensor-core products accumulated in
// the same fp32 TMEM accumulator: hi.hi + hi.lo + lo.hi (the dropped lo.lo term is 2^-16 relative).  In memory the
// halves sit side by side — weights [N][hi(Kpad) | lo(Kpad)], activations [rows][hi(Kpad) | lo(Kpad)] — and the
// kernels simply run 3 Kpad/64 k-blocks whose TMA coordinates pick (A half, W half) = (hi,hi), (hi,lo), (lo,hi); the
// epilogue emits both halves of the next layer's input.  Outputs agree with the f32 forward to ~1e-6.
// Roles per CTA (256 threads): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "azb_common.cuh"

#define TC_BM 128
#define TC_BK 64
#define TC_STAGES 4
#define TC_THREADS 256

// ---- PTX wrappers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t tc_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void tc_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(tc_smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tc_tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            tc_smem_u32(dst)),
        "l"(map), "r"(tc_smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One elected lane of a converged warp.  `if (lane == 0)` makes the issue block a divergent region, and ptxas then
// feeds every tcgen05.mma through a waterfall loop (ELECT + 7 R2UR.BROADCAST + branch per instruction, ~100 cycles
// each: the issue thread, not the tensor pipe, bounds small-N MMAs); with elect.sync it knows the block is uniform.
__device__ __forceinline__ bool tc_elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0u;
}
__device__ __forceinline__ void tc_umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor of a K-major bf16 tile written by TMA with SWIZZLE_128B (rows of 128 bytes,
// 8-row groups of 1024 bytes): start address >> 4, SBO = 1024 >> 4, version 1, layout type 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3ffffu) >> 4);
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Y = act(X W^T + b) for one [128 x BN] tile.  out_bf16: next layer's activations [rows x ld_out] (ReLU);
// out_f32: h_theta rows [rows x ld_out] (Sigmoid); exactly one of them is non-null.
__global__ void __launch_bounds__(TC_THREADS, 1)
    azb_linear_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                         const float *__restrict__ bias, __nv_bfloat16 *__restrict__ out_bf16,
                         float *__restrict__ out_f32, uint32_t ld_out, uint32_t row0, uint32_t rows_end, uint32_t n_valid,
                         uint32_t k_blocks, uint32_t bn, uint32_t nseg, uint32_t lo_out) {
    // k_blocks = k-blocks per segment; nseg = 1 (plain bf16) or 3 (bf16x3: segments (hi,hi), (hi,lo), (lo,hi); the lo
    // halves start k_blocks * 64 columns into a row); lo_out = column offset of the lo half of the output rows
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    __shared__ __align__(8) uint64_t full_bar[TC_STAGES], empty_bar[TC_STAGES], accum_bar;
    __shared__ uint32_t tmem_base_slot;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t m0 = row0 + blockIdx.y * TC_BM, n0 = blockIdx.x * bn;
    const uint32_t a_bytes = TC_BM * TC_BK * 2, b_bytes = bn * TC_BK * 2, stage_bytes = a_bytes + b_bytes;
    uint8_t *smem = (uint8_t *)(((uintptr_t)tc_smem + 1023) & ~(uintptr_t)1023);
    // TMEM columns: power of two >= BN
    const uint32_t tmem_cols = bn <= 32 ? 32 : (bn <= 64 ? 64 : (bn <= 128 ? 128 : 256));

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            tc_mbar_init(&full_bar[s], 1);
            tc_mbar_init(&empty_bar[s], 1);
        }
        tc_mbar_init(&accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&tmem_base_slot)),
                     "r"(tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = tmem_base_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (tc_elect_one()) {
            for (uint32_t kb = 0; kb < nseg * k_blocks; ++kb) {
                const uint32_t s = kb % TC_STAGES, ph = (kb / TC_STAGES) & 1u;
                const uint32_t seg = kb / k_blocks, j = kb - seg * k_blocks;
                tc_mbar_wait(&empty_bar[s], ph ^ 1u);
                uint8_t *a_dst = smem + (size_t)s * stage_bytes, *b_dst = a_dst + a_bytes;
                tc_mbar_expect_tx(&full_bar[s], stage_bytes);
                tc_tma_load_2d(a_dst, &map_x, &full_bar[s], (int)(((seg == 2u ? k_blocks : 0u) + j) * TC_BK), (int)m0);
                tc_tma_load_2d(b_dst, &map_w, &full_bar[s], (int)(((seg == 1u ? k_blocks : 0u) + j) * TC_BK), (int)n0);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        // instruction descriptor, kind::f16: D = F32, A = B = BF16, both K-major, N >> 3, M >> 4
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((bn >> 3) << 17) | ((TC_BM >> 4) << 24);
        const uint32_t kb_all = nseg * k_blocks;
        for (uint32_t kb = 0; kb < kb_all; ++kb) {
            const uint32_t s = kb % TC_STAGES, ph = (kb / TC_STAGES) & 1u;
            tc_mbar_wait(&full_bar[s], ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (tc_elect_one()) {
                const uint32_t a_addr = tc_smem_u32(smem + (size_t)s * stage_bytes), b_addr = a_addr + a_bytes;
#pragma unroll
                for (uint32_t k = 0; k < TC_BK / 16; ++k) {
                    const uint64_t adesc = tc_smem_desc(a_addr + k * 32u), bdesc = tc_smem_desc(b_addr + k * 32u);
                    tc_umma_f16(tmem_d, adesc, bdesc, idesc, (kb | k) != 0u ? 1u : 0u);
                }
                tc_umma_commit(&empty_bar[s]);                     // frees the ring slot when these MMAs retire
                if (kb + 1 == kb_all) tc_umma_commit(&accum_bar);  // accumulator complete
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> bias + activation -> global =====
        tc_mbar_wait(&accum_bar, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t q = warp & 3u;  // TMEM lane quadrant this warp may read
        const uint32_t row = m0 + q * 32u + lane;
        for (uint32_t c0 = 0; c0 < bn; c0 += 32) {
            uint32_t r[32];
            tc_tmem_ld32(tmem_d + ((q * 32u) << 16) + c0, r);
            if (row < rows_end) {
                if (out_bf16) {
                    __nv_bfloat16 *dst = out_bf16 + (size_t)row * ld_out + n0 + c0;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint32_t pk[4], pl[4];
#pragma unroll
                        for (int t = 0; t < 4; ++t) {
                            const uint32_t n = n0 + c0 + j + 2 * t;
                            float v0 = __uint_as_float(r[j + 2 * t]) + bias[n];
                            float v1 = __uint_as_float(r[j + 2 * t + 1]) + bias[n + 1];
                            v0 = v0 > 0.f ? v0 : 0.f;
                            v1 = v1 > 0.f ? v1 : 0.f;
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(v0, v1);
                            pk[t] = *reinterpret_cast<uint32_t *>(&h2);
                            // the part bf16 lost, itself rounded to bf16 (x - hi is exact in f32)
                            __nv_bfloat162 l2 = __floats2bfloat162_rn(v0 - __low2float(h2), v1 - __high2float(h2));
                            pl[t] = *reinterpret_cast<uint32_t *>(&l2);
                        }
                        *reinterpret_cast<uint4 *>(dst + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                        if (nseg == 3u) *reinterpret_cast<uint4 *>(dst + lo_out + j) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                    }
                }
            }
            if (!out_bf16) {
                // Sigmoid head, f32 rows: transpose the warp's 32x32 chunk through shared memory (the operand ring is
                // idle once the accumulator is complete) so that every store instruction writes one contiguous row piece
                float *tile = reinterpret_cast<float *>(smem) + q * (32 * 33);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const uint32_t n = n0 + c0 + j;
                    const float v = __uint_as_float(r[j]) + bias[n];
                    tile[lane * 33 + j] = __fdividef(1.0f, 1.0f + __expf(-v));
                }
                __syncwarp();
                const uint32_t n = n0 + c0 + lane;
                for (uint32_t rr = 0; rr < 32; ++rr) {
                    const uint32_t orow = m0 + q * 32u + rr;
                    if (orow < rows_end && n < n_valid) out_f32[(size_t)orow * ld_out + n] = tile[rr * 33 + lane];
                }
                __syncwarp();
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(tmem_cols) : "memory");
    }
}

// f32 rows -> bf16 rows padded to Kpad (zeros beyond K); split: the row is [hi(Kpad) | lo(Kpad)], lo = bf16(x - hi)
__global__ void azb_rows_to_bf16_kernel(const float *__restrict__ x, uint32_t ldx, uint32_t K, __nv_bfloat16 *__restrict__ y,
                                        uint32_t ldy, uint32_t rows, uint32_t Kpad, uint32_t split) {
    const uint32_t r = blockIdx.x;
    if (r >= rows) return;
    for (uint32_t k = threadIdx.x; k < Kpad; k += blockDim.x) {
        const float v = k < K ? x[(size_t)r * ldx + k] : 0.f;
        const __nv_bfloat16 hi = __float2bfloat16(v);
        y[(size_t)r * ldy + k] = hi;
        if (split) y[(size_t)r * ldy + Kpad + k] = __float2bfloat16(v - __bfloat162float(hi));
    }
}

// dfdx parameter block (weight[out][in], bias[out]) -> bf16 weight [Npad x Kpad] (split: [Npad x (hi(Kpad) | lo(Kpad))]),
// f32 bias [Npad], zero padded
__global__ void azb_params_to_bf16_kernel(const float *__restrict__ w, const float *__restrict__ b, uint32_t K, uint32_t N,
                                          __nv_bfloat16 *__restrict__ wq, float *__restrict__ bq, uint32_t Kpad, uint32_t Npad,
                                          uint32_t split) {
    const uint32_t n = blockIdx.x;
    const uint32_t ld = split ? 2u * Kpad : Kpad;
    for (uint32_t k = threadIdx.x; k < Kpad; k += blockDim.x) {
        const float v = (n < N && k < K) ? w[(size_t)n * K + k] : 0.f;
        const __nv_bfloat16 hi = __float2bfloat16(v);
        wq[(size_t)n * ld + k] = hi;
        if (split) wq[(size_t)n * ld + Kpad + k] = __float2bfloat16(v - __bfloat162float(hi));
    }
    if (threadIdx.x == 0) bq[n] = n < N ? b[n] : 0.f;
}

struct AzbMlpTc {
    bool ready;
    uint32_t split;         // 0: plain bf16; 1: bf16x3 (operands stored as [hi | lo], three products per dot product)
    uint32_t rows_pad, dims[5], kpad[4], npad[4], bn[4];
    __nv_bfloat16 *act[4];  // act[l] = input of layer l, [rows_pad x kpad[l]]
    __nv_bfloat16 *w[4];
    float *bias[4];
    CUtensorMap map_x[4], map_w[4];
    size_t smem_bytes[4];
};

typedef CUresult(CUDAAPI *azb_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                         const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                         CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline const char *azb_tc_make_map(azb_encode_fn enc, CUtensorMap *map, void *ptr, uint64_t rows, uint64_t kpad,
                                          uint32_t box_rows) {
    const cuuint64_t gdim[2] = {kpad, rows};
    const cuuint64_t gstride[1] = {kpad * 2};
    const cuuint32_t box[2] = {TC_BK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? nullptr : "cuTensorMapEncodeTiled failed";
}

static inline void azb_mlp_tc_destroy(AzbMlpTc &t) {
    for (int l = 0; l < 4; ++l) {
        if (t.act[l]) cudaFree(t.act[l]);
        if (t.w[l]) cudaFree(t.w[l]);
        if (t.bias[l]) cudaFree(t.bias[l]);
        t.act[l] = nullptr;
        t.w[l] = nullptr;
        t.bias[l] = nullptr;
    }
    t.ready = false;
}

static inline const char *azb_mlp_tc_create(AzbMlpTc &t, uint32_t rows, const uint32_t *dims, uint64_t *dev_bytes,
                                            bool split = false) {
    memset(&t, 0, sizeof(t));
    t.split = split ? 1u : 0u;
    azb_encode_fn enc = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void **)&enc, cudaEnableDefault, &qres) != cudaSuccess || !enc)
        return "cuTensorMapEncodeTiled is not available";
    t.rows_pad = (rows + TC_BM - 1) / TC_BM * TC_BM;
    for (int i = 0; i < 5; ++i) t.dims[i] = dims[i];
    for (int l = 0; l < 4; ++l) {
        t.kpad[l] = (dims[l] + TC_BK - 1) / TC_BK * TC_BK;
        // output columns of layer l are the K of layer l+1: pad to its K padding; the head pads to a multiple of 16
        const uint32_t n = dims[l + 1];
        t.npad[l] = l < 3 ? (n + TC_BK - 1) / TC_BK * TC_BK : (n + 15) / 16 * 16;
        t.bn[l] = t.npad[l] % 128 == 0 ? 128 : (t.npad[l] <= 256 ? t.npad[l] : 0);
        if (t.bn[l] == 0) {  // wide head: fall back to 64-column tiles over a 64-padded width
            t.npad[l] = (n + 63) / 64 * 64;
            t.bn[l] = 64;
        }
    }
    for (int l = 0; l < 4; ++l) {
        // weight rows are padded (zeros) to a multiple of 128 so that a 128-row TMA box never leaves the tensor
        const uint32_t kw = (t.split ? 2u : 1u) * t.kpad[l];  // row width in elements: [hi | lo] when split
        const size_t abytes = (size_t)t.rows_pad * kw * 2, wbytes = (size_t)((t.npad[l] + 127u) / 128u * 128u) * kw * 2;
        // the epilogue reads the bias 32 columns at a time and a head's npad is only a multiple of 16: the biases are
        // allocated to the next multiple of 32 floats, the tail zero (azb_params_to_bf16_kernel writes npad of them)
        const size_t bbytes = (size_t)((t.npad[l] + 31u) & ~31u) * 4;
        if (cudaMalloc((void **)&t.act[l], abytes) != cudaSuccess) return "cudaMalloc (activations) failed";
        if (cudaMalloc((void **)&t.w[l], wbytes) != cudaSuccess) return "cudaMalloc (weights) failed";
        if (cudaMalloc((void **)&t.bias[l], bbytes) != cudaSuccess) return "cudaMalloc (bias) failed";
        cudaMemset(t.act[l], 0, abytes);
        cudaMemset(t.w[l], 0, wbytes);
        cudaMemset(t.bias[l], 0, bbytes);
        if (dev_bytes) *dev_bytes += abytes + wbytes + bbytes;
        const char *why = azb_tc_make_map(enc, &t.map_x[l], t.act[l], t.rows_pad, kw, TC_BM);
        if (why) return why;
        why = azb_tc_make_map(enc, &t.map_w[l], t.w[l], t.npad[l], kw, t.bn[l]);
        if (why) return why;
        t.smem_bytes[l] = (size_t)TC_STAGES * (TC_BM + t.bn[l]) * TC_BK * 2 + 1024;
    }
    size_t mx = 0;
    for (int l = 0; l < 4; ++l) mx = t.smem_bytes[l] > mx ? t.smem_bytes[l] : mx;
    if (cudaFuncSetAttribute(azb_linear_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mx) != cudaSuccess)
        return "cudaFuncSetAttribute failed";
    t.ready = true;
    return nullptr;
}

static inline const char *azb_mlp_tc_load(AzbMlpTc &t, const float *params, cudaStream_t stream, uint64_t *launches) {
    const float *p = params;
    for (int l = 0; l < 4; ++l) {
        const uint32_t K = t.dims[l], N = t.dims[l + 1];
        azb_params_to_bf16_kernel<<<t.npad[l], 128, 0, stream>>>(p, p + (size_t)K * N, K, N, t.w[l], t.bias[l], t.kpad[l],
                                                                 t.npad[l], t.split);
        if (launches) *launches += 1;
        p += (size_t)K * N + N;
    }
    return cudaGetLastError() == cudaSuccess ? nullptr : "weight conversion launch failed";
}

// rows [row0, row0 + rows) of the batch; row0 is a multiple of 128.  x: f32 rows [.. x ldx] to convert first, or null
// when the bf16 input rows are already in place (tree_pack wrote them); y: f32 [.. x ldy]
static inline const char *azb_mlp_tc_forward(AzbMlpTc &t, const float *x, uint32_t ldx, float *y, uint32_t ldy,
                                             uint32_t row0, uint32_t rows, cudaStream_t stream, uint64_t *launches) {
    if (!t.ready) return "not created";
    const uint32_t wide = t.split ? 2u : 1u;
    if (x) {
        azb_rows_to_bf16_kernel<<<rows, 128, 0, stream>>>(x + (size_t)row0 * ldx, ldx, t.dims[0],
                                                          t.act[0] + (size_t)row0 * wide * t.kpad[0], wide * t.kpad[0], rows,
                                                          t.kpad[0], t.split);
        if (launches) *launches += 1;
    }
    for (int l = 0; l < 4; ++l) {
        dim3 grid(t.npad[l] / t.bn[l], (rows + TC_BM - 1) / TC_BM);
        const bool head = l == 3;
        azb_linear_tc_kernel<<<grid, TC_THREADS, t.smem_bytes[l], stream>>>(
            t.map_x[l], t.map_w[l], t.bias[l], head ? nullptr : t.act[l + 1], head ? y : nullptr,
            head ? ldy : wide * t.kpad[l + 1], row0, row0 + rows, t.dims[l + 1], t.kpad[l] / TC_BK, t.bn[l], t.split ? 3u : 1u,
            head ? 0u : t.kpad[l + 1]);
        if (launches) *launches += 1;
    }
    return cudaGetLastError() == cudaSuccess ? nullptr : "tensor-core forward launch failed";
}
