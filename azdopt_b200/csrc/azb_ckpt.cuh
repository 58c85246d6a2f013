// azb_ckpt.cuh — checkpoint save and load (azb_checkpoint_size / _save / _load): the kernels that move the trees between
// the arenas and a blob.  The blob format and the digest are defined in include/azb.h; DESIGN.md §4.9 has the design.
//
//   size     one thread per tree: record length from the walker header; a CUB exclusive scan makes the offset table
//   pack     up to 64 CTAs per tree, each a slice of the record: gathers walker | nodes | keys | blocks | overflow in-arcs
//            into a staging chunk and adds its digest terms to the tree's sum (an exact integer sum: any order and any
//            split give the same value); a thread per tree then writes the digest word
//   unpack   the mirror: record length against the walker header and the handle's capacities, the scatter, the digest
//            terms; a thread per tree then compares the digest.  The lowest failing global root is kept with atomicMin
//   hash     one warp per tree: clears its transposition table and inserts nodes 0..n-1 in index order with the search
//            kernel's own probe (hash_probe / hash_insert), which rebuilds the table the search built
#pragma once
#include <cub/device/device_scan.cuh>

#include "azb_common.cuh"
#include "azb_tree.cuh"

#define AZB_CKPT_WARPS 8  // hash rebuild: one warp per tree
#define AZB_CKPT_K 0x9E3779B97F4A7C15ull

// record of one tree, in 32-bit words: walker | nodes (16 words each) | keys (W each) | block units [AZB_BLK_PAD, nblk)
// (2 words each) | overflow in-arcs (2 words each), padded to an even count, then the 64-bit digest
__host__ __device__ __forceinline__ unsigned long long azb_ckpt_data_words(uint32_t WS, uint32_t W, uint32_t nn, uint32_t nblk,
                                                                           uint32_t intop) {
    const unsigned long long n = (unsigned long long)WS + (unsigned long long)nn * (16u + W) +
                                 2ull * (nblk > AZB_BLK_PAD ? nblk - AZB_BLK_PAD : 0u) + 2ull * intop;
    return (n + 1ull) & ~1ull;
}

__host__ __device__ __forceinline__ unsigned long long azb_ckpt_term(unsigned long long w, unsigned long long i) {
    return azb_mix64(w ^ (i * AZB_CKPT_K));
}

#ifdef __CUDACC__
#define AZB_CKPT_THREADS 256
#define AZB_CKPT_SLICE_BYTES 65536u  // a CTA's share of a record: records are cut into up to 64 slices of this size

// sum of the digest terms of 64-bit words [j0, j1) of w over the CTA, added to *acc (a sum mod 2^64: any order, any
// split of the words over CTAs gives the same total)
__device__ __forceinline__ void ckpt_digest_part(const unsigned long long *w, unsigned long long j0, unsigned long long j1,
                                                 unsigned long long *acc) {
    __shared__ unsigned long long red[AZB_CKPT_THREADS / 32];
    unsigned long long s = 0ull;
#pragma unroll 4
    for (unsigned long long j = j0 + threadIdx.x; j < j1; j += AZB_CKPT_THREADS) s += azb_ckpt_term(w[j], j);
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) s += shfl_xor_u64(s, m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < AZB_CKPT_THREADS / 32; ++k) s += red[k];
        atomicAdd(acc, s);
    }
}

// the five sections of a record (walker, nodes, keys, blocks, overflow in-arcs) as (arena pointer, start word, words)
struct CkptSections {
    uint32_t *p[5];
    unsigned long long a[6];  // a[k] = first record word of section k; a[5] = end of the data before the pad word
};
__device__ __forceinline__ CkptSections ckpt_sections(const AzbLayout &L, uint32_t t, uint32_t nn, uint32_t nblk, uint32_t intop) {
    CkptSections c;
    c.p[0] = L.walker + (size_t)t * L.WS;
    c.p[1] = reinterpret_cast<uint32_t *>(L.node + (size_t)t * L.cap_nodes * 4);
    c.p[2] = L.key + (size_t)t * L.cap_nodes * L.W;
    c.p[3] = reinterpret_cast<uint32_t *>(L.blk + (size_t)t * L.cap_blk + AZB_BLK_PAD);
    c.p[4] = reinterpret_cast<uint32_t *>(L.inl + (size_t)t * L.cap_in);
    c.a[0] = 0ull;
    c.a[1] = L.WS;
    c.a[2] = c.a[1] + 16ull * nn;
    c.a[3] = c.a[2] + (unsigned long long)nn * L.W;
    c.a[4] = c.a[3] + 2ull * (nblk - AZB_BLK_PAD);
    c.a[5] = c.a[4] + 2ull * intop;
    return c;
}

// this CTA's slice [lo, hi) of a record's nd data words (even bounds, so that it holds whole 64-bit words)
__device__ __forceinline__ void ckpt_slice(unsigned long long nd, unsigned long long &lo, unsigned long long &hi) {
    const unsigned long long per = 2ull * ((nd / 2ull + gridDim.y - 1u) / gridDim.y);
    lo = min(nd, per * blockIdx.y);
    hi = min(nd, lo + per);
}

// len[t] = record bytes of tree t; len[B] = 0 (the scan's last entry is then the total)
__global__ void __launch_bounds__(256) azb_ckpt_size_kernel(const AzbLayout L, unsigned long long *__restrict__ len) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > L.B) return;
    if (t == L.B) {
        len[t] = 0ull;
        return;
    }
    const uint32_t *wk = L.walker + (size_t)t * L.WS;
    len[t] = 4ull * (azb_ckpt_data_words(L.WS, L.W, wk[WK_NNODES], wk[WK_NBLK], wk[WK_INTOP]) + 2ull);
}

// grid (t1 - t0, slices): CTA (x, y) gathers slice y of tree t0 + x's record into `out`, which holds the blob's tree
// bytes from offset `base` on, and adds the slice's digest terms to acc[t]
__global__ void __launch_bounds__(AZB_CKPT_THREADS) azb_ckpt_pack_kernel(const AzbLayout L, const unsigned long long *__restrict__ off,
                                                                         uint32_t t0, unsigned long long base, uint32_t *__restrict__ out,
                                                                         unsigned long long *acc) {
    const uint32_t t = t0 + blockIdx.x;
    const uint32_t *wk = L.walker + (size_t)t * L.WS;
    const uint32_t nn = wk[WK_NNODES], nblk = wk[WK_NBLK], intop = wk[WK_INTOP];
    const unsigned long long nd = azb_ckpt_data_words(L.WS, L.W, nn, nblk, intop);
    unsigned long long lo, hi;
    ckpt_slice(nd, lo, hi);
    uint32_t *rec = out + (off[t] - base) / 4u;
    const CkptSections c = ckpt_sections(L, t, nn, nblk, intop);
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const unsigned long long s0 = max(lo, c.a[k]), s1 = min(hi, c.a[k + 1]);
        const uint32_t *src = c.p[k] - c.a[k];
#pragma unroll 4
        for (unsigned long long i = s0 + threadIdx.x; i < s1; i += AZB_CKPT_THREADS) rec[i] = src[i];
    }
    if (threadIdx.x == 0 && c.a[5] < nd && c.a[5] >= lo && c.a[5] < hi) rec[c.a[5]] = 0u;  // the pad word
    __syncthreads();
    ckpt_digest_part(reinterpret_cast<const unsigned long long *>(rec), lo / 2u, hi / 2u, acc + t);
}

// the digest word of every record of trees [t0, t1)
__global__ void __launch_bounds__(256) azb_ckpt_pack_finish_kernel(const AzbLayout L, const unsigned long long *__restrict__ off,
                                                                   uint32_t t0, uint32_t t1, unsigned long long base, uint32_t *__restrict__ out,
                                                                   const unsigned long long *__restrict__ acc) {
    const uint32_t t = t0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= t1) return;
    const uint32_t *wk = L.walker + (size_t)t * L.WS;
    const unsigned long long nd = azb_ckpt_data_words(L.WS, L.W, wk[WK_NNODES], wk[WK_NBLK], wk[WK_INTOP]);
    *reinterpret_cast<unsigned long long *>(out + (off[t] - base) / 4u + nd) = azb_mix64(acc[t] ^ (nd / 2u));
}

// record i of a blob chunk (offsets relative to its tree section, `in` = its bytes from `base` on): 0 if its length
// agrees with its walker header and it fits the handle, 1 if it is corrupt, 2 if it exceeds the capacities
__device__ __forceinline__ uint32_t ckpt_check_record(const AzbLayout &L, const unsigned long long *off, uint32_t i, unsigned long long base,
                                                      const uint32_t *in, uint32_t &nn, uint32_t &nblk, uint32_t &intop,
                                                      unsigned long long &nd) {
    const unsigned long long bytes = off[i + 1] - off[i];
    if (bytes % 8u || bytes < 4ull * (L.WS + 2u)) return 1u;
    const uint32_t *rec = in + (off[i] - base) / 4u;
    nn = rec[WK_NNODES];
    nblk = rec[WK_NBLK];
    intop = rec[WK_INTOP];
    nd = azb_ckpt_data_words(L.WS, L.W, nn, nblk, intop);
    if (nblk < AZB_BLK_PAD || nd != bytes / 4u - 2u) return 1u;
    if (nn > L.cap_nodes || nblk > L.cap_blk || intop > L.cap_in) return 2u;
    return 0u;
}

// grid (i1 - i0, slices): CTA (x, y) scatters slice y of record i0 + x into the handle's tree local0 + i0 + x and adds
// its digest terms to acc[i]; bad[0] / bad[1] = lowest global root whose record is corrupt / exceeds the capacities
__global__ void __launch_bounds__(AZB_CKPT_THREADS) azb_ckpt_unpack_kernel(const AzbLayout L, const unsigned long long *__restrict__ off,
                                                                           uint32_t i0, unsigned long long base, const uint32_t *__restrict__ in,
                                                                           uint32_t local0, unsigned long long gfirst, unsigned long long *acc,
                                                                           unsigned long long *bad) {
    const uint32_t i = i0 + blockIdx.x;
    uint32_t nn = 0, nblk = 0, intop = 0;
    unsigned long long nd = 0;
    const uint32_t why = ckpt_check_record(L, off, i, base, in, nn, nblk, intop, nd);
    if (why) {
        if (blockIdx.y == 0 && threadIdx.x == 0) atomicMin(bad + (why - 1u), gfirst + i);
        return;
    }
    unsigned long long lo, hi;
    ckpt_slice(nd, lo, hi);
    const uint32_t *rec = in + (off[i] - base) / 4u;
    const CkptSections c = ckpt_sections(L, local0 + i, nn, nblk, intop);
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const unsigned long long s0 = max(lo, c.a[k]), s1 = min(hi, c.a[k + 1]);
        uint32_t *dst = c.p[k] - c.a[k];
#pragma unroll 4
        for (unsigned long long j = s0 + threadIdx.x; j < s1; j += AZB_CKPT_THREADS) dst[j] = rec[j];
    }
    ckpt_digest_part(reinterpret_cast<const unsigned long long *>(rec), lo / 2u, hi / 2u, acc + i);
}

// the digest of every well-formed record of [i0, i1) against its digest word
__global__ void __launch_bounds__(256) azb_ckpt_unpack_finish_kernel(const AzbLayout L, const unsigned long long *__restrict__ off,
                                                                     uint32_t i0, uint32_t i1, unsigned long long base,
                                                                     const uint32_t *__restrict__ in, unsigned long long gfirst,
                                                                     const unsigned long long *__restrict__ acc, unsigned long long *bad) {
    const uint32_t i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i1) return;
    uint32_t nn, nblk, intop;
    unsigned long long nd;
    if (ckpt_check_record(L, off, i, base, in, nn, nblk, intop, nd)) return;  // reported by the unpack kernel
    const unsigned long long d = *reinterpret_cast<const unsigned long long *>(in + (off[i] - base) / 4u + nd);
    if (azb_mix64(acc[i] ^ (nd / 2u)) != d) atomicMin(bad, gfirst + i);
}

// the transposition table of every tree from its keys, nodes in index order; a key found twice (a record that passed its
// digest but repeats a node) sets bad[0] like a corrupt record
template <bool WIDE>
__global__ void __launch_bounds__(AZB_CKPT_WARPS * 32) azb_ckpt_hash_kernel(const AzbLayout L, unsigned long long *bad) {
    const int lane = threadIdx.x & 31;
    const uint32_t t = blockIdx.x * AZB_CKPT_WARPS + (threadIdx.x >> 5);
    if (t >= L.B) return;
    uint32_t *hash = L.hash + (size_t)t * L.cap_hash;
    const uint32_t *key = L.key + (size_t)t * L.cap_nodes * L.W;
#pragma unroll 4
    for (uint32_t s = lane; s < L.cap_hash; s += 32) hash[s] = 0u;
    __syncwarp();
    const uint32_t nn = L.walker[(size_t)t * L.WS + WK_NNODES];
#pragma unroll 1
    for (uint32_t i = 0; i < nn; ++i) {
        const uint32_t k0 = (uint32_t)lane < L.W ? key[(size_t)i * L.W + lane] : 0u;
        const uint32_t k1 = WIDE && (uint32_t)lane + 32 < L.W ? key[(size_t)i * L.W + lane + 32] : 0u;
        const uint32_t hv = key_hash(k0, k1, lane, L.W);
        uint32_t slot;
        if (hash_probe<WIDE>(L, hash, key, k0, k1, lane, hv, slot) >= 0) {
            if (lane == 0) atomicMin(bad, L.first_root + t);
            return;
        }
        if (lane == 0) hash_insert(hash, slot, i, hv);
        __syncwarp();
    }
}
#endif
