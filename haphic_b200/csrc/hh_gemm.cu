// Dense-block pre-expansion on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
// What it computes (scripts/HapHiC_cluster.py:2144-2149, dense mode 2035 / 2149): the one-off pre-expansion
//     M1 = M0 . M0,   M0 = normalize(link_matrix, 'l1', axis=0)
// for the part of the product that is a true GEMM.  With C the symmetric link matrix and s its column sums,
//     M1[r, c] = ( sum_k C[r, k] * M0[c, k] ) / s[c]          (C[k, c] = C[c, k],  M0[c, k] = C[c, k] / s[k])
// so S[r, c] = sum_k C[r, k] * M0[c, k] is a "TN" GEMM of two row-major (K-major) n x n operands and S is symmetric:
// only tiles on or above the diagonal are computed; the epilogue writes M1[r, c] = S / s[c] and the mirror image
// M1[c, r] = S / s[r].
//
// Precision.  The reference multiplies fp32 by fp32.  Tensor cores take bf16, so each operand is split into bf16
// "planes" whose sum is the fp32 value EXACTLY:
//   A = C      integer link counts: min(count, clip) in one plane, the excess as a sparse correction; anything else three;
//   B = M0     three planes (8 + 8 + 8 significant bits).
// A bf16 x bf16 product is exact in fp32, so the passes (plane_a, plane_b) below reproduce the fp32 product up to
// dropped terms of relative size 2^-24.  The accumulation inside the tensor core is not IEEE round-to-nearest, so a
// tile's K range is cut into chunks: each chunk accumulates in TMEM, is drained by the epilogue warps and added to fp32
// REGISTER accumulators with round-to-nearest (HH_GEMM_CHUNK k-blocks per chunk).
//
// Kernel shape (one persistent CTA pair per two SMs, cta_group::2):
//   tile 256 x 256 (128 rows of A and 128 rows of B per CTA), BLOCK_K = 64 bf16 = one 128-byte swizzle atom;
//   warp 0   TMA producer: per k-block one 128x64 box per operand plane (cp.async.bulk.tensor, SWIZZLE_128B)
//            into a ring of shared-memory stages, completion on the LEADER CTA's mbarrier;
//   warp 1   allocates TMEM; in the leader CTA one thread issues tcgen05.mma (M=256, N=256, K=16) for every pass and
//            commits to the stage's "empty" barrier (multicast to both CTAs) and to the chunk's "full" barrier;
//   warps 2-9  epilogue: tcgen05.ld the chunk (32 lanes x 128 columns per warp), add into registers, release the TMEM
//            buffer; after the last chunk scale and store the tile and its mirror image.
// HH_GEMM_CG=1 selects a single-CTA variant (tile 128 x 128, cta_group::1) with the same shared-memory layout.
#include "hh_common.cuh"
#include "hh_internal.cuh"
#include "hh_gemm.cuh"
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <algorithm>

// ---------------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t hg_cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void hg_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t hg_mapa(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void hg_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void hg_fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void hg_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void hg_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hg_mbar_arrive_local(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void hg_mbar_arrive_cluster(uint32_t remote_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}

template <int CG>
__device__ __forceinline__ void hg_tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t mbar, int c0, int c1, int c2) {
    if (CG == 2) {
        asm volatile(
            "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
            "l"(tm), "r"(mbar), "r"(c0), "r"(c1), "r"(c2)
            : "memory");
    } else {
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
                     "l"(tm), "r"(mbar), "r"(c0), "r"(c1), "r"(c2)
                     : "memory");
    }
}
__device__ __forceinline__ void hg_prefetch_tmap(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}

template <int CG>
__device__ __forceinline__ void hg_tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    if (CG == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
}
template <int CG>
__device__ __forceinline__ void hg_tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void hg_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void hg_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem]^T, bf16 operands, fp32 accumulator
template <int CG>
__device__ __forceinline__ void hg_umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (CG == 2) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// all MMAs issued so far by this thread -> arrive on an mbarrier when they have completed (both CTAs of the pair)
template <int CG>
__device__ __forceinline__ void hg_umma_commit(uint32_t bar) {
    if (CG == 2) {
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                     "h"((uint16_t)3)
                     : "memory");
    } else {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    }
}
// 32 lanes x 32 consecutive columns of TMEM -> 32 registers per thread (lane = TMEM lane, register = column)
__device__ __forceinline__ void hg_tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void hg_tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor of a K-major tile stored as [rows][64 bf16] with the 128-byte swizzle TMA applies:
// 8-row groups 1024 bytes apart (SBO), version 1 (Blackwell), layout SWIZZLE_128B.  The start address moves by 32 bytes
// per K = 16 step inside the swizzle atom.
__device__ __forceinline__ uint64_t hg_make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)1 << 16;               // leading byte offset: unused for swizzled K-major layouts
    d |= (uint64_t)(1024 >> 4) << 32;     // stride byte offset
    d |= (uint64_t)1 << 46;               // descriptor version
    d |= (uint64_t)2 << 61;               // SWIZZLE_128B
    return d;
}

// ---------------------------------------------------------------------------------------------------------------------
// the GEMM kernel
// ---------------------------------------------------------------------------------------------------------------------
#define HG_THREADS 320
#define HG_PLANE_BYTES 16384        // 128 rows x 64 bf16
#define HG_MAX_STAGES 4

struct hh_gemm_args {
    const hh_gemm_item* items;
    int n_items;
    int n;                 // matrix dimension
    int na, nb;            // planes of A / of B per k-block (1..3)
    int npass;
    int pa[8], pb[8];      // pass list: plane of A, plane of B
    int chunk_kb;          // k-blocks accumulated in TMEM before they are drained into registers
    int stages;
    float* m1;             // dense column-major [ld x (col_hi - col_lo)]
    long long ld;
    int col_lo, col_hi;
    const float* inv_s;    // 1 / column sum
    float out_scale;       // applied instead when inv_s == NULL
    int accumulate;        // 1: the epilogue adds to what the output holds (K range processed in several launches)
    uint32_t idesc_fmt;    // operand format bits of the instruction descriptor (bit 7: A is bf16, bit 10: B is bf16)
};

template <int CG>
__global__ void __launch_bounds__(HG_THREADS, 1)
hh_k_syrk(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const hh_gemm_args a) {
    constexpr int BN = 128 * CG;              // tile columns (= TMEM columns per accumulator buffer)
    constexpr int CW = BN / 2;                // columns per epilogue warp
    constexpr uint32_t TMEM_COLS = 2 * BN;    // two accumulator buffers
    // kind::f16 descriptor: fp32 accumulator (bit 4), A / B format (bits 7-9 / 10-12: 0 = f16, 1 = bf16), both K-major, N >> 3, M >> 4
    const uint32_t IDESC = (1u << 4) | a.idesc_fmt | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((128 * CG) >> 4) << 24);

    extern __shared__ uint8_t hg_smem_raw[];
    __shared__ __align__(8) uint64_t s_full[HG_MAX_STAGES];
    __shared__ __align__(8) uint64_t s_empty[HG_MAX_STAGES];
    __shared__ __align__(8) uint64_t s_tfull[2];
    __shared__ __align__(8) uint64_t s_tempty[2];
    __shared__ uint32_t s_tmem;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = (CG == 2) ? hg_cluster_ctarank() : 0u;
    const int pair = (CG == 2) ? (blockIdx.x >> 1) : blockIdx.x;
    const int npairs = (CG == 2) ? (gridDim.x >> 1) : gridDim.x;
    const uint32_t smem_base = (hg_smem_u32(hg_smem_raw) + 1023u) & ~1023u;
    const uint32_t stage_bytes = (uint32_t)(a.na + a.nb) * HG_PLANE_BYTES;
    const int S = a.stages;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            hg_mbar_init(hg_smem_u32(&s_full[s]), 1);
            hg_mbar_init(hg_smem_u32(&s_empty[s]), 1);
        }
        for (int b = 0; b < 2; ++b) {
            hg_mbar_init(hg_smem_u32(&s_tfull[b]), 1);
            hg_mbar_init(hg_smem_u32(&s_tempty[b]), 8 * CG);     // every epilogue warp of the pair
        }
        hg_fence_barrier_init();
        hg_prefetch_tmap(&tmA);
        hg_prefetch_tmap(&tmB);
    }
    __syncwarp();
    if (warp == 1) hg_tmem_alloc<CG>(hg_smem_u32(&s_tmem), TMEM_COLS);
    hg_tc_fence_before();
    if (CG == 2) hg_cluster_sync();
    else __syncthreads();
    hg_tc_fence_after();
    const uint32_t tmem_base = s_tmem;

    if (warp == 0) {
        // ------------------------------------------------------------------------------------------- TMA producer
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            const uint32_t full0 = (CG == 2) ? hg_mapa(hg_smem_u32(&s_full[0]), 0) : hg_smem_u32(&s_full[0]);
            for (int it = pair; it < a.n_items; it += npairs) {
                const hh_gemm_item w = a.items[it];
                const int rowA = w.m0 + (int)rank * 128;
                const int rowB = w.n0 + (int)rank * 128;
                for (int seg = 0; seg < 2; ++seg) {
                    for (int kb = w.kb_lo[seg]; kb < w.kb_hi[seg]; ++kb) {
                        hg_mbar_wait(hg_smem_u32(&s_empty[s]), ph ^ 1u);
                        if (rank == 0) hg_mbar_expect_tx(hg_smem_u32(&s_full[s]), stage_bytes * CG);
                        const uint32_t dst = smem_base + (uint32_t)s * stage_bytes;
                        const uint32_t bar = full0 + (uint32_t)s * 8u;
                        for (int p = 0; p < a.na; ++p) hg_tma_load_3d<CG>(dst + (uint32_t)p * HG_PLANE_BYTES, &tmA, bar, kb * 64, rowA, p);
                        for (int p = 0; p < a.nb; ++p)
                            hg_tma_load_3d<CG>(dst + (uint32_t)(a.na + p) * HG_PLANE_BYTES, &tmB, bar, kb * 64, rowB, p);
                        if (++s == S) {
                            s = 0;
                            ph ^= 1u;
                        }
                    }
                }
            }
        }
        __syncwarp();     // the other lanes wait here: the teardown barrier is .aligned
    } else if (warp == 1) {
        // ------------------------------------------------------------------------------------------- MMA issuer
        if (rank == 0 && lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            uint32_t g = 0;     // running chunk counter: TMEM buffer g & 1, phase (g >> 1) & 1
            for (int it = pair; it < a.n_items; it += npairs) {
                const hh_gemm_item w = a.items[it];
                int in_chunk = 0;
                const int total = (w.kb_hi[0] - w.kb_lo[0]) + (w.kb_hi[1] - w.kb_lo[1]);
                for (int t = 0; t < total; ++t) {
                    const uint32_t buf = g & 1u;
                    if (in_chunk == 0) {
                        hg_mbar_wait(hg_smem_u32(&s_tempty[buf]), ((g >> 1) & 1u) ^ 1u);
                        hg_tc_fence_after();
                    }
                    hg_mbar_wait(hg_smem_u32(&s_full[s]), ph);
                    hg_tc_fence_after();
                    const uint32_t st = smem_base + (uint32_t)s * stage_bytes;
                    const uint32_t d = tmem_base + buf * (uint32_t)BN;
                    uint32_t acc = in_chunk ? 1u : 0u;      // 0: the MMA overwrites the accumulator
                    for (int p = 0; p < a.npass; ++p) {
                        const uint64_t ad = hg_make_desc(st + (uint32_t)a.pa[p] * HG_PLANE_BYTES);
                        const uint64_t bd = hg_make_desc(st + (uint32_t)(a.na + a.pb[p]) * HG_PLANE_BYTES);
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            hg_umma<CG>(d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), IDESC, acc);
                            acc = 1u;
                        }
                    }
                    hg_umma_commit<CG>(hg_smem_u32(&s_empty[s]));      // the stage is free once these MMAs have read it
                    if (++s == S) {
                        s = 0;
                        ph ^= 1u;
                    }
                    if (++in_chunk == a.chunk_kb || t + 1 == total) {
                        hg_umma_commit<CG>(hg_smem_u32(&s_tfull[buf]));    // chunk complete -> epilogue
                        in_chunk = 0;
                        ++g;
                    }
                }
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------------------------------- epilogue
        const int e = warp - 2;
        const int quarter = warp & 3;          // TMEM lanes this warp may touch: 32 * (warp id % 4)
        const int half = e >> 2;               // column half of the tile
        const uint32_t lane_addr = ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * CW);
        const uint32_t tempty0 = (CG == 2) ? hg_mapa(hg_smem_u32(&s_tempty[0]), 0) : hg_smem_u32(&s_tempty[0]);
        uint32_t g = 0;
        float acc[CW];
        for (int it = pair; it < a.n_items; it += npairs) {
            const hh_gemm_item w = a.items[it];
            const int total = (w.kb_hi[0] - w.kb_lo[0]) + (w.kb_hi[1] - w.kb_lo[1]);
            const int nchunks = (total + a.chunk_kb - 1) / a.chunk_kb;
#pragma unroll
            for (int j = 0; j < CW; ++j) acc[j] = 0.f;
            for (int ch = 0; ch < nchunks; ++ch, ++g) {
                const uint32_t buf = g & 1u;
                hg_mbar_wait(hg_smem_u32(&s_tfull[buf]), (g >> 1) & 1u);
                hg_tc_fence_after();
                const uint32_t tb = tmem_base + buf * (uint32_t)BN + lane_addr;
#pragma unroll
                for (int q = 0; q < CW / 32; ++q) {
                    uint32_t v[32];
                    hg_tmem_ld32(tb + (uint32_t)(q * 32), v);
                    hg_tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[q * 32 + j] = __fadd_rn(acc[q * 32 + j], __uint_as_float(v[j]));
                }
                hg_tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CG == 2) hg_mbar_arrive_cluster(tempty0 + buf * 8u);
                    else hg_mbar_arrive_local(tempty0 + buf * 8u);
                }
            }
            // ---- scale and store: out[r, c] = D * scale[c]; mirror image out[c, r] = D * scale[r]
            const int r = w.m0 + (int)rank * 128 + quarter * 32 + lane;
            const int c0 = w.n0 + half * CW;
            if (r < w.m_end) {
                if (w.flags & HH_GEMM_DIRECT) {
                    float* __restrict__ dst = a.m1 + (ptrdiff_t)(r - w.out_row0);
#pragma unroll
                    for (int j = 0; j < CW; ++j) {
                        const int c = c0 + j;
                        if (c < w.n_end && c >= a.col_lo && c < a.col_hi) {
                            float* __restrict__ o = dst + (size_t)(c - a.col_lo) * (size_t)a.ld;
                            const float v = a.inv_s ? acc[j] * __ldg(a.inv_s + c) : acc[j] * a.out_scale;
                            *o = a.accumulate ? __fadd_rn(*o, v) : v;
                        }
                    }
                }
                if ((w.flags & HH_GEMM_MIRROR) && r >= a.col_lo && r < a.col_hi) {
                    const float sr = a.inv_s ? __ldg(a.inv_s + r) : a.out_scale;
                    float* __restrict__ dst = a.m1 + (size_t)(r - a.col_lo) * (size_t)a.ld - (ptrdiff_t)w.out_row0;
#pragma unroll
                    for (int j = 0; j < CW; j += 4) {
                        const int c = c0 + j;
                        if (c + 3 < w.n_end && w.out_row0 == 0) {
                            float4 v = make_float4(acc[j] * sr, acc[j + 1] * sr, acc[j + 2] * sr, acc[j + 3] * sr);
                            if (a.accumulate) {
                                const float4 old = *reinterpret_cast<const float4*>(dst + c);
                                v = make_float4(__fadd_rn(old.x, v.x), __fadd_rn(old.y, v.y), __fadd_rn(old.z, v.z), __fadd_rn(old.w, v.w));
                            }
                            *reinterpret_cast<float4*>(dst + c) = v;
                        } else {
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                if (c + q < w.n_end) dst[c + q] = a.accumulate ? __fadd_rn(dst[c + q], acc[j + q] * sr) : acc[j + q] * sr;
                        }
                    }
                }
            }
        }
    }

    // ---- teardown: every MMA has completed (the epilogues consumed the last chunk), free TMEM
    hg_tc_fence_before();
    if (CG == 2) hg_cluster_sync();
    else __syncthreads();
    hg_tc_fence_after();
    if (warp == 1) hg_tmem_dealloc<CG>(tmem_base, TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------------------------
// operand preparation: CSC of the symmetric link matrix -> dense row-major bf16 planes
// ---------------------------------------------------------------------------------------------------------------------
// column sums in fp64 (sklearn normalize accumulates in double, 2144) and their fp32 reciprocals
__global__ void hh_k_gemm_colsum(const int64_t* __restrict__ colptr, const float* __restrict__ val, int n, double* __restrict__ s,
                                 float* __restrict__ inv_s, int* __restrict__ flags) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const int lane = threadIdx.x & 31;
    double t = 0.0;
    for (int64_t p = colptr[c] + lane; p < colptr[c + 1]; p += 32) t += fabs((double)val[p]);
    t = hh_warp_sum(t);
    if (lane == 0) {
        s[c] = t;
        inv_s[c] = (t != 0.0) ? (float)(1.0 / t) : 1.f;
        if (t >= 8388608.0) atomicOr(flags, 4);          // 2^-e_k of the scaled f16 encoding would leave the subnormal range
    }
}

// flags[0] |= 1 if some value is not an integer in [0, 65536); |= 2 if some value exceeds 256; |= 8 if some value exceeds 2048
__global__ void hh_k_gemm_valstats(const float* __restrict__ val, int64_t nnz, int* __restrict__ flags) {
    int f = 0;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x) {
        const float v = val[p];
        if (!(v >= 0.f && v < 65536.f && v == floorf(v))) f |= 1;
        if (v > 256.f) f |= 2;
        if (v > 2048.f) f |= 8;
    }
    f = __reduce_or_sync(HH_FULL_MASK, f);
    if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

__device__ __forceinline__ void hg_split3(float x, unsigned short& h1, unsigned short& h2, unsigned short& h3) {
    const uint32_t b1 = __float_as_uint(x) & 0xFFFF0000u;          // bf16 by truncation: the remainder stays exact
    const float r1 = x - __uint_as_float(b1);
    const uint32_t b2 = __float_as_uint(r1) & 0xFFFF0000u;
    const float r2 = r1 - __uint_as_float(b2);
    h1 = (unsigned short)(b1 >> 16);
    h2 = (unsigned short)(b2 >> 16);
    h3 = (unsigned short)(__float_as_uint(r2) >> 16);              // at most 8 significant bits are left
}

// One CTA per column c of the CSC = row c of both operands.  Two encodings of  S[r, c] = sum_k C[r, k] * M0[c, k]:
//   exact bf16   A[c, k] = min(C[c, k], clip) in na planes,  B[c, k] = fp32(A[c, k] / s[k]) in three bf16 planes (8 + 8 + 8 bits);
//   scaled f16   A[c, k] = min(C[c, k], clip) * 2^-e_k  (ONE plane: an integer times a power of two is exact in bf16 up to 256 and
//                in f16 up to 2048, subnormals included while e_k <= 24),
//                B[c, k] = fp32(A / s[k]) * 2^e_k in (count, 2 count]  as TWO f16 planes hi + lo = 22 significant bits, round to
//                nearest: every product is within 2^-23 relative of the fp32 product, in two passes instead of three.
//                2^e_k is the power of two above the column sum s[k]: it cancels inside every product.
// The row is assembled in shared memory (segments of HG_SEG columns, up to three planes at a time) and written with
// coalesced 16-byte stores: every element of the padded row is written exactly once, so the planes need no memset and no
// read-modify-write of partially written sectors.
#define HG_SEG 32768
__global__ void __launch_bounds__(1024)
hh_k_gemm_densify(const int64_t* __restrict__ colptr, const int32_t* __restrict__ row, const float* __restrict__ val, int n,
                  const double* __restrict__ s, unsigned short* __restrict__ A, int na, unsigned short* __restrict__ B, int nb, long long ldk,
                  long long plane, float clip, int scaled, int a_f16, long long k0) {
    // the planes hold the K range [k0, k0 + ldk) of the operands (the whole range unless the product is cut along K)
    extern __shared__ __align__(16) unsigned short hg_row[];        // [3][HG_SEG]
    const int c = blockIdx.x;
    const int64_t p0 = colptr[c], p1 = colptr[c + 1];
    for (int group = 0; group < 2; ++group) {                       // 0: planes of A, 1: planes of B
        const int np = group ? nb : na;
        unsigned short* __restrict__ out = (group ? B : A) + (size_t)c * (size_t)ldk;
        for (long long seg0 = k0; seg0 < k0 + ldk; seg0 += HG_SEG) {
            const int seg_n = (int)((k0 + ldk - seg0 < HG_SEG) ? (k0 + ldk - seg0) : HG_SEG);      // multiple of 64
            uint4* z = reinterpret_cast<uint4*>(hg_row);
            for (int q = threadIdx.x; q < 3 * HG_SEG / 8; q += blockDim.x) z[q] = make_uint4(0u, 0u, 0u, 0u);
            __syncthreads();
            for (int64_t p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
                const long long k = row[p];
                if (k < seg0 || k >= seg0 + seg_n) continue;
                const float v = fminf(val[p], clip);      // counts above `clip` are finished by the caller's sparse correction
                const double sk = s[k];
                unsigned short h1 = 0, h2 = 0, h3 = 0;
                if (!scaled) {
                    float x = v;
                    if (group) x = (sk != 0.0) ? (float)((double)v / sk) : v;
                    hg_split3(x, h1, h2, h3);
                } else {
                    // s[k] in [2^(e-1), 2^e), 0 <= e <= 24: the exponent field of the double; 2^e and 2^-e as floats
                    const int e = (sk != 0.0) ? (int)((__double2hiint(sk) >> 20) & 0x7ff) - 1022 : 0;
                    if (!group) {
                        const float xa = v * __int_as_float((127 - e) << 23);
                        h1 = a_f16 ? __half_as_ushort(__float2half_rn(xa)) : (unsigned short)(__float_as_uint(xa) >> 16);
                    } else {
                        const float x = (sk != 0.0) ? (float)((double)v / sk) : v;
                        const float xs = x * __int_as_float((127 + e) << 23);
                        const __half hi = __float2half_rn(xs);
                        const __half lo = __float2half_rn(xs - __half2float(hi));
                        h1 = __half_as_ushort(hi);
                        h2 = __half_as_ushort(lo);
                    }
                }
                const int kk = (int)(k - seg0);
                hg_row[kk] = h1;
                if (np > 1) hg_row[HG_SEG + kk] = h2;
                if (np > 2) hg_row[2 * HG_SEG + kk] = h3;
            }
            __syncthreads();
            for (int pl = 0; pl < np; ++pl) {
                const uint4* src = reinterpret_cast<const uint4*>(hg_row + (size_t)pl * HG_SEG);
                uint4* dst = reinterpret_cast<uint4*>(out + (size_t)pl * (size_t)plane + (size_t)(seg0 - k0));
                for (int q = threadIdx.x; q < seg_n / 8; q += blockDim.x) dst[q] = src[q];
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
typedef CUresult (*hg_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int hg_encode(CUtensorMap* tm, void* base, int rows, int kdim, long long ldk, long long plane_elems, int planes, int fmt) {
    static hg_encode_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        HH_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        HH_REQUIRE(p != nullptr && q == cudaDriverEntryPointSuccess, HH_ERR_CUDA, "hh_gemm: the driver does not export cuTensorMapEncodeTiled");
        fn = reinterpret_cast<hg_encode_fn>(p);
    }
    const cuuint64_t dims[3] = {(cuuint64_t)kdim, (cuuint64_t)rows, (cuuint64_t)planes};
    const cuuint64_t strides[2] = {(cuuint64_t)ldk * 2ull, (cuuint64_t)plane_elems * 2ull};
    const cuuint32_t box[3] = {64u, 128u, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = fn(tm, fmt == HH_GEMM_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HH_REQUIRE(r == CUDA_SUCCESS, HH_ERR_CUDA, "hh_gemm: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return HH_OK;
}

static int hg_env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

template <int CG>
static int hg_launch(hh_ctx* ctx, const CUtensorMap& tmA, const CUtensorMap& tmB, const hh_gemm_args& a, size_t smem) {
    auto kern = hh_k_syrk<CG>;
    HH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    int pairs = ctx->sm_count / CG;
    if (pairs > a.n_items) pairs = a.n_items;
    if (pairs < 1) pairs = 1;
    cfg.gridDim = dim3((unsigned)(pairs * CG));
    cfg.blockDim = dim3(HG_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    HH_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, a));
    ctx->launches++;
    return HH_OK;
}

int hh_gemm_cta_group() { return hg_env_int("HH_GEMM_CG", 2) == 1 ? 1 : 2; }

int hh_gemm_run(hh_ctx* ctx, const hh_gemm_operand& A, const hh_gemm_operand& B, const hh_gemm_item* d_items, int n_items, int npass,
                const int* pa, const int* pb, int chunk_kb, float* out, long long ld, int col_lo, int col_hi, const float* scale,
                int* stages_out, float out_scale, int accumulate) {
    HH_REQUIRE(n_items >= 1 && npass >= 1 && npass <= 8, HH_ERR_ARG, "hh_gemm_run: bad work list");
    CUtensorMap tmA, tmB;
    HH_CHECK(hg_encode(&tmA, (void*)A.base, A.rows, A.kdim, A.ldk, A.plane, A.planes, A.fmt));
    HH_CHECK(hg_encode(&tmB, (void*)B.base, B.rows, B.kdim, B.ldk, B.plane, B.planes, B.fmt));
    hh_gemm_args a;
    memset(&a, 0, sizeof(a));
    a.items = d_items;
    a.n_items = n_items;
    a.na = A.planes;
    a.nb = B.planes;
    a.npass = npass;
    for (int p = 0; p < npass; ++p) {
        a.pa[p] = pa[p];
        a.pb[p] = pb[p];
    }
    a.chunk_kb = chunk_kb < 1 ? (1 << 30) : chunk_kb;           // 0 = accumulate the whole K range in TMEM
    const size_t stage_bytes = (size_t)(A.planes + B.planes) * HG_PLANE_BYTES;
    int stages = (int)((ctx->smem_optin - 2048) / stage_bytes);
    if (stages > HG_MAX_STAGES) stages = HG_MAX_STAGES;
    HH_REQUIRE(stages >= 2, HH_ERR_UNSUPPORTED, "hh_gemm: shared memory too small for two pipeline stages");
    a.stages = stages;
    if (stages_out) *stages_out = stages;
    a.m1 = out;
    a.ld = ld;
    a.col_lo = col_lo;
    a.col_hi = col_hi;
    a.inv_s = scale;
    a.out_scale = out_scale;
    a.accumulate = accumulate;
    a.idesc_fmt = (A.fmt == HH_GEMM_BF16 ? (1u << 7) : 0u) | (B.fmt == HH_GEMM_BF16 ? (1u << 10) : 0u);
    const size_t smem = (size_t)stages * stage_bytes + 1024;
    if (hh_gemm_cta_group() == 2) return hg_launch<2>(ctx, tmA, tmB, a, smem);
    return hg_launch<1>(ctx, tmA, tmB, a, smem);
}

static const int HG_P1[3][2] = {{0, 0}, {0, 1}, {0, 2}};
static const int HG_P3[6][2] = {{0, 0}, {0, 1}, {1, 0}, {0, 2}, {1, 1}, {2, 0}};

// pass list for `na` (1 or 3) planes of A against three planes of B: every product of relative size >= 2^-16 (na = 1: exact)
int hh_gemm_passes(int na, int* pa, int* pb) {
    const int(*pl)[2] = na == 1 ? HG_P1 : HG_P3;
    const int np = na == 1 ? 3 : 6;
    for (int p = 0; p < np; ++p) {
        pa[p] = pl[p][0];
        pb[p] = pl[p][1];
    }
    return np;
}

int hh_gemm_preexpand(hh_ctx* ctx, const hh_matrix* m, int col_lo, int col_hi, float* d_m1, long long ld, const hh_gemm_item* h_items,
                      int n_items, hh_gemm_stats* st) {
    const int n = m->n;
    HH_REQUIRE(n >= 1 && n_items >= 1, HH_ERR_ARG, "hh_gemm_preexpand: empty problem");
    const long long ldk = ((long long)n + 63) & ~63ll;       // row pitch in elements (128-byte multiple)
    const long long plane = ldk * (long long)n;
    double* d_s = nullptr;
    float* d_inv = nullptr;
    int* d_flags = nullptr;
    unsigned short *d_A = nullptr, *d_B = nullptr;
    hh_gemm_item* d_items = nullptr;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    int rc = [&]() -> int {
        for (int k = 0; k < 3; ++k) HH_CUDA(cudaEventCreate(&ev[k]));
        HH_CHECK(hh_dmalloc(&d_s, (size_t)n));
        HH_CHECK(hh_dmalloc(&d_inv, (size_t)n));
        HH_CHECK(hh_dmalloc(&d_flags, 1));
        HH_CUDA(cudaEventRecord(ev[0], ctx->stream));
        HH_CUDA(cudaMemsetAsync(d_flags, 0, sizeof(int), ctx->stream));
        HH_LAUNCH(ctx, hh_k_gemm_colsum, (n + 7) / 8, 256, 0, m->d_colptr, m->d_val, n, d_s, d_inv, d_flags);
        HH_LAUNCH(ctx, hh_k_gemm_valstats, ctx->sm_count * 8, 256, 0, m->d_val, m->nnz, d_flags);
        int flags = 0;
        HH_CUDA(cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        // Integer link counts (the usual case): the scaled encoding, one plane of min(count, clip) against two f16 planes of M0,
        // two passes, clip 2048; the excess over `clip` is the caller's sparse correction.  It needs column sums below 2^23 (the
        // scaled counts may be f16 subnormals, exact down to 2^-24).  Otherwise, or with HH_GEMM_FMT=bf16, the exact encoding:
        // one bf16 plane of min(count, 256) against three bf16 planes of M0, three passes.  (kind::f16 takes ONE format for both
        // operands: a bf16 count plane against f16 planes of M0 is an illegal instruction on sm_100a -- measured.)
        // Anything else (weights of --normalize_by_nlinks, allele-aware scaling): three exact bf16 planes each, six passes.
        const char* fmt_env = getenv("HH_GEMM_FMT");
        int enc = 2;                                             // 0 = exact bf16, 2 = scaled f16
        if (fmt_env && !strcmp(fmt_env, "bf16")) enc = 0;
        if (flags & (1 | 4)) enc = 0;
        const int na = (flags & 1) ? 3 : 1;
        const int nb = enc ? 2 : 3;
        const float clip = (flags & 1) ? 3.0e38f : (enc == 2 ? 2048.f : 256.f);
        const int fmt_a = enc == 2 ? HH_GEMM_F16 : HH_GEMM_BF16, fmt_b = enc ? HH_GEMM_F16 : HH_GEMM_BF16;
        // The K range is cut into equal chunks when the operand planes of the whole range would exceed ~36 GB (150k contigs:
        // 135 GB): planes of one chunk at a time, the epilogue of every chunk after the first adds to M1.  The cut depends on
        // n and the encoding only, so every rank of a sharded run cuts alike and M1 stays bit-identical for any world size.
        const double plane_bytes_all = (double)(na + nb) * (double)plane * 2.0;
        int kchunks = (int)(plane_bytes_all / 36.0e9) + 1;
        kchunks = hg_env_int("HH_GEMM_KCHUNKS", kchunks);
        if (kchunks < 1) kchunks = 1;
        const long long kw = ((((long long)n + kchunks - 1) / kchunks) + 63) & ~63ll;      // chunk width, multiple of 64
        kchunks = (int)(((long long)n + kw - 1) / kw);
        const long long plane_c = kw * (long long)n;
        HH_CHECK(hh_ws_alloc(ctx, &d_A, (size_t)plane_c * (size_t)na));
        HH_CHECK(hh_ws_alloc(ctx, &d_B, (size_t)plane_c * (size_t)nb));
        // rows [n, ld) of every M1 column stay zero
        HH_CUDA(cudaMemsetAsync(d_m1, 0, (size_t)ld * (size_t)(col_hi - col_lo) * sizeof(float), ctx->stream));
        HH_CHECK(hh_dmalloc(&d_items, (size_t)n_items));
        int pa[8], pb[8];
        int npass = hh_gemm_passes(na, pa, pb);
        if (enc) {                                               // (A, B hi), (A, B lo)
            npass = 2;
            pa[0] = pa[1] = 0;
            pb[0] = 0;
            pb[1] = 1;
        }
        // k-blocks accumulated in TMEM between two drains: the tensor core's accumulate truncates, so the bias grows with the
        // number of accumulations (4 MMAs per k-block and pass).
        // Measured at 50k contigs (one B200; GEMM time / max and mean relative error against the exact product), two f16 passes:
        //   chunk 2: 205 ms, 1.5e-6, -1.6e-8   4: 177 ms, 1.2e-6, -2.4e-8   8: 139 ms, 1.1e-6, -3.9e-8   16: 136 ms, 1.9e-6, -6.6e-8
        // every drain costs 0.5-2k clocks of tensor-pipe time, so longer chunks are faster -- but on dense inputs (every product
        // of similar size) the bias of 64 truncating accumulations reaches 2.5e-6.  Three k-blocks = 24 accumulations, the
        // same as three bf16 passes drained every second k-block, keeps every test input below 2e-6.
        // Giving the low-order pass (2^-11 of the result) the second TMEM buffer for the whole tile and chunking only the
        // high-order pass was measured bias-free (mean -1.4e-10) but, single-buffered, slower: 244 ms against 211 ms at
        // chunk 8 on the same device.
        const int chunk = hg_env_int("HH_GEMM_CHUNK", npass > 3 ? 1 : (npass == 3 ? 2 : 3));
        int stages = 0;
        float densify_ms = 0.f, gemm_ms = 0.f;
        const float stats_ms = 0.f;                              // column sums + value statistics: a fraction of a millisecond
        std::vector<hh_gemm_item> items_c(h_items, h_items + n_items);
        for (int kc = 0; kc < kchunks; ++kc) {
            const long long k0 = (long long)kc * kw;
            const long long k1 = std::min((long long)n, k0 + kw);
            HH_CUDA(cudaEventRecord(ev[0], ctx->stream));
            {
                auto kd = hh_k_gemm_densify;
                const size_t dsm = (size_t)3 * HG_SEG * sizeof(unsigned short);
                HH_CUDA(cudaFuncSetAttribute(kd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm));
                HH_LAUNCH(ctx, kd, n, 1024, dsm, m->d_colptr, m->d_row, m->d_val, n, d_s, d_A, na, d_B, nb, kw, plane_c, clip, enc ? 1 : 0,
                          enc == 2 ? 1 : 0, k0);
            }
            const int nkb_c = (int)((k1 - k0 + 63) / 64);
            for (auto& w : items_c) {
                w.kb_lo[0] = 0;
                w.kb_hi[0] = nkb_c;
            }
            HH_CUDA(cudaMemcpyAsync(d_items, items_c.data(), (size_t)n_items * sizeof(hh_gemm_item), cudaMemcpyHostToDevice, ctx->stream));
            hh_gemm_operand A = {d_A, na, n, (int)(k1 - k0), kw, plane_c, fmt_a};
            hh_gemm_operand B = {d_B, nb, n, (int)(k1 - k0), kw, plane_c, fmt_b};
            HH_CUDA(cudaEventRecord(ev[1], ctx->stream));
            HH_CHECK(hh_gemm_run(ctx, A, B, d_items, n_items, npass, pa, pb, chunk, d_m1, ld, col_lo, col_hi, d_inv, &stages, 1.0f, kc > 0 ? 1 : 0));
            HH_CUDA(cudaEventRecord(ev[2], ctx->stream));
            HH_CUDA(cudaStreamSynchronize(ctx->stream));         // items_c is rewritten for the next chunk
            float t0 = 0.f, t1 = 0.f;
            HH_CUDA(cudaEventElapsedTime(&t0, ev[0], ev[1]));
            HH_CUDA(cudaEventElapsedTime(&t1, ev[1], ev[2]));
            densify_ms += t0;
            gemm_ms += t1;
        }
        HH_CUDA(cudaEventRecord(ev[2], ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        if (st) {
            memset(st, 0, sizeof(*st));
            st->a_planes = na;
            st->clipped = (clip < 1.0e38f && (flags & (clip > 256.f ? 8 : 2))) ? 1 : 0;
            st->clip = clip;
            st->fmt_a = fmt_a;
            st->fmt_b = fmt_b;
            st->b_planes = nb;
            st->passes = npass;
            st->cta_group = hh_gemm_cta_group();
            st->stages = stages;
            st->chunk_kb = chunk < 1 ? (1 << 30) : chunk;
            st->densify_ms = densify_ms + stats_ms;
            st->gemm_ms = gemm_ms;
            st->k_chunks = kchunks;
            double kb = 0.0;
            for (int i = 0; i < n_items; ++i) kb += (double)((h_items[i].kb_hi[0] - h_items[i].kb_lo[0]) + (h_items[i].kb_hi[1] - h_items[i].kb_lo[1]));
            const double tile = 128.0 * hh_gemm_cta_group();
            st->flops = 2.0 * tile * tile * 64.0 * kb * (double)npass;
        }
        return HH_OK;
    }();
    hh_dfree(d_s);
    hh_dfree(d_inv);
    hh_dfree(d_flags);
    hh_ws_free(ctx, d_A);
    hh_ws_free(ctx, d_B);
    hh_dfree(d_items);
    for (int k = 0; k < 3; ++k)
        if (ev[k]) cudaEventDestroy(ev[k]);
    return rc;
}


// ---------------------------------------------------------------------------------------------------------------------
// block-diagonal products of the Markov-cluster iterations (hh_mcl.cu): operand planes of the component blocks
// ---------------------------------------------------------------------------------------------------------------------
// Bt[c, kk] = M[lo + kk, c] for the columns c of `list` (lo = first row of c's component): one CTA per column assembles the
// row of its planes in shared memory and writes all ldk elements (zeros beyond the component).  Two encodings:
//   three bf16 planes, the exact fp32 value (8 + 8 + 8 bits by truncation);
//   two f16 planes of M * 2^14, hi + lo = 22 significant bits (entries of a pruned column-stochastic iterate lie in
//   [pruning, 1]: scaled they are f16 normals for every pruning >= 2^-14; the product carries 2^28, removed in the epilogue).
#define HG_BLK_SHIFT 14
__global__ void __launch_bounds__(128)
hh_k_blk_densify(const int* __restrict__ len, const uint2* __restrict__ ent, int cap, const int* __restrict__ list, int nlist,
                 const int* __restrict__ comp_lo, const int* __restrict__ comp_hi, unsigned short* __restrict__ Bt, long long ldk,
                 long long plane, int f16) {
    extern __shared__ __align__(16) unsigned short hb_row[];        // [3][ldk]
    const int j = list[blockIdx.x];
    const int lo = comp_lo[j], width = comp_hi[j] - lo;
    uint4* z = reinterpret_cast<uint4*>(hb_row);
    for (int q = threadIdx.x; q < (int)(3 * ldk / 8); q += 128) z[q] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const int L = len[j];
    const uint2* __restrict__ e = ent + (size_t)j * (size_t)cap;
    for (int p = threadIdx.x; p < L; p += 128) {
        const uint2 t = e[p];
        const unsigned kk = t.x - (unsigned)lo;
        if (kk < (unsigned)width) {
            unsigned short h1, h2, h3 = 0;
            if (f16) {
                const float xs = ldexpf(__uint_as_float(t.y), HG_BLK_SHIFT);
                const __half hi = __float2half_rn(xs);
                h1 = __half_as_ushort(hi);
                h2 = __half_as_ushort(__float2half_rn(xs - __half2float(hi)));
            } else {
                hg_split3(__uint_as_float(t.y), h1, h2, h3);
            }
            hb_row[kk] = h1;
            hb_row[ldk + kk] = h2;
            hb_row[2 * ldk + kk] = h3;
        }
    }
    __syncthreads();
    for (int pl = 0; pl < (f16 ? 2 : 3); ++pl) {
        const uint4* src = reinterpret_cast<const uint4*>(hb_row + (size_t)pl * (size_t)ldk);
        uint4* dst = reinterpret_cast<uint4*>(Bt + (size_t)pl * (size_t)plane + (size_t)j * (size_t)ldk);
        for (int q = threadIdx.x; q < (int)(ldk / 8); q += 128) dst[q] = src[q];
    }
}

// A[r, kk] = M[r, lo + kk] = Bt[lo + kk, r - lo]: the transpose inside every component block; zeros beyond the component and
// for rows of components wider than ldk (those are not multiplied).  grid (ceil(n / 32), ldk / 32, 3), block (32, 8).
__global__ void __launch_bounds__(256)
hh_k_blk_transpose(const unsigned short* __restrict__ Bt, unsigned short* __restrict__ A, int n, const int* __restrict__ comp_lo,
                   const int* __restrict__ comp_hi, long long ldk, long long plane) {
    __shared__ unsigned short tile[32][34];
    const int r0 = blockIdx.x * 32, kk0 = blockIdx.y * 32;
    const unsigned short* __restrict__ src = Bt + (size_t)blockIdx.z * (size_t)plane;
    unsigned short* __restrict__ dst = A + (size_t)blockIdx.z * (size_t)plane;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int rl = min(r0 + 31, n - 1);
    const bool same = (r0 + 31 < n) && comp_lo[r0] == comp_lo[rl];
    if (same) {
        const int lo = comp_lo[r0], width = comp_hi[r0] - lo;
        const bool fits = width <= (int)ldk;
        for (int y = ty; y < 32; y += 8) {
            const int kk = kk0 + y;
            tile[y][tx] = (fits && kk < width) ? src[(size_t)(lo + kk) * (size_t)ldk + (size_t)(r0 - lo + tx)] : (unsigned short)0;
        }
        __syncthreads();
        for (int y = ty; y < 32; y += 8) dst[(size_t)(r0 + y) * (size_t)ldk + (size_t)(kk0 + tx)] = tile[tx][y];
    } else {
        for (int y = ty; y < 32; y += 8) {
            const int r = r0 + y;
            if (r >= n) continue;
            const int lo = comp_lo[r], width = comp_hi[r] - lo;
            const int kk = kk0 + tx;
            dst[(size_t)r * (size_t)ldk + (size_t)kk] =
                (width <= (int)ldk && kk < width) ? src[(size_t)(lo + kk) * (size_t)ldk + (size_t)(r - lo)] : (unsigned short)0;
        }
    }
}

float hh_gemm_blk_out_scale(int f16) { return f16 ? ldexpf(1.0f, -2 * HG_BLK_SHIFT) : 1.0f; }

int hh_gemm_blk_operands(hh_ctx* ctx, const int* d_len, const void* d_ent, int cap, const int* d_list, int nlist, const int* d_comp_lo,
                         const int* d_comp_hi, int n, unsigned short* d_A, unsigned short* d_Bt, long long ldk, int f16) {
    const long long plane = ldk * (long long)n;
    auto kd = hh_k_blk_densify;
    const size_t dsm = (size_t)3 * (size_t)ldk * sizeof(unsigned short);
    HH_CUDA(cudaFuncSetAttribute(kd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm));
    if (nlist > 0)
        HH_LAUNCH(ctx, kd, nlist, 128, dsm, d_len, reinterpret_cast<const uint2*>(d_ent), cap, d_list, nlist, d_comp_lo, d_comp_hi, d_Bt, ldk,
                  plane, f16);
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)(ldk / 32), f16 ? 2u : 3u), block(32, 8);
    hh_k_blk_transpose<<<grid, block, 0, ctx->stream>>>(d_Bt, d_A, n, d_comp_lo, d_comp_hi, ldk, plane);
    ctx->launches++;
    HH_CUDA(cudaGetLastError());
    return HH_OK;
}

int hh_gemm_tile_size() { return 128 * (hg_env_int("HH_GEMM_CG", 2) == 1 ? 1 : 2); }

// work list of the whole-matrix product: every tile pair (a <= b) on or above the diagonal whose result (columns of
// tile b) or mirror image (columns of tile a) falls into the owned column block [col_lo, col_hi).  A column shard
// computes every element exactly as the single-GPU run does (same tile, same orientation), so M1 is bit-identical
// for any number of shards.
int hh_gemm_items_full(int n, int col_lo, int col_hi, std::vector<hh_gemm_item>& out) {
    const int T = hh_gemm_tile_size();
    const int nt = (n + T - 1) / T;
    const int nkb = (n + 63) / 64;
    out.clear();
    auto owned = [&](int t) {
        const int c0 = t * T, c1 = std::min(n, c0 + T);
        return c1 > col_lo && c0 < col_hi;
    };
    // Rasterisation.  Item i runs on CTA pair (i mod pairs), so `pairs` consecutive items form a wave that streams its
    // operand panels together: the wave should be a compact block of tiles.  A panels (one bf16 plane) are three times
    // cheaper than B panels (three planes), so super-blocks are SB_M = 15 tiles tall and SB_N = 5 wide (75 tiles ~ one
    // wave of 74 pairs): per k-block a wave then reads 15 + 3 * 5 = 30 panel blocks instead of 1 + 3 * 74.
    const int SB_M = 15, SB_N = 5;
    for (int bb = 0; bb < nt; bb += SB_N) {
        for (int ba = 0; ba <= std::min(nt - 1, bb + SB_N - 1); ba += SB_M) {
            for (int ta = ba; ta < std::min(nt, ba + SB_M); ++ta) {
                for (int tb = std::max(bb, ta); tb < std::min(nt, bb + SB_N); ++tb) {
                    int flags = 0;
                    if (owned(tb)) flags |= HH_GEMM_DIRECT;
                    if (tb > ta && owned(ta)) flags |= HH_GEMM_MIRROR;
                    if (!flags) continue;
                    hh_gemm_item w;
                    memset(&w, 0, sizeof(w));
                    w.m0 = ta * T;
                    w.n0 = tb * T;
                    w.m_end = n;
                    w.n_end = n;
                    w.kb_lo[0] = 0;
                    w.kb_hi[0] = nkb;
                    w.flags = flags;
                    out.push_back(w);
                }
            }
        }
    }
    return HH_OK;
}
