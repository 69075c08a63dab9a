// Markov clustering on the GPU (scripts/HapHiC_cluster.py:1987-2062, 2132-2162).
//
// Storage: "row-blocked slotted CSC".  Column j owns a fixed slot of `cap` entries
// (idx/val at j*cap), rows ascending; blk[j*(W+1) + w] is the offset of the first entry whose
// row lies in row block w (rows [w*T, (w+1)*T)), blk[..W] == len[j].  W is the number of warps
// of the column kernel, so warp w finds "its" part of any column with two loads.
//
// One kernel template does every per-column job.  A CTA takes columns from a dynamic queue and
// keeps a dense fp32 accumulator of the whole column in shared memory (n <= 57,600; a
// global-memory accumulator otherwise).  Warp w owns accumulator rows [w*T, (w+1)*T): during
// the Gustavson expansion  C[:,j] = sum_i B[i,j] * A[:,i]  it walks the B entries in order and adds
// only the row-block-w segment of A[:,i], so every accumulator cell is updated by one warp, in
// ascending i -- no atomics, and the fp32 sums are bit-reproducible for any grid size or GPU count.
// The epilogue (inflate -> column L1 -> prune/keep-max -> column L1 -> convergence) runs on
// the accumulator in place and writes the pruned column straight into its slot: the unpruned
// product never reaches HBM.
//
//   SRC_CSC     scatter an unsorted CSC column            (dict_to_matrix output, 366-368)
//   SRC_PRODUCT expansion, A.B column product             (mkl_matrix_power, 2017-2023)
//   EPI_NORM    column L1 normalise (sklearn normalize, 2144) or raw copy (canonical CSC)
//   EPI_DUMP    write the accumulator as a dense column    (pre-expansion result, 2146-2149)
//   EPI_PRUNE   inflate + normalise (2038), prune + keep first max + normalise (1987-2014),
//               optional convergence term max(|M-L| - 1e-5|L|) (2045)
#include "hh_common.cuh"
#include "hh_internal.cuh"
#include "hh_gemm.cuh"
#include <math.h>
#include <stdlib.h>
#include <algorithm>
#include <utility>

struct hh_slotmat {
    int n;       // rows == columns
    int cap;     // entries per column slot
    int W;       // row blocks per column
    int* len;    // [n]
    int* blk;    // [n * (W+1)]
    uint2* ent;  // [n * cap]  {row index, fp32 value bits}: one 64-bit load per entry
};

// matrix.power(r) on fp32 data (2037; numpy: x * x for r == 2, powf otherwise).  Exponents that are small multiples of one
// half are evaluated with correctly rounded multiplications and square roots (at most two roundings, i.e. within one ulp
// of the exact power -- tighter than powf's bound) instead of the ~60-instruction powf: iteration 0 inflates all n^2
// entries of the dense pre-expanded matrix.
enum { HH_INFL_POW = 0, HH_INFL_SQUARE = 1, HH_INFL_X15 = 2, HH_INFL_CUBE = 3, HH_INFL_X25 = 4 };
__device__ __forceinline__ float hh_inflate(float x, float rf, int mode) {
    switch (mode) {
        case HH_INFL_SQUARE: return x * x;
        case HH_INFL_X15: return x * __fsqrt_rn(x);
        case HH_INFL_CUBE: return (x * x) * x;
        case HH_INFL_X25: return (x * x) * __fsqrt_rn(x);
        default: return powf(x, rf);
    }
}

enum { SRC_CSC = 0, SRC_PRODUCT = 1 };
enum { EPI_NORM = 0, EPI_DUMP = 1, EPI_PRUNE = 2 };
// Link counts above the clip threshold of the tensor-core encoding (hh_gemm_stats.clip: 2048 for an f16 plane, 256 for a bf16
// plane) are split: min(x, clip) goes through the GEMM as ONE exact plane, the rest through two small Gustavson corrections
// (hh_k_clip_fix, hh_mcl_create_ex).

struct hh_colargs {
    int n, T, ch_shift, n_pad;
    int col_lo, ncols;
    int* counter;
    hh_slotmat A, B, out;
    const int64_t* csc_ptr;
    const int32_t* csc_row;
    const float* csc_val;
    const float* dense_in;
    float* dense_out;
    int64_t ld;
    int raw;
    int inflate_square;
    float inflation, prune;
    int do_conv;
    int track;                   // product + prune only: keep the dirty-chunk bitmap (sparse columns)
    // cluster-contiguous relabelling ("perm space"): new index = perm[original index], orig = inverse
    const int* perm;             // SRC_CSC(slot source): scatter rows through perm
    const int* orig;             // original index of every (new) row: tie-break of the first maximum; source column lookup
    int slot_src;                // SRC_CSC: read the column from slotted matrix B (column orig[j] when orig != NULL) instead of a CSC
    const int* ncols_ptr;        // optional: number of columns to process is read from device memory (overflow list)
    const int* order;            // optional processing order of the owned columns (cluster-sorted: operand reuse in L2)
    int flat;                    // expansion inner loop: 1 = flat 32-entry walk, 0 = one segment at a time
    int l2pf;                    // expansion: prefetch the next batch's segments into L2
    hh_slotmat prev;             // EPI_PRUNE convergence test against this matrix instead of B (expansion > 2: B is M^(e-1))
    int use_prev;
    float* scratch;
    unsigned long long* stats;   // [0] nnz written  [1] products
    int* delta_bits;
    int* err;
};

__device__ __forceinline__ uint64_t hh_warp_or64(uint64_t v) {
    unsigned lo = __reduce_or_sync(HH_FULL_MASK, (unsigned)v);
    unsigned hi = __reduce_or_sync(HH_FULL_MASK, (unsigned)(v >> 32));
    return ((uint64_t)hi << 32) | lo;
}

template <int W, int SRC, int EPI, bool SMEM, bool TRACK, bool FLAT>
__global__ void __launch_bounds__(W * 32) hh_k_col(const hh_colargs a) {
    extern __shared__ __align__(16) float hh_dyn_smem[];
    __shared__ double s_d[32];
    __shared__ float s_f[32];
    __shared__ int s_k[32];
    __shared__ int s_c[32];
    __shared__ int s_o[32];
    __shared__ int s_col;

    float* __restrict__ acc = SMEM ? hh_dyn_smem : (a.scratch + (size_t)blockIdx.x * a.n_pad);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int T = a.T;
    const int tile0 = w * T;
    const int ch_shift = a.ch_shift;
    const int nch = (T + (1 << ch_shift) - 1) >> ch_shift;
    const uint64_t ALL = (nch >= 64) ? ~0ull : ((1ull << nch) - 1ull);
    const unsigned lt_mask = (1u << lane) - 1u;

    if (SMEM) {
        for (int k = threadIdx.x; k < a.n_pad; k += W * 32) acc[k] = 0.f;
    }
    __syncthreads();

    float dmax = 0.f;
    unsigned long long prod_acc = 0ull, nnz_acc = 0ull;
    const int ncols_run = a.ncols_ptr ? *a.ncols_ptr : a.ncols;

    for (;;) {
        if (threadIdx.x == 0) s_col = atomicAdd(a.counter, 1);
        __syncthreads();
        const int jj = s_col;
        if (jj >= ncols_run) break;
        const int j = a.order ? a.order[jj] : (a.col_lo + jj);
        const int jsrc = (a.orig && SRC == SRC_CSC && a.slot_src) ? a.orig[j] : j;   // source column
        const int jloc = jsrc - a.col_lo;       // position inside the owned (dense) column block
        uint64_t dirty = 0ull;

        // ------------------------------------------------------------------ source
        if (SRC == SRC_CSC) {
            if (a.slot_src) {
                // relabelling pass: column jsrc of the slotted matrix B, rows sent through perm
                const int L = a.B.len[jsrc];
                const uint2* __restrict__ se = a.B.ent + (size_t)jsrc * (size_t)a.B.cap;
                for (int p = threadIdx.x; p < L; p += W * 32) {
                    const uint2 e = se[p];
                    acc[a.perm ? a.perm[e.x] : (int)e.x] = __uint_as_float(e.y);
                }
            } else {
                const int64_t p0 = a.csc_ptr[j], p1 = a.csc_ptr[j + 1];
                for (int64_t p = p0 + threadIdx.x; p < p1; p += W * 32) atomicAdd(&acc[a.csc_row[p]], a.csc_val[p]);
            }
            __syncthreads();
            dirty = ALL;
        } else {
            // Gustavson expansion restricted to this warp's row block.  The B entries of column j are
            // taken 32 at a time (one candidate segment of A per lane); the non-empty segments are
            // compacted and their entries walked as ONE flat list, 32 entries per step, so lanes stay
            // busy whatever the segment lengths are.  Entries of one segment have distinct rows; entries
            // of different segments inside a step are applied in segment order (one round per segment),
            // which keeps every accumulator cell's additions in ascending-i order.
            const int lenB = a.B.len[j];
            const uint2* __restrict__ Bent = a.B.ent + (size_t)j * (size_t)a.B.cap;
            const uint2* __restrict__ Aent = a.A.ent;
            const int* __restrict__ Ablk = a.A.blk;
            const size_t capA = (size_t)a.A.cap;
            unsigned long long warp_prod = 0ull;
            // software pipeline over batches: B entries two batches ahead, block pointers one batch ahead
            int i1 = 0, i2 = 0, s1 = 0, e1 = 0;
            float v1 = 0.f, v2 = 0.f;
            if (lane < lenB) {
                const uint2 be = Bent[lane];
                i1 = (int)be.x;
                v1 = __uint_as_float(be.y);
            }
            if (32 + lane < lenB) {
                const uint2 be = Bent[32 + lane];
                i2 = (int)be.x;
                v2 = __uint_as_float(be.y);
            }
            if (lane < lenB) {
                const int* bp = Ablk + (size_t)i1 * (W + 1) + w;
                s1 = bp[0];
                e1 = bp[1];
            }
            for (int t0 = 0; t0 < lenB; t0 += 32) {
                // ---- current batch header (loaded during the previous trip)
                const int seg_len = (t0 + lane < lenB) ? (e1 - s1) : 0;
                const unsigned seg_base = (unsigned)((size_t)i1 * capA + (size_t)s1);
                const float seg_v = v1;
                // ---- advance the pipeline: batch +1 gets its block pointers, batch +2 its B entries
                i1 = i2;
                v1 = v2;
                s1 = 0;
                e1 = 0;
                if (t0 + 32 + lane < lenB) {
                    const int* bp = Ablk + (size_t)i1 * (W + 1) + w;
                    s1 = bp[0];
                    e1 = bp[1];
                }
                if (t0 + 64 + lane < lenB) {
                    const uint2 be = Bent[t0 + 64 + lane];
                    i2 = (int)be.x;
                    v2 = __uint_as_float(be.y);
                }
                const unsigned ne = __ballot_sync(HH_FULL_MASK, seg_len > 0);
                if (!FLAT) {
                    // ---- one segment at a time, two 32-entry chunks per trip; the first two chunks of the
                    // next segment are loaded before the current one is applied
                    unsigned rem = ne;
                    int nL = 0, nk0 = 0, nk1 = 0;
                    unsigned nb = 0;
                    float nv = 0.f, na0 = 0.f, na1 = 0.f;
                    auto preload = [&]() {
                        const int u = __ffs(rem) - 1;
                        rem &= rem - 1;
                        nL = __shfl_sync(HH_FULL_MASK, seg_len, u);
                        nb = __shfl_sync(HH_FULL_MASK, seg_base, u);
                        nv = __shfl_sync(HH_FULL_MASK, seg_v, u);
                        if (lane < nL) {
                            const uint2 e0 = Aent[nb + lane];
                            nk0 = (int)e0.x;
                            na0 = __uint_as_float(e0.y);
                        }
                        if (lane + 32 < nL) {
                            const uint2 e1x = Aent[nb + lane + 32];
                            nk1 = (int)e1x.x;
                            na1 = __uint_as_float(e1x.y);
                        }
                    };
                    if (rem) preload();
                    bool have = ne != 0;
                    while (have) {
                        const int cL = nL, ck0 = nk0, ck1 = nk1;
                        const unsigned cb = nb;
                        const float cv = nv, ca0 = na0, ca1 = na1;
                        have = rem != 0;
                        if (have) preload();
                        warp_prod += (unsigned long long)cL;
                        if (lane < cL) {
                            acc[ck0] = fmaf(cv, ca0, acc[ck0]);
                            if (TRACK) dirty |= 1ull << ((ck0 - tile0) >> ch_shift);
                        }
                        if (lane + 32 < cL) {
                            acc[ck1] = fmaf(cv, ca1, acc[ck1]);
                            if (TRACK) dirty |= 1ull << ((ck1 - tile0) >> ch_shift);
                        }
                        for (int c = 64; c < cL; c += 64) {
                            const int p0 = c + lane, p1 = c + 32 + lane;
                            int k0 = 0, k1 = 0;
                            float a0 = 0.f, a1 = 0.f;
                            if (p0 < cL) {
                                const uint2 e0 = Aent[cb + p0];
                                k0 = (int)e0.x;
                                a0 = __uint_as_float(e0.y);
                            }
                            if (p1 < cL) {
                                const uint2 e1x = Aent[cb + p1];
                                k1 = (int)e1x.x;
                                a1 = __uint_as_float(e1x.y);
                            }
                            if (p0 < cL) {
                                acc[k0] = fmaf(cv, a0, acc[k0]);
                                if (TRACK) dirty |= 1ull << ((k0 - tile0) >> ch_shift);
                            }
                            if (p1 < cL) {
                                acc[k1] = fmaf(cv, a1, acc[k1]);
                                if (TRACK) dirty |= 1ull << ((k1 - tile0) >> ch_shift);
                            }
                        }
                        __syncwarp();   // the next segment may hit the same rows from other lanes
                    }
                }
                // ---- compact the non-empty segments to the low lanes
                const int nseg = FLAT ? __popc(ne) : 0;
                if (nseg > 0) {
                const unsigned src = __fns(ne, 0, lane + 1) & 31u;
                int c_len = __shfl_sync(HH_FULL_MASK, seg_len, src);
                const unsigned c_base = __shfl_sync(HH_FULL_MASK, seg_base, src);
                const float c_v = __shfl_sync(HH_FULL_MASK, seg_v, src);
                if (lane >= nseg) c_len = 0;
                int incl = c_len;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int tt = __shfl_up_sync(HH_FULL_MASK, incl, o);
                    if (lane >= o) incl += tt;
                }
                const int excl = incl - c_len;
                const int total = __shfl_sync(HH_FULL_MASK, incl, 31);
                warp_prod += (unsigned long long)total;
                // ---- flat walk, two steps in flight
                int uf = 0;
                int uf_end = __shfl_sync(HH_FULL_MASK, incl, 0);
                // step descriptor: (valid, du, nround, v, k, a)
                bool n_valid = false;
                int n_du = 0, n_round = 0, n_k = 0;
                float n_v = 0.f, n_a = 0.f;
                auto fetch_step = [&](int q0) {
                    while (uf_end <= q0) {      // warp-uniform
                        ++uf;
                        uf_end = __shfl_sync(HH_FULL_MASK, incl, uf);
                    }
                    const bool inside = (lane > uf) && (lane < nseg) && (excl > q0) && (excl < q0 + 32);
                    const unsigned bmask = __reduce_or_sync(HH_FULL_MASK, inside ? (1u << (excl - q0)) : 0u);
                    const int q = q0 + lane;
                    n_valid = q < total;
                    n_du = __popc(bmask & (0xFFFFFFFFu >> (31 - lane)));
                    n_round = __popc(bmask) + 1;
                    const int u = (uf + n_du) & 31;
                    const unsigned b = __shfl_sync(HH_FULL_MASK, c_base, u);
                    const int o = __shfl_sync(HH_FULL_MASK, excl, u);
                    n_v = __shfl_sync(HH_FULL_MASK, c_v, u);
                    if (n_valid) {
                        const unsigned pidx = b + (unsigned)(q - o);
                        const uint2 e0 = Aent[pidx];
                        n_k = (int)e0.x;
                        n_a = __uint_as_float(e0.y);
                    }
                };
                fetch_step(0);
                for (int q0 = 0; q0 < total; q0 += 32) {
                    const bool c_valid = n_valid;
                    const int c_du = n_du, c_round = n_round, c_k = n_k;
                    const float cv = n_v, ca = n_a;
                    if (q0 + 32 < total) fetch_step(q0 + 32);
                    for (int r = 0; r < c_round; ++r) {
                        if (c_valid && c_du == r) {
                            acc[c_k] = fmaf(cv, ca, acc[c_k]);
                            if (TRACK) dirty |= 1ull << ((c_k - tile0) >> ch_shift);
                        }
                        __syncwarp();
                    }
                }
                }   // nseg > 0
                // ---- pull the next batch's segments into L2 (their block pointers arrived long ago)
                if (a.l2pf && e1 > s1) {
                    const size_t nb = (size_t)i1 * capA;
                    const char* pi = reinterpret_cast<const char*>(Aent + nb + s1);
                    const int bytes = (e1 - s1) * 8;
                    for (int o = -(int)((uintptr_t)pi & 127); o < bytes; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pi + o));
                }
            }
            if (lane == 0) prod_acc += warp_prod;
            dirty = TRACK ? hh_warp_or64(dirty) : ALL;
        }

        // ------------------------------------------------------------------ epilogue
#define HH_FOR_DIRTY_ROWS(...)                                                    \
    for (uint64_t _m = dirty; _m; _m &= _m - 1ull) {                              \
        const int _c = __ffsll((long long)_m) - 1;                                \
        const int _r0 = tile0 + (_c << ch_shift);                                 \
        const int _r1 = min(_r0 + (1 << ch_shift), tile0 + T);                    \
        for (int _r = _r0; _r < _r1; _r += 32) {                                  \
            const int k = _r + lane;                                              \
            __VA_ARGS__                                                           \
        }                                                                         \
    }

        if (EPI == EPI_DUMP) {
            float* __restrict__ col = a.dense_out + (size_t)jloc * (size_t)a.ld;
            for (int r = tile0 + lane; r < tile0 + T; r += 32) {
                if (r < a.ld) {          // rows in [n, ld) are zero padding (never accumulated)
                    col[r] = acc[r];
                    acc[r] = 0.f;
                }
            }
        } else if (EPI == EPI_NORM) {
            double s = 0.0;
            int cnt = 0;
            HH_FOR_DIRTY_ROWS({
                const float x = acc[k];
                if (x != 0.f) {
                    s += fabs((double)x);
                    cnt++;
                }
            })
            s = hh_warp_sum(s);
            cnt = hh_warp_sum(cnt);
            if (lane == 0) {
                s_d[w] = s;
                s_c[w] = cnt;
            }
            __syncthreads();
            const double sv = (lane < W) ? s_d[lane] : 0.0;
            const int cv = (lane < W) ? s_c[lane] : 0;
            const double S = hh_warp_sum(sv);
            int incl = cv;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int tt = __shfl_up_sync(HH_FULL_MASK, incl, o);
                if (lane >= o) incl += tt;
            }
            const int base = __shfl_sync(HH_FULL_MASK, incl - cv, w);
            const int total = __shfl_sync(HH_FULL_MASK, incl, 31);
            int off = base;
            uint2* __restrict__ oent = a.out.ent + (size_t)j * (size_t)a.out.cap;
            HH_FOR_DIRTY_ROWS({
                const float x = acc[k];
                const bool f = (x != 0.f);
                const unsigned bal = __ballot_sync(HH_FULL_MASK, f);
                if (f) {
                    const int pos = off + __popc(bal & lt_mask);
                    if (pos < a.out.cap) {
                        oent[pos] = make_uint2((unsigned)k, __float_as_uint((a.raw || S == 0.0) ? x : (float)((double)x / S)));
                    }
                    acc[k] = 0.f;
                }
                off += __popc(bal);
            })
            if (lane == 0) a.out.blk[(size_t)j * (W + 1) + w] = base;
            if (threadIdx.x == 0) {
                a.out.blk[(size_t)j * (W + 1) + W] = min(total, a.out.cap);
                a.out.len[j] = min(total, a.out.cap);
                if (total > a.out.cap) atomicExch(a.err, 1);
                nnz_acc += (unsigned long long)total;
            }
        } else {
            // E1: inflate (matrix.power(r), fp32) and first column sum (fp64)
            const float rf = a.inflation;
            const int im = a.inflate_square;
            double s1 = 0.0;
            HH_FOR_DIRTY_ROWS({
                const float x = acc[k];
                if (x != 0.f) {
                    const float y = hh_inflate(x, rf, im);
                    acc[k] = y;
                    s1 += (double)y;
                }
            })
            s1 = hh_warp_sum(s1);
            if (lane == 0) s_d[w] = s1;
            __syncthreads();
            const double S1 = hh_warp_sum((lane < W) ? s_d[lane] : 0.0);
            __syncthreads();   // s_d is reused below
            // E2: normalise, threshold statistics, first maximum
            const float p32 = a.prune;
            double s2 = 0.0;
            int cnt = 0;
            float vbest = 0.f;
            int kbest = 0x7fffffff, obest = 0x7fffffff;     // obest: ORIGINAL row index of kbest (first maximum = lowest original row)
            HH_FOR_DIRTY_ROWS({
                const float y = acc[k];
                if (y != 0.f) {
                    const float x1 = (S1 != 0.0) ? (float)((double)y / S1) : y;
                    acc[k] = x1;
                    if (x1 >= p32 && x1 > 0.f) {
                        cnt++;
                        s2 += (double)x1;
                    }
                    if (x1 > vbest) {
                        vbest = x1;
                        kbest = k;
                        obest = a.orig ? a.orig[k] : k;
                    } else if (x1 == vbest && a.orig) {
                        const int o = a.orig[k];
                        if (o < obest) {
                            kbest = k;
                            obest = o;
                        }
                    }
                }
            })
            s2 = hh_warp_sum(s2);
            cnt = hh_warp_sum(cnt);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(HH_FULL_MASK, vbest, o);
                const int ok = __shfl_xor_sync(HH_FULL_MASK, kbest, o);
                const int oo = __shfl_xor_sync(HH_FULL_MASK, obest, o);
                if (ov > vbest || (ov == vbest && oo < obest)) {
                    vbest = ov;
                    kbest = ok;
                    obest = oo;
                }
            }
            if (lane == 0) {
                s_d[w] = s2;
                s_c[w] = cnt;
                s_f[w] = vbest;
                s_k[w] = kbest;
                s_o[w] = obest;
            }
            __syncthreads();
            const double sv = (lane < W) ? s_d[lane] : 0.0;
            const int cv = (lane < W) ? s_c[lane] : 0;
            float vmax = (lane < W) ? s_f[lane] : 0.f;
            int kmax = (lane < W) ? s_k[lane] : 0x7fffffff;
            int omax = (lane < W) ? s_o[lane] : 0x7fffffff;
            double S2 = hh_warp_sum(sv);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(HH_FULL_MASK, vmax, o);
                const int ok = __shfl_xor_sync(HH_FULL_MASK, kmax, o);
                const int oo = __shfl_xor_sync(HH_FULL_MASK, omax, o);
                if (ov > vmax || (ov == vmax && oo < omax)) {
                    vmax = ov;
                    kmax = ok;
                    omax = oo;
                }
            }
            int incl = cv;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int tt = __shfl_up_sync(HH_FULL_MASK, incl, o);
                if (lane >= o) incl += tt;
            }
            int base = __shfl_sync(HH_FULL_MASK, incl - cv, w);
            int total = __shfl_sync(HH_FULL_MASK, incl, 31);
            // keep the column maximum when nothing reaches the threshold (2009-2013)
            const bool need_max = (total == 0) && (vmax > 0.f);
            if (need_max) {
                const int wk = kmax / T;
                base = (w > wk) ? 1 : 0;
                total = 1;
                S2 = (double)vmax;
            }
            // E3: compact the survivors in row order, second normalisation (2014)
            int off = base;
            uint2* __restrict__ oent = a.out.ent + (size_t)j * (size_t)a.out.cap;
            const bool conv = a.do_conv != 0;
            HH_FOR_DIRTY_ROWS({
                const float x1 = acc[k];
                const bool f = need_max ? (k == kmax) : (x1 >= p32 && x1 > 0.f);
                const unsigned bal = __ballot_sync(HH_FULL_MASK, f);
                float keepv = 0.f;
                if (f) {
                    const int pos = off + __popc(bal & lt_mask);
                    // the kept maximum of a column without survivors is x1 / x1 = 1 (S2 = its own x1)
                    const float x2 = need_max ? 1.0f : (float)((double)x1 / S2);
                    if (pos < a.out.cap) {
                        oent[pos] = make_uint2((unsigned)k, __float_as_uint(x2));
                    }
                    keepv = x2;
                }
                if (x1 != 0.f) acc[k] = conv ? keepv : 0.f;
                off += __popc(bal);
            })
            if (lane == 0) a.out.blk[(size_t)j * (W + 1) + w] = base;
            if (threadIdx.x == 0) {
                a.out.blk[(size_t)j * (W + 1) + W] = min(total, a.out.cap);
                a.out.len[j] = min(total, a.out.cap);
                if (total > a.out.cap) atomicExch(a.err, 1);
                nnz_acc += (unsigned long long)total;
            }
            if (SRC == SRC_PRODUCT && conv) {
                // E4: entries of the previous iterate L = B[:, j]  ->  |M - L| - 1e-5|L|  (fp32, 2045)
                __syncwarp();
                const hh_slotmat& Lm = a.use_prev ? a.prev : a.B;
                const int* bp = Lm.blk + (size_t)j * (W + 1) + w;
                const int ps = bp[0], pe = bp[1];
                const uint2* __restrict__ Lent = Lm.ent + (size_t)j * (size_t)Lm.cap;
                for (int p = ps + lane; p < pe; p += 32) {
                    const uint2 le = Lent[p];
                    const int k = (int)le.x;
                    const float l = __uint_as_float(le.y);
                    const float m = acc[k];
                    const float d = __fsub_rn(fabsf(__fsub_rn(m, l)), __fmul_rn(1e-5f, fabsf(l)));
                    dmax = fmaxf(dmax, d);
                    acc[k] = 0.f;
                }
                __syncwarp();
                // E5: entries only in M (L is an implicit zero there) and accumulator reset
                HH_FOR_DIRTY_ROWS({
                    const float m = acc[k];
                    if (m != 0.f) {
                        dmax = fmaxf(dmax, m);
                        acc[k] = 0.f;
                    }
                })
            }
        }
#undef HH_FOR_DIRTY_ROWS
        __syncthreads();
    }

    // flush per-CTA statistics
    dmax = hh_warp_max(dmax);
    if (lane == 0) {
        if (dmax > 0.f) atomicMax(a.delta_bits, __float_as_int(dmax));
        if (prod_acc) atomicAdd(a.stats + 1, prod_acc);
    }
    if (threadIdx.x == 0 && nnz_acc) atomicAdd(a.stats + 0, nnz_acc);
}

// ---------------------------------------------------------------------------------------------
// Cluster-contiguous relabelling.  Markov clustering never creates an entry between two connected
// components of the iterate's pattern, so once the vertices of a component are contiguous every later
// column lives in a window of rows = its component.  Components are found on the first pruned iterate by
// min-label hooking + pointer jumping; new index = rank of (component label, original index).
// ---------------------------------------------------------------------------------------------
__global__ void hh_k_cc_init(int* __restrict__ label, int n) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) label[v] = v;
}

__global__ void hh_k_cc_hook(const hh_slotmat m, int* __restrict__ label, int* __restrict__ changed) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < m.n; j += warps) {
        const int L = m.len[j];
        const uint2* e = m.ent + (size_t)j * (size_t)m.cap;
        int lj = label[j];
        int mn = lj;
        for (int p = lane; p < L; p += 32) mn = min(mn, label[e[p].x]);
        mn = __reduce_min_sync(HH_FULL_MASK, mn);
        bool ch = false;
        if (mn < lj) {
            if (lane == 0) atomicMin(label + j, mn);
            ch = true;
        }
        for (int p = lane; p < L; p += 32) {
            const int k = (int)e[p].x;
            if (label[k] > mn) {
                atomicMin(label + k, mn);
                ch = true;
            }
        }
        if (ch) *changed = 1;
    }
}

// same on the raw link matrix (unsorted CSC), strong links only: components of the counts >= thr graph order the
// columns of the pre-expansion so that CTAs working side by side gather the same operand columns (L2 reuse)
__global__ void hh_k_cc_hook_csc(const int64_t* __restrict__ colptr, const int32_t* __restrict__ row, const float* __restrict__ val,
                                 int n, float thr, int* __restrict__ label, int* __restrict__ changed) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += warps) {
        const int64_t p0 = colptr[j], p1 = colptr[j + 1];
        const int lj = label[j];
        int mn = lj;
        for (int64_t p = p0 + lane; p < p1; p += 32)
            if (val[p] >= thr) mn = min(mn, label[row[p]]);
        mn = __reduce_min_sync(HH_FULL_MASK, mn);
        bool ch = false;
        if (mn < lj) {
            if (lane == 0) atomicMin(label + j, mn);
            ch = true;
        }
        for (int64_t p = p0 + lane; p < p1; p += 32) {
            if (val[p] < thr) continue;
            const int k = row[p];
            if (label[k] > mn) {
                atomicMin(label + k, mn);
                ch = true;
            }
        }
        if (ch) *changed = 1;
    }
}

// keep the entries of `src` that fall into [lo, hi), order preserved (one block; n is small)
__global__ void __launch_bounds__(1024) hh_k_filter_range(const int* __restrict__ src, int n, int lo, int hi, int* __restrict__ dst) {
    __shared__ int s_warp[32];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int b = 0; b < n; b += 1024) {
        const int k = b + threadIdx.x;
        const int v = (k < n) ? src[k] : -1;
        const bool keep = v >= lo && v < hi;
        const unsigned m = __ballot_sync(HH_FULL_MASK, keep);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += s_warp[w];
        if (keep) dst[off + __popc(m & ((1u << lane) - 1u))] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < 32; ++w) t += s_warp[w];
            s_base += t;
        }
        __syncthreads();
    }
}

__global__ void hh_k_cc_jump(int* __restrict__ label, int n) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    int l = label[v];
    for (int t = 0; t < 8; ++t) {
        const int l2 = label[l];
        if (l2 == l) break;
        l = l2;
    }
    label[v] = l;
}

// perm[v] = number of vertices with a smaller (label, v) key; also component sizes
__global__ void __launch_bounds__(256) hh_k_cc_rank(const int* __restrict__ label, int n, int* __restrict__ perm,
                                                    int* __restrict__ inv, int* __restrict__ comp_size) {
    __shared__ unsigned long long tile[1024];
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long mine = (v < n) ? (((unsigned long long)(unsigned)label[v] << 32) | (unsigned)v) : ~0ull;
    int rank = 0;
    for (int base = 0; base < n; base += 1024) {
        for (int k = threadIdx.x; k < 1024; k += blockDim.x)
            tile[k] = (base + k < n) ? (((unsigned long long)(unsigned)label[base + k] << 32) | (unsigned)(base + k)) : ~0ull;
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 1024; ++k) rank += (tile[k] < mine) ? 1 : 0;
        __syncthreads();
    }
    if (v < n) {
        perm[v] = rank;
        inv[rank] = v;
        atomicAdd(comp_size + label[v], 1);
    }
}

// per NEW index: the row window of its component
__global__ void hh_k_cc_ranges(const int* __restrict__ label, const int* __restrict__ perm, const int* __restrict__ comp_size, int n,
                               int* __restrict__ comp_lo, int* __restrict__ comp_hi) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const int root = label[v];                 // the smallest original index of the component = its first new index
    const int lo = perm[root];
    comp_lo[perm[v]] = lo;
    comp_hi[perm[v]] = lo + comp_size[root];
}

// split the owned columns (new indices perm[col_lo + jj]) into window-eligible and the rest
__global__ void hh_k_cc_lists(const int* __restrict__ perm, int col_lo, int ncols, const int* __restrict__ comp_lo,
                              const int* __restrict__ comp_hi, int wmax, int* __restrict__ owned, int* __restrict__ win_list,
                              int* __restrict__ big_list, int* __restrict__ counts) {
    const int jj = blockIdx.x * blockDim.x + threadIdx.x;
    if (jj >= ncols) return;
    const int j = perm[col_lo + jj];
    owned[jj] = j;
    if (comp_hi[j] - comp_lo[j] <= wmax) win_list[atomicAdd(counts + 0, 1)] = j;
    else big_list[atomicAdd(counts + 1, 1)] = j;
}

// ---------------------------------------------------------------------------------------------
// Windowed expansion (perm space): ONE WARP per column with a private accumulator of the column's row
// window (its component).  The warp walks the column's entries in order and streams every operand column
// whole (long coalesced 64-bit loads, four in flight per lane), so each accumulator cell receives its
// additions in ascending i exactly like the accumulator kernel and like SciPy's SpGEMM -- the results are
// bit-identical to the un-windowed path.  The epilogue runs over the window only.  Dozens of such
// single-warp CTAs share an SM, and consecutive columns of the list belong to the same component, so the
// operand columns they re-read stay in L2.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) hh_k_col_win(const hh_colargs a, int W, const int* __restrict__ list, int nlist,
                                                   const int* __restrict__ comp_lo, const int* __restrict__ comp_hi, int wmax) {
    extern __shared__ __align__(16) float acc[];      // wmax floats, zero between columns
    const int lane = threadIdx.x;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint2* __restrict__ Aent = a.A.ent;
    const size_t capA = (size_t)a.A.cap;
    const float p32 = a.prune, rf = a.inflation;
    const bool conv = a.do_conv != 0;
    const int T = a.T;
    for (int k = lane; k < wmax; k += 32) acc[k] = 0.f;
    __syncwarp();
    float dmax = 0.f;
    unsigned long long prod_acc = 0ull, nnz_acc = 0ull;
    for (;;) {
        int jj = 0;
        if (lane == 0) jj = atomicAdd(a.counter, 1);
        jj = __shfl_sync(HH_FULL_MASK, jj, 0);
        if (jj >= nlist) break;
        const int j = list[jj];
        const int lo = comp_lo[j], width = comp_hi[j] - lo;
        const int lenB = a.B.len[j];
        const uint2* __restrict__ Bent = a.B.ent + (size_t)j * (size_t)a.B.cap;
        if (a.dense_in) {
            // the block product of this component came from the tensor cores (hh_mcl_step): column j of it, rows of the window
            const float* __restrict__ dcol = a.dense_in + (size_t)j * (size_t)a.ld;
            for (int r = lane; r < width; r += 32) acc[r] = dcol[r];
            prod_acc += (unsigned long long)width * (unsigned long long)width / 32ull;       // b * b multiply-adds per column (lane share)
            __syncwarp();
        }
        // ---- expansion
        for (int t0 = 0; t0 < (a.dense_in ? 0 : lenB); t0 += 32) {
            const int t = t0 + lane;
            int il = 0, Ll = 0;
            float vl = 0.f;
            if (t < lenB) {
                const uint2 be = Bent[t];
                il = (int)be.x;
                vl = __uint_as_float(be.y);
                Ll = a.A.len[il];
            }
            const int cnt = min(32, lenB - t0);
            for (int u = 0; u < cnt; ++u) {
                const int L = __shfl_sync(HH_FULL_MASK, Ll, u);
                const float v = __shfl_sync(HH_FULL_MASK, vl, u);
                const uint2* __restrict__ col = Aent + (size_t)__shfl_sync(HH_FULL_MASK, il, u) * capA;
                prod_acc += (unsigned long long)L;
                for (int p = lane; p < L; p += 128) {
                    uint2 e[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) e[q] = (p + 32 * q < L) ? col[p + 32 * q] : make_uint2(0xFFFFFFFFu, 0u);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (e[q].x != 0xFFFFFFFFu) {
                            const unsigned r = e[q].x - (unsigned)lo;
                            if (r < (unsigned)width) acc[r] = fmaf(v, __uint_as_float(e[q].y), acc[r]);
                            else atomicExch(a.err, 2);             // a row outside the component window: never silently dropped
                        }
                    }
                }
                __syncwarp();      // the next operand column may hit the same rows from other lanes
            }
        }
        // ---- E1: inflate + first column sum
        double s1 = 0.0;
        for (int r = lane; r < width; r += 32) {
            const float x = acc[r];
            if (x != 0.f) {
                const float y = hh_inflate(x, rf, a.inflate_square);
                acc[r] = y;
                s1 += (double)y;
            }
        }
        const double S1 = hh_warp_sum(s1);
        __syncwarp();
        // ---- E2: normalise, threshold statistics, first maximum (lowest ORIGINAL row among ties)
        double s2 = 0.0;
        int cnt = 0, kmax = 0x7fffffff, omax = 0x7fffffff;
        float vmax = 0.f;
        for (int r = lane; r < width; r += 32) {
            const float y = acc[r];
            if (y != 0.f) {
                const float x1 = (S1 != 0.0) ? (float)((double)y / S1) : y;
                acc[r] = x1;
                if (x1 >= p32 && x1 > 0.f) {
                    cnt++;
                    s2 += (double)x1;
                }
                if (x1 > vmax || (x1 == vmax && x1 > 0.f)) {
                    const int o = a.orig ? a.orig[lo + r] : (lo + r);
                    if (x1 > vmax || o < omax) {
                        vmax = x1;
                        kmax = lo + r;
                        omax = o;
                    }
                }
            }
        }
        double S2 = hh_warp_sum(s2);
        cnt = hh_warp_sum(cnt);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(HH_FULL_MASK, vmax, o);
            const int ok = __shfl_xor_sync(HH_FULL_MASK, kmax, o);
            const int oo = __shfl_xor_sync(HH_FULL_MASK, omax, o);
            if (ov > vmax || (ov == vmax && oo < omax)) {
                vmax = ov;
                kmax = ok;
                omax = oo;
            }
        }
        const bool need_max = (cnt == 0) && (vmax > 0.f);
        int total = cnt;
        if (need_max) {
            total = 1;
            S2 = (double)vmax;
        }
        __syncwarp();
        // ---- E3: ordered compaction into the slot; row-block pointers on the fly (rows ascend)
        uint2* __restrict__ oent = a.out.ent + (size_t)j * (size_t)a.out.cap;
        int* __restrict__ oblk = a.out.blk + (size_t)j * (W + 1);
        int bnext = 0;                       // next row-block boundary (row bnext*T) whose pointer is still unset
        int off = 0;
        for (int r0 = 0; r0 < width; r0 += 32) {
            const int r = r0 + lane;
            const float x1 = (r < width) ? acc[r] : 0.f;
            const bool f = (r < width) && (need_max ? (lo + r == kmax) : (x1 >= p32 && x1 > 0.f));
            const unsigned bal = __ballot_sync(HH_FULL_MASK, f);
            // boundaries that fall at or before the end of this 32-row step
            while (bnext <= W && (long long)bnext * T <= (long long)(lo + r0 + 31)) {
                const long long brow = (long long)bnext * T;
                // survivors of this step with row < brow
                const int nlt = (brow <= lo + r0) ? 0 : (int)(brow - (lo + r0));     // lanes [0, nlt) have row < brow
                const unsigned below = (nlt >= 32) ? 0xFFFFFFFFu : ((1u << nlt) - 1u);
                if (lane == 0) oblk[bnext] = min(off + __popc(bal & below), a.out.cap);
                bnext++;
            }
            float keepv = 0.f;
            if (f) {
                const int pos = off + __popc(bal & lt_mask);
                const float x2 = (float)((double)x1 / S2);
                if (pos < a.out.cap) oent[pos] = make_uint2((unsigned)(lo + r), __float_as_uint(x2));
                keepv = x2;
            }
            if (r < width) acc[r] = conv ? keepv : 0.f;
            off += __popc(bal);
        }
        if (lane == 0) {
            for (; bnext <= W; ++bnext) oblk[bnext] = min(total, a.out.cap);   // boundaries beyond the window
            a.out.len[j] = min(total, a.out.cap);
            if (total > a.out.cap) atomicExch(a.err, 1);
            nnz_acc += (unsigned long long)total;
        }
        __syncwarp();
        if (conv) {
            // E4: entries of the previous iterate L = B[:, j]
            for (int p = lane; p < lenB; p += 32) {
                const uint2 le = Bent[p];
                const unsigned r = le.x - (unsigned)lo;
                const float l = __uint_as_float(le.y);
                const float m = (r < (unsigned)width) ? acc[r] : 0.f;
                dmax = fmaxf(dmax, __fsub_rn(fabsf(__fsub_rn(m, l)), __fmul_rn(1e-5f, fabsf(l))));
                if (r < (unsigned)width) acc[r] = 0.f;
            }
            __syncwarp();
            // E5: entries only in M + accumulator reset
            for (int r = lane; r < width; r += 32) {
                const float m = acc[r];
                if (m != 0.f) {
                    dmax = fmaxf(dmax, m);
                    acc[r] = 0.f;
                }
            }
        }
        __syncwarp();
    }
    dmax = hh_warp_max(dmax);
    if (lane == 0) {
        if (dmax > 0.f) atomicMax(a.delta_bits, __float_as_int(dmax));
        if (prod_acc) atomicAdd(a.stats + 1, prod_acc);
        if (nnz_acc) atomicAdd(a.stats + 0, nnz_acc);
    }
}

// relabelling copy inside the component window: new column j <- old column inv[j], rows through perm (they land in
// [comp_lo[j], comp_hi[j])), re-sorted by a scatter into the window and an ordered compaction.  One warp per column.
__global__ void __launch_bounds__(32) hh_k_relabel_win(const hh_slotmat src, const hh_slotmat out, int W, int T,
                                                       const int* __restrict__ list, int nlist, const int* __restrict__ perm,
                                                       const int* __restrict__ inv, const int* __restrict__ comp_lo,
                                                       const int* __restrict__ comp_hi, int wmax, int* __restrict__ err) {
    extern __shared__ __align__(16) float acc[];      // wmax floats, zero between columns
    const int lane = threadIdx.x;
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int k = lane; k < wmax; k += 32) acc[k] = 0.f;
    __syncwarp();
    for (int jj = blockIdx.x; jj < nlist; jj += gridDim.x) {
        const int j = list[jj];
        const int lo = comp_lo[j], width = comp_hi[j] - lo;
        const int jsrc = inv[j];
        const int L = src.len[jsrc];
        const uint2* __restrict__ se = src.ent + (size_t)jsrc * (size_t)src.cap;
        for (int p = lane; p < L; p += 32) {
            const uint2 e = se[p];
            const unsigned r = (unsigned)perm[e.x] - (unsigned)lo;
            if (r < (unsigned)width) acc[r] = __uint_as_float(e.y);
            else atomicExch(err, 2);
        }
        __syncwarp();
        uint2* __restrict__ oent = out.ent + (size_t)j * (size_t)out.cap;
        int* __restrict__ oblk = out.blk + (size_t)j * (W + 1);
        int bnext = 0, off = 0;
        for (int r0 = 0; r0 < width; r0 += 32) {
            const int r = r0 + lane;
            const float x = (r < width) ? acc[r] : 0.f;
            const bool f = x != 0.f;
            const unsigned bal = __ballot_sync(HH_FULL_MASK, f);
            while (bnext <= W && (long long)bnext * T <= (long long)(lo + r0 + 31)) {
                const long long brow = (long long)bnext * T;
                const int nlt = (brow <= lo + r0) ? 0 : (int)(brow - (lo + r0));
                const unsigned below = (nlt >= 32) ? 0xFFFFFFFFu : ((1u << nlt) - 1u);
                if (lane == 0) oblk[bnext] = min(off + __popc(bal & below), out.cap);
                bnext++;
            }
            if (f) {
                const int pos = off + __popc(bal & lt_mask);
                if (pos < out.cap) oent[pos] = make_uint2((unsigned)(lo + r), __float_as_uint(x));
                acc[r] = 0.f;
            }
            off += __popc(bal);
        }
        if (lane == 0) {
            for (; bnext <= W; ++bnext) oblk[bnext] = min(off, out.cap);
            out.len[j] = min(off, out.cap);
            if (off > out.cap || off != L) atomicExch(err, 1);
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// nearly converged iterates: a column has a handful of entries, and the CTA-per-column kernel is bound
// by its per-column latency chain (one column in flight per SM).  Here ONE WARP expands a column by a
// 32-way merge of the operand columns (rows come out ascending, contributions are fused in ascending-i
// order exactly like the accumulator kernel), prunes it in shared memory and writes its slot.  Columns
// that do not fit (more than 32 entries, long operand columns, more than HH_SMALL_CAP result rows) are
// appended to an overflow list and handled by the accumulator kernel afterwards.
// ---------------------------------------------------------------------------------------------
#define HH_SMALL_CAP 256
#define HH_SMALL_MAXPROD 4096

__global__ void __launch_bounds__(256) hh_k_col_small(const hh_colargs a, int W, int* __restrict__ biglist, int* __restrict__ bigcount,
                                                      const int* __restrict__ list) {
    __shared__ int s_k[8][HH_SMALL_CAP];
    __shared__ float s_v[8][HH_SMALL_CAP];
    __shared__ int s_ok[8][32];
    const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint2* __restrict__ Aent = a.A.ent;
    const size_t capA = (size_t)a.A.cap;
    const float p32 = a.prune, rf = a.inflation;
    int* sk = s_k[wq];
    float* sv = s_v[wq];
    int* sok = s_ok[wq];
    float dmax = 0.f;
    unsigned long long prod_acc = 0ull, nnz_acc = 0ull;
    for (int jj = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; jj < a.ncols; jj += nwarps) {
        const int j = list ? list[jj] : (a.col_lo + jj);
        const int L = a.B.len[j];
        bool big = L > 32;
        int il = 0x7fffffff, lenl = 0;
        float vl = 0.f;
        size_t basel = 0;
        if (!big && lane < L) {
            const uint2 be = a.B.ent[(size_t)j * (size_t)a.B.cap + lane];
            il = (int)be.x;
            vl = __uint_as_float(be.y);
            lenl = a.A.len[il];
            basel = (size_t)il * capA;
        }
        const int tot = hh_warp_sum(lenl);
        if (tot > HH_SMALL_MAXPROD) big = true;
        int nout = 0;
        if (!big) {
            // ---- 32-way merge: every round emits the smallest pending row
            int h = 0x7fffffff, c = 0;
            float av = 0.f;
            if (lenl > 0) {
                const uint2 e = Aent[basel];
                h = (int)e.x;
                av = __uint_as_float(e.y);
            }
            for (;;) {
                const int kmin = __reduce_min_sync(HH_FULL_MASK, h);
                if (kmin == 0x7fffffff) break;
                const bool mine = (h == kmin);
                const unsigned part = __ballot_sync(HH_FULL_MASK, mine);
                float accv = 0.f;
                for (unsigned mm = part; mm; mm &= mm - 1u) {          // ascending lane == ascending i
                    const int b = __ffs(mm) - 1;
                    accv = fmaf(__shfl_sync(HH_FULL_MASK, vl, b), __shfl_sync(HH_FULL_MASK, av, b), accv);
                }
                if (lane == 0 && nout < HH_SMALL_CAP) {
                    sk[nout] = kmin;
                    sv[nout] = accv;
                }
                nout++;
                if (mine) {
                    c++;
                    if (c < lenl) {
                        const uint2 e = Aent[basel + c];
                        h = (int)e.x;
                        av = __uint_as_float(e.y);
                    } else {
                        h = 0x7fffffff;
                    }
                }
            }
            if (nout > HH_SMALL_CAP) big = true;
        }
        if (big) {
            if (lane == 0) biglist[atomicAdd(bigcount, 1)] = j;
            continue;
        }
        if (lane == 0) prod_acc += (unsigned long long)tot;
        __syncwarp();
        // ---- E1: inflate + first column sum
        double s1 = 0.0;
        for (int p = lane; p < nout; p += 32) {
            const float x = sv[p];
            if (x != 0.f) {
                const float y = hh_inflate(x, rf, a.inflate_square);
                sv[p] = y;
                s1 += (double)y;
            }
        }
        const double S1 = hh_warp_sum(s1);
        __syncwarp();
        // ---- E2: normalise, threshold statistics, first maximum
        double s2 = 0.0;
        int cnt = 0, kmax = 0x7fffffff, omax = 0x7fffffff;
        float vmax = 0.f;
        for (int p = lane; p < nout; p += 32) {
            const float y = sv[p];
            if (y != 0.f) {
                const float x1 = (S1 != 0.0) ? (float)((double)y / S1) : y;
                sv[p] = x1;
                if (x1 >= p32 && x1 > 0.f) {
                    cnt++;
                    s2 += (double)x1;
                }
                if (x1 > vmax || (x1 == vmax && x1 > 0.f)) {
                    const int o = a.orig ? a.orig[sk[p]] : sk[p];      // first maximum = lowest ORIGINAL row
                    if (x1 > vmax || o < omax) {
                        vmax = x1;
                        kmax = sk[p];
                        omax = o;
                    }
                }
            }
        }
        double S2 = hh_warp_sum(s2);
        cnt = hh_warp_sum(cnt);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(HH_FULL_MASK, vmax, o);
            const int ok = __shfl_xor_sync(HH_FULL_MASK, kmax, o);
            const int oo = __shfl_xor_sync(HH_FULL_MASK, omax, o);
            if (ov > vmax || (ov == vmax && oo < omax)) {
                vmax = ov;
                kmax = ok;
                omax = oo;
            }
        }
        const bool need_max = (cnt == 0) && (vmax > 0.f);
        int total = cnt;
        if (need_max) {
            total = 1;
            S2 = (double)vmax;
        }
        __syncwarp();
        // ---- E3: ordered compaction (in place in shared memory) + slot write
        uint2* __restrict__ oent = a.out.ent + (size_t)j * (size_t)a.out.cap;
        int off = 0;
        for (int p0 = 0; p0 < nout; p0 += 32) {
            const int p = p0 + lane;
            const float x1 = (p < nout) ? sv[p] : 0.f;
            const int k = (p < nout) ? sk[p] : 0;
            const bool f = (p < nout) && (need_max ? (k == kmax && x1 > 0.f) : (x1 >= p32 && x1 > 0.f));
            const unsigned bal = __ballot_sync(HH_FULL_MASK, f);
            __syncwarp();
            if (f) {
                const int pos = off + __popc(bal & lt_mask);
                const float x2 = (float)((double)x1 / S2);
                if (pos < a.out.cap) oent[pos] = make_uint2((unsigned)k, __float_as_uint(x2));
                sk[pos] = k;
                sv[pos] = x2;
            }
            off += __popc(bal);
            __syncwarp();
        }
        // row-block pointers of the new column
        if (lane < W) {
            const int target = lane * a.T;
            int lo = 0, hi = total;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (sk[mid] < target) lo = mid + 1;
                else hi = mid;
            }
            a.out.blk[(size_t)j * (W + 1) + lane] = lo;
        }
        if (lane == 0) {
            a.out.blk[(size_t)j * (W + 1) + W] = min(total, a.out.cap);
            a.out.len[j] = min(total, a.out.cap);
            if (total > a.out.cap) atomicExch(a.err, 1);
            nnz_acc += (unsigned long long)total;
        }
        // ---- convergence term against the previous iterate L = B[:, j] (its entries sit in the lanes)
        if (a.do_conv) {
            sok[lane] = il;                    // old rows, ascending; 0x7fffffff beyond L
            __syncwarp();
            if (lane < L) {
                int lo = 0, hi = total;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (sk[mid] < il) lo = mid + 1;
                    else hi = mid;
                }
                const float m = (lo < total && sk[lo] == il) ? sv[lo] : 0.f;
                dmax = fmaxf(dmax, __fsub_rn(fabsf(__fsub_rn(m, vl)), __fmul_rn(1e-5f, fabsf(vl))));
            }
            for (int p = lane; p < total; p += 32) {
                const int k = sk[p];
                int lo = 0, hi = L;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (sok[mid] < k) lo = mid + 1;
                    else hi = mid;
                }
                if (!(lo < L && sok[lo] == k)) dmax = fmaxf(dmax, sv[p]);
            }
        }
        __syncwarp();
    }
    dmax = hh_warp_max(dmax);
    if (lane == 0) {
        if (dmax > 0.f) atomicMax(a.delta_bits, __float_as_int(dmax));
        if (prod_acc) atomicAdd(a.stats + 1, prod_acc);
        if (nnz_acc) atomicAdd(a.stats + 0, nnz_acc);
    }
}

// ---------------------------------------------------------------------------------------------
// rank-sum statistic of filter_fragments (HapHiC_cluster.py:864-892) on the sorted slotted matrix
// (symmetric, so row a == column a).  Order of a row: links descending, ties by matrix index.
// ---------------------------------------------------------------------------------------------
#define HH_TOPN_MAX 32

// warp per fragment: the first topN columns of its sorted row
__global__ void hh_k_topn(const hh_slotmat m, int topN, int* __restrict__ top) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int a = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; a < m.n; a += warps) {
        const int L = m.len[a];
        const uint2* ent = m.ent + (size_t)a * (size_t)m.cap;
        float last_v = INFINITY;
        int last_i = -1;
        int zero_c = -1, zero_p = 0;        // cursor over the zero-valued columns (ascending index)
        for (int t = 0; t < topN; ++t) {
            // best stored entry strictly after (last_v, last_i) in (value desc, index asc) order
            float bv = -1.f;
            int bi = 0x7fffffff;
            for (int p = lane; p < L; p += 32) {
                const float v = __uint_as_float(ent[p].y);
                const int i = (int)ent[p].x;
                if (v <= 0.f) continue;
                const bool after = (v < last_v) || (v == last_v && i > last_i);
                if (after && (v > bv || (v == bv && i < bi))) {
                    bv = v;
                    bi = i;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(HH_FULL_MASK, bv, o);
                const int oi = __shfl_xor_sync(HH_FULL_MASK, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) {
                    bv = ov;
                    bi = oi;
                }
            }
            int pick;
            if (bv > 0.f) {
                pick = bi;
                last_v = bv;
                last_i = bi;
            } else {
                // no positive entry left: zero-valued columns in ascending index (the fragment itself included)
                last_v = 0.f;
                int c = zero_c + 1;
                if (lane == 0) {
                    for (;;) {
                        if (c >= m.n) break;
                        while (zero_p < L && (int)ent[zero_p].x < c) zero_p++;
                        if (zero_p < L && (int)ent[zero_p].x == c && __uint_as_float(ent[zero_p].y) > 0.f) {
                            c++;            // a positive entry: not a zero column
                            continue;
                        }
                        break;
                    }
                }
                c = __shfl_sync(HH_FULL_MASK, c, 0);
                zero_p = __shfl_sync(HH_FULL_MASK, zero_p, 0);
                zero_c = c;
                pick = (c < m.n) ? c : -1;
            }
            if (lane == 0) top[(size_t)a * topN + t] = pick;
        }
    }
}

// position of column b in the sorted row of fragment a
__device__ __forceinline__ int hh_rank_of(const hh_slotmat& m, int a, int b) {
    const int L = m.len[a];
    const uint2* ent = m.ent + (size_t)a * (size_t)m.cap;
    int lo = 0, hi = L;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int)ent[mid].x < b) lo = mid + 1;
        else hi = mid;
    }
    const bool found = lo < L && (int)ent[lo].x == b && __uint_as_float(ent[lo].y) > 0.f;
    int npos = 0, before = 0;           // positive entries in the row / positive entries left of b
    if (!found) {
        for (int p = 0; p < L; ++p) {
            const uint2 e = ent[p];
            const bool pos = __uint_as_float(e.y) > 0.f;
            npos += pos;
            before += pos && (int)e.x < b;
        }
        return npos + (b - before);     // all positive entries first, then the zero columns by index
    }
    const float v = __uint_as_float(ent[lo].y);
    int r = 0;
    for (int p = 0; p < L; ++p) {
        const uint2 e = ent[p];
        const float x = __uint_as_float(e.y);
        r += (x > v) || (x == v && (int)e.x < b);
    }
    return r;
}

// warp per fragment x: sum over the pairs of its top list of min(rank_a(b), rank_b(a))
__global__ void hh_k_rank_sum(const hh_slotmat m, int topN, const int* __restrict__ top, long long* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int npairs = topN * (topN - 1) / 2;
    for (int x = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; x < m.n; x += warps) {
        const int* tx = top + (size_t)x * topN;
        long long s = 0;
        for (int p = lane; p < npairs; p += 32) {
            // unrank pair p -> (u < v) in combinations order
            int u = 0, rem = p;
            while (rem >= topN - 1 - u) {
                rem -= topN - 1 - u;
                u++;
            }
            const int v = u + 1 + rem;
            const int a = tx[u], b = tx[v];
            if (a < 0 || b < 0) continue;
            const int r1 = hh_rank_of(m, a, b), r2 = hh_rank_of(m, b, a);
            s += (r1 < r2) ? r1 : r2;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(HH_FULL_MASK, s, o);
        if (lane == 0) out[x] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// pack / unpack of column blocks (canonical CSC export, multi-GPU exchange)
// ---------------------------------------------------------------------------------------------
__global__ void hh_k_pack(const hh_slotmat m, int col_lo, int ncols, const int64_t* __restrict__ off, int* __restrict__ len_out,
                          int* __restrict__ idx_out, float* __restrict__ val_out, const int* __restrict__ colmap) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int jj = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; jj < ncols; jj += warps) {
        const int c = colmap ? colmap[col_lo + jj] : (col_lo + jj);
        const int L = m.len[c];
        if (lane == 0 && len_out) len_out[jj] = L;
        const uint2* se = m.ent + (size_t)c * (size_t)m.cap;
        const int64_t o = off[jj];
        for (int p = lane; p < L; p += 32) {
            const uint2 e = se[p];
            idx_out[o + p] = (int)e.x;
            val_out[o + p] = __uint_as_float(e.y);
        }
    }
}

__global__ void hh_k_unpack(const hh_slotmat m, int T, int col_lo, int ncols, const int* __restrict__ len_in,
                            const int64_t* __restrict__ off, const int* __restrict__ idx_in, const float* __restrict__ val_in,
                            int* __restrict__ err, const int* __restrict__ colmap) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int W = m.W;
    for (int jj = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; jj < ncols; jj += warps) {
        const int c = colmap ? colmap[col_lo + jj] : (col_lo + jj);
        int L = len_in[jj];
        if (L > m.cap || L < 0) {
            if (lane == 0) atomicExch(err, 1);
            L = 0;
        }
        const int64_t o = off[jj];
        uint2* de = m.ent + (size_t)c * (size_t)m.cap;
        for (int p = lane; p < L; p += 32) de[p] = make_uint2((unsigned)idx_in[o + p], __float_as_uint(val_in[o + p]));
        if (lane < W) {   // first entry with row >= lane*T
            const int target = lane * T;
            int lo = 0, hi = L;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (idx_in[o + mid] < target) lo = mid + 1;
                else hi = mid;
            }
            m.blk[(size_t)c * (W + 1) + lane] = lo;
        }
        if (lane == 0) {
            m.blk[(size_t)c * (W + 1) + W] = L;
            m.len[c] = L;
        }
    }
}

__global__ void hh_k_gather_len(const int* __restrict__ len, const int* __restrict__ colmap, int col_lo, int ncols, int* __restrict__ out) {
    const int jj = blockIdx.x * blockDim.x + threadIdx.x;
    if (jj < ncols) out[jj] = len[colmap ? colmap[col_lo + jj] : (col_lo + jj)];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// per column: fp64 sum of the raw link counts and bclip[c] = fp32(HH_CLIP / sum), the image of the clip threshold in M0
__global__ void hh_k_clip_stats(const int64_t* __restrict__ colptr, const float* __restrict__ val, int n, double* __restrict__ s,
                                float* __restrict__ bclip, float clip) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const int lane = threadIdx.x & 31;
    double t = 0.0;
    for (int64_t p = colptr[c] + lane; p < colptr[c + 1]; p += 32) t += fabs((double)val[p]);
    t = hh_warp_sum(t);
    if (lane == 0) {
        s[c] = t;
        bclip[c] = (t != 0.0) ? (float)((double)clip / t) : clip;
    }
}

// The tensor-core GEMM multiplied the counts clipped to HH_CLIP: with C = Cs + Cl, Cs = min(C, HH_CLIP), it produced
// (Cs D Cs) D.  What is left of M1 = (C D C) D is
//     MODE 0:  M1[:, x] += M0l[i, x] * M0[:, i]        M0l = Cl D  (the excess of the few large counts)
//     MODE 1:  M1[x, j] += M0l[x, i] * M0s[i, j]       M0s = Cs D
// for every large entry (i, x).  One warp owns column x (MODE 0) or row x (MODE 1) of M1 and walks the large entries of
// column x of M0 in row order, so every element receives its additions in a fixed order: no atomics, bit-reproducible.
// Large entries are recognised in M0 itself (M0[i, x] > fp32(HH_CLIP / s_x) <=> count > HH_CLIP); the count is rint(M0 * s).
template <int MODE>
__global__ void __launch_bounds__(256)
hh_k_clip_fix(const hh_slotmat m0, const double* __restrict__ s, const float* __restrict__ bclip, float* __restrict__ m1, long long ld,
              int col_lo, int col_hi, unsigned long long* __restrict__ products, float clip_f) {
    const int x = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (x >= m0.n) return;
    if (MODE == 0 && (x < col_lo || x >= col_hi)) return;
    const double HH_CLIP = (double)clip_f;
    const int lane = threadIdx.x & 31;
    const int L = m0.len[x];
    const uint2* __restrict__ ex = m0.ent + (size_t)x * (size_t)m0.cap;
    const float bc = bclip[x];
    const double sx = s[x];
    unsigned long long np = 0ull;
    for (int p0 = 0; p0 < L; p0 += 32) {
        uint2 e = make_uint2(0u, 0u);
        if (p0 + lane < L) e = ex[p0 + lane];
        unsigned big = __ballot_sync(HH_FULL_MASK, (p0 + lane < L) && __uint_as_float(e.y) > bc);
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1;
            const int i = (int)__shfl_sync(HH_FULL_MASK, e.x, src);
            const double c = rint((double)__uint_as_float(__shfl_sync(HH_FULL_MASK, e.y, src)) * sx);     // C[i, x]
            const int Li = m0.len[i];
            const uint2* __restrict__ ei = m0.ent + (size_t)i * (size_t)m0.cap;
            if (MODE == 0) {
                const float vl = (float)((c - (double)HH_CLIP) / sx);                  // M0l[i, x]
                float* __restrict__ col = m1 + (size_t)(x - col_lo) * (size_t)ld;
                for (int q = lane; q < Li; q += 32) {
                    const uint2 t = ei[q];
                    col[t.x] = fmaf(vl, __uint_as_float(t.y), col[t.x]);
                }
            } else {
                const double si = s[i];
                const float vl = (float)((c - (double)HH_CLIP) / si);                  // M0l[x, i]
                for (int q = lane; q < Li; q += 32) {
                    const uint2 t = ei[q];                                             // (j, C[j, i] / s_i)
                    const int j = (int)t.x;
                    if (j < col_lo || j >= col_hi) continue;
                    const double cj = rint((double)__uint_as_float(t.y) * si);         // C[i, j]
                    const float ms = (float)(fmin(cj, (double)HH_CLIP) / s[j]);        // M0s[i, j]
                    float* __restrict__ dst = m1 + (size_t)(j - col_lo) * (size_t)ld + (size_t)x;
                    *dst = fmaf(vl, ms, *dst);
                }
            }
            np += (unsigned long long)Li;
            __syncwarp();
        }
    }
    if (lane == 0 && np) atomicAdd(products, np);
}

struct hh_mcl {
    hh_ctx* ctx;
    int n, W, T, ch_shift, n_pad;
    int64_t ld;
    int col_lo, col_hi;
    int expansion;
    bool smem_acc;
    size_t smem_bytes;
    int grid_cap;           // resident CTAs of the column kernel
    float* d_scratch;       // global accumulators (large n only)
    hh_slotmat m0;
    float* d_m1;            // dense [ld x (col_hi-col_lo)]
    hh_slotmat it[2];
    int it_cap;
    hh_slotmat pw[2];       // expansion > 2: unpruned powers M^2 .. M^(e-1) of the owned columns (slots of n entries)
    int cur;                // index of the current iterate in it[]; -1 before iteration 0
    int pending;            // buffer hh_mcl_step wrote (to be committed)
    bool have_pending;
    float inflation, prune;
    int inflate_square;
    bool begun;
    int64_t cur_nnz, pending_nnz;   // stored entries of the current / pending iterate (all columns)
    int* d_counter;
    unsigned long long* d_stats;   // [0] nnz [1] products [2] delta bits [3] err
    int64_t nnz_m0, preexp_products;
    int32_t own_lo, own_hi;        // the column block given to hh_mcl_create (dense M1 block); col_lo/col_hi = active block
    int* d_order;                  // [ncols] processing order for the next expansion
    int* d_cnt;                    // [2n] histogram + cursors
    int use_small;                 // warp-per-column kernel for nearly converged iterates
    int* d_bigcount;
    int use_window;                // cluster-contiguous relabelling + windowed expansion
    bool perm_valid;               // perm / lists below are built (once per hh_mcl, from the first pruned iterate)
    bool perm_space;               // the iterates it[] are stored in new (perm) indices
    int last_step_it;              // iteration number of the pending / last committed step
    int* d_perm;                   // [n] original -> new
    int* d_inv;                    // [n] new -> original
    int* d_comp_lo;                // [n] per new index: first row of its component
    int* d_comp_hi;                // [n]
    int* d_owned;                  // [ncols] new indices of the owned columns
    int* d_win_list;               // owned columns whose component fits the window kernel
    int* d_big_list;               // the rest
    int* d_overflow;               // [ncols] overflow list of the small kernel
    int n_win, n_big, wmax;
    std::vector<int>* h_inv;       // host copy of d_inv (result export)
    cudaEvent_t ev0, ev1;
    float create_ms[2];            // device time of the normalisation / pre-expansion kernels
    // block-diagonal iterations on the tensor cores (HH_MCL_BLOCKGEMM): work list of the window components, built with perm
    int use_blk;
    std::vector<hh_gemm_item>* blk_items;
    hh_gemm_item* d_blk_items;
    long long blk_ldk;
    double blk_flops;              // tensor flops one block iteration issues
    int64_t blk_iters;             // iterations that ran as block GEMMs (statistics)
    int preexp_mode;               // HH_PREEXP_SPARSE or HH_PREEXP_DENSE: the engine that built M1
    float clip_ms;                 // dense engine: the sparse correction for counts above HH_CLIP
    hh_gemm_stats gemm;            // tensor-core path: planes, passes, flops, times
};

static void slot_free(hh_slotmat& s) {
    hh_dfree(s.len);
    hh_dfree(s.blk);
    hh_dfree(s.ent);
    s.cap = 0;
}

static int slot_alloc(hh_slotmat& s, int n, int cap, int W) {
    memset(&s, 0, sizeof(s));
    HH_REQUIRE((unsigned long long)n * (unsigned long long)cap <= 0xFFFFFFFFull, HH_ERR_UNSUPPORTED,
               "hh_mcl: %d columns x %d slot entries exceed the 32-bit entry offsets of the expansion kernel", n, cap);
    s.n = n;
    s.cap = cap;
    s.W = W;
    int rc;
    if ((rc = hh_dmalloc(&s.len, (size_t)n)) != HH_OK || (rc = hh_dmalloc(&s.blk, (size_t)n * (W + 1))) != HH_OK ||
        (rc = hh_dmalloc(&s.ent, (size_t)n * (size_t)cap)) != HH_OK) {
        slot_free(s);
        return rc;
    }
    return HH_OK;
}

struct hh_geom {
    int W, T, ch_shift, n_pad;
    bool smem_acc;
    size_t smem_bytes;
};

static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// link count from which an edge of the input matrix is "strong": the components of the strong-link graph order the columns
// of the pre-expansion (hh_k_cc_hook_csc)
static constexpr float HH_PREORDER_STRONG = 10.f;
// largest component (rows) that gets a window: the relabelling and expansion window kernels and the block-diagonal GEMM
// take these; larger components stay on the n-row column kernel
static constexpr int HH_WINDOW_MAX = 8192;

static hh_geom geom_for(hh_ctx* ctx, int n) {
    hh_geom g;
    g.W = (n <= 12288) ? 8 : (n <= 28672 ? 16 : 32);
    int T = (n + g.W - 1) / g.W;
    T = (T + 31) & ~31;
    g.T = T;
    g.n_pad = T * g.W;
    int s = 5;
    while (((T + (1 << s) - 1) >> s) > 64) s++;
    g.ch_shift = s;
    const size_t need = (size_t)g.n_pad * sizeof(float);
    const size_t static_smem = 1024;   // s_d/s_f/s_k/s_c/s_col, rounded up
    g.smem_acc = need + static_smem <= ctx->smem_optin;
    g.smem_bytes = g.smem_acc ? need : 0;
    if (!g.smem_acc) {
        g.W = 32;
        T = (n + 31) / 32;
        T = (T + 31) & ~31;
        g.T = T;
        g.n_pad = T * 32;
        s = 5;
        while (((T + (1 << s) - 1) >> s) > 64) s++;
        g.ch_shift = s;
    }
    return g;
}

template <int W, int SRC, int EPI, bool TRACK, bool FLAT>
static int launch_col_wtf(hh_ctx* ctx, const hh_geom& g, float* d_scratch, int grid_cap, hh_colargs& a) {
    a.scratch = d_scratch;
    int grid = a.ncols < grid_cap ? a.ncols : grid_cap;
    if (grid < 1) return HH_OK;
    HH_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(int), ctx->stream));
    if (g.smem_acc) {
        auto kern = hh_k_col<W, SRC, EPI, true, TRACK, FLAT>;
        HH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem_bytes));
        HH_LAUNCH(ctx, kern, grid, W * 32, g.smem_bytes, a);
    } else {
        auto kern = hh_k_col<W, SRC, EPI, false, TRACK, FLAT>;
        HH_CUDA(cudaMemsetAsync(d_scratch, 0, (size_t)grid_cap * (size_t)g.n_pad * sizeof(float), ctx->stream));
        HH_LAUNCH(ctx, kern, grid, W * 32, 0, a);
    }
    return HH_OK;
}

// dirty-chunk tracking only pays off when a column touches a small part of the accumulator
template <int W, int SRC, int EPI>
static int launch_col_w(hh_ctx* ctx, const hh_geom& g, float* d_scratch, int grid_cap, hh_colargs& a) {
    if (SRC == SRC_PRODUCT) {
        const bool track = (EPI == EPI_PRUNE) && a.track;
        if (a.flat) {
            if (track) return launch_col_wtf<W, SRC, EPI, true, true>(ctx, g, d_scratch, grid_cap, a);
            return launch_col_wtf<W, SRC, EPI, false, true>(ctx, g, d_scratch, grid_cap, a);
        }
        if (track) return launch_col_wtf<W, SRC, EPI, true, false>(ctx, g, d_scratch, grid_cap, a);
        return launch_col_wtf<W, SRC, EPI, false, false>(ctx, g, d_scratch, grid_cap, a);
    }
    return launch_col_wtf<W, SRC, EPI, false, false>(ctx, g, d_scratch, grid_cap, a);
}

template <int SRC, int EPI>
static int launch_col(hh_ctx* ctx, const hh_geom& g, float* d_scratch, int grid_cap, hh_colargs& a) {
    a.n_pad = g.n_pad;
    a.T = g.T;
    a.ch_shift = g.ch_shift;
    switch (g.W) {
        case 8: return launch_col_w<8, SRC, EPI>(ctx, g, d_scratch, grid_cap, a);
        case 16: return launch_col_w<16, SRC, EPI>(ctx, g, d_scratch, grid_cap, a);
        default: return launch_col_w<32, SRC, EPI>(ctx, g, d_scratch, grid_cap, a);
    }
}


// ---------------------------------------------------------------------------------------------
// Iteration 0 of every mcl() call (HapHiC_cluster.py:2030-2042: no expansion, the input IS the pre-expanded dense M1):
// inflate, column L1, prune + keep first maximum, column L1 -- as a stream.  The column never sits in shared memory:
//   pass 1 (HBM)  y = x^r, fp64 column sum S1, maximum of x (x -> x1 is monotone);
//   pass 2 (L2)   only x >= xthr can reach x1 = fp32(fp64(y) / S1) >= pruning: exact quotient for those, count + fp64 sum S2;
//   pass 3 (L2)   the survivors in row order, x2 = fp32(fp64(x1) / S2), into the column's slot.
// Warp w owns row block w (rows [w * T, (w + 1) * T)), so the row-block pointers of the slotted format fall out of the
// per-warp counts.  Two CTAs per SM overlap one column's reductions with the other's loads.
// ---------------------------------------------------------------------------------------------
// x1 of one candidate (rare: a few percent of a column), kept out of line so that the streaming loops stay small -- with powf
// and the fp64 quotient inlined at every use the kernel outgrew the instruction cache and ran 3-7x slower for r != 2
__device__ __noinline__ float hh_it0_x1(float x, double S1, float rf, int sq) {
    const float y = hh_inflate(x, rf, sq);
    return (float)((double)y / S1);
}

// 8 warps per CTA and 4 CTAs per SM: 592 columns (118 MB, the whole L2) are in flight and ncu shows
// all three passes in DRAM (29.6 GB read, L2 hit 4 %) -- but fewer, larger CTAs (59 / 30 MB in flight) are not faster:
// 10.1 / 10.5 / 11.6 ms for 8 / 16 / 32 warps at r = 2.0 on the same device.  The kernel is bound by instruction issue
// (1.0e10 warp instructions, issue slots 61 % busy), not by where the re-reads come from.
// The candidates of passes 2 and 3 (a few percent of the elements) are first collected in a per-warp shared-memory
// queue and then evaluated 32 at a time.  Evaluating them where they are found costs one call of hh_it0_x1 (pow + fp64
// division, ~100 instructions) per warp and element slot that holds at least one candidate -- with 1-2 % candidates that
// is every second slot, executed with one or two active lanes: 7.5e9 of the kernel's 1.0e10 warp instructions (ncu).
constexpr int HH_IT0_WARPS = 8;
template <int W, bool SQ>      // SQ: any of the multiplicative modes (no powf in the streaming loop)
__global__ void __launch_bounds__(HH_IT0_WARPS * 32, 32 / HH_IT0_WARPS) hh_k_iter0(const hh_colargs a) {
    constexpr int QCAP = 256;                       // queue entries per warp (a trip adds at most 128)
    __shared__ float s_qx[HH_IT0_WARPS][QCAP];
    __shared__ unsigned s_qr[HH_IT0_WARPS][QCAP];
    const unsigned lt_mask = (1u << (threadIdx.x & 31)) - 1u;
    // HH_IT0_WARPS warps per CTA (several CTAs per SM keep loads of other columns in flight across the reductions); warp v
    // handles the row blocks v, v + HH_IT0_WARPS, ... of the slotted format (W blocks of T rows)
    __shared__ double s_d[HH_IT0_WARPS];
    __shared__ float s_f[HH_IT0_WARPS];
    __shared__ int s_k[HH_IT0_WARPS];
    __shared__ int s_c[32];          // survivors per row block
    __shared__ int s_col;
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    const int T = a.T;
    const float rf = a.inflation, p32 = a.prune;
    const int sq = a.inflate_square;      // HH_INFL_* mode
    constexpr int U = SQ ? 4 : 1;    // float4 per lane and trip of pass 1 (one copy of powf per component when !SQ)
    const int ld4 = (int)(a.ld >> 2);
    unsigned long long nnz_acc = 0ull;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_col = atomicAdd(a.counter, 1);
        __syncthreads();
        const int jj = s_col;
        if (jj >= a.ncols) break;
        const int j = a.order ? a.order[jj] : (a.col_lo + jj);
        const float4* __restrict__ col4 = reinterpret_cast<const float4*>(a.dense_in + (size_t)(j - a.col_lo) * (size_t)a.ld);
        // ---------------------------------------------------------------- pass 1: S1 and the maximum
        double s1 = 0.0;
        float xbest = 0.f;
        int kbest = 0x7fffffff;
        for (int b = wv; b < W; b += HH_IT0_WARPS) {
            const int r4_lo = (b * T) >> 2, r4_hi = min(((b + 1) * T) >> 2, ld4);
#pragma unroll 1
            for (int r4 = r4_lo + lane; r4 < r4_hi; r4 += 32 * U) {
                float4 x[U];
#pragma unroll
                for (int q = 0; q < U; ++q) x[q] = (r4 + 32 * q < r4_hi) ? hh_ld_stream_f4(col4 + r4 + 32 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int q = 0; q < U; ++q) {
                    const float xv[4] = {x[q].x, x[q].y, x[q].z, x[q].w};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float v = xv[c];
                        if (v != 0.f) {
                            s1 += (double)(SQ ? hh_inflate(v, rf, sq) : powf(v, rf));
                            const int k = ((r4 + 32 * q) << 2) + c;
                            if (v > xbest || (v == xbest && k < kbest)) {
                                xbest = v;
                                kbest = k;
                            }
                        }
                    }
                }
            }
        }
        s1 = hh_warp_sum(s1);
        if (lane == 0) s_d[wv] = s1;
        __syncthreads();
        const double S1 = hh_warp_sum((lane < HH_IT0_WARPS) ? s_d[lane] : 0.0);
        __syncthreads();
        // exact x1 of this lane's maximum; two different x may round to one x1: then the lower row wins (first maximum)
        float vbest = (xbest > 0.f && S1 != 0.0) ? hh_it0_x1(xbest, S1, rf, sq) : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(HH_FULL_MASK, vbest, o);
            const int ok = __shfl_xor_sync(HH_FULL_MASK, kbest, o);
            if (ov > vbest || (ov == vbest && ok < kbest)) {
                vbest = ov;
                kbest = ok;
            }
        }
        // ---------------------------------------------------------------- pass 2: survivors of the prune, S2
        // x1 >= pruning needs y >= 0.999 * pruning * S1, i.e. x >= (that)^(1/r): taken a little lower, the rest is exact
        const float thr_y = (float)(0.999 * (double)p32 * S1);
        const float xthr = (S1 != 0.0) ? 0.9999f * powf(thr_y, 1.0f / rf) : 3.0e38f;
        double s2 = 0.0;
        for (int b = wv; b < W; b += HH_IT0_WARPS) {
            const int r4_lo = (b * T) >> 2, r4_hi = min(((b + 1) * T) >> 2, ld4);
            int cnt = 0;
            int qn = 0;                                  // warp-uniform fill of this warp's queue
            auto drain2 = [&]() {
                __syncwarp();
                for (int i0 = 0; i0 < qn; i0 += 32) {
                    const int i = i0 + lane;
                    if (i < qn) {
                        const float x1 = hh_it0_x1(s_qx[wv][i], S1, rf, sq);
                        if (x1 >= p32 && x1 > 0.f) {
                            cnt++;
                            s2 += (double)x1;
                        }
                    }
                }
                __syncwarp();
                qn = 0;
            };
            for (int r4 = r4_lo; r4 < r4_hi; r4 += 128) {
                const int r4l = r4 + lane;      // warp-uniform trip count, the lane offset is added here
                float4 x[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) x[q] = (r4l + 32 * q < r4_hi) ? hh_ld_stream_f4(col4 + r4l + 32 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float xv[4] = {x[q].x, x[q].y, x[q].z, x[q].w};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const bool cand = xv[c] >= xthr;
                        const unsigned bal = __ballot_sync(HH_FULL_MASK, cand);
                        if (bal) {
                            if (cand) s_qx[wv][qn + __popc(bal & lt_mask)] = xv[c];
                            qn += __popc(bal);
                        }
                    }
                    if (qn > QCAP - 128) drain2();
                }
            }
            if (qn > 0) drain2();
            cnt = hh_warp_sum(cnt);
            if (lane == 0) s_c[b] = cnt;
        }
        s2 = hh_warp_sum(s2);
        if (lane == 0) {
            s_d[wv] = s2;
            s_f[wv] = vbest;
            s_k[wv] = kbest;
        }
        __syncthreads();
        const int cv = (lane < W) ? s_c[lane] : 0;
        double S2 = hh_warp_sum((lane < HH_IT0_WARPS) ? s_d[lane] : 0.0);
        float vmax = (lane < HH_IT0_WARPS) ? s_f[lane] : 0.f;
        int kmax = (lane < HH_IT0_WARPS) ? s_k[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(HH_FULL_MASK, vmax, o);
            const int ok = __shfl_xor_sync(HH_FULL_MASK, kmax, o);
            if (ov > vmax || (ov == vmax && ok < kmax)) {
                vmax = ov;
                kmax = ok;
            }
        }
        int incl = cv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int tt = __shfl_up_sync(HH_FULL_MASK, incl, o);
            if (lane >= o) incl += tt;
        }
        const int excl = incl - cv;                                  // lane b: first output position of row block b
        int total = __shfl_sync(HH_FULL_MASK, incl, 31);
        const bool need_max = (total == 0) && (vmax > 0.f);        // keep the column maximum (2009-2013)
        if (need_max) total = 1;
        // ---------------------------------------------------------------- pass 3: ordered write
        uint2* __restrict__ oent = a.out.ent + (size_t)j * (size_t)a.out.cap;
        if (need_max && threadIdx.x == 0) oent[0] = make_uint2((unsigned)kmax, __float_as_uint(1.0f));      // x1 / x1
        for (int b = wv; b < W; b += HH_IT0_WARPS) {
            const int base = need_max ? ((b > kmax / T) ? 1 : 0) : __shfl_sync(HH_FULL_MASK, excl, b);
            const int mine = need_max ? 0 : __shfl_sync(HH_FULL_MASK, cv, b);
            if (lane == 0) a.out.blk[(size_t)j * (W + 1) + b] = base;
            if (mine == 0) continue;
            const int r4_lo = (b * T) >> 2, r4_hi = min(((b + 1) * T) >> 2, ld4);
            int off = base;
            // candidates into the queue in row order (lane-major, then the four rows of a lane), survivors out of it in the
            // same order: position = off + rank among the survivors of the drained batch
            int qn = 0;
            auto drain3 = [&]() {
                __syncwarp();
                for (int i0 = 0; i0 < qn; i0 += 32) {
                    const int i = i0 + lane;
                    float x1 = 0.f;
                    unsigned row = 0u;
                    if (i < qn) {
                        x1 = hh_it0_x1(s_qx[wv][i], S1, rf, sq);
                        row = s_qr[wv][i];
                    }
                    const bool sv = (i < qn) && x1 >= p32 && x1 > 0.f;
                    const unsigned bal = __ballot_sync(HH_FULL_MASK, sv);
                    if (sv) {
                        const int pos = off + __popc(bal & lt_mask);
                        if (pos < a.out.cap) oent[pos] = make_uint2(row, __float_as_uint((float)((double)x1 / S2)));
                    }
                    off += __popc(bal);
                }
                __syncwarp();
                qn = 0;
            };
            for (int r4 = r4_lo; r4 < r4_hi; r4 += 32) {
                const int rr = r4 + lane;
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rr < r4_hi) x = hh_ld_stream_f4(col4 + rr);
                const float xv[4] = {x.x, x.y, x.z, x.w};
                const bool c0 = xv[0] >= xthr, c1 = xv[1] >= xthr, c2 = xv[2] >= xthr, c3 = xv[3] >= xthr;
                const unsigned b0 = __ballot_sync(HH_FULL_MASK, c0), b1 = __ballot_sync(HH_FULL_MASK, c1);
                const unsigned b2 = __ballot_sync(HH_FULL_MASK, c2), b3 = __ballot_sync(HH_FULL_MASK, c3);
                if ((b0 | b1 | b2 | b3) == 0u) continue;
                int pos = qn + __popc(b0 & lt_mask) + __popc(b1 & lt_mask) + __popc(b2 & lt_mask) + __popc(b3 & lt_mask);
                const bool cc[4] = {c0, c1, c2, c3};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (cc[q]) {
                        s_qx[wv][pos] = xv[q];
                        s_qr[wv][pos] = (unsigned)((rr << 2) + q);
                        pos++;
                    }
                }
                qn += __popc(b0) + __popc(b1) + __popc(b2) + __popc(b3);
                if (qn > QCAP - 128) drain3();
            }
            if (qn > 0) drain3();
        }
        if (threadIdx.x == 0) {
            a.out.blk[(size_t)j * (W + 1) + W] = min(total, a.out.cap);
            a.out.len[j] = min(total, a.out.cap);
            if (total > a.out.cap) atomicExch(a.err, 1);
            nnz_acc += (unsigned long long)total;
        }
    }
    if (threadIdx.x == 0 && nnz_acc) atomicAdd(a.stats + 0, nnz_acc);
}

template <int W>
static int launch_iter0_w(hh_ctx* ctx, hh_colargs& a) {
    auto kern = (a.inflate_square != HH_INFL_POW) ? hh_k_iter0<W, true> : hh_k_iter0<W, false>;
    int per_sm = 0;
    HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, HH_IT0_WARPS * 32, 0));
    if (per_sm < 1) per_sm = 1;
    int grid = per_sm * ctx->sm_count;
    if (grid > a.ncols) grid = a.ncols;
    if (grid < 1) return HH_OK;
    HH_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(int), ctx->stream));
    HH_LAUNCH(ctx, kern, grid, HH_IT0_WARPS * 32, 0, a);
    return HH_OK;
}

static int launch_iter0(hh_ctx* ctx, const hh_geom& g, hh_colargs& a) {
    a.T = g.T;
    switch (g.W) {
        case 8: return launch_iter0_w<8>(ctx, a);
        case 16: return launch_iter0_w<16>(ctx, a);
        default: return launch_iter0_w<32>(ctx, a);
    }
}

static int grid_cap_for(hh_ctx* ctx, const hh_geom& g, int* out) {
    int per_sm = 0;
    if (g.smem_acc) {
        // every instantiation has the same footprint; query the heaviest (product + prune)
        switch (g.W) {
            case 8:
                HH_CUDA(cudaFuncSetAttribute(hh_k_col<8, SRC_PRODUCT, EPI_PRUNE, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)g.smem_bytes));
                HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hh_k_col<8, SRC_PRODUCT, EPI_PRUNE, true, true, true>, 256,
                                                                     g.smem_bytes));
                break;
            case 16:
                HH_CUDA(cudaFuncSetAttribute(hh_k_col<16, SRC_PRODUCT, EPI_PRUNE, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)g.smem_bytes));
                HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hh_k_col<16, SRC_PRODUCT, EPI_PRUNE, true, true, true>, 512,
                                                                     g.smem_bytes));
                break;
            default:
                HH_CUDA(cudaFuncSetAttribute(hh_k_col<32, SRC_PRODUCT, EPI_PRUNE, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)g.smem_bytes));
                HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hh_k_col<32, SRC_PRODUCT, EPI_PRUNE, true, true, true>, 1024,
                                                                     g.smem_bytes));
                break;
        }
    } else {
        per_sm = 2;
    }
    HH_REQUIRE(per_sm >= 1, HH_ERR_UNSUPPORTED, "hh_mcl: the column kernel does not fit on an SM (W=%d, smem=%zu)", g.W, g.smem_bytes);
    *out = per_sm * ctx->sm_count;
    return HH_OK;
}

// ---------------------------------------------------------------------------------------------
// Unsorted CSC column -> row-sorted slot without an n-row accumulator: the rows present are marked in a bitmap (n bits of
// shared memory), an exclusive prefix over the bitmap words gives every row its rank, and every entry writes itself to its
// rank.  d marks + n/32 words scanned + d lookups per column, instead of 2 n rows scanned (the accumulator kernel spent
// 13 ms here at 50k contigs).  Column sum in fp64 (sklearn normalize, 2144; exact in any order for integer link counts, the
// order below is fixed).  A row stored twice in one column (only a caller's own CSC can have that) raises *dup: the caller
// then runs the accumulator kernel, which adds duplicates up.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
hh_k_slot_from_csc(const int64_t* __restrict__ colptr, const int32_t* __restrict__ row, const float* __restrict__ val, int n, int W, int T,
                   int raw, hh_slotmat out, unsigned long long* __restrict__ stats, int* __restrict__ err, int* __restrict__ dup) {
    extern __shared__ uint32_t sfc_smem[];
    const int nw = (n + 31) >> 5;
    const int nw_pad = (nw + 255) & ~255;
    uint32_t* __restrict__ bm = sfc_smem;             // [nw_pad] bitmap of the rows present
    uint32_t* __restrict__ pre = sfc_smem + nw_pad;   // [nw_pad] entries in the words before
    __shared__ double s_part[8];
    __shared__ uint32_t s_wsum[8];
    __shared__ double s_S;
    __shared__ uint32_t s_total;
    const int tid = threadIdx.x, lane = tid & 31, wv = tid >> 5;
    const int per = nw_pad >> 8;                      // bitmap words per thread in the scan
    unsigned long long nnz_acc = 0ull;
    for (int j = blockIdx.x; j < n; j += gridDim.x) {
        const int64_t p0 = colptr[j], p1 = colptr[j + 1];
        for (int w = tid; w < nw_pad; w += 256) bm[w] = 0u;
        __syncthreads();
        double s = 0.0;
        for (int64_t p = p0 + tid; p < p1; p += 256) {
            const float v = val[p];
            if (v != 0.f) {
                const uint32_t r = (uint32_t)row[p];
                const uint32_t bit = 1u << (r & 31u);
                if (atomicOr(&bm[r >> 5], bit) & bit) atomicExch(dup, 1);
                s += fabs((double)v);
            }
        }
        s = hh_warp_sum(s);
        if (lane == 0) s_part[wv] = s;
        __syncthreads();
        // exclusive prefix of popc(bm[]) : thread t owns words [t * per, (t + 1) * per)
        uint32_t mine = 0;
        for (int q = 0; q < per; ++q) mine += __popc(bm[tid * per + q]);
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(HH_FULL_MASK, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_wsum[wv] = incl;
        __syncthreads();
        if (tid == 0) {
            double S = 0.0;
            uint32_t run = 0;
            for (int k = 0; k < 8; ++k) {
                S += s_part[k];
                const uint32_t t = s_wsum[k];
                s_wsum[k] = run;
                run += t;
            }
            s_S = S;
            s_total = run;
        }
        __syncthreads();
        uint32_t run = s_wsum[wv] + incl - mine;
        for (int q = 0; q < per; ++q) {
            pre[tid * per + q] = run;
            run += __popc(bm[tid * per + q]);
        }
        __syncthreads();
        const double S = s_S;
        const int total = (int)s_total;
        uint2* __restrict__ oent = out.ent + (size_t)j * (size_t)out.cap;
        for (int64_t p = p0 + tid; p < p1; p += 256) {
            const float v = val[p];
            if (v != 0.f) {
                const uint32_t r = (uint32_t)row[p];
                const uint32_t pos = pre[r >> 5] + __popc(bm[r >> 5] & ((1u << (r & 31u)) - 1u));
                if ((int)pos < out.cap) oent[pos] = make_uint2(r, __float_as_uint((raw || S == 0.0) ? v : (float)((double)v / S)));
            }
        }
        for (int w = tid; w <= W; w += 256) {
            int b = total;
            if (w < W && w * T < n) b = (int)pre[(w * T) >> 5];        // T is a multiple of 32
            out.blk[(size_t)j * (W + 1) + w] = (w == W) ? min(total, out.cap) : b;
        }
        if (tid == 0) {
            out.len[j] = min(total, out.cap);
            if (total > out.cap) atomicExch(err, 1);
            nnz_acc += (unsigned long long)total;
        }
        __syncthreads();
    }
    if (tid == 0 && nnz_acc) atomicAdd(stats + 0, nnz_acc);
}

// unsorted CSC -> slotted (raw or column-normalised); cap must be >= the longest column
static int slot_from_csc_fast(hh_ctx* ctx, const hh_geom& g, int* d_counter, unsigned long long* d_stats, const hh_matrix* m, int raw,
                              hh_slotmat& out, bool* done) {
    *done = false;
    const int nw_pad = (((m->n + 31) >> 5) + 255) & ~255;
    const size_t smem = (size_t)nw_pad * 2 * sizeof(uint32_t);
    if (smem + 1024 > ctx->smem_optin) return HH_OK;
    auto kern = hh_k_slot_from_csc;
    HH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem));
    if (per_sm < 1) return HH_OK;
    int grid = per_sm * ctx->sm_count;
    if (grid > m->n) grid = m->n;
    HH_CUDA(cudaMemsetAsync(d_counter, 0, sizeof(int), ctx->stream));
    HH_LAUNCH(ctx, kern, grid, 256, smem, m->d_colptr, m->d_row, m->d_val, m->n, g.W, g.T, raw, out, d_stats,
              reinterpret_cast<int*>(d_stats + 3), d_counter);
    int dup = 0;
    HH_CUDA(cudaMemcpyAsync(&dup, d_counter, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    if (dup) {
        HH_CUDA(cudaMemsetAsync(d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));      // every caller zeroed it before
        return HH_OK;
    }
    *done = true;
    return HH_OK;
}

static int slot_from_csc(hh_ctx* ctx, const hh_geom& g, float* d_scratch, int grid_cap, int* d_counter, unsigned long long* d_stats,
                         const hh_matrix* m, int raw, hh_slotmat& out) {
    bool done = false;
    HH_CHECK(slot_from_csc_fast(ctx, g, d_counter, d_stats, m, raw, out, &done));
    if (done) return HH_OK;
    hh_colargs a;
    memset(&a, 0, sizeof(a));
    a.n = m->n;
    a.col_lo = 0;
    a.ncols = m->n;
    a.counter = d_counter;
    a.csc_ptr = m->d_colptr;
    a.csc_row = m->d_row;
    a.csc_val = m->d_val;
    a.out = out;
    a.raw = raw;
    a.stats = d_stats;
    a.delta_bits = reinterpret_cast<int*>(d_stats + 2);
    a.err = reinterpret_cast<int*>(d_stats + 3);
    return launch_col<SRC_CSC, EPI_NORM>(ctx, g, d_scratch, grid_cap, a);
}

static int max_col_len(hh_ctx* ctx, const hh_matrix* m, int* out) {
    std::vector<int64_t> ptr((size_t)m->n + 1);
    HH_CUDA(cudaMemcpyAsync(ptr.data(), m->d_colptr, ptr.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    int64_t mx = 1;
    for (int c = 0; c < m->n; ++c) {
        const int64_t l = ptr[c + 1] - ptr[c];
        if (l > mx) mx = l;
    }
    *out = (int)(mx < m->n ? mx : m->n);
    return HH_OK;
}

// slotted -> canonical CSC on the host
static int slot_fetch_csc(hh_ctx* ctx, const hh_slotmat& s, int col_lo, int ncols, int64_t* indptr, int32_t* indices, float* data,
                          const int* d_colmap = nullptr, const std::vector<int>* h_rowinv = nullptr) {
    int64_t* d_off = nullptr;
    int* d_idx = nullptr;
    float* d_val = nullptr;
    int* d_len = nullptr;
    HH_CHECK(hh_dmalloc(&d_off, (size_t)ncols + 1));
    int rc = [&]() -> int {
        HH_CHECK(hh_dmalloc(&d_len, (size_t)ncols));
        HH_LAUNCH(ctx, hh_k_gather_len, (ncols + 255) / 256, 256, 0, s.len, d_colmap, col_lo, ncols, d_len);
        HH_CHECK(hh_exclusive_scan_i32(ctx, d_len, d_off, ncols));
        if (indptr) HH_CUDA(cudaMemcpyAsync(indptr, d_off, ((size_t)ncols + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaMemcpyAsync(ctx->h_scratch, d_off + ncols, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        const int64_t nnz = (int64_t)ctx->h_scratch[0];
        if (nnz == 0 || (!indices && !data)) return HH_OK;
        HH_CHECK(hh_dmalloc(&d_idx, (size_t)nnz));
        HH_CHECK(hh_dmalloc(&d_val, (size_t)nnz));
        int grid = (ncols + 7) / 8;
        if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
        HH_LAUNCH(ctx, hh_k_pack, grid, 256, 0, s, col_lo, ncols, d_off, (int*)nullptr, d_idx, d_val, d_colmap);
        if (indices) HH_CUDA(cudaMemcpyAsync(indices, d_idx, (size_t)nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (data) HH_CUDA(cudaMemcpyAsync(data, d_val, (size_t)nnz * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        if (h_rowinv && indices && data && indptr) {
            // rows are new indices: translate to original ones and restore ascending order inside every column
            std::vector<std::pair<int32_t, float>> tmp;
            for (int c = 0; c < ncols; ++c) {
                const int64_t b = indptr[c], e = indptr[c + 1];
                tmp.resize((size_t)(e - b));
                for (int64_t q = b; q < e; ++q) tmp[(size_t)(q - b)] = std::make_pair((int32_t)(*h_rowinv)[(size_t)indices[q]], data[q]);
                std::sort(tmp.begin(), tmp.end(), [](const std::pair<int32_t, float>& x, const std::pair<int32_t, float>& y) { return x.first < y.first; });
                for (int64_t q = b; q < e; ++q) {
                    indices[q] = tmp[(size_t)(q - b)].first;
                    data[q] = tmp[(size_t)(q - b)].second;
                }
            }
        }
        return HH_OK;
    }();
    hh_dfree(d_off);
    hh_dfree(d_idx);
    hh_dfree(d_val);
    hh_dfree(d_len);
    return rc;
}

static int read_stats(hh_ctx* ctx, unsigned long long* d_stats, unsigned long long out[4]) {
    HH_CUDA(cudaMemcpyAsync(ctx->h_scratch + 16, d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 4; ++k) out[k] = ctx->h_scratch[16 + k];
    return HH_OK;
}

extern "C" int hh_matrix_fetch_csc(hh_matrix* m, int64_t* indptr, int32_t* indices, float* data) {
    HH_REQUIRE(m != nullptr, HH_ERR_ARG, "hh_matrix_fetch_csc: NULL handle");
    hh_scope _scope(m->ctx);
    hh_ctx* ctx = m->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    const hh_geom g = geom_for(ctx, m->n);
    int grid_cap = 0;
    HH_CHECK(grid_cap_for(ctx, g, &grid_cap));
    int cap = 0;
    HH_CHECK(max_col_len(ctx, m, &cap));
    hh_slotmat s;
    HH_CHECK(slot_alloc(s, m->n, cap, g.W));
    float* d_scratch = nullptr;
    int* d_counter = nullptr;
    unsigned long long* d_stats = nullptr;
    int rc = [&]() -> int {
        if (!g.smem_acc) HH_CHECK(hh_dmalloc(&d_scratch, (size_t)grid_cap * (size_t)g.n_pad));
        HH_CHECK(hh_dmalloc(&d_counter, 1));
        HH_CHECK(hh_dmalloc(&d_stats, 4));
        HH_CUDA(cudaMemsetAsync(d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
        HH_CHECK(slot_from_csc(ctx, g, d_scratch, grid_cap, d_counter, d_stats, m, 1, s));
        unsigned long long st[4];
        HH_CHECK(read_stats(ctx, d_stats, st));
        HH_REQUIRE((int)st[3] == 0, HH_ERR_CAPACITY, "hh_matrix_fetch_csc: column slot overflow");
        return slot_fetch_csc(ctx, s, 0, m->n, indptr, indices, data);
    }();
    hh_dfree(d_scratch);
    hh_dfree(d_counter);
    hh_dfree(d_stats);
    slot_free(s);
    return rc;
}

extern "C" int hh_matrix_rank_sums(hh_matrix* m, int topN, int64_t* rank_sum) {
    HH_REQUIRE(m && rank_sum, HH_ERR_ARG, "hh_matrix_rank_sums: NULL argument");
    hh_scope _scope(m->ctx);
    HH_REQUIRE(topN >= 2 && topN <= HH_TOPN_MAX, HH_ERR_UNSUPPORTED, "hh_matrix_rank_sums: topN must be in [2, %d]", HH_TOPN_MAX);
    HH_REQUIRE(topN <= m->n, HH_ERR_ARG, "hh_matrix_rank_sums: topN exceeds the number of fragments");
    hh_ctx* ctx = m->ctx;
    const hh_geom g = geom_for(ctx, m->n);
    int grid_cap = 0;
    HH_CHECK(grid_cap_for(ctx, g, &grid_cap));
    int cap = 0;
    HH_CHECK(max_col_len(ctx, m, &cap));
    hh_slotmat s;
    HH_CHECK(slot_alloc(s, m->n, cap, g.W));
    float* d_scratch = nullptr;
    int* d_counter = nullptr;
    unsigned long long* d_stats = nullptr;
    int* d_top = nullptr;
    long long* d_out = nullptr;
    int rc = [&]() -> int {
        if (!g.smem_acc) HH_CHECK(hh_dmalloc(&d_scratch, (size_t)grid_cap * (size_t)g.n_pad));
        HH_CHECK(hh_dmalloc(&d_counter, 1));
        HH_CHECK(hh_dmalloc(&d_stats, 4));
        HH_CHECK(hh_dmalloc(&d_top, (size_t)m->n * topN));
        HH_CHECK(hh_dmalloc(&d_out, (size_t)m->n));
        HH_CUDA(cudaMemsetAsync(d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
        HH_CHECK(slot_from_csc(ctx, g, d_scratch, grid_cap, d_counter, d_stats, m, 1, s));     // rows sorted, raw values
        int grid = (m->n + 7) / 8;
        if (grid > ctx->sm_count * 16) grid = ctx->sm_count * 16;
        HH_LAUNCH(ctx, hh_k_topn, grid, 256, 0, s, topN, d_top);
        HH_LAUNCH(ctx, hh_k_rank_sum, grid, 256, 0, s, topN, d_top, d_out);
        HH_CUDA(cudaMemcpyAsync(rank_sum, d_out, (size_t)m->n * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        unsigned long long st[4];
        HH_CHECK(read_stats(ctx, d_stats, st));
        HH_REQUIRE((int)st[3] == 0, HH_ERR_CAPACITY, "hh_matrix_rank_sums: column slot overflow");
        return HH_OK;
    }();
    hh_dfree(d_scratch);
    hh_dfree(d_counter);
    hh_dfree(d_stats);
    hh_dfree(d_top);
    hh_dfree(d_out);
    slot_free(s);
    return rc;
}

extern "C" int hh_mcl_destroy(hh_mcl* mc) {
    if (!mc) return HH_OK;
    hh_scope _scope(mc->ctx);
    cudaSetDevice(mc->ctx->device);
    cudaStreamSynchronize(mc->ctx->stream);
    slot_free(mc->m0);
    slot_free(mc->it[0]);
    slot_free(mc->it[1]);
    slot_free(mc->pw[0]);
    slot_free(mc->pw[1]);
    hh_dfree(mc->d_m1);
    hh_dfree(mc->d_scratch);
    hh_dfree(mc->d_counter);
    hh_dfree(mc->d_stats);
    hh_dfree(mc->d_order);
    hh_dfree(mc->d_cnt);
    hh_dfree(mc->d_bigcount);
    hh_dfree(mc->d_perm);
    hh_dfree(mc->d_inv);
    hh_dfree(mc->d_comp_lo);
    hh_dfree(mc->d_comp_hi);
    hh_dfree(mc->d_owned);
    hh_dfree(mc->d_win_list);
    hh_dfree(mc->d_big_list);
    hh_dfree(mc->d_overflow);
    hh_dfree(mc->d_blk_items);
    delete mc->blk_items;
    delete mc->h_inv;
    if (mc->ev0) cudaEventDestroy(mc->ev0);
    if (mc->ev1) cudaEventDestroy(mc->ev1);
    delete mc;
    return HH_OK;
}

static hh_geom mcl_geom(const hh_mcl* mc) {
    hh_geom g;
    g.W = mc->W;
    g.T = mc->T;
    g.ch_shift = mc->ch_shift;
    g.n_pad = mc->n_pad;
    g.smem_acc = mc->smem_acc;
    g.smem_bytes = mc->smem_bytes;
    return g;
}

static void mcl_base_args(hh_mcl* mc, hh_colargs& a) {
    memset(&a, 0, sizeof(a));
    a.n = mc->n;
    a.col_lo = mc->col_lo;
    a.ncols = mc->col_hi - mc->col_lo;
    a.counter = mc->d_counter;
    a.ld = mc->ld;
    a.stats = mc->d_stats;
    a.delta_bits = reinterpret_cast<int*>(mc->d_stats + 2);
    a.err = reinterpret_cast<int*>(mc->d_stats + 3);
}

// Expansion inner loop by the mean entries per (column, row block) segment of the operand A: below 16 the flat walk beats
// the segment-wise one (measured on B200, 50k contigs: 32 -> segment-wise 180 ms vs flat 267 ms; 12 -> 71 ms vs 61 ms).
// The next batch's segments are prefetched into L2 in segment-wise mode only (long segments).
static void choose_walk(const hh_mcl* mc, double nnz_operand, hh_colargs& a) {
    const double seg = nnz_operand / (double)mc->n / (double)mc->W;
    a.flat = seg < 16.0 ? 1 : 0;
    a.l2pf = !a.flat;
}

// out[:, owned] = A . B[:, owned] as an unpruned slotted matrix: one factor of mkl_matrix_power's recursion
// A . A^(k-1) (HapHiC_cluster.py:2017-2023) for --expansion k > 2
static int raw_product(hh_mcl* mc, const hh_slotmat& A, const hh_slotmat& B, double nnz_a, hh_slotmat& out) {
    hh_colargs a;
    mcl_base_args(mc, a);
    a.A = A;
    a.B = B;
    a.out = out;
    a.raw = 1;
    choose_walk(mc, nnz_a, a);
    const hh_geom g = mcl_geom(mc);
    HH_CHECK((launch_col<SRC_PRODUCT, EPI_NORM>(mc->ctx, g, mc->d_scratch, mc->grid_cap, a)));
    return HH_OK;
}

// Which engine builds M1.  The Gustavson kernel does n*d^2 multiply-adds on a scattered accumulator, the tensor-core
// GEMM 2 passes of n^3/2 (3 in the exact bf16 encoding).  AUTO picks the cheaper estimate; HH_MCL_PREEXP=sparse|dense overrides.
static int choose_preexp(const hh_matrix* m, int requested) {
    const char* e = getenv("HH_MCL_PREEXP");
    if (e && *e) {
        if (!strcmp(e, "sparse")) return HH_PREEXP_SPARSE;
        if (!strcmp(e, "dense")) return HH_PREEXP_DENSE;
    }
    if (requested == HH_PREEXP_SPARSE || requested == HH_PREEXP_DENSE) return requested;
    // measured on B200: Gustavson ~0.5e12 products/s; tensor-core GEMM ~1.9e15 flop/s issued over two f16 passes of the
    // symmetric half, plus operand planes (memset + scatter) and allocation
    const double n = (double)m->n, d = (double)m->nnz / (n > 0 ? n : 1.0);
    // (above 57,600 vertices the column accumulator no longer fits shared memory: measured 8.5 s per rank for 1/8 of the
    // columns at 150k contigs / 1B pairs, about ten times the shared-memory rate)
    const double t_sparse = n * d * d / (n > 57600.0 ? 0.05e12 : 0.5e12);
    const double t_dense = 1.2e-15 * n * n * n + 3.0e-12 * n * n + 5.0e-4;
    // the operand planes (up to six bf16 planes of n x n) must fit beside M1 and the iterates
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
        cudaGetLastError();
        free_b = 0;
    }
    // the operand planes of one K chunk (hh_gemm_preexpand cuts the K range so that a chunk stays below ~36 GB; six bf16
    // planes in the worst case) must fit beside M1 and the iterates
    const double planes_all = 6.0 * 2.0 * n * n;
    const double planes = planes_all / (double)((int)(planes_all / 36.0e9) + 1);
    if (planes > 0.5 * (double)free_b) return HH_PREEXP_SPARSE;
    return (1.2 * t_dense < t_sparse) ? HH_PREEXP_DENSE : HH_PREEXP_SPARSE;
}

extern "C" int hh_mcl_create(hh_matrix* m, int expansion, int32_t col_lo, int32_t col_hi, hh_mcl** out) {
    return hh_mcl_create_ex(m, expansion, col_lo, col_hi, HH_PREEXP_AUTO, out);
}

extern "C" int hh_mcl_create_ex(hh_matrix* m, int expansion, int32_t col_lo, int32_t col_hi, int preexp_mode, hh_mcl** out) {
    HH_REQUIRE(m && out, HH_ERR_ARG, "hh_mcl_create: NULL argument");
    hh_scope _scope(m->ctx);
    *out = nullptr;
    HH_REQUIRE(expansion >= 2 && expansion <= 8, HH_ERR_UNSUPPORTED,
               "hh_mcl_create: expansion %d is not supported (2 .. 8; the reference's default is 2)", expansion);
    HH_REQUIRE(0 <= col_lo && col_lo < col_hi && col_hi <= m->n, HH_ERR_ARG, "hh_mcl_create: bad column block [%d, %d) for n = %d",
               col_lo, col_hi, m->n);
    hh_ctx* ctx = m->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    hh_mcl* mc = new (std::nothrow) hh_mcl();
    HH_REQUIRE(mc != nullptr, HH_ERR_NOMEM, "hh_mcl_create: out of host memory");
    memset(mc, 0, sizeof(*mc));
    mc->ctx = ctx;
    mc->n = m->n;
    mc->col_lo = col_lo;
    mc->col_hi = col_hi;
    mc->own_lo = col_lo;
    mc->own_hi = col_hi;
    mc->expansion = expansion;
    mc->cur = -1;
    mc->use_small = 1;
    mc->use_window = 1;
    mc->use_blk = env_int("HH_MCL_BLOCKGEMM", 1);
    if (expansion != 2) {          // higher powers go through the plain column kernel: A . (A . (... A)), one factor at a time
        mc->use_small = 0;
        mc->use_window = 0;
        mc->use_blk = 0;
    }
    mc->blk_items = new std::vector<hh_gemm_item>();
    const hh_geom g = geom_for(ctx, m->n);
    mc->W = g.W;
    mc->T = g.T;
    mc->ch_shift = g.ch_shift;
    mc->n_pad = g.n_pad;
    mc->smem_acc = g.smem_acc;
    mc->smem_bytes = g.smem_bytes;
    mc->ld = ((int64_t)m->n + 31) & ~31ll;
    int rc = [&]() -> int {
        HH_CHECK(grid_cap_for(ctx, g, &mc->grid_cap));
        HH_CUDA(cudaEventCreate(&mc->ev0));
        HH_CUDA(cudaEventCreate(&mc->ev1));
        if (!g.smem_acc) HH_CHECK(hh_dmalloc(&mc->d_scratch, (size_t)mc->grid_cap * (size_t)g.n_pad));
        HH_CHECK(hh_dmalloc(&mc->d_counter, 1));
        HH_CHECK(hh_dmalloc(&mc->d_stats, 4));
        HH_CHECK(hh_dmalloc(&mc->d_order, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_cnt, (size_t)m->n * 2));
        HH_CHECK(hh_dmalloc(&mc->d_bigcount, 4));
        HH_CHECK(hh_dmalloc(&mc->d_perm, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_inv, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_comp_lo, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_comp_hi, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_owned, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_win_list, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_big_list, (size_t)m->n));
        HH_CHECK(hh_dmalloc(&mc->d_overflow, (size_t)m->n));
        HH_CUDA(cudaMemsetAsync(mc->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
        // 1) M0 = normalize(link_matrix, 'l1', axis=0)   (2144)
        int cap0 = 0;
        HH_CHECK(max_col_len(ctx, m, &cap0));
        HH_CHECK(slot_alloc(mc->m0, m->n, cap0, g.W));
        HH_CUDA(cudaEventRecord(mc->ev0, ctx->stream));
        HH_CHECK(slot_from_csc(ctx, g, mc->d_scratch, mc->grid_cap, mc->d_counter, mc->d_stats, m, 0, mc->m0));
        HH_CUDA(cudaEventRecord(mc->ev1, ctx->stream));
        unsigned long long st[4];
        HH_CHECK(read_stats(ctx, mc->d_stats, st));
        HH_CUDA(cudaEventElapsedTime(&mc->create_ms[0], mc->ev0, mc->ev1));
        HH_REQUIRE((int)st[3] == 0, HH_ERR_CAPACITY, "hh_mcl_create: column slot overflow while normalising");
        mc->nnz_m0 = (int64_t)st[0];
        // 2) M1 = M0 . M0 for the owned columns, kept dense and resident   (2146-2149)
        const int ncols = col_hi - col_lo;
        HH_CHECK(hh_dmalloc(&mc->d_m1, (size_t)mc->ld * (size_t)ncols));
        HH_CUDA(cudaMemsetAsync(mc->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
        mc->preexp_mode = (expansion == 2) ? choose_preexp(m, preexp_mode) : HH_PREEXP_SPARSE;
        if (expansion > 2) {
            HH_CHECK(slot_alloc(mc->pw[0], m->n, m->n, g.W));
            if (expansion > 3) HH_CHECK(slot_alloc(mc->pw[1], m->n, m->n, g.W));
        }
        if (mc->preexp_mode == HH_PREEXP_DENSE) {
            // dense-block path: the whole product as a symmetric GEMM on the tensor cores (hh_gemm.cu)
            std::vector<hh_gemm_item> items;
            HH_CHECK(hh_gemm_items_full(m->n, col_lo, col_hi, items));
            HH_CHECK(hh_gemm_preexpand(ctx, m, col_lo, col_hi, mc->d_m1, mc->ld, items.data(), (int)items.size(), &mc->gemm));
            mc->create_ms[1] = mc->gemm.densify_ms + mc->gemm.gemm_ms;
            mc->preexp_products = 0;
            if (mc->gemm.clipped) {
                // finish the few link counts above the clip threshold (hh_k_clip_fix)
                float* d_bclip = nullptr;
                double* d_s = nullptr;
                int rc2 = [&]() -> int {
                    HH_CHECK(hh_dmalloc(&d_bclip, (size_t)m->n));
                    HH_CHECK(hh_dmalloc(&d_s, (size_t)m->n));
                    HH_CUDA(cudaMemsetAsync(mc->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
                    HH_CUDA(cudaEventRecord(mc->ev0, ctx->stream));
                    const int grid = (m->n + 7) / 8;
                    HH_LAUNCH(ctx, hh_k_clip_stats, grid, 256, 0, m->d_colptr, m->d_val, m->n, d_s, d_bclip, mc->gemm.clip);
                    HH_LAUNCH(ctx, hh_k_clip_fix<0>, grid, 256, 0, mc->m0, d_s, d_bclip, mc->d_m1, (long long)mc->ld, (int)col_lo, (int)col_hi,
                              mc->d_stats + 1, mc->gemm.clip);
                    HH_LAUNCH(ctx, hh_k_clip_fix<1>, grid, 256, 0, mc->m0, d_s, d_bclip, mc->d_m1, (long long)mc->ld, (int)col_lo, (int)col_hi,
                              mc->d_stats + 1, mc->gemm.clip);
                    HH_CUDA(cudaEventRecord(mc->ev1, ctx->stream));
                    unsigned long long st2[4];
                    HH_CHECK(read_stats(ctx, mc->d_stats, st2));
                    float ms = 0.f;
                    HH_CUDA(cudaEventElapsedTime(&ms, mc->ev0, mc->ev1));
                    mc->clip_ms = ms;
                    mc->create_ms[1] += ms;
                    mc->preexp_products = (int64_t)st2[1];
                    return HH_OK;
                }();
                hh_dfree(d_bclip);
                hh_dfree(d_s);
                HH_CHECK(rc2);
            }
            return HH_OK;
        }
        // --expansion k > 2: M0^(k-1) of the owned columns first, one unpruned product per factor
        const hh_slotmat* Bp = &mc->m0;
        HH_CUDA(cudaEventRecord(mc->ev0, ctx->stream));
        for (int pwr = 2; pwr < expansion; ++pwr) {
            HH_CHECK(raw_product(mc, mc->m0, *Bp, (double)mc->nnz_m0, mc->pw[pwr & 1]));
            Bp = &mc->pw[pwr & 1];
        }
        if (expansion > 2) {
            HH_CHECK(read_stats(ctx, mc->d_stats, st));
            HH_REQUIRE((int)(st[3] & 0xffffffffull) == 0, HH_ERR_CAPACITY, "hh_mcl_create: slot overflow in a matrix power");
        }
        hh_colargs a;
        mcl_base_args(mc, a);
        a.A = mc->m0;
        a.B = *Bp;
        a.dense_out = mc->d_m1;
        choose_walk(mc, (double)mc->nnz_m0, a);
        {   // column preorder: components of the strong-link graph
            const int n = m->n;
            int* d_lab = mc->d_comp_lo;        // n-sized scratch, rewritten by mcl_build_perm later
            int* d_flag = mc->d_bigcount + 2;
            HH_LAUNCH(ctx, hh_k_cc_init, (n + 255) / 256, 256, 0, d_lab, n);
            int gridc = (n + 7) / 8;
            if (gridc > ctx->sm_count * 16) gridc = ctx->sm_count * 16;
            for (int round = 0; round < 64; ++round) {
                HH_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), ctx->stream));
                HH_LAUNCH(ctx, hh_k_cc_hook_csc, gridc, 256, 0, m->d_colptr, m->d_row, m->d_val, n, HH_PREORDER_STRONG, d_lab, d_flag);
                HH_LAUNCH(ctx, hh_k_cc_jump, (n + 255) / 256, 256, 0, d_lab, n);
                int changed = 0;
                HH_CUDA(cudaMemcpyAsync(&changed, d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
                HH_CUDA(cudaStreamSynchronize(ctx->stream));
                if (!changed) break;
            }
            HH_CUDA(cudaMemsetAsync(mc->d_cnt, 0, (size_t)n * sizeof(int), ctx->stream));
            HH_LAUNCH(ctx, hh_k_cc_rank, (n + 255) / 256, 256, 0, d_lab, n, mc->d_perm, mc->d_inv, mc->d_cnt);
            a.order = mc->d_inv;              // columns sorted by (component, index)
            if (col_lo != 0 || col_hi != n) {
                // column shard: the owned columns in the same order
                HH_LAUNCH(ctx, hh_k_filter_range, 1, 1024, 0, mc->d_inv, n, (int)col_lo, (int)col_hi, mc->d_order);
                a.order = mc->d_order;
            }
        }
        if (expansion == 2) HH_CUDA(cudaEventRecord(mc->ev0, ctx->stream));
        HH_CHECK((launch_col<SRC_PRODUCT, EPI_DUMP>(ctx, g, mc->d_scratch, mc->grid_cap, a)));
        HH_CUDA(cudaEventRecord(mc->ev1, ctx->stream));
        HH_CHECK(read_stats(ctx, mc->d_stats, st));
        HH_CUDA(cudaEventElapsedTime(&mc->create_ms[1], mc->ev0, mc->ev1));
        mc->preexp_products = (int64_t)st[1];
        return HH_OK;
    }();
    if (rc != HH_OK) {
        hh_mcl_destroy(mc);
        return rc;
    }
    *out = mc;
    return HH_OK;
}

extern "C" int hh_mcl_info(hh_mcl* mc, int32_t* n, int64_t* nnz_m0, int64_t* preexp_products, float* normalize_ms,
                           float* preexp_ms) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_info: NULL handle");
    if (n) *n = mc->n;
    if (nnz_m0) *nnz_m0 = mc->nnz_m0;
    if (preexp_products) *preexp_products = mc->preexp_products;
    if (normalize_ms) *normalize_ms = mc->create_ms[0];
    if (preexp_ms) *preexp_ms = mc->create_ms[1];
    return HH_OK;
}

extern "C" int hh_mcl_preexp_info(hh_mcl* mc, hh_preexp_info* info) {
    HH_REQUIRE(mc && info, HH_ERR_ARG, "hh_mcl_preexp_info: NULL argument");
    memset(info, 0, sizeof(*info));
    info->mode = mc->preexp_mode;
    info->total_ms = mc->create_ms[1];
    if (mc->preexp_mode == HH_PREEXP_DENSE) {
        info->a_planes = mc->gemm.a_planes;
        info->passes = mc->gemm.passes;
        info->cta_group = mc->gemm.cta_group;
        info->stages = mc->gemm.stages;
        info->chunk_kb = mc->gemm.chunk_kb;
        info->densify_ms = mc->gemm.densify_ms;
        info->gemm_ms = mc->gemm.gemm_ms;
        info->flops = mc->gemm.flops;
        info->clip_ms = mc->clip_ms;
        info->products = mc->preexp_products;
        info->clip = mc->gemm.clip;
        info->b_planes = mc->gemm.b_planes;
        info->fmt_a = mc->gemm.fmt_a;
        info->fmt_b = mc->gemm.fmt_b;
        info->k_chunks = mc->gemm.k_chunks;
    } else {
        info->products = mc->preexp_products;
    }
    return HH_OK;
}

extern "C" int hh_mcl_fetch_m0(hh_mcl* mc, int64_t* indptr, int32_t* indices, float* data) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_fetch_m0: NULL handle");
    hh_scope _scope(mc->ctx);
    HH_CUDA(cudaSetDevice(mc->ctx->device));
    return slot_fetch_csc(mc->ctx, mc->m0, 0, mc->n, indptr, indices, data);
}

extern "C" int hh_mcl_fetch_m1(hh_mcl* mc, float* dense) {
    HH_REQUIRE(mc && dense, HH_ERR_ARG, "hh_mcl_fetch_m1: NULL argument");
    HH_CUDA(cudaSetDevice(mc->ctx->device));
    const int ncols = mc->own_hi - mc->own_lo;
    HH_CUDA(cudaMemcpy2DAsync(dense, (size_t)mc->n * sizeof(float), mc->d_m1, (size_t)mc->ld * sizeof(float),
                              (size_t)mc->n * sizeof(float), (size_t)ncols, cudaMemcpyDeviceToHost, mc->ctx->stream));
    HH_CUDA(cudaStreamSynchronize(mc->ctx->stream));
    return HH_OK;
}

// components of the committed iterate's pattern -> perm / inv / component windows / column lists, then the
// iterate itself is rewritten in new indices (one pass of the column kernel)
// work list of the block-diagonal GEMM: all tiles of every window component.  Needs whole-matrix ownership (the columns of
// a shard are scattered over the components): built with the relabelling when the context owns every column, or by
// hh_mcl_set_block(0, n) when a sharded run goes on replicated.
static int mcl_build_blk_items(hh_mcl* mc) {
    hh_ctx* ctx = mc->ctx;
    const int n = mc->n;
    mc->blk_items->clear();
    mc->blk_ldk = 0;
    mc->blk_flops = 0.0;
    if (mc->use_blk && mc->col_lo == 0 && mc->col_hi == n && mc->n_win > 0) {
        std::vector<int> clo((size_t)n), chi((size_t)n);
        HH_CUDA(cudaMemcpyAsync(clo.data(), mc->d_comp_lo, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaMemcpyAsync(chi.data(), mc->d_comp_hi, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        const int T = hh_gemm_tile_size();
        int maxb = 0;
        for (int p0 = 0; p0 < n;) {
            const int lo = clo[(size_t)p0], hi = chi[(size_t)p0];
            const int b = hi - lo;
            if (b <= HH_WINDOW_MAX) {
                if (b > maxb) maxb = b;
                const int nt = (b + T - 1) / T, nkb = (b + 63) / 64;
                for (int mt = 0; mt < nt; ++mt)
                    for (int tt = 0; tt < nt; ++tt) {
                        hh_gemm_item w;
                        memset(&w, 0, sizeof(w));
                        w.m0 = lo + mt * T;
                        w.n0 = lo + tt * T;
                        w.m_end = hi;
                        w.n_end = hi;
                        w.kb_lo[0] = 0;
                        w.kb_hi[0] = nkb;
                        w.flags = HH_GEMM_DIRECT;
                        w.out_row0 = lo;
                        mc->blk_items->push_back(w);
                    }
                mc->blk_flops += 2.0 * (double)T * (double)T * 64.0 * (double)nkb * (double)nt * (double)nt * 6.0;
            }
            p0 = hi > p0 ? hi : p0 + 1;
        }
        mc->blk_ldk = ((long long)maxb + 63) & ~63ll;
        hh_dfree(mc->d_blk_items);
        if (!mc->blk_items->empty()) {
            HH_CHECK(hh_dmalloc(&mc->d_blk_items, mc->blk_items->size()));
            HH_CUDA(cudaMemcpyAsync(mc->d_blk_items, mc->blk_items->data(), mc->blk_items->size() * sizeof(hh_gemm_item),
                                    cudaMemcpyHostToDevice, ctx->stream));
            HH_CUDA(cudaStreamSynchronize(ctx->stream));
        }
    }
    return HH_OK;
}

static int mcl_build_perm(hh_mcl* mc) {
    hh_ctx* ctx = mc->ctx;
    const int n = mc->n;
    const hh_geom g = mcl_geom(mc);
    const hh_slotmat& M = mc->it[mc->cur];
    int* d_csize = mc->d_cnt;             // [n] component sizes (+ [n..2n) unused)
    int* d_flag = mc->d_bigcount + 2;
    const int ncols = mc->col_hi - mc->col_lo;
    int* d_lab = nullptr;
    HH_CHECK(hh_dmalloc(&d_lab, (size_t)n));
    int rc = [&]() -> int {
        HH_LAUNCH(ctx, hh_k_cc_init, (n + 255) / 256, 256, 0, d_lab, n);
        int grid = (n + 7) / 8;
        if (grid > ctx->sm_count * 16) grid = ctx->sm_count * 16;
        for (int round = 0; round < 64; ++round) {
            HH_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), ctx->stream));
            HH_LAUNCH(ctx, hh_k_cc_hook, grid, 256, 0, M, d_lab, d_flag);
            HH_LAUNCH(ctx, hh_k_cc_jump, (n + 255) / 256, 256, 0, d_lab, n);
            int changed = 0;
            HH_CUDA(cudaMemcpyAsync(&changed, d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            HH_CUDA(cudaStreamSynchronize(ctx->stream));
            if (!changed) break;
        }
        HH_CUDA(cudaMemsetAsync(d_csize, 0, (size_t)n * sizeof(int), ctx->stream));
        HH_LAUNCH(ctx, hh_k_cc_rank, (n + 255) / 256, 256, 0, d_lab, n, mc->d_perm, mc->d_inv, d_csize);
        HH_LAUNCH(ctx, hh_k_cc_ranges, (n + 255) / 256, 256, 0, d_lab, mc->d_perm, d_csize, n, mc->d_comp_lo, mc->d_comp_hi);
        // window size: the largest component that still fits (4 private accumulators of wmax floats, several CTAs per SM)
        if (!mc->h_inv) mc->h_inv = new std::vector<int>((size_t)n);
        HH_CUDA(cudaMemcpyAsync(mc->h_inv->data(), mc->d_inv, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        std::vector<int> csz((size_t)n);
        HH_CUDA(cudaMemcpyAsync(csz.data(), d_csize, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        int wmax = 32;
        for (int v = 0; v < n; ++v)
            if (csz[(size_t)v] <= HH_WINDOW_MAX && csz[(size_t)v] > wmax) wmax = csz[(size_t)v];
        mc->wmax = (wmax + 31) & ~31;
        // rewrite the iterate in new indices: column j' <- column inv[j'], rows through perm, rows re-sorted.
        // Columns of small components do it inside their window (one warp each); the others on the n-row accumulator.
        int all_counts[2] = {0, 0};
        HH_CUDA(cudaMemsetAsync(mc->d_bigcount, 0, 2 * sizeof(int), ctx->stream));
        HH_LAUNCH(ctx, hh_k_cc_lists, (n + 255) / 256, 256, 0, mc->d_perm, 0, n, mc->d_comp_lo, mc->d_comp_hi, HH_WINDOW_MAX, mc->d_owned,
                  mc->d_win_list, mc->d_big_list, mc->d_bigcount);
        HH_CUDA(cudaMemcpyAsync(all_counts, mc->d_bigcount, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaMemsetAsync(mc->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        hh_colargs a;
        mcl_base_args(mc, a);
        if (all_counts[0] > 0) {
            const size_t smem = (size_t)mc->wmax * sizeof(float);
            auto kern = hh_k_relabel_win;
            HH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int per_sm = 0;
            HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32, smem));
            int grid = per_sm * ctx->sm_count;
            if (grid > all_counts[0]) grid = all_counts[0];
            HH_LAUNCH(ctx, kern, grid, 32, smem, M, mc->it[mc->cur ^ 1], g.W, g.T, mc->d_win_list, all_counts[0], mc->d_perm, mc->d_inv,
                      mc->d_comp_lo, mc->d_comp_hi, mc->wmax, a.err);
        }
        if (all_counts[1] > 0) {
            a.col_lo = 0;
            a.ncols = all_counts[1];
            a.order = mc->d_big_list;
            a.B = M;
            a.slot_src = 1;
            a.perm = mc->d_perm;
            a.orig = mc->d_inv;
            a.out = mc->it[mc->cur ^ 1];
            a.raw = 1;
            HH_CHECK((launch_col<SRC_CSC, EPI_NORM>(ctx, g, mc->d_scratch, mc->grid_cap, a)));
        }
        unsigned long long st[4];
        HH_CHECK(read_stats(ctx, mc->d_stats, st));
        HH_REQUIRE((int)(st[3] & 0xffffffffull) == 0, HH_ERR_CAPACITY, "hh_mcl: slot overflow while relabelling");
        // the lists of the columns this context steps
        HH_CUDA(cudaMemsetAsync(mc->d_bigcount, 0, 2 * sizeof(int), ctx->stream));
        HH_LAUNCH(ctx, hh_k_cc_lists, (ncols + 255) / 256, 256, 0, mc->d_perm, mc->col_lo, ncols, mc->d_comp_lo, mc->d_comp_hi, HH_WINDOW_MAX,
                  mc->d_owned, mc->d_win_list, mc->d_big_list, mc->d_bigcount);
        int counts[2] = {0, 0};
        HH_CUDA(cudaMemcpyAsync(counts, mc->d_bigcount, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        mc->n_win = counts[0];
        mc->n_big = counts[1];
        mc->cur ^= 1;
        mc->perm_valid = true;
        mc->perm_space = true;
        HH_CHECK(mcl_build_blk_items(mc));
        return HH_OK;
    }();
    hh_dfree(d_lab);
    return rc;
}

extern "C" int hh_mcl_begin(hh_mcl* mc, double inflation, double pruning) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_begin: NULL handle");
    hh_scope _scope(mc->ctx);
    HH_REQUIRE(inflation > 0.0, HH_ERR_ARG, "hh_mcl_begin: inflation must be positive");
    HH_CUDA(cudaSetDevice(mc->ctx->device));
    // a column that sums to 1 holds at most 1/pruning entries >= pruning (+ slack for fp32 rounding)
    int cap = mc->n;
    if (pruning > 0.0 && 1.0 / pruning + 16.0 < (double)mc->n) cap = (int)(1.0 / pruning) + 16;
    if (cap != mc->it_cap) {
        slot_free(mc->it[0]);
        slot_free(mc->it[1]);
        mc->it_cap = 0;
        HH_CHECK(slot_alloc(mc->it[0], mc->n, cap, mc->W));
        HH_CHECK(slot_alloc(mc->it[1], mc->n, cap, mc->W));
        mc->it_cap = cap;
    }
    // matrix.power(inflation): fp32 array ** Python float = fp32 pow with the exponent cast to fp32
    mc->inflation = (float)inflation;
    mc->inflate_square = HH_INFL_POW;                 // how x^r is evaluated (hh_inflate)
    if (mc->inflation == 2.0f) mc->inflate_square = HH_INFL_SQUARE;
    else if (mc->inflation == 1.5f) mc->inflate_square = HH_INFL_X15;
    else if (mc->inflation == 3.0f) mc->inflate_square = HH_INFL_CUBE;
    else if (mc->inflation == 2.5f) mc->inflate_square = HH_INFL_X25;
    mc->prune = (float)pruning;   // `matrix >= pruning` compares in fp32
    mc->cur = -1;
    mc->have_pending = false;
    // the relabelling is rebuilt from this inflation's own first pruned iterate: its components bound every later
    // iterate of the same mcl() call, which is what makes the row windows safe
    mc->perm_valid = false;
    mc->perm_space = false;
    mc->col_lo = mc->own_lo;      // hh_mcl_set_block is per mcl() call
    mc->col_hi = mc->own_hi;
    mc->begun = true;
    return HH_OK;
}

extern "C" int hh_mcl_step(hh_mcl* mc, int it, int64_t* nnz_owned, int64_t* products, float* delta, float* kernel_ms) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_step: NULL handle");
    hh_scope _scope(mc->ctx);
    HH_REQUIRE(mc->begun, HH_ERR_STATE, "hh_mcl_step: call hh_mcl_begin first");
    HH_REQUIRE(!mc->have_pending, HH_ERR_STATE, "hh_mcl_step: previous step not committed");
    HH_REQUIRE((it == 0) == (mc->cur < 0), HH_ERR_STATE, "hh_mcl_step: iteration %d out of sequence", it);
    hh_ctx* ctx = mc->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    const hh_geom g = mcl_geom(mc);
    HH_CUDA(cudaMemsetAsync(mc->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    hh_colargs a;
    mcl_base_args(mc, a);
    a.inflation = mc->inflation;
    a.inflate_square = mc->inflate_square;
    a.prune = mc->prune;
    const int dst = (mc->cur < 0) ? 0 : (mc->cur ^ 1);
    a.out = mc->it[dst];
    HH_CUDA(cudaEventRecord(mc->ev0, ctx->stream));
    const int ncols_owned = mc->col_hi - mc->col_lo;
    if (it == 0) {
        a.dense_in = mc->d_m1;
        a.do_conv = 0;
        HH_CHECK(launch_iter0(ctx, g, a));      // original indices: the relabelling is built after iteration 0
    } else if (mc->perm_space) {
        a.A = mc->it[mc->cur];
        a.B = mc->it[mc->cur];
        a.do_conv = 1;
        a.orig = mc->d_inv;
        const double dcol = (double)mc->cur_nnz / (double)mc->n;
        a.track = (dcol * dcol * 4.0 < (double)mc->n) ? 1 : 0;
        choose_walk(mc, (double)mc->cur_nnz, a);
        a.T = g.T;
        if (mc->use_small && mc->cur_nnz <= 8ll * mc->n) {
            HH_CUDA(cudaMemsetAsync(mc->d_bigcount, 0, sizeof(int), ctx->stream));
            a.ncols = ncols_owned;
            int grid = (ncols_owned + 7) / 8;
            if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
            HH_LAUNCH(ctx, hh_k_col_small, grid, 256, 0, a, g.W, mc->d_overflow, mc->d_bigcount, mc->d_owned);
            a.order = mc->d_overflow;
            a.ncols_ptr = mc->d_bigcount;
            HH_CHECK((launch_col<SRC_PRODUCT, EPI_PRUNE>(ctx, g, mc->d_scratch, mc->grid_cap, a)));
        } else {
            // Window components whose block product is cheaper as a GEMM: both operands as three exact bf16 planes (six
            // passes), drained every k-block; the expansion of hh_k_col_win is replaced, its epilogue is not.
            unsigned short *d_blkA = nullptr, *d_blkB = nullptr;
            float* d_blk_out = nullptr;
            bool blk = false;
            // entries of the pruned iterate lie in [pruning, 1]: two f16 planes of M * 2^14 per operand (four passes) while
            // they stay f16 normals, else three exact bf16 planes (six passes); HH_GEMM_BLK_FMT=bf16 forces the latter
            const char* bf = getenv("HH_GEMM_BLK_FMT");
            const int f16 = (mc->prune >= 6.2e-5f && !(bf && !strcmp(bf, "bf16"))) ? 1 : 0;
            if (mc->n_win > 0 && mc->d_blk_items && mc->col_lo == 0 && mc->col_hi == mc->n) {
                const double est_sparse = (double)mc->cur_nnz * (double)mc->cur_nnz / (double)mc->n / 0.6e12;
                const double est_gemm = mc->blk_flops * (f16 ? 4.0 / 6.0 : 1.0) / 1.2e15 + 2.0e-3;      // blk_flops counts six passes
                blk = est_gemm < est_sparse;
            }
            if (blk) {
                const int np_op = f16 ? 2 : 3;
                const size_t plane = (size_t)mc->blk_ldk * (size_t)mc->n;
                HH_CHECK(hh_ws_alloc(ctx, &d_blkA, plane * np_op));
                HH_CHECK(hh_ws_alloc(ctx, &d_blkB, plane * np_op));
                HH_CHECK(hh_ws_alloc(ctx, &d_blk_out, plane));
                const hh_slotmat& M = mc->it[mc->cur];
                HH_CHECK(hh_gemm_blk_operands(ctx, M.len, M.ent, M.cap, mc->d_win_list, mc->n_win, mc->d_comp_lo, mc->d_comp_hi, mc->n,
                                              d_blkA, d_blkB, mc->blk_ldk, f16));
                int pa[8], pb[8];
                int npass = hh_gemm_passes(3, pa, pb);
                if (f16) {                                       // hi hi, hi lo, lo hi, lo lo: what is left is the rounding of lo, 2^-23
                    npass = 4;
                    pa[0] = 0, pb[0] = 0;
                    pa[1] = 0, pb[1] = 1;
                    pa[2] = 1, pb[2] = 0;
                    pa[3] = 1, pb[3] = 1;
                }
                const int fmt = f16 ? HH_GEMM_F16 : HH_GEMM_BF16;
                hh_gemm_operand A = {d_blkA, np_op, mc->n, (int)mc->blk_ldk, mc->blk_ldk, (long long)plane, fmt};
                hh_gemm_operand B = {d_blkB, np_op, mc->n, (int)mc->blk_ldk, mc->blk_ldk, (long long)plane, fmt};
                HH_CHECK(hh_gemm_run(ctx, A, B, mc->d_blk_items, (int)mc->blk_items->size(), npass, pa, pb,
                                     env_int("HH_GEMM_CHUNK", f16 ? 2 : 1), d_blk_out, mc->blk_ldk, 0, mc->n, nullptr, nullptr,
                                     hh_gemm_blk_out_scale(f16), 0));
                a.dense_in = d_blk_out;
                a.ld = mc->blk_ldk;
                mc->blk_iters++;
            }
            if (mc->n_win > 0) {
                const size_t smem = (size_t)mc->wmax * sizeof(float);
                auto kern = hh_k_col_win;
                HH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                int per_sm = 0;
                HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32, smem));
                int grid = per_sm * ctx->sm_count;
                if (grid > mc->n_win) grid = mc->n_win;
                if (grid < 1) grid = 1;
                HH_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(int), ctx->stream));
                HH_LAUNCH(ctx, kern, grid, 32, smem, a, g.W, mc->d_win_list, mc->n_win, mc->d_comp_lo, mc->d_comp_hi, mc->wmax);
            }
            if (blk) {
                a.dense_in = nullptr;
                a.ld = mc->ld;
                hh_ws_free(ctx, d_blkA);
                hh_ws_free(ctx, d_blkB);
                hh_ws_free(ctx, d_blk_out);
            }
            if (mc->n_big > 0) {
                a.order = mc->d_big_list;
                a.ncols = mc->n_big;
                HH_CHECK((launch_col<SRC_PRODUCT, EPI_PRUNE>(ctx, g, mc->d_scratch, mc->grid_cap, a)));
            }
        }
    } else {
        const hh_slotmat* Bp = &mc->it[mc->cur];
        for (int pwr = 2; pwr < mc->expansion; ++pwr) {           // --expansion k > 2: M^(k-1) of the owned columns, unpruned
            HH_CHECK(raw_product(mc, mc->it[mc->cur], *Bp, (double)mc->cur_nnz, mc->pw[pwr & 1]));
            Bp = &mc->pw[pwr & 1];
        }
        if (mc->expansion > 2) HH_CUDA(cudaMemsetAsync(mc->d_stats, 0, sizeof(unsigned long long), ctx->stream));   // nnz of the result only
        a.A = mc->it[mc->cur];
        a.B = *Bp;
        a.prev = mc->it[mc->cur];
        a.use_prev = mc->expansion > 2;
        a.do_conv = 1;
        // expected products per column ~ (nnz/n)^2; track dirty chunks when that is well below n
        const double dcol = (double)mc->cur_nnz / (double)mc->n;
        a.track = (dcol * dcol * 4.0 < (double)mc->n) ? 1 : 0;
        choose_walk(mc, (double)mc->cur_nnz, a);
        if (mc->use_small && mc->cur_nnz <= 8ll * mc->n) {
            // nearly converged: one warp per column; what does not fit goes to the accumulator kernel
            const int ncols = mc->col_hi - mc->col_lo;
            HH_CUDA(cudaMemsetAsync(mc->d_bigcount, 0, sizeof(int), ctx->stream));
            a.T = g.T;
            int grid = (ncols + 7) / 8;
            if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
            HH_LAUNCH(ctx, hh_k_col_small, grid, 256, 0, a, g.W, mc->d_order, mc->d_bigcount, (const int*)nullptr);
            a.order = mc->d_order;
            a.ncols_ptr = mc->d_bigcount;
        }
        HH_CHECK((launch_col<SRC_PRODUCT, EPI_PRUNE>(ctx, g, mc->d_scratch, mc->grid_cap, a)));
    }
    HH_CUDA(cudaEventRecord(mc->ev1, ctx->stream));
    unsigned long long st[4];
    HH_CHECK(read_stats(ctx, mc->d_stats, st));
    if (kernel_ms) HH_CUDA(cudaEventElapsedTime(kernel_ms, mc->ev0, mc->ev1));
    HH_REQUIRE((int)(st[3] & 0xffffffffull) == 0, HH_ERR_CAPACITY,
               "hh_mcl_step: a pruned column exceeded its slot (%d entries); pruning threshold too small for this layout", mc->it_cap);
    mc->pending_nnz = (int64_t)st[0] * (int64_t)mc->n / (int64_t)(mc->col_hi - mc->col_lo);   // owned block scaled to n
    if (nnz_owned) *nnz_owned = (int64_t)st[0];
    if (products) *products = (int64_t)st[1];
    if (delta) {
        const int bits = (int)(st[2] & 0xffffffffull);
        float d;
        memcpy(&d, &bits, sizeof(float));
        *delta = d;
    }
    mc->pending = dst;
    mc->have_pending = true;
    mc->last_step_it = it;
    return HH_OK;
}

extern "C" int hh_mcl_pack(hh_mcl* mc, int32_t* len_dev, int32_t* idx_dev, float* val_dev) {
    HH_REQUIRE(mc && len_dev, HH_ERR_ARG, "hh_mcl_pack: NULL argument");
    hh_scope _scope(mc->ctx);
    HH_REQUIRE(mc->have_pending, HH_ERR_STATE, "hh_mcl_pack: nothing to pack (call hh_mcl_step first)");
    hh_ctx* ctx = mc->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    const int ncols = mc->col_hi - mc->col_lo;
    int64_t* d_off = nullptr;
    HH_CHECK(hh_dmalloc(&d_off, (size_t)ncols + 1));
    int rc = [&]() -> int {
        const hh_slotmat& s = mc->it[mc->pending];
        const int* colmap = mc->perm_space ? mc->d_perm : nullptr;        // owned ORIGINAL columns live at perm[c]
        HH_LAUNCH(ctx, hh_k_gather_len, (ncols + 255) / 256, 256, 0, s.len, colmap, mc->col_lo, ncols, len_dev);
        HH_CHECK(hh_exclusive_scan_i32(ctx, len_dev, d_off, ncols));
        int grid = (ncols + 7) / 8;
        if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
        HH_LAUNCH(ctx, hh_k_pack, grid, 256, 0, s, mc->col_lo, ncols, d_off, len_dev, idx_dev, val_dev, colmap);
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        return HH_OK;
    }();
    hh_dfree(d_off);
    return rc;
}

extern "C" int hh_mcl_unpack(hh_mcl* mc, int32_t col_lo, int32_t col_hi, const int32_t* len_dev, const int32_t* idx_dev,
                             const float* val_dev, int64_t nnz_block) {
    HH_REQUIRE(mc && len_dev, HH_ERR_ARG, "hh_mcl_unpack: NULL argument");
    hh_scope _scope(mc->ctx);
    HH_REQUIRE(mc->have_pending, HH_ERR_STATE, "hh_mcl_unpack: no pending iterate (call hh_mcl_step first)");
    HH_REQUIRE(0 <= col_lo && col_lo < col_hi && col_hi <= mc->n, HH_ERR_ARG, "hh_mcl_unpack: bad column block");
    HH_REQUIRE(col_hi <= mc->col_lo || col_lo >= mc->col_hi, HH_ERR_ARG, "hh_mcl_unpack: block overlaps the owned columns");
    (void)nnz_block;
    hh_ctx* ctx = mc->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    const int ncols = col_hi - col_lo;
    int64_t* d_off = nullptr;
    HH_CHECK(hh_dmalloc(&d_off, (size_t)ncols + 1));
    int rc = [&]() -> int {
        HH_CUDA(cudaMemsetAsync(mc->d_stats + 3, 0, sizeof(unsigned long long), ctx->stream));
        HH_CHECK(hh_exclusive_scan_i32(ctx, len_dev, d_off, ncols));
        int grid = (ncols + 7) / 8;
        if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
        HH_LAUNCH(ctx, hh_k_unpack, grid, 256, 0, mc->it[mc->pending], mc->T, col_lo, ncols, len_dev, d_off, idx_dev, val_dev,
                  reinterpret_cast<int*>(mc->d_stats + 3), mc->perm_space ? mc->d_perm : nullptr);
        unsigned long long st[4];
        HH_CHECK(read_stats(ctx, mc->d_stats, st));
        HH_REQUIRE((int)(st[3] & 0xffffffffull) == 0, HH_ERR_CAPACITY, "hh_mcl_unpack: a peer column exceeds the slot capacity");
        return HH_OK;
    }();
    hh_dfree(d_off);
    return rc;
}

// change the block of columns the following steps compute (sparse iterations only: iteration 0 streams the dense M1
// block given to hh_mcl_create).  Column shards use it to stop exchanging once the iterate is tiny: every rank then
// computes all columns itself -- same kernels, same order of additions, so all ranks keep identical iterates.
extern "C" int hh_mcl_set_block(hh_mcl* mc, int32_t col_lo, int32_t col_hi) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_set_block: NULL handle");
    hh_scope _scope(mc->ctx);
    HH_REQUIRE(mc->begun && mc->cur >= 0 && !mc->have_pending, HH_ERR_STATE,
               "hh_mcl_set_block: only between hh_mcl_commit and the next hh_mcl_step, after iteration 0");
    HH_REQUIRE(0 <= col_lo && col_lo < col_hi && col_hi <= mc->n, HH_ERR_ARG, "hh_mcl_set_block: bad column block");
    hh_ctx* ctx = mc->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    mc->col_lo = col_lo;
    mc->col_hi = col_hi;
    if (mc->perm_space) {
        const int ncols = col_hi - col_lo;
        HH_CUDA(cudaMemsetAsync(mc->d_bigcount, 0, 2 * sizeof(int), ctx->stream));
        HH_LAUNCH(ctx, hh_k_cc_lists, (ncols + 255) / 256, 256, 0, mc->d_perm, mc->col_lo, ncols, mc->d_comp_lo, mc->d_comp_hi, HH_WINDOW_MAX,
                  mc->d_owned, mc->d_win_list, mc->d_big_list, mc->d_bigcount);
        int counts[2] = {0, 0};
        HH_CUDA(cudaMemcpyAsync(counts, mc->d_bigcount, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        mc->n_win = counts[0];
        mc->n_big = counts[1];
        // a sharded run that goes on replicated owns every column from here on: the component blocks can be multiplied on
        // the tensor cores like on a single GPU
        if (col_lo == 0 && col_hi == mc->n && mc->blk_items->empty()) HH_CHECK(mcl_build_blk_items(mc));
    }
    return HH_OK;
}

extern "C" int hh_mcl_commit(hh_mcl* mc) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_commit: NULL handle");
    HH_REQUIRE(mc->have_pending, HH_ERR_STATE, "hh_mcl_commit: nothing to commit");
    mc->cur = mc->pending;
    mc->cur_nnz = mc->pending_nnz;
    mc->have_pending = false;
    if (mc->use_window && !mc->perm_valid && mc->last_step_it == 0) {
        hh_scope _scope(mc->ctx);
        HH_CHECK(mcl_build_perm(mc));
    }
    return HH_OK;
}

extern "C" int hh_mcl_run(hh_mcl* mc, double inflation, int max_iter, double pruning, hh_mcl_result* res, int64_t* iter_nnz,
                          int64_t* iter_products, float* iter_delta, float* iter_ms) {
    HH_REQUIRE(mc && res, HH_ERR_ARG, "hh_mcl_run: NULL argument");
    HH_REQUIRE(mc->own_lo == 0 && mc->own_hi == mc->n, HH_ERR_STATE,
               "hh_mcl_run needs a context that owns every column; use the step interface for column shards");
    HH_REQUIRE(max_iter >= 1, HH_ERR_ARG, "hh_mcl_run: max_iter must be >= 1");
    HH_CHECK(hh_mcl_begin(mc, inflation, pruning));
    memset(res, 0, sizeof(*res));
    int64_t nnz_prev = 0;
    for (int it = 0; it < max_iter; ++it) {
        int64_t nnz = 0, prod = 0;
        float delta = 0.f, ms = 0.f;
        HH_CHECK(hh_mcl_step(mc, it, &nnz, &prod, &delta, &ms));
        HH_CHECK(hh_mcl_commit(mc));
        if (iter_ms) iter_ms[it] = ms;
        if (iter_nnz) iter_nnz[it] = nnz;
        if (iter_products) iter_products[it] = prod;
        if (iter_delta) iter_delta[it] = delta;
        res->rounds = it + 1;
        res->nnz = nnz;
        res->products += prod;
        // algorithmic bytes (SURVEY.md 8d): it == 0 streams the dense M1 and writes the pruned result;
        // it >= 1 reads the operand, writes the result, re-reads the operand for the convergence test
        if (it == 0) res->bytes += 4ll * mc->n * (int64_t)mc->n + 8ll * nnz;
        else res->bytes += 16ll * nnz_prev + 8ll * nnz + 12ll * ((int64_t)mc->n + 1);
        nnz_prev = nnz;
        // n > 1 and max(|M-L| - 1e-5|L|) <= 1e-8   (2044-2046)
        if (it > 1 && (double)delta <= 1e-8) {
            res->converged = 1;
            break;
        }
    }
    return HH_OK;
}

extern "C" int hh_mcl_fetch_result(hh_mcl* mc, int64_t* indptr, int32_t* indices, float* data) {
    HH_REQUIRE(mc != nullptr, HH_ERR_ARG, "hh_mcl_fetch_result: NULL handle");
    hh_scope _scope(mc->ctx);
    HH_REQUIRE(mc->cur >= 0 && !mc->have_pending, HH_ERR_STATE, "hh_mcl_fetch_result: no committed iterate");
    HH_CUDA(cudaSetDevice(mc->ctx->device));
    if (mc->perm_space) return slot_fetch_csc(mc->ctx, mc->it[mc->cur], 0, mc->n, indptr, indices, data, mc->d_perm, mc->h_inv);
    return slot_fetch_csc(mc->ctx, mc->it[mc->cur], 0, mc->n, indptr, indices, data);
}
