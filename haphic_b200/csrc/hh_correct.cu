// Assembly correction (`--correct_nrounds`): Hi-C span coverage, breakpoint detection, contig splitting and the record
// remap of the second pass.  Reference: scripts/HapHiC_cluster.py (v1.0.7) parse_pairs_for_correction 1300-1344,
// detect_break_points 943-1014, break_and_update_ctgs 1017-1197, *_generator_for_correction[_ctg] 1401-1536.
//
// Layout.  Every contig c owns the coverage bins [bin_off[c], bin_off[c+1]) of one int32 array, len//res + 1 bins as in the
// reference (1312).  A fragment made by splitting c keeps c's bin grid: it is a sub-range of c's bins, exactly the numpy view
// the reference slices out of its parent (1158, 1180).  Intra-contig read pairs are kept in a link store of int32
// {bucket, lo, hi}: `bucket` is an id the host gives to each key string of ctg_link_pos_dict, so the links move between
// buckets when a fragment is split, with the key quirk of pos_shift (1036-1052) decided on the host.
#include "hh_common.cuh"

#include <algorithm>
#include <climits>

namespace {

constexpr int CT_THREADS = 256;
constexpr int SCAN_TILE = 4096;                 // elements per CTA of the coverage scan (16 per thread)
constexpr int DET_THREADS = 256;
constexpr int DET_SMEM_BINS = 11264;            // fragments up to this many bins are staged in shared memory (44 KB: with
                                                // the static histogram it stays under the 48 KB of a launch without opt-in)

}  // namespace

struct hh_correct {
    hh_ctx* ctx;
    int32_t n_ctg;
    int32_t res;
    int64_t n_bins;                 // sum over contigs of len // res + 1
    int64_t* d_bin_off;             // [n_ctg + 1]
    int64_t* d_len;                 // [n_ctg]
    int32_t* d_diff;                // [n_bins + 1] difference array of the records added so far / of a split's subtraction
    int32_t* d_cov;                 // [n_bins] coverage, valid once `scanned`
    int32_t* d_links;               // [cap][3] {bucket, lo, hi}
    int64_t n_links, cap;
    unsigned long long* d_counters; // [0] links appended, [1] records with a position outside their contig
    int32_t* d_stage;               // staging buffer of host records (add / remap)
    int64_t stage_records;
    bool scanned;
    // piece table of the remap (set by hh_correct_set_pieces)
    int32_t* d_piece_off;           // [n_ctg + 1]
    int32_t* d_piece_start;         // [n_piece] 0-based start of every piece on its contig, ascending per contig
    int32_t* d_piece_id;            // [n_piece] id of the piece in the corrected fa_dict order
    bool have_pieces;
};

// ---------------------------------------------------------------------------------------------
// pass 1: coverage difference array + link store (1321-1343)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CT_THREADS) hh_k_correct_add(const int4* __restrict__ rec, int64_t n, int32_t n_ctg,
                                                               const int64_t* __restrict__ bin_off,
                                                               const int64_t* __restrict__ len, int32_t res,
                                                               int32_t* __restrict__ diff, int32_t* __restrict__ links,
                                                               unsigned long long* __restrict__ counters) {
    const int lane = hh_lane();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // warp-uniform trip count: every lane takes part in the ballot of the append
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < n; i0 += stride) {
        const int64_t i = i0 + lane;
        bool ok = false;
        int32_t c = 0, lo = 0, hi = 0;
        if (i < n) {
            const int4 r = hh_ld_stream(rec + i);
            if (r.x == r.z && r.x >= 0 && r.x < n_ctg) {
                c = r.x;
                lo = min(r.y, r.w);
                hi = max(r.y, r.w);
                if (lo < 0 || (int64_t)hi >= len[c]) {
                    atomicAdd(counters + 1, 1ull);
                } else {
                    ok = true;
                    const int64_t off = bin_off[c];
                    atomicAdd(diff + off + lo / res, 1);
                    atomicAdd(diff + off + hi / res + 1, -1);
                }
            }
        }
        const unsigned mask = __ballot_sync(HH_FULL_MASK, ok);
        if (mask == 0) continue;
        const int leader = __ffs(mask) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(counters, (unsigned long long)__popc(mask));
        base = __shfl_sync(HH_FULL_MASK, base, leader);
        if (ok) {
            const int64_t k = (int64_t)base + __popc(mask & ((1u << lane) - 1u));
            links[3 * k + 0] = c;
            links[3 * k + 1] = lo;
            links[3 * k + 2] = hi;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// inclusive scan of the difference array: cov = scan(diff) (SUBTRACT: cov -= scan(diff))
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CT_THREADS) hh_k_correct_tile_sums(const int32_t* __restrict__ in, int64_t n,
                                                                     int32_t* __restrict__ sums) {
    __shared__ int warp_tot[CT_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    int s = 0;
    for (int k = threadIdx.x; k < SCAN_TILE; k += CT_THREADS)
        if (base + k < n) s += in[base + k];
    s = hh_warp_sum(s);
    if (hh_lane() == 0) warp_tot[hh_warp()] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < CT_THREADS / 32; ++w) t += warp_tot[w];
        sums[blockIdx.x] = t;
    }
}

template <bool SUBTRACT>
__global__ void __launch_bounds__(CT_THREADS) hh_k_correct_tile_scan(const int32_t* __restrict__ in, int64_t n,
                                                                     const int64_t* __restrict__ tile_off,
                                                                     int32_t* __restrict__ out) {
    __shared__ int warp_tot[CT_THREADS / 32];
    constexpr int PER = SCAN_TILE / CT_THREADS;
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * PER;
    int v[PER];
    int s = 0;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        v[k] = (base + k < n) ? in[base + k] : 0;
        s += v[k];
    }
    const int lane = hh_lane(), warp = hh_warp();
    int incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(HH_FULL_MASK, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    int run = (int)tile_off[blockIdx.x] + before + incl - s;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        run += v[k];
        if (base + k < n) {
            if (SUBTRACT)
                out[base + k] -= run;
            else
                out[base + k] = run;
        }
    }
}

static int correct_scan(hh_ctx* ctx, const int32_t* d_in, int32_t* d_out, int64_t n, bool subtract) {
    if (n == 0) return HH_OK;
    const int64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    HH_REQUIRE(tiles < (1ll << 30), HH_ERR_UNSUPPORTED, "correction: %lld coverage bins are too many", (long long)n);
    int32_t* d_sums = nullptr;
    int64_t* d_off = nullptr;
    int rc = hh_dmalloc(&d_sums, (size_t)tiles);
    if (rc == HH_OK) rc = hh_dmalloc(&d_off, (size_t)tiles + 1);
    if (rc == HH_OK) {
        hh_k_correct_tile_sums<<<(unsigned)tiles, CT_THREADS, 0, ctx->stream>>>(d_in, n, d_sums);
        ctx->launches++;
        rc = cudaGetLastError() == cudaSuccess ? HH_OK : HH_ERR_CUDA;
    }
    if (rc == HH_OK) rc = hh_exclusive_scan_i32(ctx, d_sums, d_off, (int)tiles);
    if (rc == HH_OK) {
        if (subtract)
            hh_k_correct_tile_scan<true><<<(unsigned)tiles, CT_THREADS, 0, ctx->stream>>>(d_in, n, d_off, d_out);
        else
            hh_k_correct_tile_scan<false><<<(unsigned)tiles, CT_THREADS, 0, ctx->stream>>>(d_in, n, d_off, d_out);
        ctx->launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) {
            hh_set_error("correction scan: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
        }
    }
    hh_dfree(d_sums);
    hh_dfree(d_off);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// detection (detect_break_points, 943-1014): one CTA per fragment
// ---------------------------------------------------------------------------------------------

// k-th smallest of v[0, n) (0-based), radix select over the order-preserving unsigned key, 8 bits per pass
__device__ int det_select(const int32_t* v, int n, int k, unsigned* hist, unsigned* shared_state) {
    unsigned prefix = 0, mask = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const unsigned key = (unsigned)v[i] ^ 0x80000000u;
            if ((key & mask) == prefix) atomicAdd(hist + ((key >> shift) & 255u), 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned cum = 0;
            int d = 0;
            for (; d < 255; ++d) {
                if (cum + hist[d] > (unsigned)k) break;
                cum += hist[d];
            }
            shared_state[0] = (unsigned)d;
            shared_state[1] = (unsigned)k - cum;
        }
        __syncthreads();
        prefix |= shared_state[0] << shift;
        k = (int)shared_state[1];
        mask |= 255u << shift;
        __syncthreads();
    }
    return (int)(prefix ^ 0x80000000u);
}

struct det_state {
    int kept;                   // filtered high-coverage regions closed so far
    int run_start;              // first bin of the open high run, -1 = none
    int rz, rmin, rarg;         // open run: leftmost 0 bin, minimum and its first bin
    int vz, vmin, varg;         // bins after the last kept run (the valley being built)
    int nzero;                  // zero valleys written
    int best_cov, best_bin;     // deepest non-zero valley
};

__device__ __forceinline__ void det_add(int& z, int& mn, int& arg, int i, int x) {
    if (x == 0 && z < 0) z = i;
    if (x < mn) {
        mn = x;
        arg = i;
    }
}

__device__ __forceinline__ void det_close_run(det_state& s, int end, int res, double region_cut, int2* out, bool writer) {
    const int64_t span = (int64_t)(end + 1 - s.run_start) * res;     // upper - lower of the closed region
    if ((double)span >= region_cut) {
        if (s.kept >= 1) {                                            // the valley between the previous kept run and this
            if (s.vz >= 0) {
                if (writer) out[s.nzero] = make_int2(s.vz, 0);
                s.nzero++;
            } else if (s.vmin < s.best_cov) {
                s.best_cov = s.vmin;
                s.best_bin = s.varg;
            }
        }
        s.kept++;
        s.vz = -1;
        s.vmin = INT_MAX;
        s.varg = -1;
    } else {                                                          // a short high run belongs to the valley around it
        if (s.vz < 0 && s.rz >= 0) s.vz = s.rz;
        if (s.rmin < s.vmin) {
            s.vmin = s.rmin;
            s.varg = s.rarg;
        }
    }
    s.run_start = -1;
}

// cov: coverage array; fragment s is cov[seg_off[s], seg_off[s] + seg_nbins[s]) of length seg_len[s] bp.  Writes the
// breakpoints (bin relative to the fragment, coverage) to scratch[seg_base[s] ...] and their number to count[s].
__global__ void __launch_bounds__(DET_THREADS) hh_k_correct_detect(const int32_t* __restrict__ cov,
                                                                   const int64_t* __restrict__ seg_off,
                                                                   const int32_t* __restrict__ seg_nbins,
                                                                   const int64_t* __restrict__ seg_len,
                                                                   const int64_t* __restrict__ seg_base, int32_t res,
                                                                   double median_cov_ratio, double region_len_ratio,
                                                                   double min_region_cutoff, int32_t* __restrict__ count,
                                                                   int2* __restrict__ scratch) {
    extern __shared__ int32_t stage[];
    __shared__ unsigned hist[256];
    __shared__ unsigned sel[2];
    const int s = blockIdx.x;
    const int n = seg_nbins[s];
    const int32_t* v = cov + seg_off[s];
    if (n <= DET_SMEM_BINS) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) stage[i] = v[i];
        __syncthreads();
        v = stage;
    }
    // numpy.median: the middle element, or the mean of the two middle elements, in float64
    const int k1 = (n - 1) / 2, k2 = n / 2;
    const int m1 = det_select(v, n, k1, hist, sel);
    const int m2 = (k2 == k1) ? m1 : det_select(v, n, k2, hist, sel);
    const double median = (k2 == k1) ? (double)m1 : ((double)m1 + (double)m2) / 2.0;
    if (hh_warp() != 0) return;
    const int lane = hh_lane();
    if (median == 0.0) {
        if (lane == 0) count[s] = 0;
        return;
    }
    const double cut = __dmul_rn(median, median_cov_ratio);
    const double by_len = __dmul_rn((double)seg_len[s], region_len_ratio);
    const double region_cut = min_region_cutoff >= by_len ? min_region_cutoff : by_len;
    int2* out = scratch + seg_base[s];
    det_state st;
    st.kept = 0;
    st.run_start = -1;
    st.rz = -1, st.rmin = INT_MAX, st.rarg = -1;
    st.vz = -1, st.vmin = INT_MAX, st.varg = -1;
    st.nzero = 0;
    st.best_cov = INT_MAX, st.best_bin = -1;
    // one warp walks the bins in order; the lanes load a tile of 32 and every lane keeps the same (uniform) state
    for (int t0 = 0; t0 < n; t0 += 32) {
        const int x = (t0 + lane < n) ? v[t0 + lane] : 0;
        const unsigned high = __ballot_sync(HH_FULL_MASK, (double)x >= cut);
        const int m = min(32, n - t0);
        for (int j = 0; j < m; ++j) {
            const int xj = __shfl_sync(HH_FULL_MASK, x, j);
            const int i = t0 + j;
            if ((high >> j) & 1u) {
                if (st.run_start < 0) {
                    st.run_start = i;
                    st.rz = -1, st.rmin = INT_MAX, st.rarg = -1;
                }
                det_add(st.rz, st.rmin, st.rarg, i, xj);
            } else {
                if (st.run_start >= 0) det_close_run(st, i - 1, res, region_cut, out, lane == 0);
                det_add(st.vz, st.vmin, st.varg, i, xj);
            }
        }
    }
    if (st.run_start >= 0) det_close_run(st, n - 1, res, region_cut, out, lane == 0);
    if (lane == 0) {
        if (st.nzero > 0) {
            count[s] = st.nzero;
        } else if (st.kept >= 2) {
            out[0] = make_int2(st.best_bin, st.best_cov);
            count[s] = 1;
        } else {
            count[s] = 0;
        }
    }
}

__global__ void hh_k_correct_compact(int32_t n_seg, const int32_t* __restrict__ count, const int64_t* __restrict__ off,
                                     const int64_t* __restrict__ seg_base, const int2* __restrict__ scratch,
                                     int2* __restrict__ out) {
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n_seg; s += gridDim.x * blockDim.x) {
        const int c = count[s];
        for (int k = 0; k < c; ++k) out[off[s] + k] = scratch[seg_base[s] + k];
    }
}

// detection on device coverage: host segment arrays in, host counts + packed breakpoints out
static int correct_detect_dev(hh_ctx* ctx, const int32_t* d_cov, int64_t n_cov, int32_t n_seg, const int64_t* seg_off,
                              const int32_t* seg_nbins, const int64_t* seg_len, int32_t res, double median_cov_ratio,
                              double region_len_ratio, int64_t min_region_cutoff, int32_t* n_bp, int32_t* bp_bin,
                              int32_t* bp_cov, int64_t max_bp, int64_t* total_bp) {
    std::vector<int64_t> base((size_t)n_seg + 1, 0);
    for (int32_t s = 0; s < n_seg; ++s) {
        HH_REQUIRE(seg_nbins[s] >= 1 && seg_off[s] >= 0 && seg_off[s] + seg_nbins[s] <= n_cov && seg_len[s] >= 0, HH_ERR_ARG,
                   "correction detect: segment %d (offset %lld, %d bins) is not inside the %lld coverage bins", s,
                   (long long)seg_off[s], seg_nbins[s], (long long)n_cov);
        base[(size_t)s + 1] = base[(size_t)s] + seg_nbins[s];
    }
    *total_bp = 0;
    if (n_seg == 0) return HH_OK;
    int64_t *d_off = nullptr, *d_len = nullptr, *d_base = nullptr, *d_pos = nullptr;
    int32_t *d_nb = nullptr, *d_count = nullptr;
    int2 *d_scratch = nullptr, *d_out = nullptr;
    int rc = HH_OK;
    do {
        if ((rc = hh_dmalloc(&d_off, (size_t)n_seg)) || (rc = hh_dmalloc(&d_len, (size_t)n_seg)) ||
            (rc = hh_dmalloc(&d_base, (size_t)n_seg)) || (rc = hh_dmalloc(&d_nb, (size_t)n_seg)) ||
            (rc = hh_dmalloc(&d_count, (size_t)n_seg)) || (rc = hh_dmalloc(&d_pos, (size_t)n_seg + 1)) ||
            (rc = hh_dmalloc(&d_scratch, (size_t)base[(size_t)n_seg])))
            break;
        cudaStream_t st = ctx->stream;
        cudaError_t e = cudaSuccess;
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, seg_off, (size_t)n_seg * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_len, seg_len, (size_t)n_seg * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_base, base.data(), (size_t)n_seg * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_nb, seg_nbins, (size_t)n_seg * 4, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) {
            hh_set_error("correction detect: copy failed: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
            break;
        }
        hh_k_correct_detect<<<(unsigned)n_seg, DET_THREADS, DET_SMEM_BINS * sizeof(int32_t), st>>>(
            d_cov, d_off, d_nb, d_len, d_base, res, median_cov_ratio, region_len_ratio, (double)min_region_cutoff, d_count,
            d_scratch);
        ctx->launches++;
        if ((e = cudaGetLastError()) != cudaSuccess) {
            hh_set_error("hh_k_correct_detect: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
            break;
        }
        if ((rc = hh_exclusive_scan_i32(ctx, d_count, d_pos, n_seg)) != HH_OK) break;
        int64_t total = 0;
        if ((e = cudaMemcpyAsync(&total, d_pos + n_seg, 8, cudaMemcpyDeviceToHost, st)) == cudaSuccess)
            e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            hh_set_error("correction detect: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
            break;
        }
        if (total > max_bp) {
            hh_set_error("correction detect: %lld breakpoints do not fit the %lld the caller provided", (long long)total,
                         (long long)max_bp);
            rc = HH_ERR_CAPACITY;
            break;
        }
        *total_bp = total;
        if ((rc = hh_dmalloc(&d_out, (size_t)total)) != HH_OK) break;
        const int grid = (int)std::min<int64_t>((n_seg + 255) / 256, 4096);
        hh_k_correct_compact<<<grid, 256, 0, st>>>(n_seg, d_count, d_pos, d_base, d_scratch, d_out);
        ctx->launches++;
        std::vector<int2> host((size_t)total);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(n_bp, d_count, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && total)
            e = cudaMemcpyAsync(host.data(), d_out, (size_t)total * sizeof(int2), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            hh_set_error("correction detect: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
            break;
        }
        for (int64_t k = 0; k < total; ++k) {
            if (bp_bin) bp_bin[k] = host[(size_t)k].x;
            if (bp_cov) bp_cov[k] = host[(size_t)k].y;
        }
    } while (0);
    hh_dfree(d_off);
    hh_dfree(d_len);
    hh_dfree(d_base);
    hh_dfree(d_nb);
    hh_dfree(d_count);
    hh_dfree(d_pos);
    hh_dfree(d_scratch);
    hh_dfree(d_out);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// split (break_and_update_ctgs, non-last rounds, 1074-1121)
// ---------------------------------------------------------------------------------------------

// first entry of the descending list p[0, m) with coord - p >= 0 (the list ends with 0, so one always exists for coord >= 0)
__device__ __forceinline__ int split_piece(const int32_t* p, int m, int32_t coord) {
    int lo = 0, hi = m - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (coord - p[mid] >= 0)
            hi = mid;
        else
            lo = mid + 1;
    }
    return lo;
}

__global__ void __launch_bounds__(CT_THREADS) hh_k_correct_split(int32_t* __restrict__ links, int64_t n_links,
                                                                 const int32_t* __restrict__ bucket_slot, int32_t n_buckets,
                                                                 const int64_t* __restrict__ frag_off,
                                                                 const int32_t* __restrict__ list_off,
                                                                 const int32_t* __restrict__ shift_pos,
                                                                 const int32_t* __restrict__ piece_bucket,
                                                                 const uint8_t* __restrict__ frag_zero, int32_t res,
                                                                 int32_t* __restrict__ diff) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_links; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t b = links[3 * i];
        if (b < 0 || b >= n_buckets) continue;
        const int32_t f = bucket_slot[b];
        if (f < 0) continue;
        const int32_t lo = links[3 * i + 1], hi = links[3 * i + 2];
        const int32_t* p = shift_pos + list_off[f];
        const int m = list_off[f + 1] - list_off[f];
        if (!frag_zero[f]) {
            const int32_t bp = p[0];                // a non-zero breakpoint is the only one of its fragment
            if (lo <= bp + res && hi >= bp) {       // closed(lo, hi) overlaps closed(bp, bp + res): remove its coverage
                const int64_t off = frag_off[f];
                atomicAdd(diff + off + lo / res, 1);
                atomicAdd(diff + off + hi / res + 1, -1);
                links[3 * i] = -1;
                continue;
            }
        }
        const int ni = split_piece(p, m, lo), nj = split_piece(p, m, hi);
        if (ni == nj) {
            links[3 * i] = piece_bucket[list_off[f] + ni];
            links[3 * i + 1] = lo - p[ni];
            links[3 * i + 2] = hi - p[nj];
        } else {
            links[3 * i] = -1;                      // an inter-piece link is not re-filed (1100, 1116)
        }
    }
}

// ---------------------------------------------------------------------------------------------
// pass-2 record remap (convert_ctg, 1405-1411)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void remap_end(int32_t& c, int32_t& pos, int32_t n_ctg, const int32_t* __restrict__ off,
                                          const int32_t* __restrict__ start, const int32_t* __restrict__ id) {
    if (c < 0 || c >= n_ctg) {
        c = -1;
        return;
    }
    int lo = off[c], hi = off[c + 1] - 1;           // largest piece start <= pos
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (start[mid] <= pos)
            lo = mid;
        else
            hi = mid - 1;
    }
    c = id[lo];
    pos -= start[lo];
}

__global__ void __launch_bounds__(CT_THREADS) hh_k_correct_remap(int4* __restrict__ rec, int64_t n, int32_t n_ctg,
                                                                 const int32_t* __restrict__ off,
                                                                 const int32_t* __restrict__ start,
                                                                 const int32_t* __restrict__ id) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int4 r = rec[i];
        remap_end(r.x, r.y, n_ctg, off, start, id);
        remap_end(r.z, r.w, n_ctg, off, start, id);
        rec[i] = r;
    }
}

// ---------------------------------------------------------------------------------------------
// ABI
// ---------------------------------------------------------------------------------------------
static int grid_for(hh_ctx* ctx, int64_t n) {
    const int64_t want = (n + CT_THREADS - 1) / CT_THREADS;
    const int64_t cap = (int64_t)ctx->sm_count * 8;
    return (int)std::max<int64_t>(1, std::min(want, cap));
}

extern "C" int hh_correct_create(hh_ctx* ctx, int32_t n_ctg, const int64_t* ctg_len, int32_t res, hh_correct** out) {
    HH_REQUIRE(ctx && out && (ctg_len || n_ctg == 0), HH_ERR_ARG, "hh_correct_create: NULL argument");
    HH_REQUIRE(n_ctg >= 0 && res > 0, HH_ERR_ARG, "hh_correct_create: n_ctg %d, resolution %d", n_ctg, res);
    hh_scope _scope(ctx);
    *out = nullptr;
    std::vector<int64_t> off((size_t)n_ctg + 1, 0);
    for (int32_t c = 0; c < n_ctg; ++c) {
        HH_REQUIRE(ctg_len[c] >= 0 && ctg_len[c] <= INT32_MAX, HH_ERR_UNSUPPORTED,
                   "hh_correct_create: contig %d has length %lld; positions must fit int32", c, (long long)ctg_len[c]);
        off[(size_t)c + 1] = off[(size_t)c] + ctg_len[c] / res + 1;
    }
    hh_correct* hc = new (std::nothrow) hh_correct();
    HH_REQUIRE(hc != nullptr, HH_ERR_NOMEM, "hh_correct_create: out of host memory");
    hc->ctx = ctx;
    hc->n_ctg = n_ctg;
    hc->res = res;
    hc->n_bins = off[(size_t)n_ctg];
    int rc = HH_OK;
    if ((rc = hh_dmalloc(&hc->d_bin_off, (size_t)n_ctg + 1)) || (rc = hh_dmalloc(&hc->d_len, (size_t)n_ctg + 1)) ||
        (rc = hh_dmalloc(&hc->d_diff, (size_t)hc->n_bins + 1)) || (rc = hh_dmalloc(&hc->d_cov, (size_t)hc->n_bins)) ||
        (rc = hh_dmalloc(&hc->d_counters, 2))) {
        hh_correct_destroy(hc);
        return rc;
    }
    cudaError_t e = cudaMemcpyAsync(hc->d_bin_off, off.data(), off.size() * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && n_ctg)
        e = cudaMemcpyAsync(hc->d_len, ctg_len, (size_t)n_ctg * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(hc->d_diff, 0, ((size_t)hc->n_bins + 1) * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(hc->d_counters, 0, 16, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        hh_set_error("hh_correct_create: %s", cudaGetErrorString(e));
        hh_correct_destroy(hc);
        return HH_ERR_CUDA;
    }
    *out = hc;
    return HH_OK;
}

static int correct_reserve(hh_correct* hc, int64_t need) {
    if (need <= hc->cap) return HH_OK;
    int64_t cap = std::max<int64_t>(need, hc->cap + hc->cap / 2);
    int32_t* nl = nullptr;
    HH_CHECK(hh_dmalloc(&nl, (size_t)cap * 3));
    if (hc->n_links)
        HH_CUDA(cudaMemcpyAsync(nl, hc->d_links, (size_t)hc->n_links * 12, cudaMemcpyDeviceToDevice, hc->ctx->stream));
    hh_dfree(hc->d_links);
    hc->d_links = nl;
    hc->cap = cap;
    return HH_OK;
}

static int correct_stage(hh_correct* hc, int64_t records) {
    if (hc->d_stage && hc->stage_records >= records) return HH_OK;
    hh_dfree(hc->d_stage);
    hc->stage_records = records;
    return hh_dmalloc(&hc->d_stage, (size_t)records * 4);
}

extern "C" int hh_correct_add(hh_correct* hc, const int32_t* rec, int64_t n_rec, int mem) {
    HH_REQUIRE(hc && (rec || n_rec == 0) && n_rec >= 0, HH_ERR_ARG, "hh_correct_add: bad argument");
    HH_REQUIRE(mem == HH_MEM_HOST || mem == HH_MEM_DEVICE, HH_ERR_ARG, "hh_correct_add: bad mem flag %d", mem);
    HH_REQUIRE(!hc->scanned, HH_ERR_STATE, "hh_correct_add: coverage already finalised by hh_correct_detect");
    if (n_rec == 0) return HH_OK;
    hh_ctx* ctx = hc->ctx;
    hh_scope _scope(ctx);
    const int64_t CH = 1ll << 22;
    for (int64_t off = 0; off < n_rec; off += CH) {
        const int64_t m = std::min(CH, n_rec - off);
        const int4* src;
        if (mem == HH_MEM_DEVICE) {
            HH_REQUIRE((((uintptr_t)rec) & 15) == 0, HH_ERR_ARG, "hh_correct_add: records must be 16-byte aligned");
            src = reinterpret_cast<const int4*>(rec) + off;
        } else {
            HH_CHECK(correct_stage(hc, CH));
            HH_CUDA(cudaMemcpyAsync(hc->d_stage, rec + off * 4, (size_t)m * 16, cudaMemcpyHostToDevice, ctx->stream));
            src = reinterpret_cast<const int4*>(hc->d_stage);
        }
        HH_CHECK(correct_reserve(hc, hc->n_links + m));
        HH_LAUNCH(ctx, hh_k_correct_add, grid_for(ctx, m), CT_THREADS, 0, src, m, hc->n_ctg, hc->d_bin_off, hc->d_len,
                  hc->res, hc->d_diff, hc->d_links, hc->d_counters);
        unsigned long long* h = reinterpret_cast<unsigned long long*>(ctx->h_scratch);
        HH_CUDA(cudaMemcpyAsync(h, hc->d_counters, 16, cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        HH_REQUIRE(h[1] == 0, HH_ERR_ARG,
                   "hh_correct_add: %llu same-contig records have a position outside [0, contig length)", h[1]);
        hc->n_links = (int64_t)h[0];
    }
    return HH_OK;
}

static int correct_finalise(hh_correct* hc) {
    if (hc->scanned) return HH_OK;
    HH_CHECK(correct_scan(hc->ctx, hc->d_diff, hc->d_cov, hc->n_bins, false));
    hc->scanned = true;
    return HH_OK;
}

extern "C" int hh_correct_info(hh_correct* hc, int64_t* n_bins, int64_t* n_links) {
    HH_REQUIRE(hc, HH_ERR_ARG, "hh_correct_info: NULL handle");
    if (n_bins) *n_bins = hc->n_bins;
    if (n_links) *n_links = hc->n_links;
    return HH_OK;
}

extern "C" int hh_correct_fetch(hh_correct* hc, int32_t* cov, int64_t* bin_off, int32_t* links) {
    HH_REQUIRE(hc, HH_ERR_ARG, "hh_correct_fetch: NULL handle");
    hh_scope _scope(hc->ctx);
    HH_CHECK(correct_finalise(hc));
    cudaStream_t st = hc->ctx->stream;
    if (cov && hc->n_bins) HH_CUDA(cudaMemcpyAsync(cov, hc->d_cov, (size_t)hc->n_bins * 4, cudaMemcpyDeviceToHost, st));
    if (bin_off) HH_CUDA(cudaMemcpyAsync(bin_off, hc->d_bin_off, ((size_t)hc->n_ctg + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (links && hc->n_links)
        HH_CUDA(cudaMemcpyAsync(links, hc->d_links, (size_t)hc->n_links * 12, cudaMemcpyDeviceToHost, st));
    HH_CUDA(cudaStreamSynchronize(st));
    return HH_OK;
}

extern "C" int hh_correct_detect(hh_correct* hc, int32_t n_seg, const int64_t* seg_off, const int32_t* seg_nbins,
                                 const int64_t* seg_len, double median_cov_ratio, double region_len_ratio,
                                 int64_t min_region_cutoff, int32_t* n_bp, int32_t* bp_bin, int32_t* bp_cov, int64_t max_bp,
                                 int64_t* total_bp) {
    HH_REQUIRE(hc && n_seg >= 0 && n_bp && total_bp && (n_seg == 0 || (seg_off && seg_nbins && seg_len)), HH_ERR_ARG,
               "hh_correct_detect: bad argument");
    hh_scope _scope(hc->ctx);
    HH_CHECK(correct_finalise(hc));
    return correct_detect_dev(hc->ctx, hc->d_cov, hc->n_bins, n_seg, seg_off, seg_nbins, seg_len, hc->res, median_cov_ratio,
                              region_len_ratio, min_region_cutoff, n_bp, bp_bin, bp_cov, max_bp, total_bp);
}

extern "C" int hh_correct_detect_segments(hh_ctx* ctx, const int32_t* cov, int64_t n_cov, int32_t res, int32_t n_seg,
                                          const int64_t* seg_off, const int32_t* seg_nbins, const int64_t* seg_len,
                                          double median_cov_ratio, double region_len_ratio, int64_t min_region_cutoff,
                                          int32_t* n_bp, int32_t* bp_bin, int32_t* bp_cov, int64_t max_bp,
                                          int64_t* total_bp) {
    HH_REQUIRE(ctx && (cov || n_cov == 0) && n_cov >= 0 && res > 0 && n_seg >= 0 && n_bp && total_bp, HH_ERR_ARG,
               "hh_correct_detect_segments: bad argument");
    hh_scope _scope(ctx);
    int32_t* d_cov = nullptr;
    HH_CHECK(hh_dmalloc(&d_cov, (size_t)n_cov));
    int rc = HH_OK;
    cudaError_t e = n_cov ? cudaMemcpyAsync(d_cov, cov, (size_t)n_cov * 4, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
    if (e != cudaSuccess) {
        hh_set_error("hh_correct_detect_segments: %s", cudaGetErrorString(e));
        rc = HH_ERR_CUDA;
    } else {
        rc = correct_detect_dev(ctx, d_cov, n_cov, n_seg, seg_off, seg_nbins, seg_len, res, median_cov_ratio, region_len_ratio,
                                min_region_cutoff, n_bp, bp_bin, bp_cov, max_bp, total_bp);
    }
    hh_dfree(d_cov);
    return rc;
}

extern "C" int hh_correct_split(hh_correct* hc, int32_t n_frag, const int32_t* frag_bucket, const int64_t* frag_off,
                                const uint8_t* frag_zero, const int32_t* list_off, const int32_t* shift_pos,
                                const int32_t* piece_bucket, int32_t n_buckets) {
    HH_REQUIRE(hc && n_frag >= 0 && n_buckets >= 0 && (n_frag == 0 || (frag_bucket && frag_off && frag_zero && list_off &&
                                                                        shift_pos && piece_bucket)),
               HH_ERR_ARG, "hh_correct_split: bad argument");
    hh_ctx* ctx = hc->ctx;
    hh_scope _scope(ctx);
    HH_CHECK(correct_finalise(hc));
    if (n_frag == 0) return HH_OK;
    std::vector<int32_t> slot((size_t)n_buckets, -1);
    for (int32_t f = 0; f < n_frag; ++f) {
        HH_REQUIRE(frag_bucket[f] < n_buckets, HH_ERR_ARG, "hh_correct_split: bucket %d of fragment %d >= n_buckets %d",
                   frag_bucket[f], f, n_buckets);
        HH_REQUIRE(list_off[f + 1] - list_off[f] >= 2 && shift_pos[list_off[f + 1] - 1] == 0, HH_ERR_ARG,
                   "hh_correct_split: the shift list of fragment %d must hold its breakpoints and end with 0", f);
        HH_REQUIRE(frag_off[f] >= 0 && frag_off[f] < hc->n_bins, HH_ERR_ARG, "hh_correct_split: fragment %d offset", f);
        if (frag_bucket[f] >= 0) slot[(size_t)frag_bucket[f]] = f;
    }
    const int32_t n_list = list_off[n_frag];
    int32_t *d_slot = nullptr, *d_loff = nullptr, *d_pos = nullptr, *d_pb = nullptr;
    int64_t* d_foff = nullptr;
    uint8_t* d_zero = nullptr;
    int rc = HH_OK;
    do {
        if ((rc = hh_dmalloc(&d_slot, (size_t)n_buckets)) || (rc = hh_dmalloc(&d_loff, (size_t)n_frag + 1)) ||
            (rc = hh_dmalloc(&d_pos, (size_t)n_list)) || (rc = hh_dmalloc(&d_pb, (size_t)n_list)) ||
            (rc = hh_dmalloc(&d_foff, (size_t)n_frag)) || (rc = hh_dmalloc(&d_zero, (size_t)n_frag)))
            break;
        cudaStream_t st = ctx->stream;
        cudaError_t e = cudaSuccess;
        if (n_buckets) e = cudaMemcpyAsync(d_slot, slot.data(), (size_t)n_buckets * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_loff, list_off, ((size_t)n_frag + 1) * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_pos, shift_pos, (size_t)n_list * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_pb, piece_bucket, (size_t)n_list * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_foff, frag_off, (size_t)n_frag * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_zero, frag_zero, (size_t)n_frag, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(hc->d_diff, 0, ((size_t)hc->n_bins + 1) * 4, st);
        if (e != cudaSuccess) {
            hh_set_error("hh_correct_split: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
            break;
        }
        if (hc->n_links) {
            hh_k_correct_split<<<grid_for(ctx, hc->n_links), CT_THREADS, 0, st>>>(
                hc->d_links, hc->n_links, d_slot, n_buckets, d_foff, d_loff, d_pos, d_pb, d_zero, hc->res, hc->d_diff);
            ctx->launches++;
            if ((e = cudaGetLastError()) != cudaSuccess) {
                hh_set_error("hh_k_correct_split: %s", cudaGetErrorString(e));
                rc = HH_ERR_CUDA;
                break;
            }
        }
        if ((rc = correct_scan(ctx, hc->d_diff, hc->d_cov, hc->n_bins, true)) != HH_OK) break;
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) {
            hh_set_error("hh_correct_split: %s", cudaGetErrorString(e));
            rc = HH_ERR_CUDA;
        }
    } while (0);
    hh_dfree(d_slot);
    hh_dfree(d_loff);
    hh_dfree(d_pos);
    hh_dfree(d_pb);
    hh_dfree(d_foff);
    hh_dfree(d_zero);
    return rc;
}

extern "C" int hh_correct_set_pieces(hh_correct* hc, int32_t n_piece, const int32_t* piece_off, const int32_t* piece_start,
                                     const int32_t* piece_id) {
    HH_REQUIRE(hc && piece_off && n_piece >= hc->n_ctg && (n_piece == 0 || (piece_start && piece_id)), HH_ERR_ARG,
               "hh_correct_set_pieces: bad argument");
    HH_REQUIRE(piece_off[0] == 0 && piece_off[hc->n_ctg] == n_piece, HH_ERR_ARG, "hh_correct_set_pieces: piece_off");
    for (int32_t c = 0; c < hc->n_ctg; ++c) {
        HH_REQUIRE(piece_off[c + 1] > piece_off[c] && piece_start[piece_off[c]] == 0, HH_ERR_ARG,
                   "hh_correct_set_pieces: contig %d needs at least one piece, the first starting at 0", c);
        for (int32_t k = piece_off[c] + 1; k < piece_off[c + 1]; ++k)
            HH_REQUIRE(piece_start[k] > piece_start[k - 1], HH_ERR_ARG,
                       "hh_correct_set_pieces: piece starts of contig %d must ascend", c);
    }
    hh_scope _scope(hc->ctx);
    hh_dfree(hc->d_piece_off);
    hh_dfree(hc->d_piece_start);
    hh_dfree(hc->d_piece_id);
    HH_CHECK(hh_dmalloc(&hc->d_piece_off, (size_t)hc->n_ctg + 1));
    HH_CHECK(hh_dmalloc(&hc->d_piece_start, (size_t)n_piece));
    HH_CHECK(hh_dmalloc(&hc->d_piece_id, (size_t)n_piece));
    cudaStream_t st = hc->ctx->stream;
    HH_CUDA(cudaMemcpyAsync(hc->d_piece_off, piece_off, ((size_t)hc->n_ctg + 1) * 4, cudaMemcpyHostToDevice, st));
    if (n_piece) {
        HH_CUDA(cudaMemcpyAsync(hc->d_piece_start, piece_start, (size_t)n_piece * 4, cudaMemcpyHostToDevice, st));
        HH_CUDA(cudaMemcpyAsync(hc->d_piece_id, piece_id, (size_t)n_piece * 4, cudaMemcpyHostToDevice, st));
    }
    HH_CUDA(cudaStreamSynchronize(st));
    hc->have_pieces = true;
    return HH_OK;
}

extern "C" int hh_correct_remap(hh_correct* hc, int32_t* rec, int64_t n_rec, int mem) {
    HH_REQUIRE(hc && (rec || n_rec == 0) && n_rec >= 0, HH_ERR_ARG, "hh_correct_remap: bad argument");
    HH_REQUIRE(mem == HH_MEM_HOST || mem == HH_MEM_DEVICE, HH_ERR_ARG, "hh_correct_remap: bad mem flag %d", mem);
    HH_REQUIRE(hc->have_pieces, HH_ERR_STATE, "hh_correct_remap: call hh_correct_set_pieces first");
    if (n_rec == 0) return HH_OK;
    hh_ctx* ctx = hc->ctx;
    hh_scope _scope(ctx);
    const int64_t CH = 1ll << 22;
    for (int64_t off = 0; off < n_rec; off += CH) {
        const int64_t m = std::min(CH, n_rec - off);
        int4* dst;
        if (mem == HH_MEM_DEVICE) {
            HH_REQUIRE((((uintptr_t)rec) & 15) == 0, HH_ERR_ARG, "hh_correct_remap: records must be 16-byte aligned");
            dst = reinterpret_cast<int4*>(rec) + off;
        } else {
            HH_CHECK(correct_stage(hc, CH));
            HH_CUDA(cudaMemcpyAsync(hc->d_stage, rec + off * 4, (size_t)m * 16, cudaMemcpyHostToDevice, ctx->stream));
            dst = reinterpret_cast<int4*>(hc->d_stage);
        }
        HH_LAUNCH(ctx, hh_k_correct_remap, grid_for(ctx, m), CT_THREADS, 0, dst, m, hc->n_ctg, hc->d_piece_off,
                  hc->d_piece_start, hc->d_piece_id);
        if (mem == HH_MEM_HOST)
            HH_CUDA(cudaMemcpyAsync(rec + off * 4, hc->d_stage, (size_t)m * 16, cudaMemcpyDeviceToHost, ctx->stream));
    }
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    return HH_OK;
}

extern "C" int hh_correct_destroy(hh_correct* hc) {
    if (!hc) return HH_OK;
    hh_scope _scope(hc->ctx);
    hh_dfree(hc->d_bin_off);
    hh_dfree(hc->d_len);
    hh_dfree(hc->d_diff);
    hh_dfree(hc->d_cov);
    hh_dfree(hc->d_links);
    hh_dfree(hc->d_counters);
    hh_dfree(hc->d_stage);
    hh_dfree(hc->d_piece_off);
    hh_dfree(hc->d_piece_start);
    hh_dfree(hc->d_piece_id);
    cudaStreamSynchronize(hc->ctx->stream);
    delete hc;
    return HH_OK;
}
