// dict_to_matrix (scripts/HapHiC_cluster.py:310-373) on the GPU: from the compact link table to a
// symmetric fp32 CSC with self loops, in the reference's first-seen index order.
#include "hh_common.cuh"
#include "hh_internal.cuh"

__global__ void hh_k_set_tail(const int32_t* __restrict__ tail, int n_tail, int n_linked, const uint8_t* __restrict__ keep,
                              int32_t* __restrict__ index, int n_ctg, int* __restrict__ err) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tail) return;
    const int c = tail[t];
    if (c < 0 || c >= n_ctg || !keep[c] || index[c] >= 0) {
        atomicExch(err, 1);
        return;
    }
    index[c] = n_linked + t;
}

// every kept fragment must have an index by now, every dropped one must not
__global__ void hh_k_check_index(const int32_t* __restrict__ index, const uint8_t* __restrict__ keep, int n_ctg, int n,
                                 int* __restrict__ err) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_ctg) return;
    const int ix = index[c];
    if (keep[c] ? (ix < 0 || ix >= n) : (ix >= 0)) atomicExch(err, 2);
}

__global__ void hh_k_mat_count(const uint32_t* __restrict__ compact, int64_t nnz, const int32_t* __restrict__ index,
                               int* __restrict__ colcnt) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        const uint32_t* p = compact + e * 9;
        if (p[3] == 0) continue;
        const int ii = index[p[0]], jj = index[p[1]];
        if (ii < 0 || jj < 0) continue;                 // 329-330
        atomicAdd(colcnt + ii, 1);
        atomicAdd(colcnt + jj, 1);
    }
}

__global__ void hh_k_fill_i32(int* __restrict__ p, int v, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__global__ void hh_k_mat_scatter(const uint32_t* __restrict__ compact, int64_t nnz, const int32_t* __restrict__ index,
                                 const unsigned long long* __restrict__ ctg_tot, int normalize,
                                 const int64_t* __restrict__ colptr, int* __restrict__ cursor, int32_t* __restrict__ row,
                                 float* __restrict__ val) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        const uint32_t* p = compact + e * 9;
        if (p[3] == 0) continue;
        const int ii = index[p[0]], jj = index[p[1]];
        if (ii < 0 || jj < 0) continue;
        float v;
        if (normalize) {
            // links / (tot_i * tot_j) ** 0.5 in fp64 (718-724), cast to fp32 by coo_matrix(dtype=float32) (368)
            const unsigned long long prod = ctg_tot[p[0]] * ctg_tot[p[1]];
            v = (float)((double)p[3] / pow((double)prod, 0.5));
        } else {
            v = (float)p[3];
        }
        int64_t q = colptr[jj] + atomicAdd(cursor + jj, 1);    // (row ii, col jj)
        row[q] = ii;
        val[q] = v;
        q = colptr[ii] + atomicAdd(cursor + ii, 1);            // diagonal symmetry (351-353)
        row[q] = jj;
        val[q] = v;
    }
}

__global__ void hh_k_mat_diag(int n, const int64_t* __restrict__ colptr, int* __restrict__ cursor, int32_t* __restrict__ row,
                              float* __restrict__ val) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const int64_t q = colptr[c] + atomicAdd(cursor + c, 1);     // self loops = 1 (362-364)
    row[q] = c;
    val[q] = 1.0f;
}

static int matrix_alloc(hh_ctx* ctx, int32_t n, int64_t nnz, hh_matrix** out) {
    hh_matrix* m = new (std::nothrow) hh_matrix();
    HH_REQUIRE(m != nullptr, HH_ERR_NOMEM, "hh_matrix: out of host memory");
    memset(m, 0, sizeof(*m));
    m->ctx = ctx;
    m->n = n;
    m->nnz = nnz;
    int rc;
    if ((rc = hh_dmalloc(&m->d_colptr, (size_t)n + 1)) != HH_OK || (rc = hh_dmalloc(&m->d_row, (size_t)nnz)) != HH_OK ||
        (rc = hh_dmalloc(&m->d_val, (size_t)nnz)) != HH_OK) {
        hh_matrix_destroy(m);
        return rc;
    }
    *out = m;
    return HH_OK;
}

extern "C" int hh_matrix_from_links(hh_links* lk, const uint8_t* keep, const int32_t* tail, int32_t n_tail,
                                    int normalize_by_nlinks, int add_self_loops, hh_matrix** out) {
    HH_REQUIRE(lk && keep && out, HH_ERR_ARG, "hh_matrix_from_links: NULL argument");
    hh_scope _scope(hh_links_ctx(lk));
    HH_REQUIRE(n_tail >= 0 && (tail || n_tail == 0), HH_ERR_ARG, "hh_matrix_from_links: bad tail");
    HH_REQUIRE(hh_links_finished(lk), HH_ERR_STATE, "hh_matrix_from_links: call hh_links_finish first");
    *out = nullptr;
    hh_ctx* ctx = hh_links_ctx(lk);
    HH_CUDA(cudaSetDevice(ctx->device));
    const int n_ctg = hh_links_n_ctg(lk);
    // the first-seen indices for this keep mask (reused when hh_links_linked_index has just computed them)
    int32_t n_linked = 0;
    HH_CHECK(hh_links_index_for(lk, keep, &n_linked));
    int32_t* d_index = hh_links_index_dev(lk, &n_linked);
    const uint8_t* d_keep = hh_links_keep_dev(lk);
    const int n = n_linked + n_tail;
    HH_REQUIRE(n > 0, HH_ERR_ARG, "hh_matrix_from_links: empty fragment set");
    int* d_err = reinterpret_cast<int*>(ctx->d_scratch + 9);
    HH_CUDA(cudaMemsetAsync(d_err, 0, sizeof(int), ctx->stream));
    int32_t* d_tail = nullptr;
    int* d_cnt = nullptr;
    int* d_cursor = nullptr;
    hh_matrix* m = nullptr;
    int rc = [&]() -> int {
        if (n_tail) {
            HH_CHECK(hh_dmalloc(&d_tail, (size_t)n_tail));
            HH_CUDA(cudaMemcpyAsync(d_tail, tail, (size_t)n_tail * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
            hh_links_index_invalidate(lk);
            HH_LAUNCH(ctx, hh_k_set_tail, (n_tail + 255) / 256, 256, 0, d_tail, n_tail, n_linked, d_keep, d_index, n_ctg, d_err);
        }
        HH_LAUNCH(ctx, hh_k_check_index, (n_ctg + 255) / 256, 256, 0, d_index, d_keep, n_ctg, n, d_err);
        HH_CHECK(hh_dmalloc(&d_cnt, (size_t)n));
        HH_CHECK(hh_dmalloc(&d_cursor, (size_t)n));
        HH_LAUNCH(ctx, hh_k_fill_i32, (n + 255) / 256, 256, 0, d_cnt, add_self_loops ? 1 : 0, n);     // the self loop
        HH_CUDA(cudaMemsetAsync(d_cursor, 0, (size_t)n * sizeof(int), ctx->stream));
        int64_t nnz_c = 0;
        const uint32_t* compact = hh_links_compact(lk, &nnz_c);
        const int gridc = (int)((nnz_c + 255) / 256 < (int64_t)ctx->sm_count * 8 ? (nnz_c + 255) / 256 : (int64_t)ctx->sm_count * 8);
        if (nnz_c) HH_LAUNCH(ctx, hh_k_mat_count, gridc, 256, 0, compact, nnz_c, d_index, d_cnt);
        int64_t* d_ptr = nullptr;
        HH_CHECK(hh_dmalloc(&d_ptr, (size_t)n + 1));
        int rc2 = [&]() -> int {
            HH_CHECK(hh_exclusive_scan_i32(ctx, d_cnt, d_ptr, n));
            HH_CUDA(cudaMemcpyAsync(ctx->h_scratch, d_ptr + n, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            HH_CUDA(cudaMemcpyAsync(ctx->h_scratch + 1, d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            HH_CUDA(cudaStreamSynchronize(ctx->stream));
            const int err = *reinterpret_cast<int*>(ctx->h_scratch + 1);
            HH_REQUIRE(err == 0, HH_ERR_ARG,
                       err == 1 ? "hh_matrix_from_links: tail lists an id that is dropped, linked, repeated or out of range"
                                : "hh_matrix_from_links: keep mask and tail do not cover the fragment set exactly");
            const int64_t nnz = (int64_t)ctx->h_scratch[0];
            HH_CHECK(matrix_alloc(ctx, n, nnz, &m));
            HH_CUDA(cudaMemcpyAsync(m->d_colptr, d_ptr, ((size_t)n + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx->stream));
            if (nnz_c)
                HH_LAUNCH(ctx, hh_k_mat_scatter, gridc, 256, 0, compact, nnz_c, d_index, hh_links_ctg_totals(lk), normalize_by_nlinks,
                          m->d_colptr, d_cursor, m->d_row, m->d_val);
            if (add_self_loops) HH_LAUNCH(ctx, hh_k_mat_diag, (n + 255) / 256, 256, 0, n, m->d_colptr, d_cursor, m->d_row, m->d_val);
            HH_CHECK(hh_dmalloc(&m->d_index, (size_t)n_ctg));
            m->n_index = n_ctg;
            HH_CUDA(cudaMemcpyAsync(m->d_index, d_index, (size_t)n_ctg * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            HH_CUDA(cudaStreamSynchronize(ctx->stream));
            return HH_OK;
        }();
        hh_dfree(d_ptr);
        return rc2;
    }();
    hh_dfree(d_tail);
    hh_dfree(d_cnt);
    hh_dfree(d_cursor);
    if (rc != HH_OK) {
        hh_matrix_destroy(m);
        return rc;
    }
    *out = m;
    return HH_OK;
}

extern "C" int hh_matrix_from_csc(hh_ctx* ctx, int32_t n, const int64_t* indptr, const int32_t* indices, const float* data,
                                  hh_matrix** out) {
    HH_REQUIRE(ctx && indptr && out, HH_ERR_ARG, "hh_matrix_from_csc: NULL argument");
    hh_scope _scope(ctx);
    HH_REQUIRE(n > 0, HH_ERR_ARG, "hh_matrix_from_csc: n must be positive");
    *out = nullptr;
    HH_REQUIRE(indptr[0] == 0, HH_ERR_ARG, "hh_matrix_from_csc: indptr[0] must be 0");
    for (int32_t c = 0; c < n; ++c)
        HH_REQUIRE(indptr[c + 1] >= indptr[c] && indptr[c + 1] - indptr[c] <= n, HH_ERR_ARG,
                   "hh_matrix_from_csc: column %d has an invalid extent", c);
    const int64_t nnz = indptr[n];
    HH_REQUIRE(nnz == 0 || (indices && data), HH_ERR_ARG, "hh_matrix_from_csc: NULL indices/data");
    for (int64_t e = 0; e < nnz; ++e)
        HH_REQUIRE(indices[e] >= 0 && indices[e] < n, HH_ERR_ARG, "hh_matrix_from_csc: row index out of range at entry %lld",
                   (long long)e);
    HH_CUDA(cudaSetDevice(ctx->device));
    hh_matrix* m = nullptr;
    HH_CHECK(matrix_alloc(ctx, n, nnz, &m));
    int rc = [&]() -> int {
        HH_CUDA(cudaMemcpyAsync(m->d_colptr, indptr, ((size_t)n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
        if (nnz) {
            HH_CUDA(cudaMemcpyAsync(m->d_row, indices, (size_t)nnz * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
            HH_CUDA(cudaMemcpyAsync(m->d_val, data, (size_t)nnz * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        }
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        return HH_OK;
    }();
    if (rc != HH_OK) {
        hh_matrix_destroy(m);
        return rc;
    }
    *out = m;
    return HH_OK;
}

extern "C" int hh_matrix_info(hh_matrix* m, int32_t* n, int64_t* nnz) {
    HH_REQUIRE(m != nullptr, HH_ERR_ARG, "hh_matrix_info: NULL handle");
    if (n) *n = m->n;
    if (nnz) *nnz = m->nnz;
    return HH_OK;
}

extern "C" int hh_matrix_destroy(hh_matrix* m) {
    if (!m) return HH_OK;
    hh_scope _scope(m->ctx);
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    hh_dfree(m->d_colptr);
    hh_dfree(m->d_row);
    hh_dfree(m->d_val);
    hh_dfree(m->d_index);
    delete m;
    return HH_OK;
}
