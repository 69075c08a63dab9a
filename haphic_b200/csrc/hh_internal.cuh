// Internal (non-ABI) declarations shared between the translation units of libhaphic_b200.
#pragma once
#include "hh_common.cuh"

struct hh_matrix {
    hh_ctx* ctx;
    int32_t n;
    int64_t nnz;
    int64_t* d_colptr;   // [n+1]
    int32_t* d_row;      // [nnz]  rows are NOT sorted inside a column
    float* d_val;        // [nnz]
    int32_t* d_index;    // [n_index] contig id -> matrix index (-1 = absent); NULL for hh_matrix_from_csc
    int32_t n_index;
};

// hh_links accessors (hh_links.cu)
int32_t hh_links_n_ctg(hh_links* lk);
hh_ctx* hh_links_ctx(hh_links* lk);
const uint32_t* hh_links_compact(hh_links* lk, int64_t* nnz);
const unsigned long long* hh_links_ctg_totals(hh_links* lk);
int32_t* hh_links_index_dev(hh_links* lk, int32_t* n_linked);
uint8_t* hh_links_keep_dev(hh_links* lk);
bool hh_links_finished(hh_links* lk);
int hh_links_index_for(hh_links* lk, const uint8_t* keep, int32_t* n_linked);
void hh_links_index_invalidate(hh_links* lk);
