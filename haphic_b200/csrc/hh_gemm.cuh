// Internal interface of the tensor-core pre-expansion (hh_gemm.cu), used by hh_mcl.cu.
#pragma once
#include "hh_common.cuh"
#include "hh_internal.cuh"
#include <vector>

enum { HH_GEMM_DIRECT = 1, HH_GEMM_MIRROR = 2 };

// one output tile of D = A . B^T (both operands row-major, K contiguous): first row of the A rows / of the B rows it
// multiplies, the bounds beyond which nothing is stored, up to two ranges of 64-wide k-blocks that are accumulated, and where
// the result goes: element (r, c) -> out[(c - col_lo) * ld + (r - out_row0)], mirror image (c, r) likewise
struct hh_gemm_item {
    int m0, n0;
    int m_end, n_end;
    int kb_lo[2], kb_hi[2];
    int flags;
    int out_row0;
    int pad[2];
};

// dense 16-bit operand planes: element (row, k) of plane p at base[p * plane + row * ldk + k]
enum { HH_GEMM_BF16 = 0, HH_GEMM_F16 = 1 };
struct hh_gemm_operand {
    const unsigned short* base;
    int planes;
    int rows, kdim;            // extent of the tensor map (TMA zero-fills beyond it)
    long long ldk, plane;
    int fmt;                   // HH_GEMM_BF16 / HH_GEMM_F16
};

struct hh_gemm_stats {
    int a_planes, passes, cta_group, stages, chunk_kb;
    int clipped;           // 1: counts above `clip` were clipped and the caller owes the sparse correction
    float clip;
    int fmt_a, fmt_b;      // HH_GEMM_BF16 / HH_GEMM_F16 per operand
    int b_planes;
    int k_chunks;          // launches the K range was cut into (operand planes of one chunk at a time)
    float densify_ms, gemm_ms;
    double flops;          // tensor-core flops issued (2 * M * N * K * passes over all tiles)
};

int hh_gemm_tile_size();
int hh_gemm_items_full(int n, int col_lo, int col_hi, std::vector<hh_gemm_item>& out);
// M1[:, col_lo:col_hi] (dense column-major, leading dimension ld, zero-filled first) from the raw link matrix
int hh_gemm_preexpand(hh_ctx* ctx, const hh_matrix* m, int col_lo, int col_hi, float* d_m1, long long ld, const hh_gemm_item* h_items,
                      int n_items, hh_gemm_stats* st);
// the GEMM itself on prepared operands: D tiles listed in d_items (device), written to out (column-major, leading dimension
// ld, columns [col_lo, col_hi)), each element multiplied by scale[c] when scale != NULL.  The pass list multiplies plane
// pa[p] of A with plane pb[p] of B.  accumulate = 1: the epilogue adds to the values `out` holds (the K range of a product processed in several launches).
// Asynchronous on the context's stream.
int hh_gemm_run(hh_ctx* ctx, const hh_gemm_operand& A, const hh_gemm_operand& B, const hh_gemm_item* d_items, int n_items, int npass,
                const int* pa, const int* pb, int chunk_kb, float* out, long long ld, int col_lo, int col_hi, const float* scale,
                int* stages_out, float out_scale, int accumulate);
int hh_gemm_cta_group();
int hh_gemm_passes(int na, int* pa, int* pb);

// operand planes of the block-diagonal iterate (row pitch ldk, rows = all n vertices): Bt from the slotted columns of `list`,
// A by transposing inside every component.  f16 = 0: three exact bf16 planes each (six passes); f16 = 1: two f16 planes of
// M * 2^14 each (four passes, every product within 2^-22 relative); the GEMM output is multiplied by hh_gemm_blk_out_scale().
int hh_gemm_blk_operands(hh_ctx* ctx, const int* d_len, const void* d_ent, int cap, const int* d_list, int nlist, const int* d_comp_lo,
                         const int* d_comp_hi, int n, unsigned short* d_A, unsigned short* d_Bt, long long ldk, int f16);
float hh_gemm_blk_out_scale(int f16);
