// Link counting on the GPU: the per-read-pair loop of parse_alignments_for_ctgs
// (scripts/HapHiC_cluster.py:1596-1655) as a warp-aggregated atomic histogram over an
// open-addressing hash table keyed by the (name-ordered) contig pair.
//
// Per record (16 B, one 128-bit streaming load) the kernel
//   * drops ctg_a == ctg_b (generator filter, 1582 / 2862) and ids outside the FASTA (1625),
//   * orders the two ends by contig NAME rank (1629),
//   * evaluates is_flank on both 1-based coordinates and the Nx membership (1636, 299-307),
//   * evaluates the head/tail halves `coord*2 > len` (404-416),
//   * groups equal keys inside the warp with match.any so one lane issues the atomics for the
//     whole group (coordinate- or name-sorted inputs collapse 32 records into one update),
//   * updates {full, flank, HT, TH, TT} counters and the first-seen stream indices (dict
//     insertion order of full_link_dict / flank_link_dict) of the key's slot, and the two
//     per-fragment totals (ctg_link_dict, 1638-1639).
// hh_links_finish orders the distinct keys by first appearance with a scatter + stream
// compaction (no sort): order[first_full] = slot, then compact.
#include "hh_common.cuh"
#include <stdlib.h>
#include <algorithm>
#include <vector>

#define HH_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define HH_NONE32 0xFFFFFFFFu

struct __align__(32) hh_slot {
    uint32_t first_full, first_flank, full, flank, ht, th, tt, pad;
};

// Counter updates of one (warp-aggregated) group of records on a slot: plain 32-bit reductions (fire and forget).
// (Measured at 200M records: packing full|flank and ht|th into 64-bit adds and guarding the two minima with a load made the
// counting 7 % slower, not faster -- the launches are not bound by the atomics of hot pairs.)
__device__ __forceinline__ void hh_slot_update(hh_slot* v, unsigned c_full, unsigned c_fl, uint32_t first_all, uint32_t first_fl,
                                               unsigned c_ht, unsigned c_th, unsigned c_tt) {
    atomicAdd(&v->full, c_full);
    atomicMin(&v->first_full, first_all);
    if (c_fl) {
        atomicAdd(&v->flank, c_fl);
        atomicMin(&v->first_flank, first_fl);
    }
    if (c_ht) atomicAdd(&v->ht, c_ht);
    if (c_th) atomicAdd(&v->th, c_th);
    if (c_tt) atomicAdd(&v->tt, c_tt);
}

struct hh_partset {
    int4* buf;                       // [npart][pcap] records {i, j, stream index, flags}
    unsigned long long* cursor;      // [npart] records written to every region (may exceed pcap: the excess went to the spill list)
    uint64_t pcap;                   // records per partition region
    int64_t sized_for, sent;         // records the set was sized for / sent to it so far
};

struct hh_links {
    hh_ctx* ctx;
    int32_t n_ctg;                   // key space: contigs, or fragments (contigs / bins) in fragment mode
    int64_t flank_bp;
    int32_t* d_len;                  // [n_ctg] lengths of the key-space objects
    int32_t* d_rank;                 // [n_ctg] name rank of the key-space objects
    uint8_t* d_nx;
    // fragment mode (parse_alignments, HapHiC_cluster.py:1658-1752): records name SOURCE contigs, keys are fragments
    int32_t n_src;                   // number of source contigs (= n_ctg in contig mode)
    int32_t* d_src_rank;             // [n_src] name rank of the source contigs
    int32_t* d_fbase;                // [n_src + 1] first fragment id of every contig (more than one fragment = split into bins)
    int64_t bin_size;
    unsigned long long* d_ctg;       // [n_ctg] per-fragment flank-link totals
    uint64_t* d_keys;                // [cap]
    hh_slot* d_vals;                 // [cap]
    uint64_t cap;                    // power of two
    unsigned long long* d_counters;  // [0] distinct keys  [1] records used  [2] overflow flag  [3] nnz_flank
                                     // [4] largest first-seen index merged from a peer
    int64_t n_records, stream_end;
    int64_t known_unique, since_known;   // growth bookkeeping (see ensure_capacity)
    bool finished;
    bool ordered;                    // d_compact is in dict insertion order (false after hh_links_finish_partition / hh_links_adopt)
    int64_t nnz, nnz_flank, n_used;
    int64_t peer_used;               // records counted by merged peers
    uint32_t* d_compact;             // [nnz][9]  {i, j, full, flank, first_full, first_flank, HT, TH, TT}
    // host staging (double-buffered H2D)
    int4* d_stage[2];
    cudaEvent_t ev_copied[2], ev_consumed[2];
    cudaStream_t copy_stream;
    int64_t stage_records;
    // partitioned counting (contig mode, long streams; see "partition, then aggregate" below)
    int mode;                        // 0 undecided, 1 direct (one big hash table), 2 partitioned
    int npart_log;                   // log2 of the number of partitions
    uint64_t scap;                   // slots of a scratch table (power of two)
    uint64_t spill_cap;
    std::vector<hh_partset>* psets;  // partition buffers; normally one set, a new one when a later add call outgrows it
    int4* d_spill;                   // records of partitions whose region overflowed (skewed keys), with their partition id
    unsigned long long* d_spill_cursor;
    int64_t capacity_hint;
    // dict_to_matrix support
    int32_t* d_index;                // [n_ctg] matrix index of linked fragments (hh_links_linked_index)
    int32_t n_linked;
    uint8_t* d_keep;
    bool index_valid;                // d_index / n_linked / d_keep hold the result for index_keep and the current entry list
    std::vector<uint8_t>* index_keep;
};

__device__ __forceinline__ uint64_t hh_mix64(uint64_t k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return k;
}

// find-or-insert; returns slot index, sets *inserted.  Returns cap (invalid) if the table is full.
__device__ __forceinline__ uint64_t hh_probe_insert(uint64_t* __restrict__ keys, uint64_t cap, uint64_t key, bool* inserted) {
    const uint64_t mask = cap - 1;
    uint64_t slot = hh_mix64(key) & mask;
    *inserted = false;
    for (uint64_t probes = 0; probes < cap; ++probes) {
        uint64_t k = *((volatile uint64_t*)(keys + slot));
        if (k == key) return slot;
        if (k == HH_EMPTY_KEY) {
            unsigned long long prev = atomicCAS((unsigned long long*)(keys + slot), (unsigned long long)HH_EMPTY_KEY,
                                                (unsigned long long)key);
            if (prev == HH_EMPTY_KEY) {
                *inserted = true;
                return slot;
            }
            if (prev == key) return slot;
        }
        slot = (slot + 1) & mask;
    }
    return cap;
}

__global__ void hh_k_links_init(uint64_t* __restrict__ keys, hh_slot* __restrict__ vals, uint64_t cap) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += stride) {
        keys[s] = HH_EMPTY_KEY;
        uint4* v = reinterpret_cast<uint4*>(vals + s);
        v[0] = make_uint4(HH_NONE32, HH_NONE32, 0u, 0u);
        v[1] = make_uint4(0u, 0u, 0u, 0u);
    }
}

__global__ void __launch_bounds__(256)
hh_k_links_insert(const int4* __restrict__ rec, int64_t n_rec, uint32_t stream_off, int32_t n_ctg,
                  const int32_t* __restrict__ ctg_len, const int32_t* __restrict__ name_rank,
                  const uint8_t* __restrict__ in_nx, int64_t flank_bp, uint64_t* __restrict__ keys,
                  hh_slot* __restrict__ vals, uint64_t cap, unsigned long long* __restrict__ ctg_links,
                  unsigned long long* __restrict__ counters, const int32_t* __restrict__ src_rank,
                  const int32_t* __restrict__ fbase, int64_t bin_size, int32_t n_src, const uint32_t* __restrict__ pos) {
    __shared__ unsigned int s_new, s_used, s_over;
    if (threadIdx.x == 0) {
        s_new = 0;
        s_used = 0;
        s_over = 0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int my_new = 0, my_used = 0;
    // warp-uniform loop bounds: every lane of a warp runs the same number of trips
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x - lane); i0 < n_rec; i0 += stride) {
        const int64_t i = i0 + lane;
        bool ok = i < n_rec;
        int4 r = make_int4(-1, 0, -1, 0);
        if (ok) r = hh_ld_stream(rec + i);
        uint64_t key = HH_EMPTY_KEY - 1 - (uint64_t)lane;   // unique per lane: never groups, never a real key
        int ci = 0, cj = 0;
        bool fl = false, ti = false, tj = false;
        int a = r.x, b = r.z, pa = r.y, pb = r.w;
        if (fbase == nullptr) {
            ok = ok && (a != b) && ((unsigned)a < (unsigned)n_ctg) && ((unsigned)b < (unsigned)n_ctg);
            if (ok && name_rank[a] > name_rank[b]) {      // sorted(((ref,pos+1),(mref,mpos+1))), 1629
                int t = a; a = b; b = t;
                t = pa; pa = pb; pb = t;
            }
        } else {
            // fragment mode (1696-1720): records name source contigs; a contig with several fragments is split
            // into bins of bin_size bp.  n_ctg is the number of fragments here; ids are checked against fbase.
            ok = ok && ((unsigned)a < (unsigned)n_src) && ((unsigned)b < (unsigned)n_src);
            if (ok) {
                const bool split_a = fbase[a + 1] - fbase[a] > 1;
                ok = (a != b) || split_a;                  // intra-contig pairs only matter for split contigs (1699)
            }
            if (ok) {
                // sorted(((ref, pos+1), (mref, mpos+1))): by contig name, then by coordinate (1707)
                const int ra = src_rank[a], rb = src_rank[b];
                if (ra > rb || (a == b && pa > pb)) {
                    int t = a; a = b; b = t;
                    t = pa; pa = pb; pb = t;
                }
                // convert_frags (1662-1670)
                int fa = fbase[a], fb = fbase[b];
                const bool sa = fbase[a + 1] - fa > 1, sb = fbase[b + 1] - fb > 1;
                // a position outside the contig (.pairs position 0, or beyond the last bin) names a bin that does not
                // exist: the reference dies with a KeyError on frag_len_dict['ctg_binK']; here the record is refused and
                // hh_links_finish reports it
                bool bad = false;
                if (sa) {
                    const int64_t nb = ((int64_t)pa + 1 + bin_size - 1) / bin_size;
                    bad = bad || pa < 0 || nb < 1 || nb > (int64_t)(fbase[a + 1] - fa);
                    fa += (int)(nb - 1);
                    pa = (int)((int64_t)pa - (nb - 1) * bin_size);
                }
                if (sb) {
                    const int64_t nb = ((int64_t)pb + 1 + bin_size - 1) / bin_size;
                    bad = bad || pb < 0 || nb < 1 || nb > (int64_t)(fbase[b + 1] - fb);
                    fb += (int)(nb - 1);
                    pb = (int)((int64_t)pb - (nb - 1) * bin_size);
                }
                if (bad) {
                    atomicAdd(counters + 5, 1ull);
                    atomicMax(counters + 6, (unsigned long long)(pos ? pos[i] : stream_off + (uint32_t)i) + 1ull);
                }
                ok = !bad && fa != fb;                     // intra-bin links are not considered (1715)
                a = fa;
                b = fb;
                if (ok && (sa || sb) && name_rank[a] > name_rank[b]) {   // sort by bin name (1719-1720)
                    int t = a; a = b; b = t;
                    t = pa; pa = pb; pb = t;
                }
            }
        }
        if (ok) {
            ci = a;
            cj = b;
            const int64_t coord_i = (int64_t)pa + 1, coord_j = (int64_t)pb + 1;   // 1-based
            const int64_t li = ctg_len[a], lj = ctg_len[b];
            const bool fi = (flank_bp == 0) || (coord_i <= flank_bp) || (coord_i > li - flank_bp);   // is_flank, 299-307
            const bool fj = (flank_bp == 0) || (coord_j <= flank_bp) || (coord_j > lj - flank_bp);
            fl = fi && fj && in_nx[a] && in_nx[b];                                                  // 1636
            ti = coord_i * 2 > li;                                                                   // 404-416
            tj = coord_j * 2 > lj;
            key = ((uint64_t)(uint32_t)a << 32) | (uint64_t)(uint32_t)b;
            my_used++;
        }
        const unsigned peers = __match_any_sync(HH_FULL_MASK, key);
        // stream position of the record: implicit (contiguous shard) or carried along (routed records, any order)
        uint32_t first_all = stream_off + (uint32_t)i, first_fl = HH_NONE32;
        if (pos != nullptr) {
            const uint32_t mine = ok ? pos[i] : HH_NONE32;
            first_all = __reduce_min_sync(peers, mine);
            first_fl = __reduce_min_sync(peers, (ok && fl) ? mine : HH_NONE32);
        }
        const unsigned b_fl = __ballot_sync(HH_FULL_MASK, ok && fl);
        const unsigned b_ht = __ballot_sync(HH_FULL_MASK, ok && !ti && tj);
        const unsigned b_th = __ballot_sync(HH_FULL_MASK, ok && ti && !tj);
        const unsigned b_tt = __ballot_sync(HH_FULL_MASK, ok && ti && tj);
        if (ok && lane == (__ffs(peers) - 1)) {
            bool inserted;
            const uint64_t slot = hh_probe_insert(keys, cap, key, &inserted);
            if (slot >= cap) {
                s_over = 1;
            } else {
                if (inserted) my_new++;
                hh_slot* v = vals + slot;
                const unsigned c_full = __popc(peers);
                const unsigned m_fl = peers & b_fl;
                const unsigned c_fl = __popc(m_fl);
                const unsigned c_ht = __popc(peers & b_ht), c_th = __popc(peers & b_th), c_tt = __popc(peers & b_tt);
                // leader = lowest lane = earliest record
                hh_slot_update(v, c_full, c_fl, first_all, pos ? first_fl : stream_off + (uint32_t)(i0 + (__ffs(m_fl) - 1)), c_ht, c_th, c_tt);
                if (c_fl) {
                    atomicAdd(ctg_links + ci, (unsigned long long)c_fl);
                    atomicAdd(ctg_links + cj, (unsigned long long)c_fl);
                }
            }
        }
    }
    if (my_new) atomicAdd(&s_new, my_new);
    if (my_used) atomicAdd(&s_used, my_used);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_new) atomicAdd(counters + 0, (unsigned long long)s_new);
        if (s_used) atomicAdd(counters + 1, (unsigned long long)s_used);
        if (s_over) atomicExch(counters + 2, 1ull);
    }
}

// ---------------------------------------------------------------------------------------------
// Partition, then aggregate.  One big hash table costs every record a random DRAM sector for the key and another
// read-modify-write for the counters (the table is two orders of magnitude larger than L2).  For long streams the
// records are therefore first split by the high bits of the key hash into 2^npart_log partitions (one sequential read,
// one write in runs that fill whole sectors).  A partition is still far too large for shared memory, and counting the
// partitions one launch at a time in an L2-resident table is a chain of latency-bound launches, so every partition is
// split again by the next hash bits into sub-partitions of at most 512 records, and ONE launch counts all of them, a
// CTA per sub-partition in a shared-memory table, emitting compact entries (9 words, the hh_links_adopt list format).
// Integer adds and mins only: the result is identical to the direct path.
//   hh_k_part_scatter   record -> {i, j, stream index, flags} (ends ordered by name rank, is_flank / head-tail evaluated once)
//   hh_k_sub_split      level 2: every partition (region + its spilled records) split by the next hash bits into
//                       sub-partitions small enough for a shared-memory table (a histogram pass, then the scatter)
//   hh_k_sub_count      one CTA per sub-partition: count in shared memory, emit the live slots
//   hh_k_part_step      the sub-partitions whose keys did not fit the shared table: emit + clear the scratch table of the
//                       previous one, count the current one into the other
// ---------------------------------------------------------------------------------------------
#define HH_PART_TILE 4096          // records per tile of the scatter kernel (512 threads x 8)
#define HH_PART_MAX 1024

// The tile kernels below work in phases: the 8 record loads of a thread are issued together, then the lookups that depend
// on them, then the shared-memory atomics.  Written as one loop per record, the compiler keeps each record's load behind
// the previous record's atomic, and a tile waits through eight DRAM latencies one after the other.
__global__ void __launch_bounds__(512)
hh_k_part_scatter(const int4* __restrict__ rec, int64_t n_rec, uint32_t stream_off, int32_t n_ctg, const int32_t* __restrict__ ctg_len,
                  const int32_t* __restrict__ name_rank, const uint8_t* __restrict__ in_nx, int64_t flank_bp, int npart_log,
                  int4* __restrict__ pbuf, uint64_t pcap, unsigned long long* __restrict__ cursor, int4* __restrict__ spill,
                  uint64_t spill_cap, unsigned long long* __restrict__ spill_cursor, unsigned long long* __restrict__ counters) {
    __shared__ unsigned int s_cnt[HH_PART_MAX];
    __shared__ unsigned long long s_base[HH_PART_MAX];
    __shared__ unsigned int s_used;
    const int npart = 1 << npart_log;
    const int64_t tiles = (n_rec + HH_PART_TILE - 1) / HH_PART_TILE;
    unsigned int my_used = 0;
    if (threadIdx.x == 0) s_used = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        for (int k = threadIdx.x; k < npart; k += 512) s_cnt[k] = 0;
        int4 out[8];
        int part[8];
        unsigned int rnk[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int64_t i = t * HH_PART_TILE + (int64_t)k * 512 + threadIdx.x;
            out[k] = (i < n_rec) ? hh_ld_stream(rec + i) : make_int4(-1, 0, -1, 0);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            int a = out[k].x, b = out[k].z, pa = out[k].y, pb = out[k].w;
            part[k] = -1;
            if (a != b && (unsigned)a < (unsigned)n_ctg && (unsigned)b < (unsigned)n_ctg) {
                if (name_rank[a] > name_rank[b]) {      // sorted(((ref,pos+1),(mref,mpos+1))), 1629
                    int x = a; a = b; b = x;
                    x = pa; pa = pb; pb = x;
                }
                const int64_t coord_i = (int64_t)pa + 1, coord_j = (int64_t)pb + 1;
                const int64_t li = ctg_len[a], lj = ctg_len[b];
                const bool fi = (flank_bp == 0) || (coord_i <= flank_bp) || (coord_i > li - flank_bp);   // is_flank, 299-307
                const bool fj = (flank_bp == 0) || (coord_j <= flank_bp) || (coord_j > lj - flank_bp);
                const unsigned fl = (fi && fj && in_nx[a] && in_nx[b]) ? 1u : 0u;                         // 1636
                const unsigned ti = (coord_i * 2 > li) ? 2u : 0u, tj = (coord_j * 2 > lj) ? 4u : 0u;       // 404-416
                const uint64_t key = ((uint64_t)(uint32_t)a << 32) | (uint64_t)(uint32_t)b;
                const int p = (int)(hh_mix64(key) >> (64 - npart_log));
                const int64_t i = t * HH_PART_TILE + (int64_t)k * 512 + threadIdx.x;
                part[k] = p;
                out[k] = make_int4(a, b, (int)(stream_off + (uint32_t)i), (int)(fl | ti | tj | ((unsigned)p << 8)));
                my_used++;
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (part[k] >= 0) rnk[k] = atomicAdd(&s_cnt[part[k]], 1u);
        __syncthreads();
        for (int k = threadIdx.x; k < npart; k += 512)
            if (s_cnt[k]) s_base[k] = atomicAdd(cursor + k, (unsigned long long)s_cnt[k]);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (part[k] < 0) continue;
            const unsigned long long q = s_base[part[k]] + rnk[k];
            if (q < pcap) {
                pbuf[(size_t)part[k] * (size_t)pcap + (size_t)q] = out[k];
            } else {
                // the region of this partition is full (a few pairs own a large share of the stream): spill list
                const unsigned long long sq = atomicAdd(spill_cursor, 1ull);
                if (sq < spill_cap) spill[sq] = out[k];
                else atomicExch(counters + 2, 3ull);
            }
        }
        __syncthreads();
    }
    my_used = (unsigned)hh_warp_sum((int)my_used);
    if ((threadIdx.x & 31) == 0 && my_used) atomicAdd(&s_used, my_used);
    __syncthreads();
    if (threadIdx.x == 0 && s_used) atomicAdd(counters + 1, (unsigned long long)s_used);
}

#define HH_SUB_MAX_LOG 10          // at most 2^10 sub-partitions per partition
// Slots of the shared-memory table: a sub-partition is sized for <= HH_SUB_SLOTS / 2 records.  Measured at C3 on a B200, the
// count runs faster the more warps an SM holds: 2048 slots (two CTAs an SM with the record buffers) 10.9 ms, 1024 slots
// (four CTAs) 7.4 ms.
#define HH_SUB_SLOTS 1024
#define HH_SUB_CHUNK (HH_SUB_SLOTS / 2)   // records a record buffer of hh_k_sub_count holds
// two record buffers of 16 B records, u64 key + 7 u32 counters a slot, u16 live-slot list: 54 KB, four CTAs an SM
#define HH_SUB_SMEM (2 * HH_SUB_CHUNK * 16 + HH_SUB_SLOTS * (36 + 2))

__device__ __forceinline__ unsigned hh_sub_of(const int4 r, int npart_log, int sub_log) {
    const uint64_t key = ((uint64_t)(uint32_t)r.x << 32) | (uint64_t)(uint32_t)r.y;
    return (unsigned)((hh_mix64(key) >> (64 - npart_log - sub_log)) & ((1ull << sub_log) - 1ull));
}

// Level 2.  blockIdx.y = the region of a partition, or (y == npart) the spill list.  !SCATTER: sub_cnt[p << sub_log | s] +=
// records of sub-partition s of partition p.  SCATTER: record -> out[sub_off[id] + atomicAdd(sub_cnt[id])] (sub_cnt zeroed by
// hh_k_sub_offsets), ranked inside a tile in shared memory with one global atomic per sub-partition and tile, as in
// hh_k_part_scatter.
template <bool SCATTER>
__global__ void __launch_bounds__(512)
hh_k_sub_split(const int4* __restrict__ pbuf, uint64_t pcap, const unsigned long long* __restrict__ fill, int npart_log,
               const int4* __restrict__ spill, const unsigned long long* __restrict__ spill_fill, uint64_t spill_cap, int sub_log,
               unsigned int* __restrict__ sub_cnt, const int64_t* __restrict__ sub_off, int4* __restrict__ out) {
    __shared__ unsigned int s_cnt[1 << HH_SUB_MAX_LOG];
    __shared__ unsigned long long s_base[SCATTER ? (1 << HH_SUB_MAX_LOG) : 1];
    const int npart = 1 << npart_log, nsub = 1 << sub_log;
    const int seg = blockIdx.y;
    if (seg == npart) {
        // the spill list (skewed streams only): records of any partition, which they carry in their flags
        const int64_t n = (int64_t)min(*spill_fill, (unsigned long long)spill_cap);
        for (int64_t i = (int64_t)blockIdx.x * 512 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 512) {
            const int4 r = spill[i];
            const unsigned id = (((unsigned)r.w >> 8) << sub_log) | hh_sub_of(r, npart_log, sub_log);
            if (SCATTER) out[sub_off[id] + atomicAdd(sub_cnt + id, 1u)] = r;
            else atomicAdd(sub_cnt + id, 1u);
        }
        return;
    }
    const int4* src = pbuf + (size_t)seg * (size_t)pcap;
    const int64_t n = (int64_t)min(fill[seg], (unsigned long long)pcap);      // the excess is on the spill list
    unsigned int* cnt = sub_cnt + ((size_t)seg << sub_log);
    const int64_t tiles = (n + HH_PART_TILE - 1) / HH_PART_TILE;
    for (int k = threadIdx.x; k < nsub; k += 512) s_cnt[k] = 0;
    __syncthreads();
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        int4 r[8];
        int s[8];
        unsigned int rnk[8];
        // phases as in hh_k_part_scatter: all loads, then the sub-partition ids, then the atomics
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int64_t i = t * HH_PART_TILE + (int64_t)k * 512 + threadIdx.x;
            if (i < n) r[k] = hh_ld_stream(src + i);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int64_t i = t * HH_PART_TILE + (int64_t)k * 512 + threadIdx.x;
            s[k] = (i < n) ? (int)hh_sub_of(r[k], npart_log, sub_log) : -1;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (s[k] < 0) continue;
            if (SCATTER) rnk[k] = atomicAdd(&s_cnt[s[k]], 1u);
            else atomicAdd(&s_cnt[s[k]], 1u);
        }
        if (SCATTER) {
            __syncthreads();
            for (int k = threadIdx.x; k < nsub; k += 512)
                if (s_cnt[k]) s_base[k] = (unsigned long long)sub_off[((size_t)seg << sub_log) + k] + atomicAdd(cnt + k, s_cnt[k]);
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (s[k] >= 0) out[s_base[s[k]] + rnk[k]] = r[k];
            __syncthreads();
            for (int k = threadIdx.x; k < nsub; k += 512) s_cnt[k] = 0;
            __syncthreads();
        }
    }
    if (!SCATTER) {
        __syncthreads();
        for (int k = threadIdx.x; k < nsub; k += 512)
            if (s_cnt[k]) atomicAdd(cnt + k, s_cnt[k]);
    }
}

// sub_off[p << sub_log | s] = pbase[p] + records of sub-partitions 0 .. s-1 of partition p (one CTA a partition); sub_cnt is
// cleared for the scatter.  pbase = exclusive prefix of the partition totals, which the host has from the level-1 cursors.
__global__ void __launch_bounds__(1024)
hh_k_sub_offsets(unsigned int* __restrict__ sub_cnt, int sub_log, const int64_t* __restrict__ pbase, int npart,
                 int64_t* __restrict__ sub_off) {
    __shared__ unsigned int s_w[32];
    const int nsub = 1 << sub_log, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t at = ((size_t)blockIdx.x << sub_log) + threadIdx.x;
    const unsigned int v = (int)threadIdx.x < nsub ? sub_cnt[at] : 0u;
    unsigned int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(HH_FULL_MASK, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const unsigned int w = s_w[lane];
        unsigned int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(HH_FULL_MASK, wi, o);
            if (lane >= o) wi += t;
        }
        s_w[lane] = wi - w;
    }
    __syncthreads();
    if ((int)threadIdx.x < nsub) {
        sub_off[at] = pbase[blockIdx.x] + (int64_t)(s_w[warp] + incl - v);
        sub_cnt[at] = 0u;
    }
    if (blockIdx.x == npart - 1 && threadIdx.x == 0) sub_off[(size_t)npart << sub_log] = pbase[npart];
}

// 16-byte asynchronous global -> shared copies (bypassing L1), in commit groups
__device__ __forceinline__ void hh_cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void hh_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void hh_cp_async_wait_prev() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// Count + emit: a CTA takes sub-partitions in a grid stride, counts each into an open-addressing table in shared memory
// (warp aggregation with match.any as in hh_part_count, then shared-memory atomics), and emits the slots it filled with ONE
// global atomic on the entry cursor.  Nothing global is touched before the emit.  A sub-partition whose keys do not fit the
// table (skewed or adversarial keys only) is abandoned and its id appended to `fallback` (counters[7] entries) for the
// global scratch-table path (hh_k_part_step).
// The records come in chunks of HH_SUB_CHUNK (a whole sub-partition, unless it is a hot one), copied into one of two
// shared-memory buffers while the chunk before is counted from the other.  Every slot a CTA inserts is appended to a list of
// live slots: the emit walks that list (its index is the entry's output position) and resets only those slots, so the table
// is cleared once, at kernel start.
__global__ void __launch_bounds__(256)
hh_k_sub_count(const int4* __restrict__ prec, const int64_t* __restrict__ sub_off, int nsub_total, uint32_t* __restrict__ compact,
               uint64_t compact_cap, unsigned long long* __restrict__ ctg_links, unsigned long long* __restrict__ counters,
               uint32_t* __restrict__ fallback) {
    constexpr int S = HH_SUB_SLOTS, C = HH_SUB_CHUNK;
    extern __shared__ int4 s_rec[];                        // [2][C] records, then u64 keys [S], 7 x u32 [S], u16 live [S]
    uint64_t* s_keys = reinterpret_cast<uint64_t*>(s_rec + 2 * C);
    uint32_t* s_ff = reinterpret_cast<uint32_t*>(s_keys + S);
    uint32_t* s_ffl = s_ff + S;
    uint32_t* s_full = s_ffl + S;
    uint32_t* s_fl = s_full + S;
    uint32_t* s_ht = s_fl + S;
    uint32_t* s_th = s_ht + S;
    uint32_t* s_tt = s_th + S;
    uint16_t* s_live = reinterpret_cast<uint16_t*>(s_tt + S);
    __shared__ unsigned int s_over, s_nlive;
    __shared__ unsigned long long s_base;
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    unsigned int nfl = 0;
    for (int k = threadIdx.x; k < S; k += 256) {
        s_keys[k] = HH_EMPTY_KEY;
        s_ff[k] = HH_NONE32;
        s_ffl[k] = HH_NONE32;
        s_full[k] = 0u;
        s_fl[k] = 0u;
        s_ht[k] = 0u;
        s_th[k] = 0u;
        s_tt[k] = 0u;
    }
    if (threadIdx.x == 0) {
        s_over = 0u;
        s_nlive = 0u;
    }
    // the chunk being counted (sub-partition id, records [b + off, b + off + C) of its n) and the bounds of the CTA's next
    // sub-partition, loaded one sub-partition ahead
    int id = blockIdx.x;
    int64_t off = 0, b = 0, n = 0, nb = 0, nn = 0;
    if (id < nsub_total) {
        b = sub_off[id];
        n = sub_off[id + 1] - b;
        for (int k = threadIdx.x; k < (int)min(n, (int64_t)C); k += 256) hh_cp_async16(s_rec + k, prec + b + k);
    }
    hh_cp_async_commit();
    if (id + (int)gridDim.x < nsub_total) {
        nb = sub_off[id + gridDim.x];
        nn = sub_off[id + gridDim.x + 1] - nb;
    }
    int buf = 0;
    while (id < nsub_total) {
        // start the copy of the next chunk: the rest of this sub-partition, or the first chunk of the next one
        const bool last = off + C >= n;
        {
            const int64_t src = last ? nb : b + off + C;
            const int m = (int)min(last ? nn : n - off - C, (int64_t)C);
            if (!last || id + (int)gridDim.x < nsub_total)
                for (int k = threadIdx.x; k < m; k += 256) hh_cp_async16(s_rec + (buf ^ 1) * C + k, prec + src + k);
            hh_cp_async_commit();
        }
        hh_cp_async_wait_prev();
        __syncthreads();                       // the chunk is in shared memory, the table reset of the last emit is done
        const int4* rc = s_rec + buf * C;
        const int m = (int)min(n - off, (int64_t)C);
        for (int i0 = wv * 32; i0 < m; i0 += 256) {
            if (__any_sync(HH_FULL_MASK, *(volatile unsigned int*)&s_over != 0u)) break;
            const int i = i0 + lane;
            const bool ok = i < m;
            int4 r = make_int4(0, 0, 0, 0);
            if (ok) r = rc[i];
            const unsigned f = (unsigned)r.w;
            const uint64_t key = ok ? (((uint64_t)(uint32_t)r.x << 32) | (uint64_t)(uint32_t)r.y) : (HH_EMPTY_KEY - 1 - (uint64_t)lane);
            const unsigned peers = __match_any_sync(HH_FULL_MASK, key);
            const bool fl = ok && (f & 1u), ti = (f & 2u) != 0, tj = (f & 4u) != 0;
            const uint32_t idx = ok ? (uint32_t)r.z : HH_NONE32;
            const uint32_t first_all = __reduce_min_sync(peers, idx);
            const uint32_t first_fl = __reduce_min_sync(peers, fl ? idx : HH_NONE32);
            const unsigned b_fl = __ballot_sync(HH_FULL_MASK, fl);
            const unsigned b_ht = __ballot_sync(HH_FULL_MASK, ok && !ti && tj);
            const unsigned b_th = __ballot_sync(HH_FULL_MASK, ok && ti && !tj);
            const unsigned b_tt = __ballot_sync(HH_FULL_MASK, ok && ti && tj);
            if (ok && lane == (__ffs(peers) - 1)) {
                unsigned int sl = (unsigned int)hh_mix64(key) & (S - 1);     // the low hash bits; the partition ids took the high ones
                bool found = false;
                for (int q = 0; q < S; ++q) {
                    const uint64_t k = *((volatile uint64_t*)(s_keys + sl));
                    if (k == key) { found = true; break; }
                    if (k == HH_EMPTY_KEY) {
                        const unsigned long long prev = atomicCAS((unsigned long long*)(s_keys + sl), (unsigned long long)HH_EMPTY_KEY,
                                                                  (unsigned long long)key);
                        if (prev == HH_EMPTY_KEY) s_live[atomicAdd(&s_nlive, 1u)] = (uint16_t)sl;
                        if (prev == HH_EMPTY_KEY || prev == key) { found = true; break; }
                    }
                    sl = (sl + 1) & (S - 1);
                }
                if (!found) {
                    s_over = 1u;
                } else {
                    const unsigned c_fl = __popc(peers & b_fl), c_ht = __popc(peers & b_ht), c_th = __popc(peers & b_th),
                                   c_tt = __popc(peers & b_tt);
                    atomicAdd(s_full + sl, (unsigned)__popc(peers));
                    atomicMin(s_ff + sl, first_all);
                    if (c_fl) {
                        atomicAdd(s_fl + sl, c_fl);
                        atomicMin(s_ffl + sl, first_fl);
                    }
                    if (c_ht) atomicAdd(s_ht + sl, c_ht);
                    if (c_th) atomicAdd(s_th + sl, c_th);
                    if (c_tt) atomicAdd(s_tt + sl, c_tt);
                }
            }
        }
        __syncthreads();                       // every warp is done with this chunk's buffer and its table updates
        if (last) {
            // ---- emit: live slots -> compact entries {i, j, full, flank, first_full, first_flank, HT, TH, TT}, per-fragment
            // totals; every live slot is reset for the next sub-partition
            const unsigned int nl = s_nlive;
            const bool over = s_over != 0u;
            __syncthreads();
            if (threadIdx.x == 0) {
                s_base = (!over && nl) ? atomicAdd(counters + 0, (unsigned long long)nl) : 0ull;
                if (over) fallback[atomicAdd(counters + 7, 1ull)] = (uint32_t)id;
                s_nlive = 0u;
                s_over = 0u;
            }
            __syncthreads();
            for (unsigned int t = threadIdx.x; t < nl; t += 256) {
                const int sl = s_live[t];
                if (!over) {
                    const uint64_t key = s_keys[sl];
                    const uint32_t flank = s_fl[sl];
                    const unsigned long long pos = s_base + t;
                    if (pos < compact_cap) {
                        uint32_t* o = compact + pos * 9;
                        o[0] = (uint32_t)(key >> 32);
                        o[1] = (uint32_t)key;
                        o[2] = s_full[sl];
                        o[3] = flank;
                        o[4] = s_ff[sl];
                        o[5] = s_ffl[sl];
                        o[6] = s_ht[sl];
                        o[7] = s_th[sl];
                        o[8] = s_tt[sl];
                    } else {
                        atomicExch(counters + 2, 5ull);
                    }
                    if (flank) {
                        nfl++;
                        atomicAdd(ctg_links + (uint32_t)(key >> 32), (unsigned long long)flank);      // ctg_link_dict (1638-1639)
                        atomicAdd(ctg_links + (uint32_t)key, (unsigned long long)flank);
                    }
                }
                s_keys[sl] = HH_EMPTY_KEY;
                s_ff[sl] = HH_NONE32;
                s_ffl[sl] = HH_NONE32;
                s_full[sl] = 0u;
                s_fl[sl] = 0u;
                s_ht[sl] = 0u;
                s_th[sl] = 0u;
                s_tt[sl] = 0u;
            }
            id += gridDim.x;
            off = 0;
            b = nb;
            n = nn;
            if (id + (int)gridDim.x < nsub_total) {
                nb = sub_off[id + gridDim.x];
                nn = sub_off[id + gridDim.x + 1] - nb;
            }
        } else {
            off += C;
        }
        buf ^= 1;
    }
    nfl = (unsigned)hh_warp_sum((int)nfl);
    if (lane == 0 && nfl) atomicAdd(counters + 3, (unsigned long long)nfl);
}

// count `n` partitioned records ({i, j, stream index, flags}) into a scratch table
__device__ __forceinline__ void hh_part_count(const int4* __restrict__ prec, int64_t n, uint64_t* __restrict__ keys,
                                              hh_slot* __restrict__ vals, uint64_t cap, unsigned long long* __restrict__ counters) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x - lane); i0 < n; i0 += stride) {
        const int64_t i = i0 + lane;
        const bool ok = i < n;
        int4 r = make_int4(0, 0, 0, 0);
        if (ok) r = hh_ld_stream(prec + i);
        const unsigned f = (unsigned)r.w;
        const uint64_t key = ok ? (((uint64_t)(uint32_t)r.x << 32) | (uint64_t)(uint32_t)r.y) : (HH_EMPTY_KEY - 1 - (uint64_t)lane);
        const unsigned peers = __match_any_sync(HH_FULL_MASK, key);
        const bool fl = ok && (f & 1u), ti = (f & 2u) != 0, tj = (f & 4u) != 0;
        const uint32_t idx = ok ? (uint32_t)r.z : HH_NONE32;
        const uint32_t first_all = __reduce_min_sync(peers, idx);
        const uint32_t first_fl = __reduce_min_sync(peers, fl ? idx : HH_NONE32);
        const unsigned b_fl = __ballot_sync(HH_FULL_MASK, fl);
        const unsigned b_ht = __ballot_sync(HH_FULL_MASK, ok && !ti && tj);
        const unsigned b_th = __ballot_sync(HH_FULL_MASK, ok && ti && !tj);
        const unsigned b_tt = __ballot_sync(HH_FULL_MASK, ok && ti && tj);
        if (ok && lane == (__ffs(peers) - 1)) {
            bool inserted;
            const uint64_t slot = hh_probe_insert(keys, cap, key, &inserted);
            if (slot >= cap) {
                atomicExch(counters + 2, 4ull);
            } else {
                hh_slot* v = vals + slot;
                hh_slot_update(v, (unsigned)__popc(peers), (unsigned)__popc(peers & b_fl), first_all, first_fl, (unsigned)__popc(peers & b_ht),
                               (unsigned)__popc(peers & b_th), (unsigned)__popc(peers & b_tt));
            }
        }
    }
}

__global__ void __launch_bounds__(256)
hh_k_part_step(const int4* __restrict__ prec, int64_t n, uint64_t* __restrict__ ckeys, hh_slot* __restrict__ cvals, uint64_t* __restrict__ ekeys, hh_slot* __restrict__ evals, uint64_t cap,
               uint32_t* __restrict__ compact, uint64_t compact_cap, unsigned long long* __restrict__ ctg_links,
               unsigned long long* __restrict__ counters) {
    // ---- emit the table of the previous partition: live slots -> compact entries, per-fragment totals; slots are cleared.
    // A CTA takes 512 consecutive slots, two per thread: the keys are loaded together (one memory round trip instead
    // of one per slot), the live ones are ranked by a block scan, the output positions of the whole CTA are reserved with
    // ONE atomic on the global cursor, then the values are read together and written.
    if (ekeys != nullptr) {
        __shared__ unsigned int s_wtot[8];
        __shared__ unsigned long long s_base;
        const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
        unsigned int nfl = 0;
        constexpr int E = 2;
        for (uint64_t r0 = (uint64_t)blockIdx.x * (256ull * E); r0 < cap; r0 += (uint64_t)gridDim.x * (256ull * E)) {
            uint64_t key[E];
            unsigned int cnt = 0;
#pragma unroll
            for (int q = 0; q < E; ++q) {
                const uint64_t sl = r0 + (uint64_t)q * 256ull + threadIdx.x;
                key[q] = (sl < cap) ? ekeys[sl] : HH_EMPTY_KEY;
                cnt += (key[q] != HH_EMPTY_KEY) ? 1u : 0u;
            }
            unsigned int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int t = __shfl_up_sync(HH_FULL_MASK, incl, o);
                if (lane >= o) incl += t;
            }
            __syncthreads();                       // s_wtot / s_base of the previous trip have been read
            if (lane == 31) s_wtot[wv] = incl;
            __syncthreads();
            unsigned int before = 0, total = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const unsigned int t = s_wtot[k];
                before += (k < wv) ? t : 0u;
                total += t;
            }
            if (threadIdx.x == 0) s_base = total ? atomicAdd(counters + 0, (unsigned long long)total) : 0ull;
            __syncthreads();
            if (cnt) {
                unsigned long long pos = s_base + before + (incl - cnt);
                uint4 v0[E], v1[E];
#pragma unroll
                for (int q = 0; q < E; ++q) {
                    if (key[q] != HH_EMPTY_KEY) {
                        const uint4* vp = reinterpret_cast<const uint4*>(evals + (r0 + (uint64_t)q * 256ull + threadIdx.x));
                        v0[q] = vp[0];       // {first_full, first_flank, full, flank}
                        v1[q] = vp[1];       // {ht, th, tt, pad}
                    }
                }
#pragma unroll
                for (int q = 0; q < E; ++q) {
                    if (key[q] == HH_EMPTY_KEY) continue;
                    const uint64_t sl = r0 + (uint64_t)q * 256ull + threadIdx.x;
                    if (pos < compact_cap) {
                        uint32_t* o = compact + pos * 9;
                        o[0] = (uint32_t)(key[q] >> 32);
                        o[1] = (uint32_t)key[q];
                        o[2] = v0[q].z;
                        o[3] = v0[q].w;
                        o[4] = v0[q].x;
                        o[5] = v0[q].y;
                        o[6] = v1[q].x;
                        o[7] = v1[q].y;
                        o[8] = v1[q].z;
                    } else {
                        atomicExch(counters + 2, 5ull);
                    }
                    pos++;
                    if (v0[q].w) {
                        nfl++;
                        atomicAdd(ctg_links + (uint32_t)(key[q] >> 32), (unsigned long long)v0[q].w);      // ctg_link_dict (1638-1639)
                        atomicAdd(ctg_links + (uint32_t)key[q], (unsigned long long)v0[q].w);
                    }
                    ekeys[sl] = HH_EMPTY_KEY;
                    uint4* vw = reinterpret_cast<uint4*>(evals + sl);
                    vw[0] = make_uint4(HH_NONE32, HH_NONE32, 0u, 0u);
                    vw[1] = make_uint4(0u, 0u, 0u, 0u);
                }
            }
        }
        nfl = (unsigned)hh_warp_sum((int)nfl);
        if (lane == 0 && nfl) atomicAdd(counters + 3, (unsigned long long)nfl);
    }
    // ---- count the current sub-partition
    if (ckeys != nullptr && n > 0) hh_part_count(prec, n, ckeys, cvals, cap, counters);
}

// re-insert every live slot of the old table into a (larger) new one
__global__ void hh_k_links_rehash(const uint64_t* __restrict__ okeys, const hh_slot* __restrict__ ovals, uint64_t ocap,
                                  uint64_t* __restrict__ keys, hh_slot* __restrict__ vals, uint64_t cap,
                                  unsigned long long* __restrict__ counters) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < ocap; s += stride) {
        const uint64_t k = okeys[s];
        if (k == HH_EMPTY_KEY) continue;
        bool inserted;
        const uint64_t slot = hh_probe_insert(keys, cap, k, &inserted);
        if (slot >= cap) {
            atomicExch(counters + 2, 1ull);
            continue;
        }
        const uint4* src = reinterpret_cast<const uint4*>(ovals + s);
        uint4* dst = reinterpret_cast<uint4*>(vals + slot);
        dst[0] = src[0];
        dst[1] = src[1];
    }
}

// merge a peer's export (9 x u32 per entry) into this table
__global__ void hh_k_links_merge(const uint32_t* __restrict__ ent, int64_t n_ent, uint64_t* __restrict__ keys,
                                 hh_slot* __restrict__ vals, uint64_t cap, unsigned long long* __restrict__ counters) {
    __shared__ unsigned int s_new;
    if (threadIdx.x == 0) s_new = 0;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int my_new = 0, my_last = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_ent; e += stride) {
        const uint32_t* p = ent + e * 9;
        const uint64_t key = ((uint64_t)p[0] << 32) | (uint64_t)p[1];
        bool inserted;
        const uint64_t slot = hh_probe_insert(keys, cap, key, &inserted);
        if (slot >= cap) {
            atomicExch(counters + 2, 1ull);
            continue;
        }
        if (inserted) my_new++;
        hh_slot* v = vals + slot;
        atomicAdd(&v->full, p[2]);
        if (p[3]) atomicAdd(&v->flank, p[3]);
        atomicMin(&v->first_full, p[4]);
        atomicMin(&v->first_flank, p[5]);
        my_last = max(my_last, p[4]);
        if (p[6]) atomicAdd(&v->ht, p[6]);
        if (p[7]) atomicAdd(&v->th, p[7]);
        if (p[8]) atomicAdd(&v->tt, p[8]);
    }
    if (my_new) atomicAdd(&s_new, my_new);
    my_last = __reduce_max_sync(HH_FULL_MASK, my_last);
    if ((threadIdx.x & 31) == 0 && my_last) atomicMax(counters + 4, (unsigned long long)my_last);
    __syncthreads();
    if (threadIdx.x == 0 && s_new) atomicAdd(counters + 0, (unsigned long long)s_new);
}

__global__ void hh_k_add_u64(unsigned long long* __restrict__ dst, const int64_t* __restrict__ src, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += (unsigned long long)src[i];
}

// ---------------------------------------------------------------------------------------------
// multi-GPU routing: every contig pair has ONE owner rank, so the partition tables are disjoint and no
// counter is ever reduced across ranks
// ---------------------------------------------------------------------------------------------
#define HH_MAX_WORLD 64

__device__ __forceinline__ int hh_owner(int a, int b, int world) {
    const uint32_t lo = (uint32_t)min(a, b), hi = (uint32_t)max(a, b);
    return (int)(hh_mix64(((uint64_t)lo << 32) | (uint64_t)hi) % (uint64_t)world);
}

// destination of a record, -1 = can never be used (same contig in contig mode, ids outside the FASTA)
__device__ __forceinline__ int hh_route_dest(const int4 r, int n_src, bool contig_mode, int world) {
    if ((unsigned)r.x >= (unsigned)n_src || (unsigned)r.z >= (unsigned)n_src) return -1;
    if (contig_mode && r.x == r.z) return -1;
    return hh_owner(r.x, r.z, world);
}

__global__ void __launch_bounds__(256)
hh_k_route_count(const int4* __restrict__ rec, int64_t n_rec, int n_src, int contig_mode, int world,
                 unsigned long long* __restrict__ counts) {
    __shared__ unsigned int s_cnt[HH_MAX_WORLD];
    if (threadIdx.x < HH_MAX_WORLD) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += stride) {
        const int d = hh_route_dest(hh_ld_stream(rec + i), n_src, contig_mode != 0, world);
        if (d >= 0) atomicAdd(&s_cnt[d], 1u);
    }
    __syncthreads();
    if (threadIdx.x < world && s_cnt[threadIdx.x]) atomicAdd(counts + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

// scatter into the destination groups; cursor[d] starts at the group's base.  One tile of 256 records per trip:
// shared-memory ranks inside the tile, one global atomic per destination and tile.
__global__ void __launch_bounds__(256)
hh_k_route_scatter(const int4* __restrict__ rec, int64_t n_rec, uint32_t stream_off, int n_src, int contig_mode, int world,
                   unsigned long long* __restrict__ cursor, int4* __restrict__ rec_out, uint32_t* __restrict__ pos_out) {
    __shared__ unsigned int s_cnt[HH_MAX_WORLD];
    __shared__ unsigned long long s_base[HH_MAX_WORLD];
    const int64_t tiles = (n_rec + 255) / 256;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        if (threadIdx.x < HH_MAX_WORLD) s_cnt[threadIdx.x] = 0;
        __syncthreads();
        const int64_t i = t * 256 + threadIdx.x;
        int4 r = make_int4(-1, 0, -1, 0);
        int d = -1;
        unsigned int my = 0;
        if (i < n_rec) {
            r = hh_ld_stream(rec + i);
            d = hh_route_dest(r, n_src, contig_mode != 0, world);
            if (d >= 0) my = atomicAdd(&s_cnt[d], 1u);
        }
        __syncthreads();
        if (threadIdx.x < world && s_cnt[threadIdx.x])
            s_base[threadIdx.x] = atomicAdd(cursor + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
        __syncthreads();
        if (d >= 0) {
            const unsigned long long q = s_base[d] + my;
            rec_out[q] = r;
            pos_out[q] = stream_off + (uint32_t)i;
        }
        __syncthreads();
    }
}

// order[s] = s for live slots (unordered compaction of a partition table re-uses the compaction kernels)
__global__ void hh_k_links_mark_slots(const uint64_t* __restrict__ keys, uint64_t cap, uint32_t* __restrict__ order) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += stride)
        order[s] = (keys[s] == HH_EMPTY_KEY) ? HH_NONE32 : (uint32_t)s;
}

// adopted (unordered) entry list -> order[first_full] = entry index; and the flank count
__global__ void hh_k_list_scatter_order(const uint32_t* __restrict__ ent, int64_t nnz, uint32_t* __restrict__ order, int64_t stream_end,
                                        unsigned long long* __restrict__ counters) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        const uint32_t f = ent[e * 9 + 4];
        if ((int64_t)f < stream_end) order[f] = (uint32_t)e;
        else atomicExch(counters + 2, 2ull);
    }
}

__global__ void hh_k_list_count_flank(const uint32_t* __restrict__ ent, int64_t nnz, unsigned long long* __restrict__ counters) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int c = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) c += ent[e * 9 + 3] ? 1u : 0u;
    c = hh_warp_sum((int)c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(counters + 3, (unsigned long long)c);
}

// order[first_full] = slot
__global__ void hh_k_links_scatter_order(const uint64_t* __restrict__ keys, const hh_slot* __restrict__ vals, uint64_t cap,
                                         uint32_t* __restrict__ order, int64_t stream_end,
                                         unsigned long long* __restrict__ counters) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += stride) {
        if (keys[s] == HH_EMPTY_KEY) continue;
        const uint32_t f = vals[s].first_full;
        if ((int64_t)f < stream_end) order[f] = (uint32_t)s;
        else atomicExch(counters + 2, 2ull);
    }
}

#define HH_CMP_TILE 2048   // elements per block in the compaction kernels (256 threads x 8)

__global__ void __launch_bounds__(256)
hh_k_compact_count(const uint32_t* __restrict__ order, int64_t n, int* __restrict__ block_cnt) {
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * HH_CMP_TILE + (int64_t)threadIdx.x * 8;
    int c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int64_t e = base + k;
        if (e < n && order[e] != HH_NONE32) c++;
    }
    c = hh_warp_sum(c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) block_cnt[blockIdx.x] = s_cnt;
}

__global__ void __launch_bounds__(256)
hh_k_compact_gather(const uint32_t* __restrict__ order, int64_t n, const int64_t* __restrict__ block_off,
                    const uint64_t* __restrict__ keys, const hh_slot* __restrict__ vals,
                    uint32_t* __restrict__ compact, unsigned long long* __restrict__ counters) {
    __shared__ int s_warp[8];
    __shared__ unsigned int s_flank;
    if (threadIdx.x == 0) s_flank = 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * HH_CMP_TILE + (int64_t)threadIdx.x * 8;
    uint32_t slot[8];
    int c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int64_t e = base + k;
        slot[k] = (e < n) ? order[e] : HH_NONE32;
        if (slot[k] != HH_NONE32) c++;
    }
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(HH_FULL_MASK, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += s_warp[w];
    int64_t q = block_off[blockIdx.x] + woff + incl - c;
    unsigned int nfl = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (slot[k] == HH_NONE32) continue;
        if (keys == nullptr) {
            // source is an entry list (hh_links_adopt): plain copy of the 9 words
            const uint32_t* src = reinterpret_cast<const uint32_t*>(vals) + (size_t)slot[k] * 9;
            uint32_t* o = compact + q * 9;
#pragma unroll
            for (int w = 0; w < 9; ++w) o[w] = src[w];
            q++;
            continue;
        }
        const uint64_t key = keys[slot[k]];
        const uint4* v = reinterpret_cast<const uint4*>(vals + slot[k]);
        const uint4 v0 = v[0], v1 = v[1];   // {first_full, first_flank, full, flank} {ht, th, tt, pad}
        uint32_t* o = compact + q * 9;
        o[0] = (uint32_t)(key >> 32);
        o[1] = (uint32_t)key;
        o[2] = v0.z;
        o[3] = v0.w;
        o[4] = v0.x;
        o[5] = v0.y;
        o[6] = v1.x;
        o[7] = v1.y;
        o[8] = v1.z;
        if (v0.w) nfl++;
        q++;
    }
    if (nfl) atomicAdd(&s_flank, nfl);
    __syncthreads();
    if (threadIdx.x == 0 && s_flank) atomicAdd(counters + 3, (unsigned long long)s_flank);
}

// ---------------------------------------------------------------------------------------------
// dict_to_matrix index assignment (327-349): first touch of each fragment in flank-dict order
// ---------------------------------------------------------------------------------------------
__global__ void hh_k_touch(const uint32_t* __restrict__ compact, int64_t nnz, const uint8_t* __restrict__ keep,
                           unsigned long long* __restrict__ touch) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        const uint32_t* p = compact + e * 9;
        if (p[3] == 0) continue;                       // not in flank_link_dict
        const uint32_t i = p[0], j = p[1];
        if (!keep[i] || !keep[j]) continue;            // 329-330
        const unsigned long long t = (unsigned long long)p[5] * 2ull;
        atomicMin(touch + i, t);
        atomicMin(touch + j, t + 1ull);
    }
}

// index[c] = number of touched fragments touched earlier than c (touch values are unique): the position of c in a sort of
// the (touch, fragment) pairs.  Untouched fragments (touch ~0) sort after every touched one.  A stable LSD radix sort,
// 8-bit digits, tiles of 1024 pairs (one per thread): touch < 2^33, so five passes over bits 0..39 order it.
#define HH_RADIX_TILE 1024
#define HH_RADIX_PASSES 5

__global__ void __launch_bounds__(HH_RADIX_TILE)
hh_k_rank_init(const unsigned long long* __restrict__ touch, int n, unsigned long long* __restrict__ key, int32_t* __restrict__ val,
               int* __restrict__ n_linked) {
    const int c = blockIdx.x * HH_RADIX_TILE + threadIdx.x;
    int touched = 0;
    if (c < n) {
        key[c] = touch[c];
        val[c] = c;
        touched = touch[c] != ~0ull;
    }
    touched = hh_warp_sum(touched);
    if ((threadIdx.x & 31) == 0 && touched) atomicAdd(n_linked, touched);
}

// cnt[digit * n_tiles + tile] = pairs of the tile with that digit
__global__ void __launch_bounds__(HH_RADIX_TILE)
hh_k_radix_hist(const unsigned long long* __restrict__ key, int n, int shift, int* __restrict__ cnt) {
    __shared__ int s_h[256];
    if (threadIdx.x < 256) s_h[threadIdx.x] = 0;
    __syncthreads();
    const int i = blockIdx.x * HH_RADIX_TILE + threadIdx.x;
    if (i < n) atomicAdd(&s_h[(key[i] >> shift) & 255u], 1);
    __syncthreads();
    if (threadIdx.x < 256) cnt[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = s_h[threadIdx.x];
}

// stable scatter: off = exclusive scan of cnt; inside the tile, the rank among equal digits of the lower warps and lanes
__global__ void __launch_bounds__(HH_RADIX_TILE)
hh_k_radix_scatter(const unsigned long long* __restrict__ key, const int32_t* __restrict__ val, int n, int shift,
                   const int64_t* __restrict__ off, unsigned long long* __restrict__ key_out, int32_t* __restrict__ val_out) {
    __shared__ int s_w[32][256];               // digit counts of every warp, then their exclusive prefix over the warps
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = threadIdx.x; k < 32 * 256; k += HH_RADIX_TILE) s_w[k >> 8][k & 255] = 0;
    __syncthreads();
    const int i = blockIdx.x * HH_RADIX_TILE + threadIdx.x;
    const bool ok = i < n;
    const unsigned long long k = ok ? key[i] : 0ull;
    const int d = ok ? (int)((k >> shift) & 255u) : -1;
    const unsigned peers = __match_any_sync(HH_FULL_MASK, d);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (ok && rank == 0) s_w[warp][d] = __popc(peers);
    __syncthreads();
    if (threadIdx.x < 256) {
        int run = 0;
        for (int w = 0; w < 32; ++w) {
            const int t = s_w[w][threadIdx.x];
            s_w[w][threadIdx.x] = run;
            run += t;
        }
    }
    __syncthreads();
    if (ok) {
        const int64_t q = off[(size_t)d * gridDim.x + blockIdx.x] + s_w[warp][d] + rank;
        key_out[q] = k;
        val_out[q] = val[i];
    }
}

__global__ void hh_k_rank_index(const int32_t* __restrict__ val, int n, const int* __restrict__ n_linked, int32_t* __restrict__ index) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) index[val[r]] = (r < *n_linked) ? r : -1;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static inline int hh_grid(hh_ctx* ctx, int per_sm) { return ctx->sm_count * per_sm; }

static int links_alloc_table(hh_links* lk, uint64_t cap, uint64_t** keys, hh_slot** vals) {
    HH_CHECK(hh_dmalloc(keys, cap));
    int rc = hh_dmalloc(vals, cap);
    if (rc != HH_OK) {
        hh_dfree(*keys);
        return rc;
    }
    HH_LAUNCH(lk->ctx, hh_k_links_init, hh_grid(lk->ctx, 8), 256, 0, *keys, *vals, cap);
    return HH_OK;
}

static int links_read_counters(hh_links* lk, unsigned long long out[8]) {
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaMemcpyAsync(ctx->h_scratch, lk->d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 8; ++k) out[k] = ctx->h_scratch[k];
    return HH_OK;
}

// the big hash table of the direct path is allocated on first use (the partitioned path never needs it)
static int links_need_table(hh_links* lk) {
    if (lk->d_keys) return HH_OK;
    uint64_t cap = 1ull << 16;
    const double want = lk->capacity_hint > 0 ? (double)lk->capacity_hint / 0.5 : 0.0;
    while ((double)cap < want) cap <<= 1;
    HH_CHECK(links_alloc_table(lk, cap, &lk->d_keys, &lk->d_vals));
    lk->cap = cap;
    return HH_OK;
}

// make sure `incoming` more distinct keys fit under a 0.7 load factor
static int links_ensure_capacity(hh_links* lk, int64_t incoming) {
    const double max_load = 0.7;
    HH_CHECK(links_need_table(lk));
    if ((double)(lk->known_unique + lk->since_known + incoming) <= max_load * (double)lk->cap) return HH_OK;
    unsigned long long c[8];
    HH_CHECK(links_read_counters(lk, c));
    HH_REQUIRE(c[2] == 0, HH_ERR_CAPACITY, "hh_links: hash table overflow (capacity %llu slots)", (unsigned long long)lk->cap);
    lk->known_unique = (int64_t)c[0];
    lk->since_known = 0;
    if ((double)(lk->known_unique + incoming) <= max_load * (double)lk->cap) return HH_OK;
    uint64_t ncap = lk->cap;
    while ((double)(lk->known_unique + incoming) > max_load * (double)ncap) ncap <<= 1;
    uint64_t* nkeys;
    hh_slot* nvals;
    HH_CHECK(links_alloc_table(lk, ncap, &nkeys, &nvals));
    HH_LAUNCH(lk->ctx, hh_k_links_rehash, hh_grid(lk->ctx, 8), 256, 0, lk->d_keys, lk->d_vals, lk->cap, nkeys, nvals, ncap,
              lk->d_counters);
    HH_CUDA(cudaStreamSynchronize(lk->ctx->stream));
    hh_dfree(lk->d_keys);
    hh_dfree(lk->d_vals);
    lk->d_keys = nkeys;
    lk->d_vals = nvals;
    lk->cap = ncap;
    return HH_OK;
}

static int links_create_common(hh_ctx* ctx, int32_t n_key, const int64_t* key_len, const int32_t* key_rank, const uint8_t* in_nx,
                               int64_t flank_bp, int64_t capacity_hint, int32_t n_src, const int32_t* src_rank,
                               const int32_t* frag_base, int64_t bin_size, hh_links** out) {
    *out = nullptr;
    std::vector<int32_t> len32(n_key);
    for (int32_t c = 0; c < n_key; ++c) {
        HH_REQUIRE(key_len[c] > 0 && key_len[c] <= 0x7fffffffLL, HH_ERR_UNSUPPORTED,
                   "hh_links_create: object %d has length %lld; records carry int32 positions (pos_int_type int32, "
                   "HapHiC_cluster.py:116-147)", c, (long long)key_len[c]);
        HH_REQUIRE(key_rank[c] >= 0 && key_rank[c] < n_key, HH_ERR_ARG, "hh_links_create: name_rank[%d] out of range", c);
        len32[c] = (int32_t)key_len[c];
    }
    hh_links* lk = new (std::nothrow) hh_links();
    HH_REQUIRE(lk != nullptr, HH_ERR_NOMEM, "hh_links_create: out of host memory");
    memset(lk, 0, sizeof(*lk));
    lk->ctx = ctx;
    lk->n_ctg = n_key;
    lk->n_src = frag_base ? n_src : n_key;
    lk->bin_size = bin_size;
    lk->flank_bp = flank_bp;
    int rc = HH_OK;
    do {
        if ((rc = hh_dmalloc(&lk->d_len, n_key)) != HH_OK) break;
        if ((rc = hh_dmalloc(&lk->d_rank, n_key)) != HH_OK) break;
        if ((rc = hh_dmalloc(&lk->d_nx, n_key)) != HH_OK) break;
        if ((rc = hh_dmalloc(&lk->d_ctg, n_key)) != HH_OK) break;
        if ((rc = hh_dmalloc(&lk->d_counters, 8)) != HH_OK) break;
        if ((rc = hh_dmalloc(&lk->d_index, n_key)) != HH_OK) break;
        if ((rc = hh_dmalloc(&lk->d_keep, n_key)) != HH_OK) break;
        if (frag_base) {
            if ((rc = hh_dmalloc(&lk->d_src_rank, n_src)) != HH_OK) break;
            if ((rc = hh_dmalloc(&lk->d_fbase, (size_t)n_src + 1)) != HH_OK) break;
        }
    } while (0);
    if (rc != HH_OK) {
        hh_links_destroy(lk);
        return rc;
    }
    cudaStream_t st = ctx->stream;
    HH_CUDA(cudaMemcpyAsync(lk->d_len, len32.data(), n_key * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    HH_CUDA(cudaMemcpyAsync(lk->d_rank, key_rank, n_key * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    HH_CUDA(cudaMemcpyAsync(lk->d_nx, in_nx, n_key * sizeof(uint8_t), cudaMemcpyHostToDevice, st));
    HH_CUDA(cudaMemsetAsync(lk->d_ctg, 0, n_key * sizeof(unsigned long long), st));
    HH_CUDA(cudaMemsetAsync(lk->d_counters, 0, 8 * sizeof(unsigned long long), st));
    if (frag_base) {
        HH_CUDA(cudaMemcpyAsync(lk->d_src_rank, src_rank, (size_t)n_src * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        HH_CUDA(cudaMemcpyAsync(lk->d_fbase, frag_base, ((size_t)n_src + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    }
    HH_CUDA(cudaStreamSynchronize(st));   // host temporaries go out of scope
    lk->capacity_hint = capacity_hint;
    lk->psets = new std::vector<hh_partset>();
    lk->index_keep = new std::vector<uint8_t>();
    HH_CUDA(cudaStreamCreateWithFlags(&lk->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
        HH_CUDA(cudaEventCreateWithFlags(&lk->ev_copied[k], cudaEventDisableTiming));
        HH_CUDA(cudaEventCreateWithFlags(&lk->ev_consumed[k], cudaEventDisableTiming));
    }
    *out = lk;
    return HH_OK;
}

extern "C" int hh_links_create(hh_ctx* ctx, int32_t n_ctg, const int64_t* ctg_len, const int32_t* name_rank,
                               const uint8_t* in_nx, int64_t flank_bp, int64_t capacity_hint, hh_links** out) {
    HH_REQUIRE(ctx && out && ctg_len && name_rank && in_nx, HH_ERR_ARG, "hh_links_create: NULL argument");
    HH_REQUIRE(n_ctg > 0, HH_ERR_ARG, "hh_links_create: n_ctg must be positive");
    HH_REQUIRE(flank_bp >= 0, HH_ERR_ARG, "hh_links_create: flank_bp must be >= 0");
    hh_scope _scope(ctx);
    return links_create_common(ctx, n_ctg, ctg_len, name_rank, in_nx, flank_bp, capacity_hint, n_ctg, nullptr, nullptr, 0, out);
}

extern "C" int hh_links_create_frags(hh_ctx* ctx, int32_t n_ctg, const int32_t* ctg_rank, const int32_t* frag_base,
                                     int32_t n_frag, const int64_t* frag_len, const int32_t* frag_rank, const uint8_t* frag_in_nx,
                                     int64_t bin_size, int64_t flank_bp, int64_t capacity_hint, hh_links** out) {
    HH_REQUIRE(ctx && out && ctg_rank && frag_base && frag_len && frag_rank && frag_in_nx, HH_ERR_ARG,
               "hh_links_create_frags: NULL argument");
    HH_REQUIRE(n_ctg > 0 && n_frag >= n_ctg, HH_ERR_ARG, "hh_links_create_frags: need n_frag >= n_ctg > 0");
    HH_REQUIRE(flank_bp >= 0 && bin_size > 0, HH_ERR_ARG, "hh_links_create_frags: flank_bp >= 0 and bin_size > 0 required");
    HH_REQUIRE(frag_base[0] == 0 && frag_base[n_ctg] == n_frag, HH_ERR_ARG, "hh_links_create_frags: frag_base must span [0, n_frag]");
    for (int32_t c = 0; c < n_ctg; ++c) {
        HH_REQUIRE(frag_base[c + 1] > frag_base[c], HH_ERR_ARG, "hh_links_create_frags: contig %d has no fragment", c);
        HH_REQUIRE(ctg_rank[c] >= 0 && ctg_rank[c] < n_ctg, HH_ERR_ARG, "hh_links_create_frags: ctg_rank[%d] out of range", c);
    }
    hh_scope _scope(ctx);
    return links_create_common(ctx, n_frag, frag_len, frag_rank, frag_in_nx, flank_bp, capacity_hint, n_ctg, ctg_rank, frag_base,
                               bin_size, out);
}

static int links_env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// a new set of partition regions sized for `n_rec` more records
static int links_new_partset(hh_links* lk, int64_t n_rec) {
    const int npart = 1 << lk->npart_log;
    hh_partset ps;
    memset(&ps, 0, sizeof(ps));
    ps.pcap = (uint64_t)((double)n_rec / npart * 1.5) + 4096;
    ps.sized_for = n_rec;
    HH_CHECK(hh_ws_alloc(lk->ctx, &ps.buf, (size_t)npart * (size_t)ps.pcap));
    int rc = hh_dmalloc(&ps.cursor, (size_t)npart);
    if (rc != HH_OK) {
        hh_ws_free(lk->ctx, ps.buf);
        return rc;
    }
    HH_CUDA(cudaMemsetAsync(ps.cursor, 0, (size_t)npart * sizeof(unsigned long long), lk->ctx->stream));
    lk->psets->push_back(ps);
    return HH_OK;
}

// first records of the stream: direct hash table or partition-then-aggregate.  `total` = records the caller is about to
// stream in this call (the sizing of the partition regions)
static int links_choose_mode(hh_links* lk, int64_t total) {
    if (lk->mode) return HH_OK;
    const int want = links_env_int("HH_LINKS_PARTITION", -1);          // 0 = never, 1 = always (contig mode), -1 = by size
    const bool can = lk->d_fbase == nullptr && lk->d_keys == nullptr;
    const bool big = total >= (16ll << 20) && lk->n_ctg >= 2048;
    if (!can || want == 0 || (want < 0 && !big)) {
        lk->mode = 1;
        return HH_OK;
    }
    lk->mode = 2;
    int lg = 4;
    while (lg < 9 && ((int64_t)400000 << lg) < total) lg++;            // ~400k records per partition, at most 512 partitions
    lk->npart_log = links_env_int("HH_LINKS_NPART_LOG", lg);
    if (lk->npart_log < 1) lk->npart_log = 1;
    if (lk->npart_log > 10) lk->npart_log = 10;
    HH_CHECK(links_new_partset(lk, total));
    lk->spill_cap = (uint64_t)(total / 8) + (4u << 20);
    HH_CHECK(hh_ws_alloc(lk->ctx, &lk->d_spill, (size_t)lk->spill_cap));
    HH_CHECK(hh_dmalloc(&lk->d_spill_cursor, 1));
    HH_CUDA(cudaMemsetAsync(lk->d_spill_cursor, 0, sizeof(unsigned long long), lk->ctx->stream));
    return HH_OK;
}

static int links_launch_insert(hh_links* lk, const int4* d_rec, int64_t n_rec, int64_t stream_offset,
                               const uint32_t* d_pos = nullptr) {
    hh_ctx* ctx = lk->ctx;
    if (lk->mode == 2 && d_pos == nullptr) {
        // one wave of resident CTAs, each taking tiles in a grid stride
        const int64_t tiles = (n_rec + HH_PART_TILE - 1) / HH_PART_TILE;
        int per_sm = 0;
        HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hh_k_part_scatter, 512, 0));
        const int grid = (int)std::max<int64_t>(1, std::min(tiles, (int64_t)hh_grid(ctx, std::max(per_sm, 1))));
        const hh_partset& ps = lk->psets->back();
        HH_LAUNCH(ctx, hh_k_part_scatter, grid, 512, 0, d_rec, n_rec, (uint32_t)stream_offset, lk->n_ctg, lk->d_len, lk->d_rank, lk->d_nx,
                  lk->flank_bp, lk->npart_log, ps.buf, ps.pcap, ps.cursor, lk->d_spill, lk->spill_cap, lk->d_spill_cursor,
                  lk->d_counters);
        return HH_OK;
    }
    HH_CHECK(links_need_table(lk));
    int64_t blocks = (n_rec + 255) / 256;
    int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
    if (grid < 1) grid = 1;
    HH_LAUNCH(ctx, hh_k_links_insert, grid, 256, 0, d_rec, n_rec, (uint32_t)stream_offset, lk->n_ctg, lk->d_len, lk->d_rank,
              lk->d_nx, lk->flank_bp, lk->d_keys, lk->d_vals, lk->cap, lk->d_ctg, lk->d_counters, lk->d_src_rank, lk->d_fbase,
              lk->bin_size, lk->n_src, d_pos);
    return HH_OK;
}

// partitioned mode: a call that would outgrow the current set (sized for the first call) gets a set of its own
static int links_part_room(hh_links* lk, int64_t n_rec) {
    hh_partset& ps = lk->psets->back();
    if (ps.sent > 0 && ps.sent + n_rec > ps.sized_for + ps.sized_for / 8) {
        HH_CHECK(links_new_partset(lk, n_rec));
        lk->psets->back().sent = n_rec;
        return HH_OK;
    }
    ps.sent += n_rec;
    return HH_OK;
}

extern "C" int hh_links_add_async(hh_links* lk, const int32_t* rec_dev, int64_t n_rec, int64_t stream_offset) {
    HH_REQUIRE(lk && (rec_dev || n_rec == 0), HH_ERR_ARG, "hh_links_add_async: NULL argument");
    hh_scope _scope(lk->ctx);
    HH_REQUIRE(!lk->finished, HH_ERR_STATE, "hh_links_add_async: stream already finished");
    HH_REQUIRE(n_rec >= 0 && stream_offset >= 0 && stream_offset + n_rec <= 0xFFFFFFFELL, HH_ERR_UNSUPPORTED,
               "hh_links_add: stream indices must fit 32 bits (offset %lld + %lld records)", (long long)stream_offset,
               (long long)n_rec);
    HH_REQUIRE(((uintptr_t)rec_dev & 15) == 0, HH_ERR_ARG, "hh_links_add: records must be 16-byte aligned");
    if (n_rec == 0) return HH_OK;
    HH_CUDA(cudaSetDevice(lk->ctx->device));
    HH_CHECK(links_choose_mode(lk, n_rec));
    if (lk->mode == 2) HH_CHECK(links_part_room(lk, n_rec));
    HH_CHECK(links_launch_insert(lk, reinterpret_cast<const int4*>(rec_dev), n_rec, stream_offset));
    lk->n_records += n_rec;
    lk->since_known += n_rec;
    if (stream_offset + n_rec > lk->stream_end) lk->stream_end = stream_offset + n_rec;
    return HH_OK;
}

extern "C" int hh_links_add(hh_links* lk, const int32_t* rec, int64_t n_rec, int64_t stream_offset, int mem) {
    HH_REQUIRE(lk && (rec || n_rec == 0), HH_ERR_ARG, "hh_links_add: NULL argument");
    hh_scope _scope(lk->ctx);
    HH_REQUIRE(!lk->finished, HH_ERR_STATE, "hh_links_add: stream already finished");
    HH_REQUIRE(mem == HH_MEM_HOST || mem == HH_MEM_DEVICE, HH_ERR_ARG, "hh_links_add: bad mem flag %d", mem);
    HH_REQUIRE(n_rec >= 0 && stream_offset >= 0 && stream_offset + n_rec <= 0xFFFFFFFELL, HH_ERR_UNSUPPORTED,
               "hh_links_add: stream indices must fit 32 bits (offset %lld + %lld records)", (long long)stream_offset,
               (long long)n_rec);
    if (n_rec == 0) return HH_OK;
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    const int64_t CH = 1ll << 23;   // 8 Mi records = 128 MiB per chunk
    HH_CHECK(links_choose_mode(lk, n_rec));
    if (lk->mode == 2) HH_CHECK(links_part_room(lk, n_rec));
    if (mem == HH_MEM_DEVICE) {
        HH_REQUIRE(((uintptr_t)rec & 15) == 0, HH_ERR_ARG, "hh_links_add: records must be 16-byte aligned");
        for (int64_t off = 0; off < n_rec; off += CH) {
            const int64_t m = (n_rec - off < CH) ? (n_rec - off) : CH;
            if (lk->mode != 2) HH_CHECK(links_ensure_capacity(lk, m));
            HH_CHECK(links_launch_insert(lk, reinterpret_cast<const int4*>(rec) + off, m, stream_offset + off));
            lk->since_known += m;
        }
    } else {
        if (!lk->d_stage[0]) {
            lk->stage_records = CH;
            HH_CUDA(cudaMalloc((void**)&lk->d_stage[0], (size_t)CH * sizeof(int4)));   // plain cudaMalloc: also used by copy_stream
            HH_CUDA(cudaMalloc((void**)&lk->d_stage[1], (size_t)CH * sizeof(int4)));
        }
        int buf = 0;
        for (int64_t off = 0; off < n_rec; off += CH, buf ^= 1) {
            const int64_t m = (n_rec - off < CH) ? (n_rec - off) : CH;
            // the copy engine may not overwrite a staging buffer the insert kernel still reads
            HH_CUDA(cudaStreamWaitEvent(lk->copy_stream, lk->ev_consumed[buf], 0));
            HH_CUDA(cudaMemcpyAsync(lk->d_stage[buf], rec + off * 4, (size_t)m * 16, cudaMemcpyHostToDevice, lk->copy_stream));
            HH_CUDA(cudaEventRecord(lk->ev_copied[buf], lk->copy_stream));
            if (lk->mode != 2) HH_CHECK(links_ensure_capacity(lk, m));
            HH_CUDA(cudaStreamWaitEvent(ctx->stream, lk->ev_copied[buf], 0));
            HH_CHECK(links_launch_insert(lk, lk->d_stage[buf], m, stream_offset + off));
            HH_CUDA(cudaEventRecord(lk->ev_consumed[buf], ctx->stream));
            lk->since_known += m;
        }
        HH_CUDA(cudaStreamSynchronize(ctx->stream));   // the caller may reuse `rec` on return
    }
    lk->n_records += n_rec;
    if (stream_offset + n_rec > lk->stream_end) lk->stream_end = stream_offset + n_rec;
    return HH_OK;
}

// partitioned counting, second phase: level-2 split, shared-memory count + emit, and the scratch-table fallback
static void links_free_partsets(hh_links* lk) {
    if (lk->psets) {
        for (size_t k = 0; k < lk->psets->size(); ++k) {
            hh_ws_free(lk->ctx, (*lk->psets)[k].buf);
            hh_dfree((*lk->psets)[k].cursor);
        }
        lk->psets->clear();
    }
    hh_ws_free(lk->ctx, lk->d_spill);
    hh_dfree(lk->d_spill_cursor);
}

static int links_finish_partitioned(hh_links* lk) {
    hh_ctx* ctx = lk->ctx;
    const int npart = 1 << lk->npart_log;
    const size_t nsets = lk->psets->size();
    // one read-back: the counters, the level-1 region fill levels and the spill count
    std::vector<unsigned long long> fill(nsets * (size_t)npart);
    unsigned long long n_spill = 0;
    HH_CUDA(cudaMemcpyAsync(ctx->h_scratch, lk->d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    for (size_t k = 0; k < nsets; ++k)
        HH_CUDA(cudaMemcpyAsync(fill.data() + k * (size_t)npart, (*lk->psets)[k].cursor, (size_t)npart * sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, ctx->stream));
    HH_CUDA(cudaMemcpyAsync(&n_spill, lk->d_spill_cursor, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    unsigned long long c[8];
    for (int k = 0; k < 8; ++k) c[k] = ctx->h_scratch[k];
    HH_REQUIRE(c[2] == 0, HH_ERR_CAPACITY,
               "hh_links_finish: the spill list of the partitioned counting overflowed (a few contig pairs own most of the stream): "
               "set HH_LINKS_PARTITION=0 to use the direct hash table");
    lk->n_used = lk->peer_used + (int64_t)c[1];
    // partition totals (a cursor counts every record of its partition, the spilled ones included), their exclusive prefix
    // (where each partition starts in the level-2 buffer), and the level-2 fan-out: the fullest partition split into
    // sub-partitions of at most HH_SUB_SLOTS / 2 records, so that even all-distinct keys fill the shared table at most half
    std::vector<int64_t> pbase((size_t)npart + 1, 0);
    int64_t worst = 1, region = (int64_t)n_spill;
    for (int p = 0; p < npart; ++p) {
        int64_t t = 0;
        for (size_t k = 0; k < nsets; ++k) {
            const unsigned long long f = fill[k * (size_t)npart + p];
            t += (int64_t)f;
            region = std::max(region, (int64_t)std::min(f, (unsigned long long)(*lk->psets)[k].pcap));
        }
        pbase[p + 1] = pbase[p] + t;
        worst = std::max(worst, t);
    }
    const int sub_max = std::min(HH_SUB_MAX_LOG, std::max(0, links_env_int("HH_LINKS_SUB_LOG_MAX", HH_SUB_MAX_LOG)));
    int sub_log = 0;
    while (sub_log < sub_max && (worst >> sub_log) > HH_SUB_SLOTS / 2) sub_log++;
    const int nsub = npart << sub_log;
    const int64_t total = pbase[npart];
    const uint64_t compact_cap = (uint64_t)(lk->n_used > 0 ? lk->n_used : 1);       // distinct pairs <= usable records
    hh_dfree(lk->d_compact);
    int4* d_rec2 = nullptr;                       // level-2 buffer: sub-partition id after sub-partition id
    uint32_t* d_stage_compact = nullptr;          // workspace; the exact-size list is cut from it
    unsigned int* d_cnt = nullptr;
    int64_t* d_off = nullptr;
    int64_t* d_pbase = nullptr;
    uint32_t* d_fb = nullptr;
    uint64_t* skeys[2] = {nullptr, nullptr};
    hh_slot* svals[2] = {nullptr, nullptr};
    int rc = [&]() -> int {
        HH_CHECK(hh_ws_alloc(ctx, &d_rec2, (size_t)(total > 0 ? total : 1)));
        HH_CHECK(hh_ws_alloc(ctx, &d_stage_compact, (size_t)compact_cap * 9));
        HH_CHECK(hh_dmalloc(&d_cnt, (size_t)nsub));
        HH_CHECK(hh_dmalloc(&d_off, (size_t)nsub + 1));
        HH_CHECK(hh_dmalloc(&d_pbase, (size_t)npart + 1));
        HH_CHECK(hh_dmalloc(&d_fb, (size_t)nsub));
        HH_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)nsub * sizeof(unsigned int), ctx->stream));
        HH_CUDA(cudaMemcpyAsync(d_pbase, pbase.data(), ((size_t)npart + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
        HH_CUDA(cudaMemsetAsync(lk->d_counters + 0, 0, sizeof(unsigned long long), ctx->stream));     // entry cursor
        HH_CUDA(cudaMemsetAsync(lk->d_counters + 3, 0, sizeof(unsigned long long), ctx->stream));     // nnz_flank
        HH_CUDA(cudaMemsetAsync(lk->d_counters + 7, 0, sizeof(unsigned long long), ctx->stream));     // fallback sub-partitions
        // level 2: histogram, offsets, scatter (the spill list goes with the first set)
        const int gx = (int)std::min<int64_t>(64, (region + HH_PART_TILE - 1) / HH_PART_TILE + 1);
        for (int pass = 0; pass < 2; ++pass) {
            if (pass == 1) HH_LAUNCH(ctx, hh_k_sub_offsets, npart, 1024, 0, d_cnt, sub_log, d_pbase, npart, d_off);
            for (size_t k = 0; k < nsets; ++k) {
                const hh_partset& ps = (*lk->psets)[k];
                const dim3 grid(gx, npart + (k == 0 ? 1 : 0));
                if (pass == 0)
                    HH_LAUNCH(ctx, hh_k_sub_split<false>, grid, 512, 0, ps.buf, ps.pcap, ps.cursor, lk->npart_log, lk->d_spill,
                              lk->d_spill_cursor, lk->spill_cap, sub_log, d_cnt, (const int64_t*)nullptr, (int4*)nullptr);
                else
                    HH_LAUNCH(ctx, hh_k_sub_split<true>, grid, 512, 0, ps.buf, ps.pcap, ps.cursor, lk->npart_log, lk->d_spill,
                              lk->d_spill_cursor, lk->spill_cap, sub_log, d_cnt, d_off, d_rec2);
            }
        }
        // count + emit in shared memory
        HH_CUDA(cudaFuncSetAttribute(hh_k_sub_count, cudaFuncAttributeMaxDynamicSharedMemorySize, HH_SUB_SMEM));
        int per_sm = 0;
        HH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hh_k_sub_count, 256, HH_SUB_SMEM));
        const int grid = (int)std::min<int64_t>(nsub, (int64_t)ctx->sm_count * std::max(per_sm, 1));
        HH_LAUNCH(ctx, hh_k_sub_count, grid, 256, HH_SUB_SMEM, d_rec2, d_off, nsub, d_stage_compact, compact_cap, lk->d_ctg,
                  lk->d_counters, d_fb);
        HH_CHECK(links_read_counters(lk, c));
        lk->scap = HH_SUB_SLOTS;
        if (c[7] && c[2] == 0) {
            // sub-partitions whose keys did not fit the shared table, one after the other through a global scratch table
            // (two tables, so the emit of one and the count of the next share a launch)
            const size_t nfb = (size_t)c[7];
            std::vector<uint32_t> fb(nfb);
            std::vector<int64_t> off((size_t)nsub + 1);
            HH_CUDA(cudaMemcpyAsync(fb.data(), d_fb, nfb * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            HH_CUDA(cudaMemcpyAsync(off.data(), d_off, ((size_t)nsub + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            HH_CUDA(cudaStreamSynchronize(ctx->stream));
            int64_t big = 1;
            for (size_t f = 0; f < nfb; ++f) big = std::max(big, off[fb[f] + 1] - off[fb[f]]);
            uint64_t scap = 1ull << 12;
            while ((double)scap * 0.6 < (double)big) scap <<= 1;          // load factor <= 0.6 even for all-distinct keys
            lk->scap = scap;
            for (int b = 0; b < 2; ++b) HH_CHECK(links_alloc_table(lk, scap, &skeys[b], &svals[b]));
            const int grid2 = hh_grid(ctx, 8);
            for (size_t f = 0; f <= nfb; ++f) {
                const int cb = (int)(f & 1), eb = cb ^ 1;
                const bool cur = f < nfb;
                const int64_t b0 = cur ? off[fb[f]] : 0, n = cur ? off[fb[f] + 1] - b0 : 0;
                HH_LAUNCH(ctx, hh_k_part_step, grid2, 256, 0, cur ? d_rec2 + b0 : nullptr, n, cur ? skeys[cb] : nullptr,
                          cur ? svals[cb] : nullptr, f > 0 ? skeys[eb] : nullptr, f > 0 ? svals[eb] : nullptr, scap, d_stage_compact,
                          compact_cap, lk->d_ctg, lk->d_counters);
            }
            HH_CHECK(links_read_counters(lk, c));
        }
        HH_REQUIRE(c[2] == 0, HH_ERR_CAPACITY,
                   "hh_links_finish: a table of the partitioned counting overflowed (code %llu): set HH_LINKS_PARTITION=0", c[2]);
        lk->nnz = (int64_t)c[0];
        lk->nnz_flank = (int64_t)c[3];
        HH_CHECK(hh_dmalloc(&lk->d_compact, (size_t)(lk->nnz > 0 ? lk->nnz : 1) * 9));
        if (lk->nnz)
            HH_CUDA(cudaMemcpyAsync(lk->d_compact, d_stage_compact, (size_t)lk->nnz * 9 * sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                                    ctx->stream));
        return HH_OK;
    }();
    hh_ws_free(ctx, d_rec2);
    hh_ws_free(ctx, d_stage_compact);
    hh_dfree(d_cnt);
    hh_dfree(d_off);
    hh_dfree(d_pbase);
    hh_dfree(d_fb);
    for (int b = 0; b < 2; ++b) {
        hh_dfree(skeys[b]);
        hh_dfree(svals[b]);
    }
    links_free_partsets(lk);
    HH_CHECK(rc);
    lk->finished = true;
    lk->ordered = false;        // dict insertion order is restored by the first hh_links_fetch (links_order_list)
    lk->index_valid = false;
    return HH_OK;
}

extern "C" int hh_links_finish(hh_links* lk, hh_links_info* info) {
    HH_REQUIRE(lk != nullptr, HH_ERR_ARG, "hh_links_finish: NULL handle");
    hh_scope _scope(lk->ctx);
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    if (!lk->finished && lk->mode == 2) HH_CHECK(links_finish_partitioned(lk));
    if (!lk->finished) {
        HH_CHECK(links_need_table(lk));
        unsigned long long c[8];
        HH_CHECK(links_read_counters(lk, c));
        HH_REQUIRE(c[2] == 0, HH_ERR_CAPACITY,
                   "hh_links_finish: hash table overflow (capacity %llu slots): pass a larger capacity_hint or use hh_links_add",
                   (unsigned long long)lk->cap);
        HH_REQUIRE(c[5] == 0, HH_ERR_ARG,
                   "hh_links_finish: %llu records have a position outside their contig's bins (e.g. record %llu of the stream): "
                   "positions must lie in [0, contig length)", c[5], c[6] - 1ull);
        lk->nnz = (int64_t)c[0];
        lk->n_used = lk->peer_used + (int64_t)c[1];
        HH_CUDA(cudaMemsetAsync(lk->d_counters + 3, 0, sizeof(unsigned long long), ctx->stream));
        if (lk->nnz > 0 && (int64_t)c[4] + 1 > lk->stream_end) lk->stream_end = (int64_t)c[4] + 1;   // merged peers
        const int64_t S = lk->stream_end;
        hh_dfree(lk->d_compact);
        HH_CHECK(hh_dmalloc(&lk->d_compact, (size_t)(lk->nnz > 0 ? lk->nnz : 1) * 9));
        if (lk->nnz > 0) {
            uint32_t* d_order = nullptr;
            int* d_bcnt = nullptr;
            int64_t* d_boff = nullptr;
            const int64_t nb = (S + HH_CMP_TILE - 1) / HH_CMP_TILE;
            int rc = HH_OK;
            do {
                if ((rc = hh_dmalloc(&d_order, (size_t)S)) != HH_OK) break;
                if ((rc = hh_dmalloc(&d_bcnt, (size_t)nb)) != HH_OK) break;
                if ((rc = hh_dmalloc(&d_boff, (size_t)nb + 1)) != HH_OK) break;
            } while (0);
            if (rc == HH_OK) {
                rc = [&]() -> int {
                    HH_CUDA(cudaMemsetAsync(d_order, 0xFF, (size_t)S * sizeof(uint32_t), ctx->stream));
                    HH_LAUNCH(ctx, hh_k_links_scatter_order, hh_grid(ctx, 8), 256, 0, lk->d_keys, lk->d_vals, lk->cap, d_order, S,
                              lk->d_counters);
                    HH_LAUNCH(ctx, hh_k_compact_count, (unsigned)nb, 256, 0, d_order, S, d_bcnt);
                    HH_CHECK(hh_exclusive_scan_i32(ctx, d_bcnt, d_boff, (int)nb));
                    HH_LAUNCH(ctx, hh_k_compact_gather, (unsigned)nb, 256, 0, d_order, S, d_boff, lk->d_keys, lk->d_vals,
                              lk->d_compact, lk->d_counters);
                    HH_CHECK(links_read_counters(lk, c));
                    return HH_OK;
                }();
            }
            hh_dfree(d_order);
            hh_dfree(d_bcnt);
            hh_dfree(d_boff);
            HH_CHECK(rc);
            HH_REQUIRE(c[2] == 0, HH_ERR_STATE, "hh_links_finish: first-seen index beyond the stream end (stream_offset misuse)");
            lk->nnz_flank = (int64_t)c[3];
        }
        lk->finished = true;
        lk->ordered = true;
        lk->index_valid = false;
    }
    if (info) {
        info->n_records = lk->n_records;
        info->n_used = lk->n_used;
        info->nnz_full = lk->nnz;
        info->nnz_flank = lk->nnz_flank;
        info->table_slots = (int64_t)(lk->mode == 2 ? lk->scap : lk->cap);
    }
    return HH_OK;
}

// AoS compact entries -> the 7 output arrays (SoA), so each goes to the host with one plain copy
__global__ void hh_k_links_split(const uint32_t* __restrict__ compact, int64_t nnz, uint32_t* __restrict__ soa, int64_t ht_off) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        const uint32_t* p = compact + e * 9;
        soa[0 * nnz + e] = p[0];
        soa[1 * nnz + e] = p[1];
        soa[2 * nnz + e] = p[2];
        soa[3 * nnz + e] = p[3];
        soa[4 * nnz + e] = p[4];
        soa[5 * nnz + e] = p[5];
        uint4 h;
        h.y = p[6];
        h.z = p[7];
        h.w = p[8];
        h.x = p[2] - p[6] - p[7] - p[8];          // HH = full - HT - TH - TT
        reinterpret_cast<uint4*>(soa + ht_off)[e] = h;
    }
}

// ---------------------------------------------------------------------------------------------
// routed multi-GPU counting (SURVEY.md 8e): route -> [all-to-all] -> add_routed -> finish_partition ->
// export -> [all-gather] -> adopt
// ---------------------------------------------------------------------------------------------
extern "C" int hh_links_route(hh_links* lk, const int32_t* rec_dev, int64_t n_rec, int64_t stream_offset, int world,
                              int32_t* rec_out_dev, uint32_t* pos_out_dev, int64_t* counts) {
    HH_REQUIRE(lk && counts && (n_rec == 0 || (rec_dev && rec_out_dev && pos_out_dev)), HH_ERR_ARG, "hh_links_route: NULL argument");
    HH_REQUIRE(world >= 1 && world <= HH_MAX_WORLD, HH_ERR_ARG, "hh_links_route: world must be in [1, %d]", HH_MAX_WORLD);
    HH_REQUIRE(n_rec >= 0 && stream_offset >= 0 && stream_offset + n_rec <= 0xFFFFFFFELL, HH_ERR_UNSUPPORTED,
               "hh_links_route: stream indices must fit 32 bits (offset %lld + %lld records)", (long long)stream_offset,
               (long long)n_rec);
    HH_REQUIRE((((uintptr_t)rec_dev | (uintptr_t)rec_out_dev) & 15) == 0, HH_ERR_ARG, "hh_links_route: records must be 16-byte aligned");
    hh_scope _scope(lk->ctx);
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    for (int d = 0; d < world; ++d) counts[d] = 0;
    if (n_rec == 0) return HH_OK;
    unsigned long long* d_cnt = nullptr;
    HH_CHECK(hh_dmalloc(&d_cnt, 2 * HH_MAX_WORLD));
    int rc = [&]() -> int {
        HH_CUDA(cudaMemsetAsync(d_cnt, 0, 2 * HH_MAX_WORLD * sizeof(unsigned long long), ctx->stream));
        const int contig_mode = lk->d_fbase == nullptr;
        int64_t blocks = (n_rec + 255) / 256;
        int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
        const int4* rec4 = reinterpret_cast<const int4*>(rec_dev);
        HH_LAUNCH(ctx, hh_k_route_count, grid, 256, 0, rec4, n_rec, lk->n_src, contig_mode, world, d_cnt);
        unsigned long long h[HH_MAX_WORLD];
        HH_CUDA(cudaMemcpyAsync(h, d_cnt, (size_t)world * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        unsigned long long base[HH_MAX_WORLD], acc = 0;
        for (int d = 0; d < world; ++d) {
            counts[d] = (int64_t)h[d];
            base[d] = acc;
            acc += h[d];
        }
        HH_CUDA(cudaMemcpyAsync(d_cnt + HH_MAX_WORLD, base, (size_t)world * sizeof(unsigned long long), cudaMemcpyHostToDevice,
                                ctx->stream));
        HH_LAUNCH(ctx, hh_k_route_scatter, grid, 256, 0, rec4, n_rec, (uint32_t)stream_offset, lk->n_src, contig_mode, world,
                  d_cnt + HH_MAX_WORLD, reinterpret_cast<int4*>(rec_out_dev), pos_out_dev);
        HH_CUDA(cudaStreamSynchronize(ctx->stream));      // `base` is a host temporary; the caller hands the buffers to NCCL next
        return HH_OK;
    }();
    hh_dfree(d_cnt);
    HH_CHECK(rc);
    lk->n_records += n_rec;          // records this rank read from the stream (used or not)
    if (stream_offset + n_rec > lk->stream_end) lk->stream_end = stream_offset + n_rec;
    return HH_OK;
}

extern "C" int hh_links_add_routed(hh_links* lk, const int32_t* rec_dev, const uint32_t* pos_dev, int64_t n_rec) {
    HH_REQUIRE(lk && (n_rec == 0 || (rec_dev && pos_dev)), HH_ERR_ARG, "hh_links_add_routed: NULL argument");
    hh_scope _scope(lk->ctx);
    HH_REQUIRE(!lk->finished, HH_ERR_STATE, "hh_links_add_routed: stream already finished");
    HH_REQUIRE(n_rec >= 0, HH_ERR_ARG, "hh_links_add_routed: negative record count");
    HH_REQUIRE(((uintptr_t)rec_dev & 15) == 0, HH_ERR_ARG, "hh_links_add_routed: records must be 16-byte aligned");
    if (n_rec == 0) return HH_OK;
    HH_CUDA(cudaSetDevice(lk->ctx->device));
    HH_REQUIRE(lk->mode != 2, HH_ERR_STATE, "hh_links_add_routed: this table counts a partitioned stream (hh_links_add of a long stream)");
    lk->mode = 1;
    const int64_t CH = 1ll << 23;
    for (int64_t off = 0; off < n_rec; off += CH) {
        const int64_t m = (n_rec - off < CH) ? (n_rec - off) : CH;
        HH_CHECK(links_ensure_capacity(lk, m));
        HH_CHECK(links_launch_insert(lk, reinterpret_cast<const int4*>(rec_dev) + off, m, 0, pos_dev + off));
        lk->since_known += m;
    }
    return HH_OK;
}

// compact list of a partition table in slot order (no first-seen ordering: the union is ordered lazily by hh_links_fetch)
extern "C" int hh_links_finish_partition(hh_links* lk, hh_links_info* info) {
    HH_REQUIRE(lk != nullptr, HH_ERR_ARG, "hh_links_finish_partition: NULL handle");
    hh_scope _scope(lk->ctx);
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    if (!lk->finished && lk->mode == 2) HH_CHECK(links_finish_partitioned(lk));     // already an unordered entry list
    if (!lk->finished) {
        HH_CHECK(links_need_table(lk));
        unsigned long long c[8];
        HH_CHECK(links_read_counters(lk, c));
        HH_REQUIRE(c[2] == 0, HH_ERR_CAPACITY, "hh_links_finish_partition: hash table overflow (capacity %llu slots)",
                   (unsigned long long)lk->cap);
        HH_REQUIRE(c[5] == 0, HH_ERR_ARG,
                   "hh_links_finish_partition: %llu records have a position outside their contig's bins (e.g. record %llu of the stream)",
                   c[5], c[6] - 1ull);
        lk->nnz = (int64_t)c[0];
        lk->n_used = lk->peer_used + (int64_t)c[1];
        HH_CUDA(cudaMemsetAsync(lk->d_counters + 3, 0, sizeof(unsigned long long), ctx->stream));
        hh_dfree(lk->d_compact);
        HH_CHECK(hh_dmalloc(&lk->d_compact, (size_t)(lk->nnz > 0 ? lk->nnz : 1) * 9));
        if (lk->nnz > 0) {
            HH_REQUIRE(lk->cap <= 0xFFFFFFFFull, HH_ERR_UNSUPPORTED, "hh_links_finish_partition: table too large");
            const int64_t S = (int64_t)lk->cap;
            uint32_t* d_order = nullptr;
            int* d_bcnt = nullptr;
            int64_t* d_boff = nullptr;
            const int64_t nb = (S + HH_CMP_TILE - 1) / HH_CMP_TILE;
            int rc = HH_OK;
            do {
                if ((rc = hh_dmalloc(&d_order, (size_t)S)) != HH_OK) break;
                if ((rc = hh_dmalloc(&d_bcnt, (size_t)nb)) != HH_OK) break;
                if ((rc = hh_dmalloc(&d_boff, (size_t)nb + 1)) != HH_OK) break;
            } while (0);
            if (rc == HH_OK) {
                rc = [&]() -> int {
                    HH_LAUNCH(ctx, hh_k_links_mark_slots, hh_grid(ctx, 8), 256, 0, lk->d_keys, lk->cap, d_order);
                    HH_LAUNCH(ctx, hh_k_compact_count, (unsigned)nb, 256, 0, d_order, S, d_bcnt);
                    HH_CHECK(hh_exclusive_scan_i32(ctx, d_bcnt, d_boff, (int)nb));
                    HH_LAUNCH(ctx, hh_k_compact_gather, (unsigned)nb, 256, 0, d_order, S, d_boff, lk->d_keys, lk->d_vals,
                              lk->d_compact, lk->d_counters);
                    HH_CHECK(links_read_counters(lk, c));
                    return HH_OK;
                }();
            }
            hh_dfree(d_order);
            hh_dfree(d_bcnt);
            hh_dfree(d_boff);
            HH_CHECK(rc);
            lk->nnz_flank = (int64_t)c[3];
        }
        lk->finished = true;
        lk->ordered = false;
        lk->index_valid = false;
    }
    if (info) {
        info->n_records = lk->n_records;
        info->n_used = lk->n_used;
        info->nnz_full = lk->nnz;
        info->nnz_flank = lk->nnz_flank;
        info->table_slots = (int64_t)lk->cap;
    }
    return HH_OK;
}

// the table becomes the union of disjoint partitions: `entries_dev` is the concatenation of every rank's export,
// `ctg_links_dev` / n_records / n_used the sums over ranks, stream_end the length of the whole stream
extern "C" int hh_links_adopt(hh_links* lk, const uint32_t* entries_dev, int64_t n_entries, const int64_t* ctg_links_dev,
                              int64_t n_records, int64_t n_used, int64_t stream_end) {
    HH_REQUIRE(lk && ctg_links_dev && (entries_dev || n_entries == 0), HH_ERR_ARG, "hh_links_adopt: NULL argument");
    HH_REQUIRE(n_entries >= 0 && stream_end >= 0 && stream_end <= 0xFFFFFFFELL, HH_ERR_ARG, "hh_links_adopt: bad sizes");
    hh_scope _scope(lk->ctx);
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    // the hash table is not needed any more: every consumer works on the entry list
    hh_dfree(lk->d_keys);
    hh_dfree(lk->d_vals);
    lk->d_keys = nullptr;
    lk->d_vals = nullptr;
    lk->cap = 0;
    hh_dfree(lk->d_compact);
    lk->d_compact = nullptr;
    HH_CHECK(hh_dmalloc(&lk->d_compact, (size_t)(n_entries > 0 ? n_entries : 1) * 9));
    HH_CUDA(cudaMemsetAsync(lk->d_counters + 2, 0, 2 * sizeof(unsigned long long), ctx->stream));
    if (n_entries) {
        HH_CUDA(cudaMemcpyAsync(lk->d_compact, entries_dev, (size_t)n_entries * 9 * sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                                ctx->stream));
        int64_t blocks = (n_entries + 255) / 256;
        int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
        HH_LAUNCH(ctx, hh_k_list_count_flank, grid, 256, 0, lk->d_compact, n_entries, lk->d_counters);
    }
    HH_CUDA(cudaMemcpyAsync(lk->d_ctg, ctg_links_dev, (size_t)lk->n_ctg * sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx->stream));
    unsigned long long c[8];
    HH_CHECK(links_read_counters(lk, c));
    lk->nnz = n_entries;
    lk->nnz_flank = (int64_t)c[3];
    lk->n_records = n_records;
    lk->n_used = n_used;
    lk->peer_used = 0;
    lk->stream_end = stream_end;
    lk->finished = true;
    lk->ordered = false;
    lk->index_valid = false;
    return HH_OK;
}

// put an adopted / partition list into dict insertion order (first_full ascending; the values are unique stream indices)
static int links_order_list(hh_links* lk) {
    if (lk->ordered || lk->nnz == 0) {
        lk->ordered = true;
        return HH_OK;
    }
    hh_ctx* ctx = lk->ctx;
    const int64_t S = lk->stream_end;
    const int64_t nb = (S + HH_CMP_TILE - 1) / HH_CMP_TILE;
    uint32_t *d_order = nullptr, *d_sorted = nullptr;
    int* d_bcnt = nullptr;
    int64_t* d_boff = nullptr;
    int rc = HH_OK;
    do {
        if ((rc = hh_dmalloc(&d_order, (size_t)S)) != HH_OK) break;
        if ((rc = hh_dmalloc(&d_sorted, (size_t)lk->nnz * 9)) != HH_OK) break;
        if ((rc = hh_dmalloc(&d_bcnt, (size_t)nb)) != HH_OK) break;
        if ((rc = hh_dmalloc(&d_boff, (size_t)nb + 1)) != HH_OK) break;
    } while (0);
    unsigned long long c[8] = {0};
    if (rc == HH_OK) {
        rc = [&]() -> int {
            HH_CUDA(cudaMemsetAsync(d_order, 0xFF, (size_t)S * sizeof(uint32_t), ctx->stream));
            HH_CUDA(cudaMemsetAsync(lk->d_counters + 2, 0, sizeof(unsigned long long), ctx->stream));
            int64_t blocks = (lk->nnz + 255) / 256;
            int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
            HH_LAUNCH(ctx, hh_k_list_scatter_order, grid, 256, 0, lk->d_compact, lk->nnz, d_order, S, lk->d_counters);
            HH_LAUNCH(ctx, hh_k_compact_count, (unsigned)nb, 256, 0, d_order, S, d_bcnt);
            HH_CHECK(hh_exclusive_scan_i32(ctx, d_bcnt, d_boff, (int)nb));
            HH_LAUNCH(ctx, hh_k_compact_gather, (unsigned)nb, 256, 0, d_order, S, d_boff, (const uint64_t*)nullptr,
                      reinterpret_cast<const hh_slot*>(lk->d_compact), d_sorted, lk->d_counters);
            HH_CHECK(links_read_counters(lk, c));
            return HH_OK;
        }();
    }
    hh_dfree(d_order);
    hh_dfree(d_bcnt);
    hh_dfree(d_boff);
    if (rc == HH_OK && c[2] != 0) {
        hh_dfree(d_sorted);
        HH_REQUIRE(false, HH_ERR_STATE, "hh_links: first-seen index beyond the stream end (stream_end misuse in hh_links_adopt)");
    }
    if (rc != HH_OK) {
        hh_dfree(d_sorted);
        return rc;
    }
    hh_dfree(lk->d_compact);
    lk->d_compact = d_sorted;
    lk->ordered = true;
    return HH_OK;
}

extern "C" int hh_links_fetch(hh_links* lk, int32_t* key_i, int32_t* key_j, uint32_t* full, uint32_t* flank,
                              uint32_t* first_full, uint32_t* first_flank, uint32_t* ht) {
    HH_REQUIRE(lk != nullptr, HH_ERR_ARG, "hh_links_fetch: NULL handle");
    hh_scope _scope(lk->ctx);
    HH_REQUIRE(lk->finished, HH_ERR_STATE, "hh_links_fetch: call hh_links_finish first");
    if (lk->nnz == 0) return HH_OK;
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    HH_CHECK(links_order_list(lk));
    const int64_t nnz = lk->nnz;
    uint32_t* d_soa = nullptr;
    HH_CHECK(hh_dmalloc(&d_soa, (size_t)nnz * 10 + 4));
    int rc = [&]() -> int {
        uint32_t* base = d_soa;
        const int64_t ht_off = (6 * nnz + 3) & ~3ll;      // the 4-wide HT block is written with 16-byte stores
        int64_t blocks = (nnz + 255) / 256;
        int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
        HH_LAUNCH(ctx, hh_k_links_split, grid, 256, 0, lk->d_compact, nnz, base, ht_off);
        void* dst[6] = {key_i, key_j, full, flank, first_full, first_flank};
        for (int k = 0; k < 6; ++k)
            if (dst[k])
                HH_CUDA(cudaMemcpyAsync(dst[k], base + (size_t)k * nnz, (size_t)nnz * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (ht) HH_CUDA(cudaMemcpyAsync(ht, base + ht_off, (size_t)nnz * 16, cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        return HH_OK;
    }();
    hh_dfree(d_soa);
    return rc;
}

extern "C" int hh_links_fetch_ctg(hh_links* lk, int64_t* ctg_links) {
    HH_REQUIRE(lk && ctg_links, HH_ERR_ARG, "hh_links_fetch_ctg: NULL argument");
    HH_CUDA(cudaSetDevice(lk->ctx->device));
    HH_CUDA(cudaMemcpyAsync(ctg_links, lk->d_ctg, (size_t)lk->n_ctg * sizeof(int64_t), cudaMemcpyDeviceToHost, lk->ctx->stream));
    HH_CUDA(cudaStreamSynchronize(lk->ctx->stream));
    return HH_OK;
}

extern "C" int hh_links_export(hh_links* lk, uint32_t* entries_dev, int64_t* ctg_links_dev) {
    HH_REQUIRE(lk != nullptr, HH_ERR_ARG, "hh_links_export: NULL handle");
    HH_REQUIRE(lk->finished, HH_ERR_STATE, "hh_links_export: call hh_links_finish first");
    HH_CUDA(cudaSetDevice(lk->ctx->device));
    if (entries_dev && lk->nnz)
        HH_CUDA(cudaMemcpyAsync(entries_dev, lk->d_compact, (size_t)lk->nnz * 9 * sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                                lk->ctx->stream));
    if (ctg_links_dev)
        HH_CUDA(cudaMemcpyAsync(ctg_links_dev, lk->d_ctg, (size_t)lk->n_ctg * sizeof(int64_t), cudaMemcpyDeviceToDevice,
                                lk->ctx->stream));
    HH_CUDA(cudaStreamSynchronize(lk->ctx->stream));
    return HH_OK;
}

extern "C" int hh_links_merge(hh_links* lk, const uint32_t* entries_dev, int64_t n_entries, const int64_t* ctg_links_dev,
                              int64_t n_records, int64_t n_used) {
    HH_REQUIRE(lk != nullptr, HH_ERR_ARG, "hh_links_merge: NULL handle");
    hh_scope _scope(lk->ctx);
    HH_REQUIRE(lk->mode != 2 && !(lk->finished && lk->d_keys == nullptr), HH_ERR_STATE,
               "hh_links_merge: this table holds an entry list (hh_links_adopt / partitioned counting), not a hash table");
    lk->mode = 1;
    HH_CHECK(links_need_table(lk));
    lk->finished = false;   // a finished table is re-opened: the next hh_links_finish rebuilds the ordered view
    lk->index_valid = false;
    HH_REQUIRE(n_entries >= 0 && (entries_dev || n_entries == 0), HH_ERR_ARG, "hh_links_merge: bad entries");
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    if (n_entries) {
        HH_CHECK(links_ensure_capacity(lk, n_entries));
        int64_t blocks = (n_entries + 255) / 256;
        int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
        HH_LAUNCH(ctx, hh_k_links_merge, grid, 256, 0, entries_dev, n_entries, lk->d_keys, lk->d_vals, lk->cap, lk->d_counters);
        lk->since_known += n_entries;
    }
    if (ctg_links_dev)
        HH_LAUNCH(ctx, hh_k_add_u64, (lk->n_ctg + 255) / 256, 256, 0, lk->d_ctg, ctg_links_dev, lk->n_ctg);
    HH_CUDA(cudaStreamSynchronize(ctx->stream));
    lk->n_records += n_records;
    lk->peer_used += n_used;
    return HH_OK;
}

extern "C" int hh_links_linked_index(hh_links* lk, const uint8_t* keep, int32_t* index, int32_t* n_linked) {
    HH_REQUIRE(lk && keep, HH_ERR_ARG, "hh_links_linked_index: NULL argument");
    hh_scope _scope(lk->ctx);
    HH_REQUIRE(lk->finished, HH_ERR_STATE, "hh_links_linked_index: call hh_links_finish first");
    hh_ctx* ctx = lk->ctx;
    HH_CUDA(cudaSetDevice(ctx->device));
    lk->index_valid = false;
    const int n = lk->n_ctg;
    const int nb = (n + HH_RADIX_TILE - 1) / HH_RADIX_TILE;
    unsigned long long* d_touch = nullptr;
    unsigned long long* d_key[2] = {nullptr, nullptr};
    int32_t* d_val[2] = {nullptr, nullptr};
    int* d_cnt = nullptr;
    int64_t* d_off = nullptr;
    int rc = [&]() -> int {
        HH_CHECK(hh_dmalloc(&d_touch, (size_t)n));
        for (int b = 0; b < 2; ++b) {
            HH_CHECK(hh_dmalloc(&d_key[b], (size_t)n));
            HH_CHECK(hh_dmalloc(&d_val[b], (size_t)n));
        }
        HH_CHECK(hh_dmalloc(&d_cnt, (size_t)nb * 256));
        HH_CHECK(hh_dmalloc(&d_off, (size_t)nb * 256 + 1));
        HH_CUDA(cudaMemcpyAsync(lk->d_keep, keep, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        HH_CUDA(cudaMemsetAsync(d_touch, 0xFF, (size_t)n * sizeof(unsigned long long), ctx->stream));
        int* d_nl = reinterpret_cast<int*>(ctx->d_scratch + 8);
        HH_CUDA(cudaMemsetAsync(d_nl, 0, sizeof(int), ctx->stream));
        if (lk->nnz) {
            int64_t blocks = (lk->nnz + 255) / 256;
            int grid = (int)(blocks < (int64_t)hh_grid(ctx, 8) ? blocks : (int64_t)hh_grid(ctx, 8));
            HH_LAUNCH(ctx, hh_k_touch, grid, 256, 0, lk->d_compact, lk->nnz, lk->d_keep, d_touch);
        }
        HH_LAUNCH(ctx, hh_k_rank_init, nb, HH_RADIX_TILE, 0, d_touch, n, d_key[0], d_val[0], d_nl);
        for (int pass = 0; pass < HH_RADIX_PASSES; ++pass) {
            const int src = pass & 1;
            HH_LAUNCH(ctx, hh_k_radix_hist, nb, HH_RADIX_TILE, 0, d_key[src], n, 8 * pass, d_cnt);
            HH_CHECK(hh_exclusive_scan_i32(ctx, d_cnt, d_off, nb * 256));
            HH_LAUNCH(ctx, hh_k_radix_scatter, nb, HH_RADIX_TILE, 0, d_key[src], d_val[src], n, 8 * pass, d_off, d_key[src ^ 1],
                      d_val[src ^ 1]);
        }
        HH_LAUNCH(ctx, hh_k_rank_index, (n + 255) / 256, 256, 0, d_val[HH_RADIX_PASSES & 1], n, d_nl, lk->d_index);
        HH_CUDA(cudaMemcpyAsync(ctx->h_scratch + 8, d_nl, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        if (index)
            HH_CUDA(cudaMemcpyAsync(index, lk->d_index, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        HH_CUDA(cudaStreamSynchronize(ctx->stream));
        lk->n_linked = *reinterpret_cast<int*>(ctx->h_scratch + 8);
        return HH_OK;
    }();
    hh_dfree(d_touch);
    for (int b = 0; b < 2; ++b) {
        hh_dfree(d_key[b]);
        hh_dfree(d_val[b]);
    }
    hh_dfree(d_cnt);
    hh_dfree(d_off);
    HH_CHECK(rc);
    lk->index_keep->assign(keep, keep + n);
    lk->index_valid = true;
    if (n_linked) *n_linked = lk->n_linked;
    return HH_OK;
}

// the first-seen index for `keep` on the device (d_index, d_keep): the one hh_links_linked_index left there when it was
// computed for the same mask and entry list, else computed now
int hh_links_index_for(hh_links* lk, const uint8_t* keep, int32_t* n_linked) {
    if (lk->index_valid && memcmp(lk->index_keep->data(), keep, (size_t)lk->n_ctg) == 0) {
        *n_linked = lk->n_linked;
        return HH_OK;
    }
    return hh_links_linked_index(lk, keep, nullptr, n_linked);
}

// d_index was changed in place (the matrix build appends the tail fragments to it)
void hh_links_index_invalidate(hh_links* lk) { lk->index_valid = false; }

extern "C" int hh_links_destroy(hh_links* lk) {
    if (!lk) return HH_OK;
    hh_scope _scope(lk->ctx);
    cudaSetDevice(lk->ctx->device);
    cudaStreamSynchronize(lk->ctx->stream);
    if (lk->copy_stream) {
        cudaStreamSynchronize(lk->copy_stream);
        cudaStreamDestroy(lk->copy_stream);
    }
    for (int k = 0; k < 2; ++k) {
        if (lk->ev_copied[k]) cudaEventDestroy(lk->ev_copied[k]);
        if (lk->ev_consumed[k]) cudaEventDestroy(lk->ev_consumed[k]);
        if (lk->d_stage[k]) cudaFree(lk->d_stage[k]);
    }
    hh_dfree(lk->d_src_rank);
    hh_dfree(lk->d_fbase);
    hh_dfree(lk->d_len);
    hh_dfree(lk->d_rank);
    hh_dfree(lk->d_nx);
    hh_dfree(lk->d_ctg);
    hh_dfree(lk->d_keys);
    hh_dfree(lk->d_vals);
    hh_dfree(lk->d_counters);
    hh_dfree(lk->d_compact);
    hh_dfree(lk->d_index);
    hh_dfree(lk->d_keep);
    links_free_partsets(lk);
    delete lk->psets;
    delete lk->index_keep;
    delete lk;
    return HH_OK;
}

// accessors used by hh_matrix.cu
int32_t hh_links_n_ctg(hh_links* lk) { return lk->n_ctg; }
hh_ctx* hh_links_ctx(hh_links* lk) { return lk->ctx; }
const uint32_t* hh_links_compact(hh_links* lk, int64_t* nnz) { *nnz = lk->nnz; return lk->d_compact; }
const unsigned long long* hh_links_ctg_totals(hh_links* lk) { return lk->d_ctg; }
int32_t* hh_links_index_dev(hh_links* lk, int32_t* n_linked) { *n_linked = lk->n_linked; return lk->d_index; }
uint8_t* hh_links_keep_dev(hh_links* lk) { return lk->d_keep; }
bool hh_links_finished(hh_links* lk) { return lk->finished; }
