#!/usr/bin/env python3
"""`haphic cluster` on the B200 -- a drop-in for scripts/HapHiC_cluster.py of zengxiaofei/HapHiC.

Same command line, same ``parse_arguments() / run(args, log_file) / main()`` entry points, same
files written into the working directory (HT_links.pkl, paired_links.clm, full_links.pkl,
inflation_*/mcl_inflation_*.clusters.txt, inflation_*/group*.txt, inflation_*/*_statistics.txt,
alignments.bed, HapHiC_cluster.log) and the same log messages (`haphic pipeline` greps the log for
"You could try inflation from ...", HapHiC_pipeline.py:385), so reassign / sort / build run
unchanged.  The per-read-pair link counting, dict_to_matrix and the Markov-cluster loop run in
libhaphic_b200.so on the GPU; file parsing, fragment statistics, filters on per-fragment scalars,
result interpretation and the writers are host Python, as in the reference.

``--correct_nrounds`` (assembly correction, 943-1297) runs on the GPU as well (haphic_b200/correct.py, hh_correct.cu).

Not supported (raise, never silently degrade): ``--ul``, ``--gfa`` (out of the hot-path scope, SURVEY.md section 2).

Reference line numbers below refer to scripts/HapHiC_cluster.py (v1.0.7).
"""

from __future__ import annotations

import argparse
import logging
import os
import pickle
import random
import sys
import time
from collections import OrderedDict, defaultdict
from itertools import combinations
from math import ceil, inf

import numpy as np

__version__ = "1.0.7-b200.1"
__update_time__ = "2026.09.24"

logging.basicConfig(format="%(asctime)s <%(filename)s> [%(funcName)s] %(message)s", datefmt="%Y-%m-%d %H:%M:%S")
logger = logging.getLogger(__name__)
logger.setLevel(logging.INFO)


# ------------------------------------------------------------------------------------------------
# FASTA / fragment statistics (host; lines 56-147, 188-296)
# ------------------------------------------------------------------------------------------------

def parse_RE_sites(sites):
    """Expand every 'N' of the recognition sites into A/T/C/G (56-72)."""
    todo, done = list(sites), []
    while todo:
        s = todo.pop(0)
        if "N" in s:
            todo[0:0] = [s.replace("N", b, 1) for b in "ATCG"]
        else:
            done.append(s)
    return done


def count_RE_sites(seq, RE):
    sites = [s.strip().upper() for s in RE.split(",") if s.strip()]
    return sum(seq.count(s) for s in parse_RE_sites(sites))


def parse_fasta(fasta, RE="GATC", keep_letter_case=False, logger=logger):
    """{ctg: [seq, length, RE sites + 1]} in file order (87-113)."""
    logger.info("Parsing input FASTA file...")
    chunks = OrderedDict()
    with open(fasta) as f:
        cur = None
        for line in f:
            s = line.strip()
            if not s:
                continue
            if line.startswith(">"):
                cur = line.split()[0][1:]
                chunks[cur] = []
            else:
                chunks[cur].append(s if keep_letter_case else s.upper())
    fa_dict = dict()
    for ctg, parts in chunks.items():
        seq = "".join(parts)
        fa_dict[ctg] = [seq, len(seq), count_RE_sites(seq, RE) + 1]     # pseudo-count as ALLHiC does
    return fa_dict


def determine_int_type(fa_dict, logger=logger):
    """int32 / int64 for positions and CLM distances (116-147)."""
    lens = sorted(info[1] for info in fa_dict.values())
    longest = lens[-1]
    second = lens[-2] if len(lens) > 1 else 0
    limit = 2 ** 31 - 1
    pos_t = "int64" if longest > limit else "int32"
    dist_t = "int64" if longest + second > limit else "int32"
    logger.info("The longest and second longest contigs are {} bp and {} bp, respectively. The data types for "
                "contig positions and CLM distances are calculated to be {} and {}, respectively.".format(
                    longest, second, pos_t, dist_t))
    if pos_t == "int64":
        logger.warning("Found at least one contig longer than {} bp in the input assembly. There could be a problem "
                       "when visualizing it in Juicebox".format(limit))
    return pos_t, dist_t


def parse_gfa(gfa_list, fa_dict, logger=logger):
    raise NotImplementedError("haphic_b200: --gfa (hifiasm read depth / phasing, HapHiC_cluster.py:150-185) is not supported")


def remove_allelic_HiC_links(fa_dict, ctg_coord_dict, full_link_dict, args, flank_link_dict=None, filtered_frags=None,
                             ctg_pair_to_frag=None, logger=logger):
    """474-692, see haphic_b200/allelic.py (HapHiC_reassign.py:23 imports this name)."""
    from . import allelic
    return allelic.remove_allelic_HiC_links(fa_dict, ctg_coord_dict, full_link_dict, args, flank_link_dict, filtered_frags,
                                            ctg_pair_to_frag, logger=logger, dict_to_matrix=dict_to_matrix)


def stat_fragments(fa_dict, RE, read_depth_dict, whitelist, nchrs=0, flank=0, Nx=100, bin_size=0, logger=logger):
    """Fragment lengths, flank RE counts, bins and the Nx set (188-296).  Returns the reference's
    7-tuple (sorted_frag_list, bin_set, bin_size, frag_len_dict, Nx_frag_set, RE_site_dict, split_ctg_set)."""
    logger.info("Making some statistics of fragments (contigs / bins)")
    flank_bp = flank * 1000

    def flank_RE(seq, length):
        if not flank_bp or length <= 2 * flank_bp:
            return count_RE_sites(seq, RE) + 1
        return count_RE_sites(seq[:flank_bp], RE) + count_RE_sites(seq[length - flank_bp:], RE) + 1

    total_len = sum(info[1] for info in fa_dict.values())
    if not bin_size:
        logger.info("bin_size is set to {}, no fragments will be split".format(bin_size))
        bin_size = inf
    elif bin_size < 0:
        bin_size = max(min(int(total_len / nchrs / 30), 2000000), 100000)
        logger.info("bin_size is calculated to be {} bp".format(bin_size))
    else:
        bin_size *= 1000
        logger.info("bin_size is manually designated to {} bp".format(bin_size))

    frags, bin_set, split_ctg_set = [], set(), set()
    RE_site_dict, frag_len_dict = dict(), dict()
    for ctg, (seq, ctg_len, RE_sites) in fa_dict.items():
        if ctg_len > bin_size:
            split_ctg_set.add(ctg)
            nbins = ceil(ctg_len / bin_size)
            for m in range(nbins):
                name = "{}_bin{}".format(ctg, m + 1)
                assert name not in fa_dict
                frags.append(name)
                bin_set.add(name)
                last = m + 1 == nbins
                blen = ctg_len - m * bin_size if last else bin_size
                bseq = seq[m * bin_size:] if last else seq[m * bin_size:(m + 1) * bin_size]
                RE_site_dict[name] = flank_RE(bseq, blen)
                frag_len_dict[name] = blen
                if read_depth_dict:
                    read_depth_dict[name] = read_depth_dict[ctg]
            if read_depth_dict:
                del read_depth_dict[ctg]
        else:
            frags.append(ctg)
            frag_len_dict[ctg] = ctg_len
            RE_site_dict[ctg] = RE_sites if (not flank_bp or ctg_len <= 2 * flank_bp) else flank_RE(seq, ctg_len)
        fa_dict[ctg][0] = None          # sequences are not needed any more

    # seeded shuffle before the stable sort so equal-length fragments are not biased (273-275)
    random.seed(12345)
    random.shuffle(frags)
    sorted_frag_list = sorted(((f, frag_len_dict[f]) for f in frags), key=lambda x: x[1], reverse=True)
    len_sum = 0
    Nx_frag_set = set()
    for frag, flen in sorted_frag_list:
        len_sum += flen
        if len_sum / total_len * 100 < Nx or Nx == 100:
            Nx_frag_set.add(frag)
    if Nx != 100:
        Nx_frag_set.add(sorted_frag_list[len(Nx_frag_set)][0])
    if whitelist:
        for frag, _ in sorted_frag_list:
            if frag.rsplit("_bin", 1)[0] in whitelist:
                Nx_frag_set.add(frag)
    return sorted_frag_list, bin_set, bin_size, frag_len_dict, Nx_frag_set, RE_site_dict, split_ctg_set


def is_flank(coord, length, flank):
    """1-based ``coord`` inside the flanking regions (299-307)."""
    return (not flank) or coord <= flank or coord > length - flank


# ------------------------------------------------------------------------------------------------
# link counting on the GPU (1596-1655)
# ------------------------------------------------------------------------------------------------

_CTX = None


def _context():
    global _CTX
    if _CTX is None:
        from ._lib import Context
        _CTX = Context(_gpu_list()[0])
    return _CTX


def _gpu_list():
    """Devices of this run: ``HAPHIC_GPUS`` = a count ("8" -> devices 0..7) or a comma list ("0,2,5"); default one device,
    ``HAPHIC_DEVICE`` (0).  With several devices the inflation sweep of run_mcl_clustering is spread over them (every
    mcl() call is independent and shares only the input matrix, HapHiC_cluster.py:2155-2158): one host thread per GPU, no
    exchange, results identical to a single-GPU run by construction."""
    spec = os.environ.get("HAPHIC_GPUS", "").strip()
    if not spec:
        return [int(os.environ.get("HAPHIC_DEVICE", "0"))]
    if "," in spec:
        devs = [int(x) for x in spec.split(",") if x.strip()]
    else:
        first = int(os.environ.get("HAPHIC_DEVICE", "0"))
        devs = list(range(first, first + max(1, int(spec))))
    if not devs:
        raise ValueError("HAPHIC_GPUS names no device")
    return devs


def count_links(batches, names, ctg_len, Nx_ctg_set, flank_kb, want_clm=True, frag_table=None):
    """Stream record batches through the GPU link table(s).  Returns (table, clm_records) where
    clm_records is the concatenation of the usable inter-contig records (for the CLM writer) or None.
    ``frag_table`` (fragment mode) receives every batch as well."""
    from .links import LinkTable, name_rank
    ctx = _context()
    in_nx = np.fromiter((n in Nx_ctg_set for n in names), dtype=np.uint8, count=len(names))
    table = LinkTable(ctx, ctg_len, name_rank(names), in_nx, flank_kb * 1000)
    kept = []
    n = len(names)
    for rec in batches:
        table.add(rec)
        if frag_table is not None:
            frag_table.add(rec)
        if want_clm:
            ok = (rec[:, 0] != rec[:, 2]) & (rec[:, 0] >= 0) & (rec[:, 2] >= 0) & (rec[:, 0] < n) & (rec[:, 2] < n)
            kept.append(rec[ok])
    table.finish()
    if frag_table is not None:
        frag_table.finish()
    clm_rec = (np.concatenate(kept) if kept else np.zeros((0, 4), np.int32)) if want_clm else None
    return table, clm_rec


def fragment_layout(fa_dict, bin_size, frag_len_dict, Nx_frag_set, split_ctg_set):
    """Fragment ids for fragment mode: contig c (FASTA order) owns ids [frag_base[c], frag_base[c+1]); a split
    contig's bins are '{ctg}_bin{k}' (stat_fragments, 229-248)."""
    from .links import name_rank
    frag_names, frag_base = [], [0]
    for ctg, info in fa_dict.items():
        if ctg in split_ctg_set:
            nbins = ceil(info[1] / bin_size)
            frag_names += ["{}_bin{}".format(ctg, k + 1) for k in range(nbins)]
        else:
            frag_names.append(ctg)
        frag_base.append(len(frag_names))
    frag_len = np.array([frag_len_dict[f] for f in frag_names], dtype=np.int64)
    in_nx = np.fromiter((f in Nx_frag_set for f in frag_names), dtype=np.uint8, count=len(frag_names))
    return frag_names, np.asarray(frag_base, np.int32), frag_len, name_rank(frag_names), in_nx


# run() sets this to --min_read_pairs (unless --verbose): contig pairs with fewer links only get a debug line in
# remove_allelic_HiC_links, so their coordinate arrays are not materialised.  0 = the reference's complete dict.
_COORD_SKIP = [0]


def _stream_bins(alignments, fa_dict, args, bin_size, frag_len_dict, Nx_frag_set, split_ctg_set):
    """Count one pass of the alignments into the contig-level table (full / HT links) and the fragment-level table
    (flank links, per-fragment totals).  Returns a dict with both tables, the usable records and the fragment layout."""
    from .links import LinkTable, name_rank
    names = list(fa_dict.keys())
    ctg_len = np.array([fa_dict[n][1] for n in names], dtype=np.int64)
    frag_names, frag_base, frag_len, frag_rank, frag_nx = fragment_layout(fa_dict, bin_size, frag_len_dict, Nx_frag_set,
                                                                          split_ctg_set)
    ftab = LinkTable(_context(), frag_len, frag_rank, frag_nx, args.flank * 1000,
                     frags=dict(ctg_rank=name_rank(names), frag_base=frag_base, bin_size=int(bin_size)))
    batches = _as_batches(alignments, names)
    # contig-level table: Nx membership is irrelevant there (flank links are counted per fragment)
    table, clm_rec = count_links(batches, names, ctg_len, set(), args.flank, frag_table=ftab)
    return dict(table=table, ftab=ftab, clm_rec=clm_rec, names=names, ctg_len=ctg_len, rank=name_rank(names),
                frag_names=frag_names, frag_base=frag_base, frag_rank=frag_rank)


def parse_alignments(alignments, fa_dict, args, bin_size, frag_len_dict, Nx_frag_set, split_ctg_set, pos_int_type, dist_int_type,
                     build_clm=True):
    """Signature and return value of the reference function for the case that some contigs are split into
    bins (1658-1752): flank links and per-fragment totals are keyed by FRAGMENTS (second device table in
    fragment mode), full / HT / clm stay contig-level."""
    logger.info("Parsing input alignments...")
    from .links import link_dicts
    st = _stream_bins(alignments, fa_dict, args, bin_size, frag_len_dict, Nx_frag_set, split_ctg_set)
    table, ftab, clm_rec, names, ctg_len, rank = st["table"], st["ftab"], st["clm_rec"], st["names"], st["ctg_len"], st["rank"]
    frag_names = st["frag_names"]
    full_link_dict, _unused_flank, HT_link_dict, _unused_tot = link_dicts(table, names)
    table.close()
    _unused_full, flank_link_dict, _unused_ht, frag_link_dict = link_dicts(ftab, frag_names)
    clm_dict = build_clm_dict(clm_rec, names, ctg_len, rank, dist_int_type) if build_clm else defaultdict(list)
    parse_alignments.last_clm = (clm_rec, names, ctg_len, rank)
    parse_alignments.last_table = ftab
    parse_alignments.frag_names = frag_names
    ctg_coord_dict, ctg_pair_to_frag = defaultdict(list), defaultdict(set)
    if args.remove_allelic_links or args.remove_concentrated_links:
        from . import allelic
        ctg_coord_dict = allelic.coord_pair_dict(clm_rec, names, ctg_len, rank, args, pos_int_type, skip_below=_COORD_SKIP[0])
        if args.remove_allelic_links:
            ctg_pair_to_frag = allelic.ctg_pair_to_frag_dict(clm_rec, names, rank, frag_names, st["frag_base"], st["frag_rank"],
                                                             int(bin_size))
    return full_link_dict, flank_link_dict, HT_link_dict, clm_dict, frag_link_dict, ctg_coord_dict, ctg_pair_to_frag


def clm_arrays(clm_rec, n_names, ctg_len, rank, sort_within=True):
    """(key_i, key_j, offsets, dist[4, total]) of update_clm_dict (395-401): contig pairs in first-seen order;
    every pair's four distance rows sorted ascending (output_clm sorts them, 388).  Vectorised numpy for now
    (SURVEY.md f-2 moves the distances and the segmented sort to the GPU)."""
    if len(clm_rec) == 0:
        z = np.zeros(0, np.int32)
        return z, z, np.zeros(1, np.int64), np.zeros((4, 0), np.int64)
    r = clm_rec.astype(np.int64)
    swap = rank[r[:, 0]] > rank[r[:, 2]]
    i = np.where(swap, r[:, 2], r[:, 0])
    j = np.where(swap, r[:, 0], r[:, 2])
    a0 = np.where(swap, r[:, 3], r[:, 1])
    b0 = np.where(swap, r[:, 1], r[:, 3])
    li, lj = ctg_len[i], ctg_len[j]
    key = i * n_names + j
    order = np.argsort(key, kind="stable")
    ks = key[order]
    starts = np.concatenate([[0], np.nonzero(np.diff(ks))[0] + 1])
    lens = np.diff(np.concatenate([starts, [len(ks)]]))
    first = order[starts]                          # stable sort: first element of a run = first seen
    seg_order = np.argsort(first, kind="stable")
    offsets = np.concatenate([[0], np.cumsum(lens[seg_order])]).astype(np.int64)
    # position of every sorted element in the output: segments re-ordered by first appearance
    new_start = np.empty(len(starts), np.int64)
    new_start[seg_order] = offsets[:-1]
    seg_id = np.repeat(np.arange(len(starts)), lens)
    dest = new_start[seg_id] + (np.arange(len(ks)) - starts[seg_id])
    dist = np.empty((4, len(ks)), np.int64)
    rows = (li - a0 + b0, li - a0 + lj - b0, a0 + b0, a0 + lj - b0)
    for k in range(4):
        dk = rows[k][order]
        if sort_within:
            dk = dk[np.lexsort((dk, seg_id))]       # ascending inside every segment
        dist[k, dest] = dk                          # else: stream order inside the segment (stable key sort)
    uk = ks[starts][seg_order]
    return (uk // n_names).astype(np.int32), (uk % n_names).astype(np.int32), offsets, dist


def build_clm_dict(clm_rec, names, ctg_len, rank, dist_int_type="int32"):
    """clm_dict {(ctg_i, ctg_j): array of 4 distances per link} as the reference returns it (395-401), in
    first-seen key order, distances in stream order."""
    from array import array
    code = "i" if dist_int_type == "int32" else "l"
    clm = defaultdict(lambda: array(code))
    ki, kj, off, dist = clm_arrays(clm_rec, len(names), ctg_len, rank, sort_within=False)
    for e in range(len(ki)):
        s, t = int(off[e]), int(off[e + 1])
        clm[(names[ki[e]], names[kj[e]])] = array(code, dist[:, s:t].T.reshape(-1).tolist())
    return clm


def write_clm(clm_rec, names, ctg_len, rank, path="paired_links.clm", threads=0):
    """paired_links.clm straight from the records: grouping by contig pair, the per-pair distance sorts and the text
    are native and threaded (hh_clm_from_records)."""
    from . import hicio
    from ._lib import check, load, ptr
    logger.info("Writing clm_dict to paired_links.clm...")
    rec = np.ascontiguousarray(clm_rec, dtype=np.int32)
    check(load().hh_clm_from_records(os.fsencode(path), hicio.names_blob(names), len(names), ptr(rec) if len(rec) else None,
                                     len(rec), ptr(np.ascontiguousarray(ctg_len, dtype=np.int64)),
                                     ptr(np.ascontiguousarray(rank, dtype=np.int32)), int(threads)))


def _stream_contigs(alignments, fa_dict, args, ctg_len_dict, Nx_ctg_set):
    """Count one pass of the alignments into the device table; returns table, usable records and the id space."""
    from .links import name_rank
    names = list(fa_dict.keys())
    ctg_len = np.array([ctg_len_dict[n] for n in names], dtype=np.int64)
    batches = _as_batches(alignments, names)
    table, clm_rec = count_links(batches, names, ctg_len, Nx_ctg_set, args.flank)
    return dict(table=table, ftab=None, clm_rec=clm_rec, names=names, ctg_len=ctg_len, rank=name_rank(names))


def parse_alignments_for_ctgs(alignments, fa_dict, args, ctg_len_dict, Nx_ctg_set, pos_int_type, dist_int_type,
                              build_clm=True):
    """Signature and return value of the reference function (1596-1655).  ``alignments`` is an
    iterable of int32 record batches (hicio.pairs_batches / hicio.bam_batches) or of
    (ref, mref, pos, mpos) tuples as the reference's generators yield.  ``build_clm=False`` (used by run())
    leaves clm_dict empty and keeps the usable records in ``.last_clm`` for the native CLM writer."""
    logger.info("Parsing input alignments...")
    from .links import link_dicts
    st = _stream_contigs(alignments, fa_dict, args, ctg_len_dict, Nx_ctg_set)
    table, clm_rec, names, ctg_len, rank = st["table"], st["clm_rec"], st["names"], st["ctg_len"], st["rank"]
    full_link_dict, flank_link_dict, HT_link_dict, ctg_link_dict = link_dicts(table, names)
    clm_dict = build_clm_dict(clm_rec, names, ctg_len, rank, dist_int_type) if build_clm else defaultdict(list)
    parse_alignments_for_ctgs.last_table = table          # run() keeps using the device table
    parse_alignments_for_ctgs.last_clm = (clm_rec, names, ctg_len, rank)
    ctg_coord_dict = defaultdict(list)
    if args.remove_allelic_links or args.remove_concentrated_links:
        from . import allelic
        ctg_coord_dict = allelic.coord_pair_dict(clm_rec, names, ctg_len, rank, args, pos_int_type, skip_below=_COORD_SKIP[0])
    return full_link_dict, flank_link_dict, HT_link_dict, clm_dict, ctg_link_dict, ctg_coord_dict


def _as_batches(alignments, names, batch=1 << 20):
    it = iter(alignments)
    try:
        first = next(it)
    except StopIteration:
        return
    if isinstance(first, np.ndarray):
        yield first
        for rec in it:
            yield rec
        return
    ids = {n: i for i, n in enumerate(names)}
    buf = []

    def flush():
        out = np.array(buf, dtype=np.int32).reshape(-1, 4)
        buf.clear()
        return out

    def push(t):
        ref, mref, pos, mpos = t
        buf.append((ids.get(ref, -1), pos, ids.get(mref, -1), mpos))

    push(first)
    for t in it:
        push(t)
        if len(buf) >= batch:
            yield flush()
    if buf:
        yield flush()


# ------------------------------------------------------------------------------------------------
# writers (376-392, 710-715)
# ------------------------------------------------------------------------------------------------

def output_pickle(dict_, from_, to):
    logger.info("Writing {} to {}...".format(from_, to))
    with open(to, "wb") as f:
        pickle.dump(dict_, f)


def output_clm(clm_dict):
    """paired_links.clm: contig pairs with >= 2 links, four orientation lines each, every sorted
    distance printed twice and the count doubled (376-392)."""
    logger.info("Writing clm_dict to paired_links.clm...")
    signs = (("+", "+"), ("+", "-"), ("-", "+"), ("-", "-"))
    with open("paired_links.clm", "w") as fout:
        for (ci, cj), values in clm_dict.items():
            if len(values) < 8:
                continue
            arr = np.asarray(values).reshape(-1, 4)
            for k, (si, sj) in enumerate(signs):
                d = np.sort(arr[:, k]).tolist()
                fout.write("{}{} {}{}\t{}\t{}\n".format(ci, si, cj, sj, 2 * len(d), " ".join("{0} {0}".format(v) for v in d)))


def normalize_by_nlinks(flank_link_dict, frag_link_dict):
    """links / sqrt(tot_i * tot_j) on the host dict (718-724); the device matrix applies the same
    formula inside hh_matrix_from_links."""
    logger.info("Normalizing flank_link_dict by the number of links to other contigs...")
    for key in flank_link_dict:
        flank_link_dict[key] /= (frag_link_dict[key[0]] * frag_link_dict[key[1]]) ** 0.5


# ------------------------------------------------------------------------------------------------
# fragment filtering (741-940) -- per-fragment scalars on the host; the rank-sum part works on the
# dense fragment x fragment matrix (numpy here; SURVEY.md f-1 moves it to the GPU)
# ------------------------------------------------------------------------------------------------

def check_param(param, string, suffix, true_suffix=""):
    """'0.2X' -> (0.2, 'X'); '0.3' -> (0.3, '') with range check (2481-2507)."""
    if len(string) == 0:
        logger.error("Parameter {} is empty".format(param))
        raise RuntimeError("Parameter check failed")
    if len(string) > 1 and suffix and string[-1] in suffix:
        return check_param(param, string[:-1], None, string[-1])
    try:
        num = float(string)
    except ValueError:
        num = None
    if num is None or (not true_suffix and not 0 <= num <= 1):
        logger.error("Parameter {} {} is illegal".format(param, string + true_suffix))
        raise RuntimeError("Parameter check failed")
    return num, true_suffix


def _cut_index(sorted_pairs, limit, inclusive):
    """First position whose value reaches (>=, inclusive) / exceeds (>) ``limit``; len() if none."""
    for pos, (_f, v) in enumerate(sorted_pairs):
        if (v >= limit) if inclusive else (v > limit):
            return pos
    return len(sorted_pairs)


def device_matrix(table, names, frag_set, normalize_by_nlinks=False, add_self_loops=True):
    """dict_to_matrix (310-373) on the device table: (LinkMatrix, frag_index_dict).  Linked fragments get their
    first-seen index on the GPU; kept-but-unlinked ones follow in the reference's set-iteration order (355-359)."""
    keep = np.fromiter((n in frag_set for n in names), dtype=np.uint8, count=len(names))
    index, n_linked = table.linked_index(keep)
    order = np.argsort(np.where(index >= 0, index, np.iinfo(np.int32).max), kind="stable")[:n_linked]
    frags_in_dict = set()
    for c in order.tolist():                    # same insertion order as 332-333
        frags_in_dict.add(names[c])
    ids = {n: i for i, n in enumerate(names)}
    tail = [ids[f] for f in frag_set - frags_in_dict]
    matrix = table.to_matrix(keep, tail, normalize_by_nlinks=normalize_by_nlinks, add_self_loops=add_self_loops)
    frag_index = {names[c]: int(index[c]) for c in order.tolist()}
    for k, c in enumerate(tail):
        frag_index[names[c]] = n_linked + k
    return matrix, frag_index


def filter_fragments(Nx_frag_set, RE_site_dict, RE_site_cutoff, frag_link_dict, density_lower, density_upper,
                     topN, rank_sum_upper, rank_sum_hard_cutoff, flank_link_dict, read_depth_dict, read_depth_upper,
                     whitelist, device_table=None, device_names=None, normalized=False):
    """Same decisions and log lines as the reference's filter_fragments (741-940).  With ``device_table`` the
    O(n^2 log n) rank-sum part (864-892) runs on the GPU (hh_matrix_rank_sums); otherwise on the host."""
    logger.info("Filtering fragments...")
    if read_depth_dict:
        raise NotImplementedError("haphic_b200: read-depth filtering (--gfa) is not supported")
    wl_frags = set()
    density = []
    total_links, total_RE = 0, 1
    for frag in Nx_frag_set:
        RE_sites = RE_site_dict[frag]
        if RE_sites > RE_site_cutoff:
            if frag in frag_link_dict:
                links = frag_link_dict[frag]
                total_links += links
                total_RE += RE_sites - 1
                density.append((frag, links / RE_sites))
            else:
                density.append((frag, 0))
        if whitelist and frag.rsplit("_bin", 1)[0] in whitelist:
            wl_frags.add(frag)
    n_nx = len(Nx_frag_set)
    logger.info("[Nx filtering] {} fragments kept".format(n_nx))
    logger.info("[RE sites filtering] {} fragments removed, {} fragments kept".format(n_nx - len(density), len(density)))

    density.sort(key=lambda x: x[1])
    p_lo = check_param("--density_lower", density_lower, {"X", "x"})
    p_hi = check_param("--density_upper", density_upper, {"X", "x"})
    remaining = len(density)
    avg = total_links / total_RE
    if p_lo[-1] in {"X", "x"}:
        lower = _cut_index(density, avg * p_lo[0], True)
        logger.info('[link density filtering] Parameter --density_lower {} is set to "multiple" mode and equivalent to {} in "fraction" mode'.format(
            density_lower, lower / remaining))
    else:
        lower = int(remaining * float(density_lower))
        logger.info('[link density filtering] Parameter --density_lower {} is set to "fraction" mode and equivalent to {}X in "multiple" mode'.format(
            density_lower, density[max(0, lower - 1)][1] / avg))
    if p_hi[-1] in {"X", "x"}:
        upper = _cut_index(density, avg * p_hi[0], False)
        logger.info('[link density filtering] Parameter --density_upper {} is set to "multiple" mode and equivalent to {} in "fraction" mode'.format(
            density_upper, upper / remaining))
    else:
        upper = int(remaining * float(density_upper))
        logger.info('[link density filtering] Parameter --density_upper {} is set to "fraction" mode and equivalent to {}X in "multiple" mode'.format(
            density_upper, density[max(0, upper - 1)][1] / avg))
    filtered = {frag for frag, _ in density[lower:upper]}
    logger.info("[link density filtering] {} fragments removed, {} fragments kept".format(remaining - len(filtered), len(filtered)))
    for frag, d in density[:lower] + density[upper:]:
        logger.debug("[link density filtering] Fragment {} is removed, density={}".format(frag, d))
    density = density[lower:upper]

    # rank-sum of the topN nearest fragments (864-927)
    if device_table is not None:
        dmat, frag_index = device_matrix(device_table, device_names, filtered, normalize_by_nlinks=normalized,
                                         add_self_loops=False)
        # `[:topN]` of the reference just truncates (874-878): fewer fragments than topN use them all, and fewer than two
        # neighbours have no pair to rank (rank sum 0)
        eff_top = min(int(topN), len(filtered))
        device_rs = dmat.rank_sums(eff_top) if eff_top >= 2 else np.zeros(dmat.n, np.int64)
        dmat.close()
    else:
        matrix, frag_index = dict_to_matrix(flank_link_dict, filtered)
        n = matrix.shape[0]
        # descending stable sort of every row: ties keep index order, exactly list.sort(reverse=True)
        order = np.argsort(-matrix, axis=1, kind="stable")
        rank_of = np.empty((n, n), dtype=np.int32)
        rows = np.arange(n)[:, None]
        rank_of[rows, order] = np.arange(n, dtype=np.int32)[None, :]
    rank_sums = []
    hard = 0
    for frag, _ in density:
        if device_table is not None:
            rs = int(device_rs[frag_index[frag]])
        else:
            top = order[frag_index[frag], :topN].tolist()
            rs = 0
            for a, b in combinations(top, 2):
                rs += min(int(rank_of[a, b]), int(rank_of[b, a]))
        if rank_sum_hard_cutoff and rs > rank_sum_hard_cutoff:
            hard += 1
            logger.debug("[rank sum filtering] Fragment {} is removed by hard filtering, rank sum={}".format(frag, rs))
            continue
        rank_sums.append((frag, rs))
    rank_sums.sort(key=lambda x: x[1])
    remaining = len(rank_sums)
    if rank_sum_hard_cutoff:
        logger.info("[rank sum filtering] {} fragments removed by hard filtering, {} fragments kept".format(hard, remaining))
    p_rs = check_param("--rank_sum_upper", rank_sum_upper, {"X", "x"})
    q1, med, q3 = np.quantile([v for _, v in rank_sums], (0.25, 0.5, 0.75))
    iqr = q3 - q1
    logger.info("[rank sum filtering] Q1={}, median={}, Q3={}, IQR=Q3-Q1={}".format(q1, med, q3, iqr))
    if p_rs[-1]:
        upper = _cut_index(rank_sums, q3 + p_rs[0] * iqr, False)
        logger.info('[rank sum filtering] Parameter --rank_sum_upper {} is set to "multiple" mode and equivalent to {} in "fraction" mode'.format(
            rank_sum_upper, upper / remaining))
    else:
        upper = int(remaining * float(rank_sum_upper))
        logger.info('[rank sum filtering] Parameter --rank_sum_upper {} is set to "fraction" mode and equivalent to {}X in "multiple" mode'.format(
            rank_sum_upper, (rank_sums[max(0, upper - 1)][1] - q3) / iqr))
    filtered = {frag for frag, _ in rank_sums[:upper]}
    logger.info("[rank sum filtering] {} fragments removed, {} fragments kept".format(len(rank_sums) - len(filtered), len(filtered)))
    for frag, rs in rank_sums[upper:]:
        logger.debug("[rank sum filtering] Fragment {} is removed, rank sum={}".format(frag, rs))
    if wl_frags:
        added = 0
        for frag in wl_frags:
            if frag not in filtered:
                added += 1
                logger.debug("[rank sum filtering] Fragment {} is added since it is on the whitelist".format(frag))
                filtered.add(frag)
        logger.info("[rank sum filtering] {} fragments added, {} fragments are used to perform Markov clustering".format(
            added, len(filtered)))
    return filtered


def dict_to_matrix(link_dict, frag_set, dense_matrix=True, add_self_loops=False):
    """Host version with the reference's signature and return (310-373) -- `haphic reassign` imports
    it (HapHiC_reassign.py:23).  The cluster step itself builds the matrix on the device
    (hh_matrix_from_links)."""
    from scipy.sparse import coo_matrix
    frag_index = dict()
    rows, cols, vals = [], [], []
    linked = set()
    for (fi, fj), links in link_dict.items():
        if fi not in frag_set or fj not in frag_set:
            continue
        linked.add(fi)
        linked.add(fj)
        i = frag_index.setdefault(fi, len(frag_index))
        j = frag_index.setdefault(fj, len(frag_index))
        rows += (i, j)
        cols += (j, i)
        vals += (links, links)
    for frag in frag_set - linked:
        frag_index[frag] = len(frag_index)
    shape = len(frag_set)
    if add_self_loops:
        rows += range(shape)
        cols += range(shape)
        vals += [1] * shape
    m = coo_matrix((vals, (rows, cols)), shape=(shape, shape), dtype=np.float32)
    return (m.toarray() if dense_matrix else m.tocsc()), frag_index


# ------------------------------------------------------------------------------------------------
# Markov clustering (2026-2242): matrix work on the GPU, interpretation / files on the host
# ------------------------------------------------------------------------------------------------

def interpret_result(result_matrix, dense_matrix=False):
    from .mcl import interpret_result as _ir
    return _ir(result_matrix)


def get_main_groups(result_clusters, len_ratio):
    for k in range(len(result_clusters) - 1):
        if result_clusters[k + 1][1] / result_clusters[k][1] < len_ratio:
            return k + 1
    return len(result_clusters)


def recommend_inflation(result_stat, nchrs, len_ratio):
    """Smallest inflation whose main-group count reaches nchrs (2110-2129).  The message format is
    machine-read by `haphic pipeline`."""
    ok = sorted(infl for infl, groups in result_stat if groups >= nchrs)
    if ok:
        logger.info("You could try inflation from {} (length ratio = {})".format(ok[0], len_ratio))
        return True
    if len_ratio > 0.5:
        logger.info("The length ratio ({}) might be too strict, trying a lower one...".format(len_ratio))
        return False
    logger.info("It seems that some chromosomes were grouped together (length ratio = {}) "
                "You could check whether the parameters used are correct / appropriate and "
                "then try to tune the parameters for assembly correction, contig / Hi-C link "
                "filtration, or Markov clustering".format(len_ratio))
    return True


def mcl(engine, expansion, inflation, iters, pruning, dense_matrix=False, _done=None):
    """One inflation on the device engine; logs the reference's convergence line (2047-2060) -- from a function called
    `mcl`, because the log format carries the function name.  ``_done`` = (statistics, result) of a run that another
    GPU already made (multi-GPU sweep)."""
    if _done is None:
        st = engine.run(inflation, iters, pruning)
        result = None
    else:
        st, result = _done
    if st["converged"]:
        logger.info("The matrix has converged after {} rounds of iterations "
                    "(expansion: {}, inflation: {}, maximum iterations: {}, pruning threshold: {})".format(
                        st["rounds"], expansion, inflation, iters, pruning))
    else:
        logger.info("The matrix does not converge after {} rounds of iterations "
                    "(expansion: {}, inflation: {}, maximum iterations: {}, pruning threshold: {})".format(
                        st["rounds"], expansion, inflation, iters, pruning))
    return engine.result() if result is None else result


def _mcl_sweep_multi_gpu(link_matrix, devices, expansion, inflations, max_iter, pruning, preexp):
    """The inflation sweep (2155-2158) over several GPUs of one process: every device gets the same canonical CSC of the
    link matrix, builds M0 / M1 itself and runs the inflations k, k + N, k + 2N, ... on its own host thread (the library
    calls release the GIL).  Yields (inflation, result matrix) in sweep order, logging like the single-GPU loop."""
    import threading
    from ._lib import Context
    from .links import LinkMatrix
    from .mcl import Mcl
    host = link_matrix.to_scipy()                 # canonical (row-sorted) CSC: the same input on every device
    results = [None] * len(inflations)
    errors = []

    def worker(k, dev):
        try:
            ctx = _context() if dev == devices[0] else Context(dev)
            mat = LinkMatrix.from_csc(ctx, host)
            engine = Mcl(mat, expansion, preexp=preexp)
            for idx in range(k, len(inflations), len(devices)):
                st = engine.run(float(inflations[idx]), max_iter, pruning)
                results[idx] = (st, engine.result())
            engine.close()
            mat.close()
            if dev != devices[0]:
                ctx.close()
        except Exception as exc:                  # surfaced by the consumer below
            errors.append(exc)

    threads = [threading.Thread(target=worker, args=(k, dev), daemon=True) for k, dev in enumerate(devices)]
    for t in threads:
        t.start()
    logger.debug("Markov clustering: {} inflations over GPUs {}".format(len(inflations), devices))
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    for inflation, done in zip(inflations, results):
        yield inflation, mcl(None, expansion, float(inflation), max_iter, pruning, _done=done)


def run_mcl_clustering(link_matrix, bin_set, frag_len_dict, frag_index_dict, expansion, min_inflation,
                       max_inflation, inflation_step, max_iter, pruning, fa_dict, nchrs, dense_matrix):
    """run_mcl_clustering (2132-2242).  ``link_matrix`` is a device LinkMatrix (or anything scipy can
    turn into CSC, which is uploaded).  Writes inflation_*/ files, logs the recommendation."""
    from .links import LinkMatrix
    from .mcl import Mcl, inflation_values
    logger.info("Performing Markov clustering...")
    if not isinstance(link_matrix, LinkMatrix):
        link_matrix = LinkMatrix.from_csc(_context(), link_matrix)
    index_frag = {i: f for f, i in frag_index_dict.items()}
    # normalise + pre-expand once for the whole sweep.  --dense_matrix selects the reference's dense mode (2035 / 2149,
    # numpy.linalg.matrix_power): here the pre-expansion as a dense GEMM on the tensor cores; without the flag the
    # engine is chosen from the matrix (HH_MCL_PREEXP overrides).  Results agree within fp32 rounding either way.
    preexp = "dense" if dense_matrix else "auto"
    inflations = inflation_values(min_inflation, max_inflation, inflation_step)
    devices = _gpu_list()
    engine = None
    if len(devices) > 1 and len(inflations) > 1:
        sweep = _mcl_sweep_multi_gpu(link_matrix, devices, expansion, inflations, max_iter, pruning, preexp)
    else:
        engine = Mcl(link_matrix, expansion, preexp=preexp)
        logger.debug("Pre-expansion engine: {} ({:.1f} ms)".format(engine.preexp["mode"], engine.preexp["total_ms"]))
        sweep = ((inflation, mcl(engine, expansion, float(inflation), max_iter, pruning, dense_matrix)) for inflation in inflations)
    result_clusters_list = []
    mcl_nrounds = 0
    for inflation, result in sweep:
        mcl_nrounds += 1
        clusters = interpret_result(result)
        if not clusters:
            logger.info("Some fragments are missing / redundant, result of inflation {} will NOT be output".format(inflation))
            continue
        groups = defaultdict(lambda: [[], 0])
        bin_votes = defaultdict(dict)
        for gid, members in enumerate(clusters):
            for i in members:
                frag = index_frag[i]
                if frag in bin_set:
                    ctg = frag.rsplit("_bin", 1)[0]
                    bin_votes[ctg][gid] = bin_votes[ctg].get(gid, 0) + frag_len_dict[frag]
                else:
                    groups[gid][0].append(frag)
                    groups[gid][1] += fa_dict[frag][1]
        for ctg, votes in bin_votes.items():
            best = sorted(votes.keys(), key=lambda g: votes[g], reverse=True)[0]
            groups[best][0].append(ctg)
            groups[best][1] += fa_dict[ctg][1]
        result_clusters = sorted(tuple(groups.values()), key=lambda x: x[1], reverse=True)
        outdir = "inflation_{}".format(inflation)
        os.makedirs(outdir, exist_ok=True)
        with open("{0}/mcl_{0}.clusters.txt".format(outdir), "w") as fout:
            fout.write("#Group\tnContigs\tContigs\n")
            for k, (ctgs, glen) in enumerate(result_clusters, 1):
                ctgs.sort(key=lambda c: fa_dict[c][1], reverse=True)
                fout.write("group{}_{}bp\t{}\t{}\n".format(k, glen, len(ctgs), " ".join(ctgs)))
        for k, (ctgs, glen) in enumerate(result_clusters, 1):
            with open("{}/group{}_{}bp.txt".format(outdir, k, glen), "w") as fout:
                fout.write("#Contig\tRECounts\tLength\n")
                for ctg in ctgs:
                    fout.write("{}\t{}\t{}\n".format(ctg, fa_dict[ctg][2], fa_dict[ctg][1]))
        result_clusters_list.append((inflation, result_clusters))
    if engine is not None:
        engine.close()

    max_nclusters = max(len(rc) for _, rc in result_clusters_list)
    if max_nclusters < nchrs:
        logger.warning("The maximum number of clusters ({}) is even less than the expected number of "
                       "chromosomes ({}). You could try higher inflation.".format(max_nclusters, nchrs))
    else:
        for len_ratio in (0.75, 0.7, 0.65, 0.6, 0.55, 0.5):
            stat = [(infl, get_main_groups(rc, len_ratio)) for infl, rc in result_clusters_list]
            if recommend_inflation(stat, nchrs, len_ratio):
                break
    return result_clusters_list, mcl_nrounds


# ------------------------------------------------------------------------------------------------
# statistics for the reassignment step (2245-2478, text files; plots need matplotlib)
# ------------------------------------------------------------------------------------------------

def add_ungrouped_ctgs(fa_dict, ctg_group_dict):
    for ctg in fa_dict:
        ctg_group_dict.setdefault(ctg, "ungrouped")


def parse_link_dict(link_dict, ctg_group_dict):
    out = defaultdict(dict)
    for (ci, cj), links in link_dict.items():
        gi, gj = ctg_group_dict[ci], ctg_group_dict[cj]
        if gj != "ungrouped":
            out[ci][gj] = out[ci].get(gj, 0) + links
        if gi != "ungrouped":
            out[cj][gi] = out[cj].get(gi, 0) + links
    return out


class LinkArrays:
    """full_link_dict as the arrays the device table hands out (entry order = dict insertion order): run() keeps the
    links in this form so that no 10^7-entry Python dict is ever built; `to_dict()` gives the reference's object."""

    def __init__(self, names, key_i, key_j, values):
        self.names = names
        self.key_i = np.ascontiguousarray(key_i, dtype=np.int32)
        self.key_j = np.ascontiguousarray(key_j, dtype=np.int32)
        self.values = np.ascontiguousarray(values, dtype=np.int64)

    def __len__(self):
        return len(self.key_i)

    def directed(self):
        """(L, ctg, other): the symmetric link matrix as CSR (int64 values) and the 2 * nnz directed entries interleaved in the
        order parse_link_dict (2245-2258) visits them (first end of entry 0, second end of entry 0, first end of entry 1,
        ...); built once, shared by every inflation's statistics."""
        if getattr(self, "_directed", None) is None:
            import scipy.sparse as sp
            n = len(self.names)
            ctg = np.empty(2 * len(self.key_i), np.int32)
            oth = np.empty(2 * len(self.key_i), np.int32)
            ctg[0::2], ctg[1::2] = self.key_i, self.key_j
            oth[0::2], oth[1::2] = self.key_j, self.key_i
            L = sp.csr_matrix((np.repeat(self.values, 2), (ctg, oth)), shape=(n, n))
            self._directed = (L, ctg, oth)
        return self._directed

    def directed_device(self, dev):
        """The interleaved directed entries as int64 CUDA tensors (contig, other end, links); built once."""
        if getattr(self, "_directed_dev", None) is None or self._directed_dev[0].device != dev:
            import torch
            ki = torch.from_numpy(self.key_i).to(dev).to(torch.int64)
            kj = torch.from_numpy(self.key_j).to(dev).to(torch.int64)
            v = torch.from_numpy(self.values).to(dev)
            ctg = torch.stack([ki, kj], dim=1).reshape(-1)
            oth = torch.stack([kj, ki], dim=1).reshape(-1)
            self._directed_dev = (ctg, oth, torch.stack([v, v], dim=1).reshape(-1))
        return self._directed_dev

    def to_dict(self):
        d = defaultdict(int)
        names = self.names
        for a, b, v in zip(self.key_i.tolist(), self.key_j.tolist(), self.values.tolist()):
            d[(names[a], names[b])] = v
        return d

    def write_pickle(self, path, ht=None):
        """full_links.pkl (or HT_links.pkl when the [n, 4] HT counters are given) with the native writer."""
        from . import hicio
        from ._lib import check, load, ptr
        n = len(self.key_i)
        check(load().hh_pickle_links(os.fsencode(path), hicio.names_blob(self.names), len(self.names), ptr(self.key_i) if n else None,
                                     ptr(self.key_j) if n else None, n, ptr(self.values) if ht is None else None, None,
                                     ptr(np.ascontiguousarray(ht, dtype=np.uint32)) if ht is not None else None))


def ranked_group_links(link_dict, ctg_group_dict):
    """For every contig with links to grouped contigs: [(group, links), ...] ranked by links descending, ties in the
    order parse_link_dict (2245-2258) first meets the group -- what output_statistics sorts out of it (2373)."""
    if not isinstance(link_dict, LinkArrays):
        return {ctg: sorted(groups.items(), key=lambda x: x[1], reverse=True)
                for ctg, groups in parse_link_dict(link_dict, ctg_group_dict).items()}
    arr = _ranked_group_arrays(link_dict, ctg_group_dict)
    if arr is None:
        return {}
    return _ranked_lists(link_dict.names, *arr[1:])


def _ranked_group_arrays(link_dict, ctg_group_dict):
    """(gid, contig, group, links) of the same ranking as flat arrays ordered by (contig, rank); None when nothing is linked to
    a group.  gid[c] = group of contig c (-1 = ungrouped)."""
    names = link_dict.names
    n = len(names)
    gid = np.array([-1 if ctg_group_dict[nm] == "ungrouped" else ctg_group_dict[nm] for nm in names], dtype=np.int64)
    if len(link_dict) == 0 or gid.max() < 0:
        return None
    ng = int(gid.max()) + 1
    if _CTX is not None and os.environ.get("HAPHIC_STATS_DEVICE", "1") != "0":
        return (gid,) + tuple(_ranked_group_links_device(link_dict, gid, ng, _CTX.device))
    # links of every contig into every group = (symmetric link matrix) x (contig -> group indicator): one sparse product per
    # inflation instead of a sort of all 2 * nnz directed entries (20 sorts of 1.2e8 keys took 15 min at 50k contigs)
    import scipy.sparse as sp
    L, ctg_dir, oth_dir = link_dict.directed()
    grouped = np.nonzero(gid >= 0)[0]
    G = sp.csr_matrix((np.ones(len(grouped), np.int64), (grouped, gid[grouped])), shape=(n, ng))
    S = sp.csr_matrix(L @ G)
    S.eliminate_zeros()
    c_of = np.repeat(np.arange(n, dtype=np.int64), np.diff(S.indptr))
    g_of = S.indices.astype(np.int64)
    sums = S.data.astype(np.int64)
    # ties between groups of one contig are ranked by where parse_link_dict first meets the group, i.e. by the smallest
    # position in the interleaved list (first end of entry 0, second end of entry 0, first end of entry 1, ...).  Only the
    # contigs that have such a tie need it: their directed entries are written into a (tie rows x groups) table in DESCENDING
    # position order, so the smallest position is what remains (one pass, no sort).
    first = np.zeros(len(sums), np.int64)
    pre = np.lexsort((-sums, c_of))
    cs, ss = c_of[pre], sums[pre]
    tie = np.zeros(n, bool)
    eq = (cs[1:] == cs[:-1]) & (ss[1:] == ss[:-1])
    tie[cs[1:][eq]] = True
    if tie.any():
        nt = int(tie.sum())
        trow = np.full(n, nt, np.int64)                            # contigs without a tie share one dump row
        trow[tie] = np.arange(nt)
        g_oth = gid[oth_dir]
        key = trow[ctg_dir] * ng + np.where(g_oth >= 0, g_oth, 0)
        key[g_oth < 0] = nt * ng                                   # links to ungrouped contigs: into the dump row as well
        tab = np.full((nt + 1) * ng, -1, np.int64)
        tab[key[::-1]] = np.arange(len(key) - 1, -1, -1, dtype=np.int64)
        mine = np.nonzero(tie[c_of])[0]
        first[mine] = tab[trow[c_of[mine]] * ng + g_of[mine]]
    rank = np.lexsort((first, -sums, c_of))
    return gid, c_of[rank], g_of[rank], sums[rank]


def _ranked_lists(names, c_of, g_of, sums):
    """{contig: [(group, links), ...]} from arrays already ordered by (contig, rank)."""
    if len(c_of) == 0:
        return {}
    cuts = np.concatenate([[0], np.nonzero(np.diff(c_of))[0] + 1, [len(c_of)]])
    out = {}
    g_list, s_list = g_of.tolist(), sums.tolist()
    for k in range(len(cuts) - 1):
        lo, hi = int(cuts[k]), int(cuts[k + 1])
        out[names[int(c_of[lo])]] = list(zip(g_list[lo:hi], s_list[lo:hi]))
    return out


def _ranked_group_links_device(link_dict, gid, ng, device):
    """The same ranking with the 2 * nnz directed entries resident on the GPU (torch tensor ops as plumbing: gather, unique,
    integer index_add, scatter-min, stable sorts; integer arithmetic only, so the result is the numpy path's bit for bit).
    At 50k contigs / 5.9e7 pairs the host version needs ~10 s per inflation, this one some tens of milliseconds."""
    import torch
    dev = device if isinstance(device, torch.device) else torch.device("cuda", device)
    ctg, oth, val = link_dict.directed_device(dev)
    g = torch.from_numpy(gid).to(dev)[oth]
    idx = torch.nonzero(g >= 0).squeeze(1)                   # position in parse_link_dict's visiting order
    key = ctg[idx] * ng + g[idx]
    uk, inv = torch.unique(key, return_inverse=True)
    sums = torch.zeros(len(uk), dtype=torch.int64, device=dev).index_add_(0, inv, val[idx])
    first = torch.full((len(uk),), 1 << 62, dtype=torch.int64, device=dev).scatter_reduce_(0, inv, idx, "amin", include_self=True)
    c_of = torch.div(uk, ng, rounding_mode="floor")
    g_of = uk - c_of * ng
    o = torch.argsort(first, stable=True)
    o = o[torch.argsort(-sums[o], stable=True)]
    o = o[torch.argsort(c_of[o], stable=True)]
    return c_of[o].cpu().numpy(), g_of[o].cpu().numpy(), sums[o].cpu().numpy()


def cal_link_density(max_group, current_group, max_links, group_RE_sites, ctg_RE_sites):
    if max_group == current_group:
        return max_links / group_RE_sites
    return max_links / (group_RE_sites + ctg_RE_sites - 1)


def _best_group_statistics(fa_dict, link_dict, ctg_group, group_RE):
    """The three per-contig lists of output_statistics (2373-2400: links to the best group, link density to it, density ratio
    best / average of the others) from the ranked (contig, group, links) arrays instead of 10^7 Python tuples.  Same
    arithmetic in the same order: int / int true divisions become float64 divisions of the same integers (both correctly
    rounded), and the sum over ranked[1:] is accumulated position by position, left to right, like sum()."""
    names = link_dict.names
    arr = _ranked_group_arrays(link_dict, ctg_group)
    zero = [(ctg, 0) for ctg in fa_dict]
    if arr is None:
        return zero, list(zero), list(zero)
    gid, c_of, g_of, sums = arr
    n_groups = len(group_RE)
    RE_g = np.array([group_RE[g] for g in range(int(gid.max()) + 1)], dtype=np.int64)
    RE_c = np.array([fa_dict[nm][2] for nm in names], dtype=np.int64)
    starts = np.concatenate([[0], np.nonzero(np.diff(c_of))[0] + 1])
    seg_len = np.diff(np.concatenate([starts, [len(c_of)]]))
    seg_c = c_of[starts]
    # per-entry attributes of the entry's contig: c_of is sorted, so np.repeat over the segments replaces two random gathers
    denom = RE_g[g_of] + np.repeat(RE_c[seg_c] - 1, seg_len)              # cal_link_density: other group
    same = np.nonzero(g_of == np.repeat(gid[seg_c], seg_len))[0]          # ... the contig's own group (few entries)
    denom[same] = RE_g[g_of[same]]
    dens = sums.astype(np.float64) / denom.astype(np.float64)
    # sum(): left to right; CPython >= 3.12 adds floats with Neumaier's compensated summation (bltinmodule.c), earlier
    # versions plainly -- the statistics files hold the repr of these sums, so the same algorithm is applied here
    acc = np.zeros(len(starts), np.float64)
    comp = np.zeros(len(starts), np.float64)
    neumaier = sys.version_info >= (3, 12)
    for pos in range(1, int(seg_len.max())):
        m = np.nonzero(seg_len > pos)[0]
        x = dens[starts[m] + pos]
        f = acc[m]
        t = f + x
        if neumaier:
            comp[m] += np.where(np.abs(f) >= np.abs(x), (f - t) + x, (x - t) + f)
        acc[m] = t
    if neumaier:
        fix = (comp != 0) & np.isfinite(comp)
        acc[fix] += comp[fix]
    others = acc / (n_groups - 1) if n_groups > 1 else np.zeros(len(starts))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = dens[starts] / others
    has = {int(c): k for k, c in enumerate(c_of[starts].tolist())}
    top_links, top_dens = sums[starts].tolist(), dens[starts].tolist()
    others_l, ratio_l = others.tolist(), ratio.tolist()
    name_idx = {nm: i for i, nm in enumerate(names)}
    best_links, best_density, best_ratio = [], [], []
    for ctg in fa_dict:
        k = has.get(name_idx.get(ctg, -1))
        if k is None:
            best_links.append((ctg, 0))
            best_density.append((ctg, 0))
            best_ratio.append((ctg, 0))
            continue
        best_links.append((ctg, top_links[k]))
        best_density.append((ctg, top_dens[k]))
        best_ratio.append((ctg, ratio_l[k] if others_l[k] else 1000000))
    return best_links, best_density, best_ratio


def output_statistics(fa_dict, link_dict, result_clusters_list):
    logger.info("Making some statistics for the next HapHiC reassignment step...")
    total_n = len(fa_dict)
    total_len = sum(info[1] for info in fa_dict.values())

    def axes(sorted_list):
        n_at, len_at = OrderedDict({0: 0}), OrderedDict({0: 0})
        last = 0
        for ctg, v in sorted_list:
            if v in n_at:
                n_at[v] += 1
                len_at[v] += fa_dict[ctg][1]
            else:
                n_at[v] = n_at[last] + 1
                len_at[v] = len_at[last] + fa_dict[ctg][1]
                last = v
        x = list(n_at.keys())
        return x, [n_at[k] / total_n * 100 for k in x], [(total_len - len_at[k]) / total_len * 100 for k in x]

    def write(x, y1, y2, title, inflation):
        with open("inflation_{}/{}_statistics.txt".format(inflation, title), "w") as fout:
            fout.write("{}\tFiltered_ctg_n\tRest_ctg_len\n".format(title))
            for k, v in enumerate(x):
                fout.write(">{}\t{}\t{}\n".format(v, y1[k], y2[k]))

    re_axes = axes(sorted(((c, info[2]) for c, info in fa_dict.items()), key=lambda x: x[1]))
    try:
        import matplotlib
        matplotlib.use("Agg")
        import matplotlib.pyplot as plt
        have_plt = True
    except Exception:
        have_plt = False
        logger.warning("Module matplotlib is not correctly installed, HapHiC will NOT draw statistical plots")

    for inflation, result_clusters in result_clusters_list:
        write(*re_axes, "RE_site_threshold", inflation)
        ctg_group, group_RE = dict(), dict()
        for gid, (ctgs, _) in enumerate(result_clusters):
            group_RE[gid] = 1
            for ctg in ctgs:
                ctg_group[ctg] = gid
                group_RE[gid] += fa_dict[ctg][2] - 1
        add_ungrouped_ctgs(fa_dict, ctg_group)
        if isinstance(link_dict, LinkArrays):
            best_links, best_density, best_ratio = _best_group_statistics(fa_dict, link_dict, ctg_group, group_RE)
            group_links = None
        else:
            group_links = ranked_group_links(link_dict, ctg_group)
            best_links, best_density, best_ratio = [], [], []
        for ctg in (fa_dict if group_links is not None else ()):
            if ctg not in group_links:
                best_links.append((ctg, 0))
                best_density.append((ctg, 0))
                best_ratio.append((ctg, 0))
                continue
            ranked = group_links[ctg]
            top_group, top_links = ranked[0]
            cur = ctg_group[ctg]
            ctg_RE = fa_dict[ctg][2]
            dens = cal_link_density(top_group, cur, top_links, group_RE[top_group], ctg_RE)
            if len(group_RE) > 1:
                others = sum(cal_link_density(g, cur, l, group_RE[g], ctg_RE) for g, l in ranked[1:]) / (len(group_RE) - 1)
            else:
                others = 0
            best_links.append((ctg, top_links))
            best_density.append((ctg, dens))
            best_ratio.append((ctg, dens / others if others else 1000000))
        curves = {}
        for title, lst in (("Link_threshold", best_links), ("Link_density_threshold", best_density),
                           ("Link_density_ratio_threshold", best_ratio)):
            lst.sort(key=lambda x: x[1])
            curves[title] = axes(lst)
            write(*curves[title], title, inflation)
        if have_plt:
            fig = plt.figure(figsize=(8, 7))
            panels = ((221, re_axes, "RE site threshold", "Number of RE sites", [0, 500]),
                      (222, curves["Link_threshold"], "Hi-C link threshold", "Number of links to the best group", [0, 500]),
                      (223, curves["Link_density_threshold"], "Link density threshold", "Link density to the best group", [0, 0.001]),
                      (224, curves["Link_density_ratio_threshold"], "Link density ratio threshold",
                       "Link density ratio (best/average)", [0, 20]))
            for pos, (x, y1, y2), title, xlabel, xlim in panels:
                ax = fig.add_subplot(pos)
                ax.plot(x, y1, "b")
                ax.tick_params(axis="y", colors="b")
                ax.set_xlim(xlim)
                ax.set_ylim([0, 50])
                ax.set_ylabel("Number of contigs filtered out (%)", color="b")
                ax.set_title(title)
                ax.set_xlabel(xlabel)
                ax2 = ax.twinx()
                ax2.plot(x, y2, "r")
                ax2.tick_params(axis="y", colors="r")
                ax2.set_ylim([90, 100])
                ax2.set_ylabel("Length of remaining contigs (%)", color="r")
            fig.tight_layout(w_pad=1, h_pad=1)
            plt.savefig("inflation_{}/statistics.pdf".format(inflation))
            plt.close()


# ------------------------------------------------------------------------------------------------
# command line (2510-2735) and the run driver (2738-2959)
# ------------------------------------------------------------------------------------------------

def detect_format(args):
    table = ((".bam", "bam", "BAM"), (".pairs", "pairs", "pairs"), (".pairs.gz", "bgzipped_pairs", "bgzipped pairs"))
    for suffix, fmt, label in table:
        if args.alignments.endswith(suffix):
            args.aln_format = fmt
            logger.info("The file for Hi-C read alignments is detected as being in {} format".format(label))
            return
    raise RuntimeError("Unknown file format for Hi-C read alignments")


_FLAGS = (
    # (group, name, kwargs) -- same names, types and defaults as the reference's parser (2530-2735)
    ("input", "--aln_format", dict(choices={"bam", "pairs", "bgzipped_pairs", "auto"}, default="auto")),
    ("input", "--RE", dict(default="GATC")),
    ("input", "--quick_view", dict(default=False, action="store_true")),
    ("input", "--gfa", dict(default=None)),
    ("input", "--ul", dict(default=None)),
    ("correct", "--correct_nrounds", dict(type=int, default=0)),
    ("correct", "--correct_resolution", dict(type=int, default=500)),
    ("correct", "--median_cov_ratio", dict(type=float, default=0.2)),
    ("correct", "--region_len_ratio", dict(type=float, default=0.1)),
    ("correct", "--min_region_cutoff", dict(type=int, default=5000)),
    ("filter", "--Nx", dict(type=int, default=80)),
    ("filter", "--RE_site_cutoff", dict(type=int, default=5)),
    ("filter", "--density_lower", dict(default="0.2X")),
    ("filter", "--density_upper", dict(default="1.9X")),
    ("filter", "--read_depth_upper", dict(default="1.5X")),
    ("filter", "--topN", dict(type=int, default=10)),
    ("filter", "--rank_sum_hard_cutoff", dict(type=int, default=0)),
    ("filter", "--rank_sum_upper", dict(default="1.5X")),
    ("filter", "--remove_allelic_links", dict(type=int, default=0)),
    ("filter", "--concordance_ratio_cutoff", dict(type=float, default=0.2)),
    ("filter", "--nwindows", dict(type=int, default=50)),
    ("filter", "--remove_concentrated_links", dict(default=False, action="store_true")),
    ("filter", "--max_read_pairs", dict(type=int, default=200)),
    ("filter", "--min_read_pairs", dict(type=int, default=20)),
    ("filter", "--phasing_weight", dict(type=float, default=1.0)),
    ("ul", "--min_ul_mapq", dict(type=int, default=30)),
    ("ul", "--min_ul_alignment_length", dict(type=int, default=10000)),
    ("ul", "--max_distance_to_end", dict(type=int, default=100)),
    ("ul", "--max_overlap_ratio", dict(type=float, default=0.5)),
    ("ul", "--max_gap_len", dict(type=int, default=10000)),
    ("ul", "--min_ul_support", dict(type=int, default=2)),
    ("mcl", "--bin_size", dict(type=int, default=-1)),
    ("mcl", "--flank", dict(type=int, default=500)),
    ("mcl", "--normalize_by_nlinks", dict(default=False, action="store_true")),
    ("mcl", "--expansion", dict(type=int, default=2)),
    ("mcl", "--min_inflation", dict(type=float, default=1.1)),
    ("mcl", "--max_inflation", dict(type=float, default=3.0)),
    ("mcl", "--inflation_step", dict(type=float, default=0.1)),
    ("mcl", "--max_iter", dict(type=int, default=200)),
    ("mcl", "--pruning", dict(type=float, default=0.0001)),
    ("mcl", "--skip_clustering", dict(default=False, action="store_true")),
    ("perf", "--threads", dict(type=int, default=8)),
    ("perf", "--dense_matrix", dict(default=False, action="store_true")),
    ("log", "--verbose", dict(default=False, action="store_true")),
)

_GROUP_TITLES = {
    "input": ">>> Parameters for parsing input files and pipeline control",
    "correct": ">>> Parameters for assembly correction",
    "filter": ">>> Parameters for preprocessing (contig / Hi-C link filtration) before clustering",
    "ul": ">>> Parameters for parsing ultra-long reads",
    "mcl": ">>> Parameters for adjacency matrix construction and Markov Clustering",
    "perf": ">>> Parameters for performance",
    "log": ">>> Parameters for logging",
}


def build_parser():
    parser = argparse.ArgumentParser(prog="haphic cluster")
    groups = {k: parser.add_argument_group(t) for k, t in _GROUP_TITLES.items()}
    groups["input"].add_argument("fasta", help="draft genome in FASTA format")
    groups["input"].add_argument("alignments", help="filtered Hi-C read alignments in BAM/pairs format (DO NOT sort it by coordinate)")
    groups["input"].add_argument("nchrs", type=int, help="expected number of chromosomes")
    for group, name, kw in _FLAGS:
        kw = dict(kw)
        kw.setdefault("help", "same meaning as in `haphic cluster` of HapHiC, default: %(default)s")
        groups[group].add_argument(name, **kw)
    return parser


def parse_arguments(argv=None):
    return build_parser().parse_args(argv)


def run(args, log_file=None):
    if log_file:
        handler = logging.FileHandler(log_file, "w")
        handler.setFormatter(logging.Formatter(fmt="%(asctime)s <%(filename)s> [%(funcName)s] %(message)s",
                                               datefmt="%Y-%m-%d %H:%M:%S"))
        logger.addHandler(handler)
    start_time = time.time()
    logger.info("Program started, HapHiC version: {} (update: {})".format(__version__, __update_time__))
    logger.info("Python version: {}".format(sys.version.replace("\n", "")))
    logger.info("Command: {}".format(" ".join(sys.argv)))
    if args.verbose:
        logger.setLevel(logging.DEBUG)
    for flag in ("density_lower", "density_upper", "read_depth_upper", "rank_sum_upper"):
        check_param("--" + flag, getattr(args, flag), {"X", "x"})
    if args.dense_matrix:
        logger.info("--dense_matrix is set: the pre-expansion runs as a dense GEMM on the tensor cores (tcgen05); "
                    "the iterates are stored sparsely in either mode")
    if args.aln_format == "auto":
        detect_format(args)
    if args.correct_nrounds and args.ul:
        args.ul = None
        logger.warning("Ultra-long data are not supported now when assembly correction is enabled")
    unsupported = [("--ul", args.ul), ("--gfa", args.gfa)]
    for flag, val in unsupported:
        if val:
            raise NotImplementedError("haphic_b200: {} is not supported (out of the hot-path scope)".format(flag))
    if args.quick_view:
        args.bin_size = 0
        args.Nx = 100
        args.remove_allelic_links = 0
        args.remove_concentrated_links = False

    fa_dict = parse_fasta(args.fasta, RE=args.RE)
    pos_int_type, dist_int_type = determine_int_type(fa_dict)
    from . import hicio

    def read_alignments(names, inter_only):
        name_index = hicio.NameIndex(names)
        if args.aln_format == "bam":
            return hicio.bam_batches(args.alignments, name_index, inter_only=inter_only, logger=logger, threads=args.threads)
        return hicio.pairs_batches(args.alignments, args.aln_format, name_index, inter_only=inter_only, threads=args.threads)

    corrected = None
    if args.correct_nrounds:
        # one read of all read1 pairs serves both passes of the reference (1300-1398 and 2835-2851): the batches stay on the
        # host, the same-contig ones feed the coverage, and the remapped batches are the second pass.  alignments.bed is
        # written during this read, with the original names and coordinates, as the reference's second pass writes it.
        from . import correct
        logger.info("Parsing input {} file for contig correction...".format("BAM" if args.aln_format == "bam" else "pairs"))
        corrected, _ = correct.run_correction(_context(), fa_dict, read_alignments(list(fa_dict), False), args)
    read_depth_dict = dict()
    whitelist = set()
    args.whitelist = whitelist
    _, bin_set, bin_size, frag_len_dict, Nx_frag_set, RE_site_dict, split_ctg_set = stat_fragments(
        fa_dict, args.RE, read_depth_dict, whitelist, nchrs=args.nchrs, flank=args.flank, Nx=args.Nx, bin_size=args.bin_size)
    names = list(fa_dict.keys())
    if corrected is not None:
        alignments = corrected
    else:
        alignments = read_alignments(names, inter_only=not split_ctg_set)      # bins need the intra-contig pairs too (2849-2856)

    # Two ways through the host side.  With --remove_allelic_links / --remove_concentrated_links the link dicts are
    # edited on the host, so they are built as the reference's Python objects.  Otherwise nothing on the host needs
    # them: the links stay arrays (LinkArrays), the pickles are written natively and no 10^7-entry dict is built.
    edits_dicts = bool(args.remove_allelic_links or args.remove_concentrated_links)
    ctg_coord_dict, ctg_pair_to_frag, flank_link_dict = None, None, None
    # pairs that reach max_read_pairs are always evaluated by the reference, whatever min_read_pairs says
    _COORD_SKIP[0] = 0 if (args.verbose or args.remove_concentrated_links) else min(int(args.min_read_pairs), int(args.max_read_pairs))
    if edits_dicts:
        if split_ctg_set:
            full_link_dict, flank_link_dict, HT_link_dict, clm_dict, frag_link_dict, ctg_coord_dict, ctg_pair_to_frag = parse_alignments(
                alignments, fa_dict, args, bin_size, frag_len_dict, Nx_frag_set, split_ctg_set, pos_int_type, dist_int_type,
                build_clm=False)
            table = parse_alignments.last_table
            clm_src = parse_alignments.last_clm
            names = parse_alignments.frag_names         # the matrix lives in fragment space from here on
        else:
            full_link_dict, flank_link_dict, HT_link_dict, clm_dict, frag_link_dict, ctg_coord_dict = parse_alignments_for_ctgs(
                alignments, fa_dict, args, frag_len_dict, Nx_frag_set, pos_int_type, dist_int_type, build_clm=False)
            table = parse_alignments_for_ctgs.last_table
            clm_src = parse_alignments_for_ctgs.last_clm
        output_pickle(HT_link_dict, "HT_link_dict", "HT_links.pkl")
        del HT_link_dict, clm_dict
    else:
        logger.info("Parsing input alignments...")
        if split_ctg_set:
            st = _stream_bins(alignments, fa_dict, args, bin_size, frag_len_dict, Nx_frag_set, split_ctg_set)
        else:
            st = _stream_contigs(alignments, fa_dict, args, frag_len_dict, Nx_frag_set)
        fetched = st["table"].fetch()
        full_link_dict = LinkArrays(st["names"], fetched["key_i"], fetched["key_j"], fetched["full"])
        logger.info("Writing {} to {}...".format("HT_link_dict", "HT_links.pkl"))
        full_link_dict.write_pickle("HT_links.pkl", ht=fetched["ht"])
        del fetched
        clm_src = (st["clm_rec"], st["names"], st["ctg_len"], st["rank"])
        if split_ctg_set:
            st["table"].close()                         # full / HT links were contig-level; the rest is fragment-level
            table, names = st["ftab"], st["frag_names"]
        else:
            table = st["table"]
        totals = table.fetch_ctg()
        frag_link_dict = {names[c]: int(totals[c]) for c in np.nonzero(totals)[0].tolist()}
        del st
    if args.quick_view:
        logger.info("Program finished in {}s".format(time.time() - start_time))
        return None
    # paired_links.clm (same file as output_clm(clm_dict), from the records, native) depends on nothing below and nothing
    # below depends on it: it is written by a host thread while the GPU filters, builds the matrix and clusters
    import threading
    clm_error = []

    def _clm_job(src=clm_src):
        try:
            write_clm(*src, threads=args.threads)
        except BaseException as exc:       # re-raised by the main thread once the run is through
            clm_error.append(exc)

    clm_thread = threading.Thread(target=_clm_job, name="write_clm")
    clm_thread.start()
    del clm_src

    if args.normalize_by_nlinks and edits_dicts:
        normalize_by_nlinks(flank_link_dict, frag_link_dict)          # (the device normalises its own copy)
    if args.remove_concentrated_links:                      # 2899-2902
        for ctg_name_pair, data in ctg_coord_dict.items():
            if isinstance(data, list):
                full_link_dict[ctg_name_pair] *= data[1]
    filtered_frags = filter_fragments(
        Nx_frag_set, RE_site_dict, args.RE_site_cutoff, frag_link_dict, args.density_lower, args.density_upper,
        args.topN, args.rank_sum_upper, args.rank_sum_hard_cutoff, flank_link_dict, read_depth_dict,
        args.read_depth_upper, whitelist, device_table=table, device_names=names, normalized=args.normalize_by_nlinks)
    if args.remove_allelic_links:                           # 2910-2919
        filtered_frags = remove_allelic_HiC_links(fa_dict, ctg_coord_dict, full_link_dict, args, flank_link_dict, filtered_frags,
                                                  ctg_pair_to_frag if split_ctg_set else None)
    del ctg_coord_dict
    if isinstance(full_link_dict, LinkArrays):
        logger.info("Writing {} to {}...".format("full_link_dict", "full_links.pkl"))
        full_link_dict.write_pickle("full_links.pkl")
    else:
        output_pickle(full_link_dict, "full_link_dict", "full_links.pkl")

    if args.remove_allelic_links:
        # the host edited flank_link_dict: the matrix comes from the edited dict (hh_matrix_from_csc), same
        # first-seen indexing as the reference's dict_to_matrix
        from .links import LinkMatrix
        host_matrix, frag_index_dict = dict_to_matrix(flank_link_dict, filtered_frags, dense_matrix=False, add_self_loops=True)
        link_matrix = LinkMatrix.from_csc(_context(), host_matrix)
    else:
        # dict_to_matrix on the device: first-seen indices from the table, unlinked fragments appended in
        # the reference's set-iteration order (355-359)
        link_matrix, frag_index_dict = device_matrix(table, names, filtered_frags, normalize_by_nlinks=args.normalize_by_nlinks,
                                                     add_self_loops=True)
    table.close()
    matrix_time = time.time()
    logger.info("Hi-C linking matrix was constructed in {}s".format(matrix_time - start_time))

    if not args.skip_clustering:
        result_clusters_list, mcl_nrounds = run_mcl_clustering(
            link_matrix, bin_set, frag_len_dict, frag_index_dict, args.expansion, args.min_inflation, args.max_inflation,
            args.inflation_step, args.max_iter, args.pruning, fa_dict, args.nchrs, args.dense_matrix)
        clustering_time = time.time()
        logger.info("{} round(s) of Markov clustering finished in {}s, average {}s per round".format(
            mcl_nrounds, clustering_time - matrix_time, (clustering_time - matrix_time) / mcl_nrounds))
        output_statistics(fa_dict, full_link_dict, result_clusters_list)
    link_matrix.close()
    clm_thread.join()
    if clm_error:
        raise clm_error[0]
    logger.info("Program finished in {}s".format(time.time() - start_time))


def main():
    run(parse_arguments(), "HapHiC_cluster.log")


if __name__ == "__main__":
    main()
