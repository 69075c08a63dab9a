"""Assembly correction (`--correct_nrounds`) of `haphic cluster`: correct_assembly / break_and_update_ctgs /
detect_break_points of scripts/HapHiC_cluster.py (v1.0.7, 943-1297).

The per-read-pair work runs on the GPU (hh_correct_* in libhaphic_b200.so): the span coverage of every intra-contig pair,
the link store, breakpoint detection, the removal of the links that span a breakpoint and the re-filing of the others, and
the remap of every record of the second pass.  The host keeps what is per breakpoint: fragment names, the
final_break_pos_dict / final_break_frag_dict of the reference, sequences and RE counts of the pieces, and the two files.
"""

from __future__ import annotations

import ctypes as C
import logging
import os
import time

import numpy as np

from . import _lib
from ._lib import check, load, ptr

logger = logging.getLogger("haphic_b200.cluster")


class Corrector:
    """Device state of one correction run (hh_correct): coverage over len // res + 1 bins per contig and the link store."""
    _close_order = 0

    def __init__(self, ctx, ctg_len, res: int):
        self.ctx = ctx
        self.res = int(res)
        self.n_ctg = len(ctg_len)
        self._h = C.c_void_p()
        self._len = np.ascontiguousarray(ctg_len, dtype=np.int64)
        check(load().hh_correct_create(ctx.handle, self.n_ctg, ptr(self._len), self.res, C.byref(self._h)))
        ctx.adopt(self)
        self.bin_off = np.concatenate([[0], np.cumsum(self._len // self.res + 1)]).astype(np.int64)

    @staticmethod
    def _records(rec):
        """(pointer owner, mem flag) of an int32 [P, 4] numpy array or torch tensor."""
        if isinstance(rec, np.ndarray):
            if rec.dtype != np.int32 or rec.ndim != 2 or rec.shape[1] != 4 or not rec.flags.c_contiguous:
                raise ValueError("records must be a C-contiguous int32 [P, 4] array")
            return rec, _lib.HH_MEM_HOST
        import torch
        if rec.dtype != torch.int32 or rec.dim() != 2 or rec.shape[1] != 4 or not rec.is_contiguous():
            raise ValueError("records must be a contiguous int32 [P, 4] tensor")
        if rec.is_cuda:
            torch.cuda.current_stream(rec.device).synchronize()
            return rec, _lib.HH_MEM_DEVICE
        return rec, _lib.HH_MEM_HOST

    def add(self, rec):
        """Pass 1 (parse_pairs_for_correction, 1300-1344): same-contig records add their span to the coverage."""
        if len(rec):
            rec, mem = self._records(rec)
            check(load().hh_correct_add(self._h, ptr(rec), len(rec), mem))

    def fetch(self):
        """(coverage int32 [n_bins], bin_off int64 [n_ctg + 1], links int32 [n_links, 3] = {bucket, lo, hi})."""
        n_bins, n_links = C.c_int64(), C.c_int64()
        check(load().hh_correct_info(self._h, C.byref(n_bins), C.byref(n_links)))
        cov = np.empty(n_bins.value, np.int32)
        off = np.empty(self.n_ctg + 1, np.int64)
        links = np.empty((n_links.value, 3), np.int32)
        check(load().hh_correct_fetch(self._h, ptr(cov), ptr(off), ptr(links)))
        return cov, off, links

    def detect(self, seg_off, seg_nbins, seg_len, args):
        """detect_break_points (943-1014) on coverage segments: (n_bp [n_seg], bp_bin, bp_cov)."""
        return _detect(lambda *a: load().hh_correct_detect(self._h, *a), seg_off, seg_nbins, seg_len, args)

    def split(self, frag_bucket, frag_off, frag_zero, list_off, shift_pos, piece_bucket, n_buckets):
        check(load().hh_correct_split(self._h, len(frag_bucket), ptr(_i32(frag_bucket)), ptr(_i64(frag_off)),
                                      ptr(np.ascontiguousarray(frag_zero, dtype=np.uint8)), ptr(_i32(list_off)),
                                      ptr(_i32(shift_pos)), ptr(_i32(piece_bucket)), int(n_buckets)))

    def set_pieces(self, piece_off, piece_start, piece_id):
        check(load().hh_correct_set_pieces(self._h, len(piece_start), ptr(_i32(piece_off)), ptr(_i32(piece_start)),
                                           ptr(_i32(piece_id))))

    def remap(self, rec):
        """Pass 2 (convert_ctg, 1405-1411): {ctg, pos} -> {piece id, pos - piece start}, in place."""
        if len(rec):
            rec, mem = self._records(rec)
            check(load().hh_correct_remap(self._h, ptr(rec), len(rec), mem))
        return rec

    def close(self):
        if self._h:
            load().hh_correct_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _detect(call, seg_off, seg_nbins, seg_len, args):
    seg_off, seg_nbins, seg_len = _i64(seg_off), _i32(seg_nbins), _i64(seg_len)
    n_seg = len(seg_off)
    cap = max(1, int(seg_nbins.astype(np.int64).sum()))
    n_bp = np.zeros(n_seg, np.int32)
    bp_bin = np.empty(cap, np.int32)
    bp_cov = np.empty(cap, np.int32)
    total = C.c_int64()
    check(call(n_seg, ptr(seg_off), ptr(seg_nbins), ptr(seg_len), float(args.median_cov_ratio), float(args.region_len_ratio),
               int(args.min_region_cutoff), ptr(n_bp), ptr(bp_bin), ptr(bp_cov), cap, C.byref(total)))
    return n_bp, bp_bin[:total.value].copy(), bp_cov[:total.value].copy()


def detect_segments(ctx, cov, res, seg_off, seg_nbins, seg_len, args):
    """hh_correct_detect_segments: detect_break_points on a caller's coverage array (no state)."""
    cov = np.ascontiguousarray(cov, dtype=np.int32)
    return _detect(lambda *a: load().hh_correct_detect_segments(ctx.handle, ptr(cov), len(cov), int(res), *a),
                   seg_off, seg_nbins, seg_len, args)


def pos_shift_key(ctg, n, pos_shift_list, ctg_len, unbroken):
    """The ctg_link_pos_dict key pos_shift (1036-1052) files a link of piece index n under.  For a fragment that starts
    after position 1 every key but the last piece's has a relative end, as in the reference; such links are lost later."""
    if ctg in unbroken:
        start, end = 1, ctg_len
    else:
        ctg, rng = ctg.rsplit(":", 1)
        start, end = [int(p) for p in rng.split("-")]
    p = pos_shift_list[n]
    if n:
        return "{}:{}-{}".format(ctg, p + start, pos_shift_list[n - 1])
    return "{}:{}-{}".format(ctg, p + start, end)


def detect_break_points(examined, fa_dict, corr, args):
    """{fragment: [(breakpoint, coverage), ...]} for the fragments under examination, in their order (943-1014)."""
    names = list(examined)
    if not names:
        return {}
    seg = np.array([examined[n] for n in names], dtype=np.int64).reshape(-1, 2)
    seg_len = np.array([fa_dict[n][1] for n in names], dtype=np.int64)
    n_bp, bp_bin, bp_cov = corr.detect(seg[:, 0], seg[:, 1], seg_len, args)
    res = args.correct_resolution
    out = {}
    k = 0
    for name, m in zip(names, n_bp.tolist()):
        if m:
            out[name] = [(int(b) * res, int(c)) for b, c in zip(bp_bin[k:k + m].tolist(), bp_cov[k:k + m].tolist())]
            k += m
    return out


def break_and_update_ctgs(ctg_break_point_dict, examined, buckets, corr, frag_source_dict, final_break_pos_dict,
                          final_break_frag_dict, fa_dict, unbroken_ctgs, args, last_round=False):
    """One round of 1017-1197.  Returns the fragments to examine in the next round: {piece: (first bin, bins)}."""
    from .cluster import count_RE_sites
    logger.info("Breaking contigs and updating data...")
    res = args.correct_resolution
    nxt = dict()
    split = ([], [], [], [0], [], [])       # frag_bucket, frag_off, frag_zero, list_off, shift_pos, piece_bucket

    def update_fa_dict(ctg, new_frag, start, end):
        new_seq = fa_dict[ctg][0][start:end]
        fa_dict[new_frag] = [new_seq, end - start, count_RE_sites(new_seq, args.RE)]       # no pseudo-count (1029)
        return end

    for ctg, break_points in ctg_break_point_dict.items():
        off, nbins = examined[ctg]
        if not last_round:
            pos_shift_list = [point for point, _cv in break_points][::-1] + [0]
            split[0].append(buckets.get(ctg, -1))
            split[1].append(off)
            split[2].append(1 if break_points[0][1] == 0 else 0)
            for n in range(len(pos_shift_list)):
                key = pos_shift_key(ctg, n, pos_shift_list, fa_dict[ctg][1], unbroken_ctgs)
                split[5].append(buckets.setdefault(key, len(buckets)))
            split[4].extend(pos_shift_list)
            split[3].append(len(split[4]))

        start = 0
        frag_source = frag_source_dict[ctg]
        father_index = final_break_frag_dict[frag_source].index(ctg)
        father_pos = final_break_pos_dict[frag_source][father_index]
        final_break_frag_dict[frag_source].pop(father_index)
        final_break_pos_dict[frag_source].pop(father_index)
        if ctg not in unbroken_ctgs:
            raw_ctg, pos_range = ctg.rsplit(":", 1)
            shift = int(pos_range.split("-")[0]) - 1
        else:
            raw_ctg, shift = ctg, 0
        last_point = 0
        for n, (point, _) in enumerate(break_points, 1):
            s = 1 if n == 1 else last_point + 1
            last_point = point
            new_frag = "{}:{}-{}".format(raw_ctg, s + shift, point + shift)
            frag_source_dict[new_frag] = frag_source
            final_break_frag_dict[frag_source].insert(father_index, new_frag)
            final_break_pos_dict[frag_source].insert(father_index, father_pos + start)
            if not last_round:
                nxt[new_frag] = (off + start // res, point // res - start // res)
            start = update_fa_dict(ctg, new_frag, start, point)
        ctg_len = fa_dict[ctg][1]
        new_frag = "{}:{}-{}".format(raw_ctg, shift + last_point + 1, shift + ctg_len)
        frag_source_dict[new_frag] = frag_source
        final_break_frag_dict[frag_source].insert(father_index, new_frag)
        final_break_pos_dict[frag_source].insert(father_index, father_pos + start)
        if not last_round:
            nxt[new_frag] = (off + start // res, nbins - start // res)
        update_fa_dict(ctg, new_frag, start, ctg_len)
        del fa_dict[ctg]

    if not last_round and split[0]:
        corr.split(split[0], split[1], split[2], split[3], split[4], split[5], len(buckets))
    return nxt


def correct_assembly(fa_dict, corr, args):
    """correct_assembly (1200-1297) on the device state of pass 1; edits fa_dict in place and writes corrected_asm.fa and
    corrected_ctgs.txt.  Returns (nbroken_ctgs, final_break_pos_dict, final_break_frag_dict)."""
    logger.info("Performing assembly correction...")
    names = list(fa_dict)
    unbroken_ctgs = set(names)
    frag_source_dict, final_break_pos_dict, final_break_frag_dict = dict(), dict(), dict()
    examined = {n: (int(corr.bin_off[i]), int(corr.bin_off[i + 1] - corr.bin_off[i])) for i, n in enumerate(names)}
    buckets = {n: i for i, n in enumerate(names)}       # ctg_link_pos_dict key -> bucket of the device link store
    nbroken_ctgs = 0
    for nround in range(args.correct_nrounds):
        ctg_break_point_dict = detect_break_points(examined, fa_dict, corr, args)
        logger.info("Correction round {}, breakpoints are detected in {} contig(s)".format(nround + 1, len(ctg_break_point_dict)))
        if nround == 0:
            nbroken_ctgs = len(ctg_break_point_dict)
        if not ctg_break_point_dict:
            break
        if nround == 0:
            for ctg in ctg_break_point_dict:
                frag_source_dict[ctg] = ctg
                final_break_pos_dict[ctg] = [0]
                final_break_frag_dict[ctg] = [ctg]
        last_round = nround + 1 == args.correct_nrounds
        examined = break_and_update_ctgs(ctg_break_point_dict, examined, buckets, corr, frag_source_dict,
                                         final_break_pos_dict, final_break_frag_dict, fa_dict, unbroken_ctgs, args, last_round)
        unbroken_ctgs -= set(ctg_break_point_dict.keys())

    # corrected_asm.fa and corrected_ctgs.txt (1264-1287), logged from this function as in the reference; an existing
    # corrected_asm.fa is renamed to .bak.{time} first
    corrected_assembly_file = "corrected_asm.fa"
    corrected_ctgs_file = "corrected_ctgs.txt"
    logger.info("Generating corrected assembly file...")
    if os.path.exists(corrected_assembly_file):
        bak_assembly_file = "{}.bak.{}".format(corrected_assembly_file, time.time())
        logger.info("File {} already exists! Rename it as {}".format(corrected_assembly_file, bak_assembly_file))
        os.rename(corrected_assembly_file, bak_assembly_file)
    if nbroken_ctgs:
        logger.info("{} contigs were broken into {} contigs. Writing corrected assembly to {}...".format(
            nbroken_ctgs, len(fa_dict) - len(unbroken_ctgs), corrected_assembly_file))
        with open(corrected_assembly_file, "w") as f:
            for ctg, ctg_info in fa_dict.items():
                f.write(">{}\n{}\n".format(ctg, ctg_info[0]))
        with open(corrected_ctgs_file, "w") as f:
            for ctg in fa_dict:
                if ctg not in unbroken_ctgs:
                    f.write(ctg + "\n")
    else:
        logger.info("No corrected contigs were found. Simply create a symbolic link of the input assembly")
        os.symlink(args.fasta, corrected_assembly_file)
        with open(corrected_ctgs_file, "w"):
            pass
    return nbroken_ctgs, final_break_pos_dict, final_break_frag_dict


def piece_table(orig_names, fa_dict, final_break_pos_dict, final_break_frag_dict):
    """(piece_off, piece_start, piece_id) of hh_correct_set_pieces: the pieces of every original contig with ascending
    starts (final_break_pos_dict is descending) and their ids in the corrected fa_dict order."""
    new_id = {n: i for i, n in enumerate(fa_dict)}
    off, start, pid = [0], [], []
    for name in orig_names:
        if name in final_break_frag_dict:
            start += final_break_pos_dict[name][::-1]
            pid += [new_id[f] for f in final_break_frag_dict[name][::-1]]
        else:
            start.append(0)
            pid.append(new_id[name])
        off.append(len(start))
    return np.array(off, np.int32), np.array(start, np.int32), np.array(pid, np.int32)


def run_correction(ctx, fa_dict, batches, args):
    """Pass 1 over the record batches (kept on the host), correction, and the pass-2 remap of the same batches.  Returns
    the batches of the second pass and the number of contigs broken in round 1."""
    names = list(fa_dict)
    corr = Corrector(ctx, np.array([fa_dict[n][1] for n in names], np.int64), args.correct_resolution)
    try:
        kept = []
        for rec in batches:
            corr.add(rec)
            kept.append(rec)
        nbroken, final_pos, final_frag = correct_assembly(fa_dict, corr, args)
        if nbroken:
            corr.set_pieces(*piece_table(names, fa_dict, final_pos, final_frag))
            for rec in kept:
                corr.remap(rec)
    finally:
        corr.close()
    return kept, nbroken
