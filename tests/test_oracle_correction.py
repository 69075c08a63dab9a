"""CPU checks of assembly correction: the numpy oracle (tests/correction_oracle.py) against the fixtures the unmodified
reference wrote (tests/golden/make_correction_golden.py), and the host bookkeeping of haphic_b200/correct.py driven by a
numpy stand-in of the device state that follows the same bucket / segment protocol as hh_correct."""

import argparse
import json
import os

import numpy as np
import pytest

from tests import correction_oracle as co
from tests.util import load_golden

ARGS = dict(correct_resolution=500, median_cov_ratio=0.2, region_len_ratio=0.1, min_region_cutoff=5000, RE="GATC")


def _misjoined():
    from haphic_b200 import synth
    shape = json.loads(str(load_golden("correct_rounds.npz")["shape"]))
    asm = synth.make_assembly(shape["nchr"], shape["n_contigs"], shape["mean_len"], seed=shape["seed"])
    pairs = synth.make_pairs(asm, shape["n_pairs"], seed=shape["seed"] + 1).numpy()
    return synth.make_misjoined(asm, pairs, frac=shape["frac"], seed=shape["mis_seed"]), shape


def test_oracle_detect_matches_reference():
    g = load_golden("correct_detect.npz")
    want = json.loads(str(g["breakpoints"]))
    got = {}
    off = g["cov_off"]
    for k, (name, length) in enumerate(zip(g["names"].tolist(), g["lengths"].tolist())):
        r = co.detect_one(g["cov"][off[k]:off[k + 1]], length, 500, 0.2, 0.1, 5000)
        if r:
            got[name] = [list(p) for p in r]
    assert got == want


def test_oracle_pass1_and_rounds_match_reference():
    g = load_golden("correct_rounds.npz")
    mis, _ = _misjoined()
    for nr in (1, 2, 3):
        r = co.correct(mis.pairs, mis.asm.names, mis.asm.lengths, 500, nr)
        if nr == 1:
            assert np.array_equal(r["cov"], g["cov"])
            assert np.array_equal(np.bincount(r["link_ctg"], minlength=mis.asm.n), g["link_count"])
            mine = np.stack([r["link_ctg"], r["link_lo"], r["link_hi"]], 1)
            ref_c = np.repeat(np.arange(mis.asm.n), g["link_count"])
            want = np.concatenate([ref_c[:, None], g["links"]], 1)
            assert np.array_equal(mine[np.lexsort(mine.T[::-1])], want[np.lexsort(want.T[::-1])])
        rounds = [{k: [list(p) for p in v] for k, v in rr.items()} for rr in r["rounds"]]
        assert rounds == json.loads(str(g["rounds_{}".format(nr)]))
        assert r["final_pos"] == json.loads(str(g["final_pos_{}".format(nr)]))
        assert r["final_frag"] == json.loads(str(g["final_frag_{}".format(nr)]))
        order = json.loads(str(g["order_{}".format(nr)]))
        assert r["names"] == [o[0] for o in order] and r["lengths"] == [o[1] for o in order]
        assert r["nbroken"] == int(g["nbroken_{}".format(nr)])
    assert len(g["quirk_frags"]) > 0


class HostCorrector:
    """numpy stand-in of hh_correct with the same protocol: coverage segments, a {bucket, lo, hi} link store, splits by
    bucket and shift lists.  Lets the host bookkeeping of haphic_b200.correct run without a GPU."""

    def __init__(self, rec, lengths, res):
        self.res = res
        cov, off, c, lo, hi = co.pass1(rec, lengths, res)
        self.cov, self.bin_off = cov.astype(np.int64), off
        self.links = np.stack([c, lo, hi], 1).astype(np.int64)

    def detect(self, seg_off, seg_nbins, seg_len, args):
        n_bp, bins, covs = [], [], []
        for o, n, L in zip(seg_off.tolist(), seg_nbins.tolist(), seg_len.tolist()):
            r = co.detect_one(self.cov[o:o + n].astype(np.int32), L, self.res, args.median_cov_ratio, args.region_len_ratio,
                              args.min_region_cutoff) or []
            n_bp.append(len(r))
            bins += [p // self.res for p, _ in r]
            covs += [cv for _, cv in r]
        return np.array(n_bp, np.int32), np.array(bins, np.int32), np.array(covs, np.int32)

    def split(self, frag_bucket, frag_off, frag_zero, list_off, shift_pos, piece_bucket, n_buckets):
        b, lo, hi = self.links[:, 0].copy(), self.links[:, 1].copy(), self.links[:, 2].copy()
        diff = np.zeros(len(self.cov) + 1, np.int64)
        for f, bucket in enumerate(frag_bucket):
            sel = np.nonzero(self.links[:, 0] == bucket)[0] if bucket >= 0 else np.zeros(0, np.int64)
            p = np.array(shift_pos[list_off[f]:list_off[f + 1]], np.int64)
            L, H = self.links[sel, 1], self.links[sel, 2]
            if not frag_zero[f]:
                span = (L <= p[0] + self.res) & (H >= p[0])
                np.add.at(diff, frag_off[f] + L[span] // self.res, 1)
                np.add.at(diff, frag_off[f] + H[span] // self.res + 1, -1)
                b[sel[span]] = -1
                sel, L, H = sel[~span], L[~span], H[~span]
            ni = len(p) - np.searchsorted(p[::-1], L, side="right")
            nj = len(p) - np.searchsorted(p[::-1], H, side="right")
            pb = np.array(piece_bucket[list_off[f]:list_off[f + 1]], np.int64)
            b[sel] = np.where(ni == nj, pb[ni], -1)
            lo[sel], hi[sel] = L - p[ni], H - p[nj]
        self.links = np.stack([b, lo, hi], 1)
        self.cov -= np.cumsum(diff[:-1])


def _fa_dict(mis, seq_len_only=False):
    return {n: ["A" * int(L), int(L), 1] for n, L in zip(mis.asm.names, mis.asm.lengths.tolist())}


@pytest.mark.parametrize("nrounds", [1, 2, 3])
def test_host_bookkeeping_matches_reference(tmp_path, monkeypatch, nrounds):
    from haphic_b200 import correct
    g = load_golden("correct_rounds.npz")
    mis, _ = _misjoined()
    monkeypatch.chdir(tmp_path)
    fa = _fa_dict(mis)
    args = argparse.Namespace(fasta=str(tmp_path / "in.fa"), correct_nrounds=nrounds, **ARGS)
    hc = HostCorrector(mis.pairs, mis.asm.lengths, 500)
    nb, fpos, ffrag = correct.correct_assembly(fa, hc, args)
    assert nb == int(g["nbroken_{}".format(nrounds)])
    assert fpos == json.loads(str(g["final_pos_{}".format(nrounds)]))
    assert ffrag == json.loads(str(g["final_frag_{}".format(nrounds)]))
    order = json.loads(str(g["order_{}".format(nrounds)]))
    assert [[k, v[1]] for k, v in fa.items()] == [o[:2] for o in order]
    for v in fpos.values():
        assert v == sorted(v, reverse=True)
    with open("corrected_ctgs.txt") as f:
        listed = f.read().split()
    assert listed == [k for k in fa if ":" in k]
    for name in listed:
        raw, rng = name.rsplit(":", 1)
        s, e = map(int, rng.split("-"))
        assert 1 <= s <= e and fa[name][1] == e - s + 1
    with open("corrected_asm.fa") as f:
        assert f.read().count(">") == len(fa)


def test_remap_table_matches_oracle():
    from haphic_b200 import correct
    mis, _ = _misjoined()
    r = co.correct(mis.pairs, mis.asm.names, mis.asm.lengths, 500, 2)
    fa = {n: None for n in r["names"]}
    off, start, pid = correct.piece_table(mis.asm.names, fa, r["final_pos"], r["final_frag"])
    rec = mis.pairs.astype(np.int64)
    out = rec.copy()
    for e in (0, 2):
        c, pos = rec[:, e], rec[:, e + 1]
        for i in range(mis.asm.n):
            sel = c == i
            st = start[off[i]:off[i + 1]]
            k = np.searchsorted(st, pos[sel], side="right") - 1
            out[sel, e] = pid[off[i]:off[i + 1]][k]
            out[sel, e + 1] = pos[sel] - st[k]
    assert np.array_equal(out.astype(np.int32), co.remap(mis.pairs, mis.asm.names, r))


def test_existing_output_is_renamed_and_no_break_links_input(tmp_path, monkeypatch):
    from haphic_b200 import correct
    monkeypatch.chdir(tmp_path)
    (tmp_path / "in.fa").write_text(">a\nACGT\n")
    (tmp_path / "corrected_asm.fa").write_text("old")
    args = argparse.Namespace(fasta=str(tmp_path / "in.fa"), correct_nrounds=2, **ARGS)
    rec = np.array([[0, 10, 0, 4000]], np.int32)
    hc = HostCorrector(rec, np.array([20000]), 500)
    nb, fpos, ffrag = correct.correct_assembly({"a": ["A" * 20000, 20000, 1]}, hc, args)
    assert nb == 0 and fpos == {} and ffrag == {}
    baks = [p for p in os.listdir(tmp_path) if p.startswith("corrected_asm.fa.bak.")]
    assert len(baks) == 1 and (tmp_path / baks[0]).read_text() == "old"
    assert os.path.islink(tmp_path / "corrected_asm.fa") and os.readlink(tmp_path / "corrected_asm.fa") == args.fasta
    assert (tmp_path / "corrected_ctgs.txt").read_text() == ""


def test_pos_shift_key_reproduces_relative_end():
    from haphic_b200.correct import pos_shift_key
    shift = [60000, 2000, 0]
    assert pos_shift_key("c:1001-100000", 0, shift, 99000, set()) == "c:61001-100000"
    assert pos_shift_key("c:1001-100000", 1, shift, 99000, set()) == "c:3001-60000"        # relative end (quirk)
    assert pos_shift_key("c:1001-100000", 2, shift, 99000, set()) == "c:1001-2000"
    assert pos_shift_key("c", 1, shift, 99000, {"c"}) == "c:2001-60000"
