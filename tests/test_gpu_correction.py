"""GPU assembly correction (hh_correct_*, haphic_b200/correct.py), bit-exact against the fixtures the unmodified reference
wrote (tests/golden/correct_*.npz) and against the numpy oracle (tests/correction_oracle.py)."""

import argparse
import hashlib
import json
import logging
import os
import pickle
import subprocess
import sys
import time

import numpy as np
import pytest

from tests import correction_oracle as co
from tests.util import load_golden

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = dict(correct_resolution=500, median_cov_ratio=0.2, region_len_ratio=0.1, min_region_cutoff=5000, RE="GATC")
log = logging.getLogger(__name__)


@pytest.fixture(scope="module")
def ctx():
    from haphic_b200._lib import Context
    c = Context(0)
    yield c
    c.close()


def _misjoined(shape=None):
    from haphic_b200 import synth
    shape = shape or json.loads(str(load_golden("correct_rounds.npz")["shape"]))
    asm = synth.make_assembly(shape["nchr"], shape["n_contigs"], shape["mean_len"], seed=shape["seed"])
    pairs = synth.make_pairs(asm, shape["n_pairs"], seed=shape["seed"] + 1).numpy()
    if not shape["frac"]:
        return synth.Misjoined(asm, pairs, {})
    return synth.make_misjoined(asm, pairs, frac=shape["frac"], seed=shape["mis_seed"])


def _sorted_rows(a):
    a = np.asarray(a, np.int64)
    return a[np.lexsort(a.T[::-1])]


def test_pass1_coverage_and_links(ctx):
    from haphic_b200.correct import Corrector
    g = load_golden("correct_rounds.npz")
    mis = _misjoined()
    corr = Corrector(ctx, mis.asm.lengths, 500)
    half = len(mis.pairs) // 2
    corr.add(np.ascontiguousarray(mis.pairs[:half]))
    import torch
    corr.add(torch.from_numpy(np.ascontiguousarray(mis.pairs[half:])).cuda())
    cov, off, links = corr.fetch()
    corr.close()
    assert np.array_equal(cov, g["cov"])
    assert np.array_equal(off, np.concatenate([[0], np.cumsum(mis.asm.lengths // 500 + 1)]))
    ref_c = np.repeat(np.arange(mis.asm.n), g["link_count"])
    assert np.array_equal(_sorted_rows(links), _sorted_rows(np.concatenate([ref_c[:, None], g["links"]], 1)))


def test_detect_segments_hand_made_cases(ctx):
    from haphic_b200.correct import detect_segments
    g = load_golden("correct_detect.npz")
    off = g["cov_off"]
    args = argparse.Namespace(**ARGS)
    n_bp, bins, covs = detect_segments(ctx, g["cov"], 500, off[:-1], np.diff(off), g["lengths"], args)
    got, k = {}, 0
    for name, m in zip(g["names"].tolist(), n_bp.tolist()):
        if m:
            got[name] = [[int(b) * 500, int(c)] for b, c in zip(bins[k:k + m], covs[k:k + m])]
            k += m
    assert got == json.loads(str(g["breakpoints"]))


def test_detect_segments_large_random_fragments(ctx):
    """Fragments above the shared-memory staging size (global-memory select) and many tiny ones, against the oracle."""
    from haphic_b200.correct import detect_segments
    rng = np.random.default_rng(5)
    nb = [200001, 11264, 11265, 1, 2, 3] + rng.integers(1, 400, size=300).tolist()
    covs = []
    for n in nb:
        c = rng.integers(0, 60, size=n).astype(np.int32)
        c[rng.random(n) < 0.3] = 50
        covs.append(c)
    cov = np.concatenate(covs)
    off = np.concatenate([[0], np.cumsum(nb)]).astype(np.int64)
    lengths = np.array([(n - 1) * 500 + int(rng.integers(0, 500)) for n in nb], np.int64)
    args = argparse.Namespace(**dict(ARGS, min_region_cutoff=1500, region_len_ratio=0.0))
    n_bp, bins, cv = detect_segments(ctx, cov, 500, off[:-1], np.diff(off), lengths, args)
    k = 0
    for s, n in enumerate(nb):
        want = co.detect_one(covs[s], int(lengths[s]), 500, 0.2, 0.0, 1500) or []
        m = int(n_bp[s])
        assert [(int(b) * 500, int(c)) for b, c in zip(bins[k:k + m], cv[k:k + m])] == want, s
        k += m


@pytest.mark.parametrize("nrounds", [1, 2, 3])
def test_rounds_final_dicts_and_remap(ctx, tmp_path, monkeypatch, nrounds):
    from haphic_b200 import correct
    g = load_golden("correct_rounds.npz")
    mis = _misjoined()
    monkeypatch.chdir(tmp_path)
    fa = {n: ["A" * int(L), int(L), 1] for n, L in zip(mis.asm.names, mis.asm.lengths.tolist())}
    args = argparse.Namespace(fasta=str(tmp_path / "in.fa"), correct_nrounds=nrounds, **ARGS)
    rounds = []
    orig = correct.detect_break_points

    def spy(*a, **k):
        r = orig(*a, **k)
        rounds.append({kk: [list(p) for p in v] for kk, v in r.items()})
        return r

    monkeypatch.setattr(correct, "detect_break_points", spy)
    # run_correction remaps the batches in place: hand it copies
    batches, nb = correct.run_correction(ctx, fa, [b.copy() for b in np.array_split(mis.pairs, 3)], args)
    assert rounds == json.loads(str(g["rounds_{}".format(nrounds)]))
    assert nb == int(g["nbroken_{}".format(nrounds)])
    order = json.loads(str(g["order_{}".format(nrounds)]))
    assert [[k, v[1]] for k, v in fa.items()] == [o[:2] for o in order]
    r = co.correct(mis.pairs, mis.asm.names, mis.asm.lengths, 500, nrounds)
    assert np.array_equal(np.concatenate(batches), co.remap(mis.pairs, mis.asm.names, r))


DRIVER = r"""
import json, os, sys
sys.path.insert(0, {repo!r})
sys.path.insert(0, os.path.join({repo!r}, "tests", "golden"))
from haphic_b200 import cluster, synth, hicio
shape = json.loads({shape!r})
asm = synth.make_assembly(shape["nchr"], shape["n_contigs"], shape["mean_len"], seed=shape["seed"])
pairs = synth.make_pairs(asm, shape["n_pairs"], seed=shape["seed"] + 1).numpy()
mis = synth.make_misjoined(asm, pairs, frac=shape["frac"], seed=shape["mis_seed"]) if shape["frac"] else synth.Misjoined(asm, pairs, {{}})
synth.write_fasta(mis.asm, "asm.fa", seed=shape["seed"] + 3)
if {bam!r}:
    hicio.write_bam("aln.bam", mis.asm.names, mis.asm.lengths.tolist(), mis.pairs)
    aln = "aln.bam"
else:
    synth.write_pairs(mis.asm, mis.pairs, "aln.pairs")
    aln = "aln.pairs"
args = cluster.parse_arguments(["asm.fa", aln, str(shape["nchr"])] + {extra!r})
args.fasta = os.path.abspath("asm.fa")
cluster.run(args, log_file="HapHiC_cluster.log")
"""


@pytest.mark.parametrize("tag,bam", [("ctgs", False), ("ctgs", True), ("bins", False), ("bins", True), ("none", False),
                                     ("quick", False)])
def test_cluster_run_with_correction_matches_reference(tmp_path, tag, bam):
    g = load_golden("correct_run_{}.npz".format(tag))
    kw = json.loads(str(g["argkw"]))
    extra = []
    for k, v in kw.items():
        if v is True:
            extra.append("--" + k)
        else:
            extra += ["--" + k, str(v)]
    code = DRIVER.format(repo=REPO, shape=str(g["shape"]), bam=bam, extra=extra)
    env = dict(os.environ, PYTHONHASHSEED="0")
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]

    def sha(b):
        return hashlib.sha1(b).hexdigest()

    want = json.loads(str(g["files_json"]))
    got = {}
    for root, _d, files in os.walk(tmp_path):
        for fn in files:
            p = os.path.relpath(os.path.join(root, fn), tmp_path)
            if p.startswith("inflation_") and p.endswith(".txt"):
                with open(os.path.join(root, fn)) as f:
                    got[p] = f.read()
    assert sorted(got) == sorted(want)
    for p in sorted(want):
        assert got[p] == want[p], p
    with open(tmp_path / "HapHiC_cluster.log") as f:
        text = f.read()
    keep = ("[recommend_inflation]", "[mcl]", "[correct_assembly]", "[break_and_update_ctgs]")
    lines = [ln.split("] ", 1)[1] for ln in text.splitlines() if any(k in ln for k in keep)]
    assert lines == g["log_lines"].tolist()
    with open(tmp_path / "HT_links.pkl", "rb") as f:
        ht = pickle.load(f)
    assert sha(json.dumps(sorted([[a, b, int(v)] for (a, b), v in ht.items()])).encode()) == str(g["HT_links_sha1"])
    if "full_links_sha1" in g:
        with open(tmp_path / "full_links.pkl", "rb") as f:
            full = pickle.load(f)
        assert sha(json.dumps(sorted([[a, b, int(v)] for (a, b), v in full.items()])).encode()) == str(g["full_links_sha1"])
        with open(tmp_path / "paired_links.clm", "rb") as f:
            assert sha(f.read()) == str(g["clm_sha1"])
    if not bam:
        with open(tmp_path / "alignments.bed", "rb") as f:
            assert sha(f.read()) == str(g["bed_sha1"])
    assert os.path.islink(tmp_path / "corrected_asm.fa") == bool(g["asm_is_link"])
    if not bool(g["asm_is_link"]):
        with open(tmp_path / "corrected_asm.fa", "rb") as f:
            assert sha(f.read()) == str(g["asm_sha1"])
    with open(tmp_path / "corrected_ctgs.txt") as f:
        assert f.read() == str(g["corrected_ctgs"])


def c3_inputs(device="cuda"):
    """C3 shape: 50 000 contigs, 200M pairs generated on the device, about 1 % of the contigs in misjoined groups."""
    from haphic_b200 import synth
    asm = synth.make_assembly(24, 50000, 20000, seed=2024)
    pairs = synth.make_pairs(asm, 200_000_000, seed=2025, device=device)
    mis = synth.make_misjoined(asm, pairs.cpu().numpy(), frac=0.004, seed=2026)
    return mis


def test_c3_shape_breakpoints_and_remap(ctx, tmp_path, monkeypatch):
    from haphic_b200 import correct
    mis = c3_inputs()
    monkeypatch.chdir(tmp_path)
    t0 = time.time()
    r = co.correct(mis.pairs, mis.asm.names, mis.asm.lengths, 500, 2)
    want = co.remap(mis.pairs, mis.asm.names, r)
    t_oracle = time.time() - t0
    import torch
    fa = {n: ["A" * 0, int(L), 1] for n, L in zip(mis.asm.names, mis.asm.lengths.tolist())}
    args = argparse.Namespace(fasta=str(tmp_path / "in.fa"), correct_nrounds=2, **ARGS)
    rounds = []
    orig = correct.detect_break_points

    def spy(*a, **k):
        out = orig(*a, **k)
        rounds.append(out)
        return out

    monkeypatch.setattr(correct, "detect_break_points", spy)
    dev = torch.from_numpy(mis.pairs).cuda()
    t0 = time.time()
    batches, nb = correct.run_correction(ctx, fa, [dev], args)
    torch.cuda.synchronize()
    t_gpu = time.time() - t0
    assert [{k: [tuple(p) for p in v] for k, v in rr.items()} for rr in rounds] == \
        [{k: [tuple(p) for p in v] for k, v in rr.items()} for rr in r["rounds"]]
    assert list(fa) == r["names"]
    assert torch.equal(batches[0].cpu(), torch.from_numpy(want))
    # planted junctions found within 2 kb
    found = 0
    total = sum(len(v) for v in mis.junctions.values())
    for name, cuts in mis.junctions.items():
        starts = r["final_pos"].get(name, [0])
        for j in cuts:
            found += any(abs(s - j) <= 2000 for s in starts if s)
    log.warning("C3 correction: %d contigs broken, %d of %d planted junctions within 2 kb; run_correction %.1f s "
                "(host copies included), oracle %.1f s", nb, found, total, t_gpu, t_oracle)
    assert found >= 0.5 * total
