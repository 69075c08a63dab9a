"""The UNMODIFIED reference (scripts/HapHiC_cluster.py of zengxiaofei/HapHiC) as a CPU baseline.

Test / bench infrastructure only (like everything under oracle/): nothing in haphic_b200/ imports this.

The reference is pure Python.  `install()` (called by __graft_entry__.build() where a checkout of the reference is
present) byte-compiles the two files the hot path needs -- scripts/HapHiC_cluster.py and scripts/_version.py -- into
oracle/_ref/ (git-ignored build output that stays with the built tree, so the CPU legs run where the checkout is
absent).  `load()` imports those modules with import stubs for `pysam` and `portion` (neither is in the image, neither is
touched on the .pairs path; SURVEY.md 8c) and, because Intel MKL / sparse_dot_mkl are not in the image either, with
`dot_product_mkl := lambda a, b: a @ b` (SciPy's SpGEMM standing in for MKL's) when the sparse mode is asked for --
stated wherever a number from it is reported.
"""

from __future__ import annotations

import os
import py_compile
import sys
import time
import types

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(REPO, "oracle", "_ref")
# scripts/ of a zengxiaofei/HapHiC v1.0.7 checkout
SRC_DIR = os.path.join(os.environ.get("HAPHIC_REFERENCE", "/root/reference"), "scripts")
MODULES = ("HapHiC_cluster", "_version")

_mod = None


def _built(name):
    return os.path.join(REF_DIR, name + ".pyc")


def install() -> bool:
    """Byte-compile the reference's two modules into oracle/_ref/ (no-op when the reference checkout is absent)."""
    if not os.path.isdir(SRC_DIR):
        return available()
    os.makedirs(REF_DIR, exist_ok=True)
    for name in MODULES:
        src, dst = os.path.join(SRC_DIR, name + ".py"), _built(name)
        if not os.path.exists(dst) or os.path.getmtime(dst) < os.path.getmtime(src):
            py_compile.compile(src, cfile=dst, doraise=True)
    return True


def available() -> bool:
    return all(os.path.exists(_built(name)) for name in MODULES)


def load(sparse_stand_in: bool = True):
    """Import the unmodified reference module from oracle/_ref/."""
    global _mod
    if _mod is not None:
        return _mod
    if not available():
        raise RuntimeError("the reference is not built: run __graft_entry__.build() with a HapHiC checkout at {} "
                           "(HAPHIC_REFERENCE)".format(os.path.dirname(SRC_DIR)))
    pysam = types.ModuleType("pysam")
    pysam.set_verbosity = lambda *_a, **_k: 0
    pysam.AlignmentFile = None
    portion = types.ModuleType("portion")
    portion.closed = lambda *_a, **_k: None
    portion.empty = lambda *_a, **_k: None
    sys.modules.setdefault("pysam", pysam)
    sys.modules.setdefault("portion", portion)
    sys.path.insert(0, REF_DIR)
    try:
        import HapHiC_cluster as ref          # noqa: the unmodified reference
    finally:
        sys.path.remove(REF_DIR)
    if sparse_stand_in and not getattr(ref, "INTEL_MKL", False):
        ref.INTEL_MKL = True
        ref.dot_product_mkl = lambda a, b: a @ b
    ref.logger.setLevel(100)                  # the reference logs every mcl() call; keep the bench output one JSON line
    _mod = ref
    return ref


def ref_args(**kw):
    import argparse
    d = dict(flank=500, remove_allelic_links=0, remove_concentrated_links=False, max_read_pairs=200, min_read_pairs=20,
             nwindows=50, concordance_ratio_cutoff=0.2)
    d.update(kw)
    return argparse.Namespace(**d)


def write_pairs(path, names, records):
    """.pairs text of int32 records {ctg_a, pos_a, ctg_b, pos_b} (0-based positions -> 1-based columns)."""
    with open(path, "w") as f:
        f.write("## pairs format v1.0\n#columns: readID chr1 pos1 chr2 pos2 strand1 strand2\n")
        f.write("".join("r{}\t{}\t{}\t{}\t{}\t+\t-\n".format(k, names[a], pa + 1, names[b], pb + 1)
                        for k, (a, pa, b, pb) in enumerate(records.tolist())))


def time_pair_loop(names, lengths, pairs_path, workdir):
    """Wall time of the reference's own hot loop #1 on a .pairs file:
    parse_alignments_for_ctgs(pairs_generator_inter_ctgs(...)) (HapHiC_cluster.py:1596-1655 over 1562-1583), exactly as
    run() calls it for .pairs input without bins (2862-2873).  Returns (seconds, len(full_link_dict))."""
    ref = load()
    fa_dict = {nm: [None, int(ln), 1] for nm, ln in zip(names, lengths)}
    ctg_len_dict = {nm: int(ln) for nm, ln in zip(names, lengths)}
    nx = set(names)
    cwd = os.getcwd()
    os.chdir(workdir)                      # the generator writes alignments.bed into the working directory (1549)
    try:
        t0 = time.perf_counter()
        out = ref.parse_alignments_for_ctgs(ref.pairs_generator_inter_ctgs(pairs_path, "pairs"), fa_dict, ref_args(), ctg_len_dict,
                                            nx, "int32", "int32")
        dt = time.perf_counter() - t0
    finally:
        os.chdir(cwd)
    return dt, len(out[0]), out


def time_mcl_sweep(link_csc, inflations, max_iter, pruning, dense=False, expansion=2):
    """Wall time of the reference's hot loop #2: normalize + pre-expansion (2144-2149) + mcl() per inflation (2026-2062),
    the body of run_mcl_clustering without its file output.  Returns (seconds, total iterations, per-inflation rounds)."""
    import io
    import logging
    import re
    ref = load(sparse_stand_in=not dense)
    from sklearn.preprocessing import normalize
    import numpy as np
    # iteration counts come from the reference's own log line (2047-2060)
    buf = io.StringIO()
    h = logging.StreamHandler(buf)
    old_handlers, old_prop = ref.logger.handlers[:], ref.logger.propagate
    ref.logger.handlers = [h]
    ref.logger.propagate = False
    ref.logger.setLevel(logging.INFO)
    try:
        t0 = time.perf_counter()
        m = link_csc.toarray() if dense else link_csc
        matrix = normalize(m, norm="l1", axis=0)
        if dense:
            matrix = np.linalg.matrix_power(matrix, expansion)
        else:
            matrix = ref.mkl_matrix_power(matrix, expansion)
        results = []
        for r in inflations:
            results.append(ref.mcl(matrix, expansion, float(r), max_iter, pruning, dense))
        dt = time.perf_counter() - t0
    finally:
        ref.logger.handlers = old_handlers
        ref.logger.propagate = old_prop
        ref.logger.setLevel(100)
    rounds = [int(x) for x in re.findall(r"after (\d+) rounds", buf.getvalue())]
    return dt, sum(rounds), rounds, results
