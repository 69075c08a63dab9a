#!/usr/bin/env python3
"""Generate the assembly-correction fixtures (tests/golden/correct_*.npz) by running the REFERENCE's own code.

Build container only (needs the reference checkout):

    python tests/golden/make_correction_golden.py

``portion`` (interval arithmetic used by detect_break_points / break_and_update_ctgs) is not installed, so a faithful
stand-in for the part of its API the reference uses is installed under that name (closed / empty, `|` merging touching
closed intervals, `-` leaving open intervals, overlaps, lower / upper, iteration and len); META.json records it.
``pysam`` is stubbed as in make_golden.py (the .pairs path never touches it).
"""

import json
import os
import sys
import tempfile
import types

if os.environ.get("PYTHONHASHSEED") != "0":
    os.environ["PYTHONHASHSEED"] = "0"
    os.execv(sys.executable, [sys.executable] + sys.argv)

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference/scripts"
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402

INF = float("inf")


class Interval:
    """Union of disjoint atomic intervals (lo, hi, lo_closed, hi_closed), kept sorted and merged like portion does."""

    def __init__(self, atoms=()):
        self.atoms = self._merge([a for a in atoms if self._nonempty(a)])

    @staticmethod
    def _nonempty(a):
        return a[0] < a[1] or (a[0] == a[1] and a[2] and a[3])

    @staticmethod
    def _merge(atoms):
        out = []
        for a in sorted(atoms, key=lambda a: (a[0], not a[2])):
            if out:
                b = out[-1]
                if a[0] < b[1] or (a[0] == b[1] and (a[2] or b[3])):
                    if a[1] > b[1] or (a[1] == b[1] and a[3]):
                        out[-1] = (b[0], a[1], b[2], a[3])
                    continue
            out.append(a)
        return out

    @property
    def lower(self):
        return self.atoms[0][0] if self.atoms else INF

    @property
    def upper(self):
        return self.atoms[-1][1] if self.atoms else -INF

    def __or__(self, other):
        return Interval(self.atoms + other.atoms)

    def __sub__(self, other):
        parts = list(self.atoms)
        for b in other.atoms:
            nxt = []
            for a in parts:
                if not self._intersect(a, b):
                    nxt.append(a)
                    continue
                left = (a[0], b[0], a[2], not b[2])
                right = (b[1], a[1], not b[3], a[3])
                if b[0] > a[0] or (b[0] == a[0] and a[2] and not b[2]):
                    nxt.append(left)
                if b[1] < a[1] or (b[1] == a[1] and a[3] and not b[3]):
                    nxt.append(right)
            parts = [p for p in nxt if self._nonempty(p)]
        return Interval(parts)

    @staticmethod
    def _intersect(a, b):
        if a[0] > b[0]:
            lo, lc = a[0], a[2]
        elif a[0] < b[0]:
            lo, lc = b[0], b[2]
        else:
            lo, lc = a[0], a[2] and b[2]
        if a[1] < b[1]:
            hi, hc = a[1], a[3]
        elif a[1] > b[1]:
            hi, hc = b[1], b[3]
        else:
            hi, hc = a[1], a[3] and b[3]
        return lo < hi or (lo == hi and lc and hc)

    def overlaps(self, other):
        return any(self._intersect(a, b) for a in self.atoms for b in other.atoms)

    def __iter__(self):
        return iter([Interval([a]) for a in self.atoms])

    def __len__(self):
        return len(self.atoms)


def import_reference():
    pysam = types.ModuleType("pysam")
    pysam.set_verbosity = lambda *_a, **_k: 0
    pysam.AlignmentFile = None
    portion = types.ModuleType("portion")
    portion.closed = lambda lo, hi: Interval([(lo, hi, True, True)])
    portion.empty = lambda: Interval()
    sys.modules["pysam"] = pysam
    sys.modules["portion"] = portion
    sys.path.insert(0, REF)
    import HapHiC_cluster as ref
    return ref


def self_check():
    """The stand-in on the cases the reference relies on."""
    c, e = sys.modules["portion"].closed, sys.modules["portion"].empty
    u = e() | c(0, 500) | c(500, 1000) | c(1500, 2000)
    assert [(a[0], a[1]) for a in u.atoms] == [(0, 1000), (1500, 2000)] and len(u) == 2
    v = c(u.lower, u.upper) - u
    assert v.atoms == [(1000, 1500, False, False)]
    assert c(999, 1000).overlaps(c(1000, 1500)) and not c(0, 999).overlaps(c(1000, 1500))
    assert [(i.lower, i.upper) for i in u] == [(0, 1000), (1500, 2000)]
    assert len(e()) == 0


def detect_cases():
    """Hand-made coverage arrays: (name, length, cov) with res = 500 and the reference defaults."""
    R = 500
    cases = []

    def add(name, length, cov):
        cov = np.asarray(cov, np.int32)
        assert len(cov) == length // R + 1, name
        cases.append((name, length, cov))

    hi = [30] * 12
    add("odd_bins", 24 * R + 7, hi + [3, 2, 4, 2, 5] + hi[:7] + [0][:0] + [9])           # 25 bins
    add("even_bins", 25 * R + 1, hi + [3, 2, 4, 2] + hi[:9] + [30])                       # 26 bins
    add("median_zero", 20 * R + 3, [0] * 12 + [40] * 9)
    add("single_run", 20 * R + 3, [1] * 5 + [30] * 16)
    add("short_run", 30 * R + 3, [30] * 12 + [1] * 4 + [30] * 3 + [1] * 2 + [30] * 10)
    add("valley_with_short_high", 40 * R + 3, [30] * 12 + [2, 1, 30, 30, 3, 2] + [30] * 23)
    add("zero_valleys", 51 * R + 3, [30] * 12 + [2, 0, 1] + [30] * 12 + [0, 0, 5] + [30] * 12 + [3, 1] + [30] * 8)
    add("argmin_tie", 40 * R + 3, [30] * 12 + [4, 2, 3, 2, 5] + [30] * 12 + [6, 2, 2] + [30] * 9)
    add("valley_tie", 40 * R + 3, [30] * 12 + [4, 1, 3] + [30] * 12 + [1, 5] + [30] * 12)
    add("partial_last_bin", 30 * R + 499, [30] * 12 + [1, 2] + [30] * 17)
    add("len_multiple_of_res", 30 * R, [30] * 12 + [1, 3] + [30] * 16 + [0])
    add("long_fragment", 400 * R + 3, [20] * 150 + [2] * 30 + [20] * 100 + [0, 1] + [20] * 119)
    return cases


def run_detect(ref, make_args):
    args = make_args()
    cases = detect_cases()
    fa = {n: [None, L, 0] for n, L, _ in cases}
    got = ref.detect_break_points({n: cov for n, _L, cov in cases}, fa, args)
    out = {"names": np.array([n for n, _, _ in cases]), "lengths": np.array([L for _, L, _ in cases], np.int64),
           "cov_off": np.concatenate([[0], np.cumsum([len(c) for _, _, c in cases])]).astype(np.int64),
           "cov": np.concatenate([c for _, _, c in cases]).astype(np.int32),
           "breakpoints": np.array(json.dumps({k: [list(map(int, p)) for p in v] for k, v in got.items()}))}
    assert any(v[0][1] == 0 and len(v) > 1 for v in got.values()) and any(v[0][1] != 0 for v in got.values())
    np.savez_compressed(os.path.join(HERE, "correct_detect.npz"), **out)
    print("correct_detect:", {k: v for k, v in got.items()})


MIS = dict(nchr=4, n_contigs=200, mean_len=40000, n_pairs=80000, seed=303, frac=0.05, mis_seed=9)


def misjoined_inputs(tmp, shape=MIS):
    from haphic_b200 import synth
    asm = synth.make_assembly(shape["nchr"], shape["n_contigs"], shape["mean_len"], seed=shape["seed"])
    pairs = synth.make_pairs(asm, shape["n_pairs"], seed=shape["seed"] + 1).numpy()
    if shape["frac"]:
        mis = synth.make_misjoined(asm, pairs, frac=shape["frac"], seed=shape["mis_seed"])
    else:
        mis = synth.Misjoined(asm, pairs, {})
    synth.write_fasta(mis.asm, os.path.join(tmp, "asm.fa"), seed=shape["seed"] + 3)
    synth.write_pairs(mis.asm, mis.pairs, os.path.join(tmp, "aln.pairs"))
    return mis


def run_rounds(ref, make_args):
    """parse_pairs_for_correction + correct_assembly for 1, 2 and 3 rounds on a C1-shaped misjoined assembly."""
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        cwd = os.getcwd()
        os.chdir(tmp)
        try:
            mis = misjoined_inputs(tmp)
            names = mis.asm.names
            for nr in (1, 2, 3):
                args = make_args(fasta=os.path.join(tmp, "asm.fa"), alignments=os.path.join(tmp, "aln.pairs"),
                                 aln_format="pairs", correct_nrounds=nr)
                fa_dict = ref.parse_fasta(args.fasta, RE=args.RE)
                cov, links = ref.parse_pairs_for_correction(fa_dict, args)
                if nr == 1:
                    out["cov"] = np.concatenate([cov[n] for n in names]).astype(np.int32)
                    out["link_count"] = np.array([len(links[n]) // 2 for n in names], np.int64)
                    out["links"] = np.concatenate([np.asarray(links[n], np.int64) for n in names]).reshape(-1, 2)
                rounds = []
                orig = ref.detect_break_points

                def rec_detect(*a, **k):
                    r = orig(*a, **k)
                    rounds.append({kk: [list(map(int, p)) for p in v] for kk, v in r.items()})
                    return r

                ref.detect_break_points = rec_detect
                try:
                    nb, fpos, ffrag = ref.correct_assembly(cov, links, fa_dict, dict(), args)
                finally:
                    ref.detect_break_points = orig
                os.remove("corrected_asm.fa")
                out["rounds_{}".format(nr)] = np.array(json.dumps(rounds))
                out["final_pos_{}".format(nr)] = np.array(json.dumps(fpos, default=int))
                out["final_frag_{}".format(nr)] = np.array(json.dumps(ffrag))
                out["order_{}".format(nr)] = np.array(json.dumps([[k, v[1], v[2]] for k, v in fa_dict.items()], default=int))
                out["nbroken_{}".format(nr)] = np.int64(nb)
                if nr == 3:
                    # the pos_shift key quirk: a fragment with start > 1 broken in round 2 files links under relative-end keys
                    quirk = [f for f in rounds[1] if ":" in f and int(f.rsplit(":", 1)[1].split("-")[0]) > 1]
                    assert quirk and len(rounds) == 3, rounds
                    out["quirk_frags"] = np.array(quirk)
            zero = any(p[1] == 0 for r in json.loads(str(out["rounds_3"])) for v in r.values() for p in v)
            nonzero = any(p[1] != 0 for r in json.loads(str(out["rounds_3"])) for v in r.values() for p in v)
            assert zero and nonzero
            out["shape"] = np.array(json.dumps(MIS))
        finally:
            os.chdir(cwd)
    np.savez_compressed(os.path.join(HERE, "correct_rounds.npz"), **out)
    print("correct_rounds:", [len(r) for r in json.loads(str(out["rounds_3"]))])


def run_whole(ref, make_args, tag, shape, **argkw):
    import hashlib
    import pickle
    out = {}

    def sha(b):
        return hashlib.sha1(b).hexdigest()

    with tempfile.TemporaryDirectory() as tmp:
        cwd = os.getcwd()
        os.chdir(tmp)
        try:
            misjoined_inputs(tmp, shape)
            args = make_args(fasta=os.path.join(tmp, "asm.fa"), alignments=os.path.join(tmp, "aln.pairs"),
                             nchrs=shape["nchr"], **argkw)
            ref.INTEL_MKL = True
            ref.dot_product_mkl = lambda a, b: a @ b
            ref.run(args, log_file="HapHiC_cluster.log")
            files = {}
            for root, _dirs, fnames in os.walk("."):
                for fn in fnames:
                    p = os.path.join(root, fn)[2:]
                    if p.endswith(".txt") and p.startswith("inflation_"):
                        with open(p) as f:
                            files[p] = f.read()
            with open("HapHiC_cluster.log") as f:
                log = f.read()
            keep = ("[recommend_inflation]", "[mcl]", "[correct_assembly]", "[break_and_update_ctgs]")
            out["log_lines"] = np.array([ln.split("] ", 1)[1] for ln in log.splitlines() if any(k in ln for k in keep)])
            with open("HT_links.pkl", "rb") as f:
                HT = pickle.load(f)
            out["HT_links_sha1"] = np.array(sha(json.dumps(sorted([[a, b, int(v)] for (a, b), v in HT.items()])).encode()))
            if not args.quick_view:
                with open("full_links.pkl", "rb") as f:
                    full = pickle.load(f)
                out["full_links_sha1"] = np.array(sha(json.dumps(sorted([[a, b, int(v)] for (a, b), v in full.items()])).encode()))
                with open("paired_links.clm", "rb") as f:
                    out["clm_sha1"] = np.array(sha(f.read()))
            with open("alignments.bed", "rb") as f:
                out["bed_sha1"] = np.array(sha(f.read()))
            out["asm_is_link"] = np.array(os.path.islink("corrected_asm.fa"))
            with open("corrected_asm.fa", "rb") as f:
                out["asm_sha1"] = np.array(sha(f.read()))
            with open("corrected_ctgs.txt") as f:
                out["corrected_ctgs"] = np.array(f.read())
            out["files_json"] = np.array(json.dumps(files, sort_keys=True))
            out["argkw"] = np.array(json.dumps(argkw, sort_keys=True))
            out["shape"] = np.array(json.dumps(shape))
        finally:
            os.chdir(cwd)
    np.savez_compressed(os.path.join(HERE, "correct_run_{}.npz".format(tag)), **out)
    print("correct_run_{}: {} files, {}".format(tag, len(files), out["log_lines"].tolist()[:4]))


def main():
    from make_golden import make_args
    ref = import_reference()
    self_check()
    only = set(sys.argv[1:])

    def want(g):
        return not only or g in only

    if want("detect"):
        run_detect(ref, make_args)
    if want("rounds"):
        run_rounds(ref, make_args)
    if want("run"):
        common = dict(Nx=100, min_inflation=1.4, max_inflation=2.2, inflation_step=0.4)
        run_whole(ref, make_args, "ctgs", MIS, correct_nrounds=2, bin_size=0, **common)
        run_whole(ref, make_args, "bins", dict(MIS, n_contigs=60, mean_len=150000, n_pairs=120000, seed=505),
                  correct_nrounds=2, bin_size=100, flank=60, **common)
        run_whole(ref, make_args, "none", dict(MIS, frac=0.0), correct_nrounds=2, bin_size=0, **common)
        run_whole(ref, make_args, "quick", MIS, correct_nrounds=1, quick_view=True, **common)
    meta = {"portion_stand_in": "tests/golden/make_correction_golden.py Interval: closed/empty, | (merges touching closed "
                                "intervals), - (open remainders), overlaps, lower/upper, iteration, len",
            "reference": "zengxiaofei/HapHiC scripts/HapHiC_cluster.py (v1.0.7), imported unmodified",
            "PYTHONHASHSEED": "0"}
    with open(os.path.join(HERE, "META_correction.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
