#!/usr/bin/env python3
"""bench.py -- the `haphic cluster` hot path on B200: Hi-C pairs/sec through the link-matrix build
and MCL iterations/sec, on the synthetic 50k-contig / 200M-pair workload (BASELINE.json configs[2]).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                          # the UNMODIFIED reference (oracle/_ref) on the host cores
    python bench.py --dump-outputs DIR [...]                        # also write the last timed step's outputs as DIR/*.npy

One "step" = one pass of the hot path over the whole synthetic input:
    link counting (200M records) -> first-seen index -> symmetric CSC -> column normalise ->
    pre-expansion M0.M0 -> Markov-cluster sweep over `--inflations`.
`value` = pairs/s through the matrix build with the records already resident in HBM (CUDA events on
the library's stream); `mcl.value` = MCL iterations/s over the sweep (normalise + pre-expansion +
all iterations, the reference's own definition, HapHiC_cluster.py:2951-2953); `e2e` = the same
quantities through the public host API with HOST (pinned) buffers, H2D and D2H inside the timed
region.  Rank 0 prints ONE JSON line.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np

REF_MISSING = "the unmodified reference is not built into oracle/_ref (__graft_entry__.build() with a HapHiC checkout)"


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", choices=["b200", "reference"], default="b200")
    p.add_argument("--contigs", type=int, default=50000)
    p.add_argument("--pairs", type=int, default=200_000_000)
    p.add_argument("--nchr", type=int, default=24)
    p.add_argument("--mean-len", type=int, default=20000)
    p.add_argument("--inflations", default="1.5,2.0,3.0")
    p.add_argument("--max-iter", type=int, default=200)
    p.add_argument("--pruning", type=float, default=1e-4)
    p.add_argument("--seed", type=int, default=12345)
    p.add_argument("--e2e-steps", type=int, default=3)
    p.add_argument("--cpu-sample-pairs", type=int, default=1_500_000)
    p.add_argument("--cpu-sample-cols", type=int, default=24)
    p.add_argument("--ingest-lines", type=int, default=1_000_000,
                   help="lines of .pairs text for the host ingest measurement (0 = skip)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-default-sweep", action="store_true", help="skip the 20-inflation default sweep figure")
    p.add_argument("--verbose", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write what the last timed step computed as DIR/<name>.npy (float64, seeded samples of the large "
                        "arrays, at most 64 MB in all), so that two builds can be compared output for output")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "b200":
        p.error("--dump-outputs applies to --impl b200")
    return a


def workload_name(a):
    return "{}k contigs / {}M pairs synthetic (nchr={}, mean_len={}, Nx=100, bin_size=0)".format(
        a.contigs // 1000, a.pairs // 1_000_000, a.nchr, a.mean_len)


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s: the sustained figure (the GEMM is timed inside a long step, under the power cap)."""
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return float(d["bf16_tflops_sustained"]), float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json: sustained / burst)"
    except Exception:
        return 1400.0, 1590.0, "fallback (B200_PROFILING.md)"


def preexp_roofline(pre, n, nnz_m0, ncols, traffic):
    """Roofline of the pre-expansion launch, the dominant kernel of the step.
    dense engine (hh_k_syrk, tcgen05): tensor bound.  achieved = 16-bit tensor flops the launch issues (2 * 256 * 256 * 64 per
    tile k-block and pass) / its CUDA-event time (summed over the K chunks when the K range is cut); the algorithmic figure of
    SURVEY.md 8(d) (2 b^3 for the block product, fp32 accuracy needing `passes` 16-bit passes) is reported beside it -- the
    symmetric half is skipped, so issued = passes * b^3.
    sparse engine (hh_k_col<SRC_PRODUCT,EPI_DUMP>): HBM bound, operand once + dense result once."""
    peak_hbm, src_hbm = measured_peaks()
    if pre["mode"] == "dense":
        sus, burst, src = measured_tensor_peak()
        ach = pre["flops"] / (pre["gemm_ms"] / 1000.0) / 1e12
        alg = 2.0 * float(n) * float(n) * float(ncols)
        return {"kernel": "hh_k_syrk<cta_group::{}> (tcgen05.mma + TMA + TMEM; pre-expansion M0*M0 -> dense M1, one launch per step)"
                .format(pre["cta_group"]), "bound": "tensor", "achieved": ach, "peak": sus, "unit": "TFLOP/s", "frac": ach / sus,
                "peak_burst": burst, "traffic": traffic.get("hh_k_syrk"), "issued_flops": pre["flops"], "passes": pre["passes"],
                "algorithmic_flops": alg, "algorithmic_frac_8d": alg / (pre["gemm_ms"] / 1000.0) / (sus * 1e12 / pre["passes"]),
                "launch_ms": pre["gemm_ms"], "densify_ms": pre["densify_ms"], "clip_correction_ms": pre["clip_ms"],
                "k_chunks": pre.get("k_chunks", 1),
                "peak_source": src, "note": "algorithmic_frac_8d = 2 n^2 ncols / t / (peak / passes); above 1 because S = C D C is "
                "symmetric and only tiles on or above the diagonal are computed.  frac can exceed 1: `peak` is the measured cuBLAS "
                "bf16 figure on dense data under the power cap, these operand planes are ~95 % zeros (the nominal dense peak is "
                "2250 TFLOP/s)"}
    alg = 8 * nnz_m0 + 4 * n * ncols
    ach = alg / (pre["total_ms"] / 1000.0) / 1e9
    return {"kernel": "hh_k_col<SRC_PRODUCT,EPI_DUMP> (pre-expansion M0*M0 -> dense M1, one launch per step)", "bound": "hbm",
            "achieved": ach, "peak": peak_hbm, "unit": "GB/s", "frac": ach / peak_hbm, "traffic": traffic.get("hh_k_col_preexpansion"),
            "algorithmic_bytes": alg, "launch_ms": pre["total_ms"], "peak_source": src_hbm,
            "gather_GBps": 8.0 * pre["products"] / (pre["total_ms"] / 1000.0) / 1e9}


def cpu_baseline_block(a, asm, rank, in_nx, rec):
    """CPU legs on this box's host cores, bounded samples of the same stream: the unmodified reference's pair loop
    (kind "reference"), and beside it the single-core C port of the same loop (oracle/haphic_oracle.c)."""
    import tempfile
    from oracle import refimpl
    if refimpl.available():
        n_ref = min(int(rec.shape[0]), a.cpu_sample_pairs)
        sample = rec[:n_ref].cpu().numpy()
        with tempfile.TemporaryDirectory() as tmp:
            v, dt, nnz = ref_pairs_per_sec(asm, sample, tmp)
        cpu = {"value": v, "unit": "pairs/s", "cores": 1, "kind": "reference",
               "sample": "first {} records as .pairs text through the unmodified HapHiC_cluster.parse_alignments_for_ctgs("
                         "pairs_generator_inter_ctgs(...)) from oracle/_ref, {:.1f} s (single-threaded Python by construction; "
                         "host has {} cores)".format(len(sample), dt, os.cpu_count())}
    else:
        cpu = {"unavailable": REF_MISSING}
    try:
        big = rec[: 8_000_000].cpu().numpy()
        vc, dtc = cpu_c_pairs_per_sec(asm, rank, in_nx, big)
        cpu["c_port"] = {"value": vc, "unit": "pairs/s", "cores": 1, "kind": "port",
                         "sample": "first {} records through oracle/haphic_oracle.c, warm call {:.1f} s (single-core C port of the "
                                   "same loop, not the reference's speed)".format(len(big), dtc)}
    except Exception as exc:                       # no gcc on the box: the reference number above stands
        cpu["c_port"] = {"unavailable": str(exc)[:200]}
    return cpu


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.proc = None
        self.device = device

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            cols = [c.strip() for c in line.split(",")]
            if len(cols) < 6:
                continue
            try:
                sm.append(float(cols[0]))
                mx = float(cols[1])
            except ValueError:
                continue
            for nm, c in zip(names, cols[2:6]):
                if c.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU port of the reference path (oracle) -- the `--impl reference` arm and the cpu_baseline leg
# --------------------------------------------------------------------------------------------------

def cpu_pairs_per_sec(asm, rank, in_nx, sample):
    """The reference's per-read-pair Python loop (HapHiC_cluster.py:1622-1653) restated in
    oracle/haphic_oracle.py, single thread by construction, on a bounded sample of the stream."""
    from oracle import haphic_oracle as orc
    t0 = time.perf_counter()
    orc.count_links_loop(sample, asm.lengths, rank, in_nx, 500000)
    dt = time.perf_counter() - t0
    return len(sample) / dt, dt


def ref_pairs_per_sec(asm, sample, tmp):
    """The reference's OWN per-read-pair loop, unmodified (oracle/_ref/HapHiC_cluster imported by oracle/refimpl.py):
    parse_alignments_for_ctgs over pairs_generator_inter_ctgs on a .pairs text of the sample (1562-1583, 1596-1655),
    single-threaded by construction.  Returns (pairs/s, seconds, distinct pairs)."""
    from oracle import refimpl
    path = os.path.join(tmp, "sample_{}.pairs".format(len(sample)))
    if not os.path.exists(path):
        refimpl.write_pairs(path, asm.names, sample)
    dt, nnz, _ = refimpl.time_pair_loop(asm.names, asm.lengths, path, tmp)
    return len(sample) / dt, dt, nnz


def ref_mcl_small(a, inflations):
    """The reference's own normalize + pre-expansion + mcl() (2144-2149, 2026-2062) on a 2,000-contig instance of the same
    generator (the 50k-contig problem is hours of CPU and a 10 GB dense intermediate): iterations/s in the reference's sparse
    mode (SciPy '@' standing in for the absent Intel MKL) and in its dense mode (what it falls back to without MKL, 2764-2766)."""
    from haphic_b200 import synth
    from haphic_b200.links import name_rank
    from oracle import haphic_oracle as orc
    from oracle import refimpl
    small = synth.make_assembly(max(2, a.nchr // 8), 2000, a.mean_len, seed=a.seed)
    sp_pairs = synth.make_pairs(small, min(a.pairs // max(1, a.contigs // 2000), 2_000_000), seed=a.seed + 1).numpy()
    r = orc.count_links_numpy(sp_pairs, small.lengths, name_rank(small.names), np.ones(small.n, np.uint8), 500000)
    m, _ = orc.dict_to_matrix(r["flank_keys"], r["flank_vals"], np.ones(small.n, np.uint8))
    out = {}
    for tag, dense in (("sparse", False), ("dense", True)):
        dt, iters, rounds, _ = refimpl.time_mcl_sweep(m, inflations, a.max_iter, a.pruning, dense=dense)
        out[tag] = {"value": iters / dt, "unit": "iter/s", "iterations": iters, "rounds": rounds, "seconds": round(dt, 2)}
    out["sample"] = ("unmodified reference normalize + matrix power + mcl() over inflations {} on a 2,000-contig / {}-pair instance "
                     "of the same generator; sparse = SciPy '@' standing in for MKL's SpGEMM, dense = numpy matrix_power".format(
                         inflations, len(sp_pairs)))
    out["kind"] = "reference"
    out["host_cores"] = os.cpu_count()
    return out


def cpu_c_pairs_per_sec(asm, rank, in_nx, sample):
    """The same loop as a single-core C port (oracle/haphic_oracle.c: hash table, entries in first-seen order,
    software-prefetched): what an optimised CPU implementation of the counting step does.  Second of two calls (the
    first one pays the page faults of the fresh buffers)."""
    from oracle import haphic_oracle as orc
    dt = None
    for _ in range(2):
        t0 = time.perf_counter()
        orc.count_links_c(sample, asm.lengths, rank, in_nx, 500000)
        dt = time.perf_counter() - t0
    return len(sample) / dt, dt


def cpu_mcl_iter_per_sec(m_csc, n_cols, inflation, pruning, seed=0):
    """One MCL iteration (expand -> inflate -> normalise -> prune, HapHiC_cluster.py:2029-2042) of the CPU
    port (scipy SpGEMM standing in for MKL) on a random sample of columns of the given iterate;
    the full-iteration time is the sample time scaled by n / n_cols (every step is column-local)."""
    from oracle import haphic_oracle as orc
    n = m_csc.shape[0]
    rng = np.random.default_rng(seed)
    # size the sample for ~4e9 Gustavson products (about ten seconds of scipy SpGEMM)
    per_col = max(1.0, (m_csc.nnz / n) ** 2)
    n_cols = int(min(n, max(n_cols, 4e9 / per_col)))
    cols = np.sort(rng.choice(n, size=min(n_cols, n), replace=False))
    sub = m_csc[:, cols]
    t0 = time.perf_counter()
    prod = (m_csc @ sub).tocsc()
    prod = orc.inflate(prod, inflation)
    orc.prune(prod, pruning)
    dt = time.perf_counter() - t0
    full = dt * n / len(cols)
    return 1.0 / full, dt, len(cols)


def ingest_rate(asm, sample, threads=0):
    """Host side of the file -> records path (SURVEY.md 8d reports it beside the device numbers): the native
    threaded tokenizer (hh_pairs_*) on a .pairs text of the sample, with the alignments.bed side product."""
    import tempfile
    from haphic_b200 import hicio
    names = asm.names
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "sample.pairs")
        with open(path, "w") as f:
            f.write("## pairs format v1.0\n#columns: readID chr1 pos1 chr2 pos2 strand1 strand2\n")
            f.write("".join("r{}\t{}\t{}\t{}\t{}\t+\t-\n".format(k, names[a], pa + 1, names[b], pb + 1)
                            for k, (a, pa, b, pb) in enumerate(sample.tolist())))
        size = os.path.getsize(path)
        idx = hicio.NameIndex(names)
        out = {}
        for tag, bed in (("with_bed", os.path.join(tmp, "alignments.bed")), ("without_bed", None)):
            t0 = time.perf_counter()
            n = sum(len(b) for b in hicio.pairs_batches(path, "pairs", idx, bed_path=bed, threads=threads))
            dt = time.perf_counter() - t0
            out[tag] = len(sample) / dt
        return {"unit": "lines/s", "pairs_text": out, "lines": len(sample), "text_bytes": size,
                "threads": max(1, min(16, os.cpu_count() or 1)) if threads <= 0 else threads,
                "note": "native tokenizer + name lookup (+ alignments.bed writer), page-cache resident file"}


def make_inputs(a, device, rank_id=0, world=1):
    """Synthetic assembly (host) and this rank's shard of the pair stream (on `device`)."""
    import torch
    from haphic_b200 import synth
    from haphic_b200.links import name_rank
    asm = synth.make_assembly(a.nchr, a.contigs, a.mean_len, seed=a.seed)
    rank = name_rank(asm.names)
    in_nx = np.ones(asm.n, np.uint8)                     # --Nx 100
    per = a.pairs // world
    lo = rank_id * per
    hi = a.pairs if rank_id == world - 1 else lo + per
    rec = synth.make_pairs_range(asm, lo, hi, seed=a.seed + 1, device=device)      # same stream for any world size
    return asm, rank, in_nx, rec, lo


# --------------------------------------------------------------------------------------------------
# --dump-outputs: the arrays a caller of the timed path receives, as float64 (exact for every integer here)
# --------------------------------------------------------------------------------------------------

DUMP_ROWS = 1 << 18           # rows kept of the link table and of the link matrix
DUMP_MCL_ROWS = 1 << 20       # entries kept of the final MCL matrices, shared by the inflations
DUMP_LIMIT = 64 << 20         # bytes over all files


def sample_index(n, cap, seed):
    """0 .. n-1, or `cap` of them drawn with a fixed seed, ascending: the same positions for the same n in every run."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=cap, replace=False))


def csc_sample(m, cap, seed):
    """[k, 3] (row, column, value) of the stored entries of a scipy CSC matrix, all or a seeded sample, in storage order."""
    k = sample_index(m.nnz, cap, seed)
    col = np.searchsorted(m.indptr, k, side="right") - 1
    return np.stack([m.indices[k].astype(np.float64), col.astype(np.float64), m.data[k].astype(np.float64)], axis=1)


def dump_mcl_result(dump, inflation, st, result, cap):
    name = "mcl_inflation_{}".format(inflation)
    dump[name] = csc_sample(result, cap, 3)
    dump[name + "_iterations"] = np.stack([st["iter_nnz"], st["iter_delta"]], axis=1)        # nnz and delta per round
    dump.setdefault("mcl_summary", []).append([inflation, st["rounds"], st["converged"], result.nnz])


def dump_links(dump, tab, info, index, n_linked, mat, mc):
    f = tab.fetch()
    k = sample_index(int(info.nnz_full), DUMP_ROWS, 1)
    # full_link_dict entries in insertion order: key_i, key_j, full, flank, first_full, first_flank, HH, HT, TH, TT
    dump["links"] = np.column_stack([f[c][k].astype(np.float64) for c in ("key_i", "key_j", "full", "flank", "first_full",
                                                                          "first_flank")] + [f["ht"][k].astype(np.float64)])
    dump["ctg_links"] = tab.fetch_ctg()
    dump["matrix_index"] = index
    dump["matrix"] = csc_sample(mat.to_scipy(), DUMP_ROWS, 2)
    dump["counts"] = [info.n_records, info.n_used, info.nnz_full, info.nnz_flank, n_linked, mat.n, mat.nnz, mc.nnz_m0]


def write_dump(path, dump):
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in dump.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: {} bytes exceed the limit of {}".format(total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for k, v in sorted(arrays.items()):
        np.save(os.path.join(path, k + ".npy"), v)


def run_reference(a):
    """`--impl reference`: the unmodified reference's hot loops on the host cores, bounded samples of the same workload."""
    rank_id = int(os.environ.get("RANK", "0"))
    if rank_id != 0:
        return
    import tempfile
    from haphic_b200 import synth
    from oracle import refimpl
    if not refimpl.available():
        print(json.dumps({"impl": "reference", "unavailable": REF_MISSING}))
        return
    asm = synth.make_assembly(a.nchr, a.contigs, a.mean_len, seed=a.seed)
    inflations = [float(x) for x in a.inflations.split(",")]
    # every step is a bounded sample of the stream; the whole --steps/--warmup run is sized for about two minutes of the
    # reference's single-threaded loop (~10 us per record on this class of host, text parsing and BED writing included)
    per_step = max(100_000, min(a.cpu_sample_pairs, int(110.0 / max(1, a.steps + a.warmup) / 10e-6)))
    sample = synth.make_pairs_range(asm, 0, per_step, seed=a.seed + 1, device="cpu").numpy()
    times = []
    with tempfile.TemporaryDirectory() as tmp:
        for s in range(a.warmup + a.steps):
            _v, dt, nnz = ref_pairs_per_sec(asm, sample, tmp)
            if s >= a.warmup:
                times.append(dt)
    ms = 1000.0 * sum(times) / len(times)
    value = len(sample) / (ms / 1000.0)
    mcl = ref_mcl_small(a, inflations)
    line = {
        "impl": "reference", "metric": "hic_pairs_per_sec_matrix_build", "value": value, "unit": "pairs/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int32 counts / fp32 matrix", "data": "synthetic",
        "config": {"workload": workload_name(a), "inflations": inflations, "max_iter": a.max_iter, "pruning": a.pruning,
                   "sample": "first {} records of the stream per step, as .pairs text".format(len(sample))},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": 1, "kind": "reference",
                         "sample": "{} records per step through the unmodified HapHiC_cluster.parse_alignments_for_ctgs("
                                   "pairs_generator_inter_ctgs(...)) (single-threaded Python by construction; host has {} cores)"
                                   .format(len(sample), os.cpu_count())},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "mcl": {"metric": "mcl_iterations_per_sec", "value": mcl["sparse"]["value"], "unit": "iter/s", "reference": mcl},
    }
    print(json.dumps(line))


def ncu_traffic(workload):
    """DRAM bytes per launch from the committed ncu capture (profiles/traffic.json); only valid for the workload it
    was captured on."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
    except OSError:
        return {}
    return t if t.get("workload") == workload else {}


def run_b200(a):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank_id = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        if a.dump_outputs:
            raise SystemExit("--dump-outputs: the multi-process run does not write outputs")
        from haphic_b200 import dist as hdist
        return hdist.bench_multi(a, world, rank_id, local)

    from haphic_b200._lib import Context
    from haphic_b200.links import LinkTable
    from haphic_b200.mcl import Mcl, interpret_result

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    inflations = [float(x) for x in a.inflations.split(",")]
    asm, rank, in_nx, rec, _ = make_inputs(a, dev)
    n = asm.n
    P = int(rec.shape[0])
    keep = np.ones(n, np.uint8)
    ctx = Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    hint = int(min(P, n * (n - 1) // 2) * (0.45 if P > 4_000_000 else 1.0))     # distinct contig pairs the table is sized for
    torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def one_step(timed, dump=None):
        """Resident-input pass.  Returns per-stage device times (ms) and statistics.  With a `dump` dict, also copies what
        the pass computed into it; the copying is reported as `dump_s` and left out of the stage and step times."""
        e = [ev() for _ in range(4)]
        e[0].record(stream)
        tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=hint)
        tab.add(rec, asynchronous=True)
        info = tab.finish()
        e[1].record(stream)
        index, n_linked = tab.linked_index(keep)
        tail = np.nonzero(index < 0)[0].astype(np.int32)
        mat = tab.to_matrix(keep, tail)
        e[2].record(stream)
        mc = Mcl(mat)
        iters, kernel_ms, alg_bytes, products = 0, mc.normalize_ms + mc.preexp_ms, 0, mc.preexp_products
        per_infl = []
        dump_ms, dump_s, dump_launches = 0.0, 0.0, 0
        for r in inflations:
            st = mc.run(r, a.max_iter, a.pruning)
            iters += st["rounds"]
            kernel_ms += float(st["iter_ms"].sum())
            alg_bytes += st["bytes"]
            products += st["products"]
            per_infl.append({"inflation": r, "rounds": st["rounds"], "converged": st["converged"],
                             "ms": float(st["iter_ms"].sum()), "nnz_iter": st["iter_nnz"][:6].tolist(),
                             "ms_iter": [round(float(x), 3) for x in st["iter_ms"][:6]]})
            if dump is not None:
                # the next inflation overwrites this result: fetch it now, between two events the stage time leaves out
                t0, l0, f = time.perf_counter(), ctx.launches, [ev(), ev()]
                f[0].record(stream)
                dump_mcl_result(dump, r, st, mc.result(), DUMP_MCL_ROWS // len(inflations))
                f[1].record(stream)
                f[1].synchronize()
                dump_ms += f[0].elapsed_time(f[1])
                dump_s += time.perf_counter() - t0
                dump_launches += ctx.launches - l0
        e[3].record(stream)
        e[3].synchronize()
        if dump is not None:
            t0, l0 = time.perf_counter(), ctx.launches
            dump_links(dump, tab, info, index, n_linked, mat, mc)
            dump_s += time.perf_counter() - t0
            dump_launches += ctx.launches - l0
        out = {
            "dump_s": dump_s, "dump_launches": dump_launches,
            "build_ms": e[0].elapsed_time(e[1]), "matrix_ms": e[1].elapsed_time(e[2]),
            "mcl_ms": e[2].elapsed_time(e[3]) - dump_ms,
            "iters": iters, "kernel_ms": kernel_ms, "alg_bytes": alg_bytes, "products": products,
            "nnz_full": int(info.nnz_full), "nnz_flank": int(info.nnz_flank), "n_used": int(info.n_used),
            "nnz_m0": mc.nnz_m0, "preexp_ms": mc.preexp_ms, "preexp_products": mc.preexp_products,
            "normalize_ms": mc.normalize_ms, "per_inflation": per_infl, "n_matrix": mat.n, "preexp": dict(mc.preexp),
        }
        mc.close()
        mat.close()
        tab.close()
        return out

    for _ in range(a.warmup):
        one_step(False)
    sampler = ClockSampler(0)
    sampler.start()
    l0 = ctx.launches
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    dump = {} if a.dump_outputs else None
    steps = [one_step(True, dump if s == a.steps - 1 else None) for s in range(a.steps)]
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0 - sum(s["dump_s"] for s in steps)
    launches = ctx.launches - l0 - sum(s["dump_launches"] for s in steps)
    clocks = sampler.stop()
    if dump is not None:
        write_dump(a.dump_outputs, dump)

    if a.verbose:
        print("per-step ms:", [(round(s["build_ms"], 1), round(s["matrix_ms"], 1), round(s["mcl_ms"], 1)) for s in steps], file=sys.stderr)
    build_ms = sum(s["build_ms"] for s in steps) / len(steps)
    matrix_ms = sum(s["matrix_ms"] for s in steps) / len(steps)
    mcl_ms = sum(s["mcl_ms"] for s in steps) / len(steps)
    s0 = steps[-1]
    pairs_per_s = P / ((build_ms + matrix_ms) / 1000.0)
    iters_per_s = s0["iters"] / (mcl_ms / 1000.0)
    peak, peak_src = measured_peaks()
    # dominant kernel launch: the pre-expansion (one launch per step), see preexp_roofline()
    pre_bytes = 8 * s0["nnz_m0"] + 4 * s0["n_matrix"] ** 2
    # all launches of the column kernels of the sweep (pre-expansion + every iteration), same definition
    mcl_bytes = s0["alg_bytes"] + pre_bytes
    mcl_achieved = mcl_bytes / (s0["kernel_ms"] / 1000.0) / 1e9
    traffic = ncu_traffic(workload_name(a))
    build_bytes = 16 * P + 12 * s0["nnz_full"] + 12 * s0["nnz_flank"] + 4 * n
    build_achieved = build_bytes / (build_ms / 1000.0) / 1e9

    # ---- end to end through the host API: pinned host records in, host results out ------------------
    rec_host = torch.empty(rec.shape, dtype=torch.int32, pin_memory=True)
    rec_host.copy_(rec)
    torch.cuda.synchronize()
    e2e_build, e2e_mcl, d2h = [], [], 0
    for s in range(1 + a.e2e_steps):
        t0 = time.perf_counter()
        tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=hint)
        tab.add(rec_host)                                   # H2D inside, double-buffered
        ta = time.perf_counter()
        info = tab.finish()
        tb = time.perf_counter()
        table = tab.fetch(pinned=True)                                 # D2H: the link dicts' arrays
        tot = tab.fetch_ctg()
        tc = time.perf_counter()
        index, n_linked = tab.linked_index(keep)
        tail = np.nonzero(index < 0)[0].astype(np.int32)
        mat = tab.to_matrix(keep, tail)
        ctx.sync()
        t1 = time.perf_counter()
        if a.verbose:
            print("e2e pass {} ms: add(H2D) {:.1f} finish {:.1f} fetch(D2H) {:.1f} index+matrix {:.1f}".format(
                s, 1e3 * (ta - t0), 1e3 * (tb - ta), 1e3 * (tc - tb), 1e3 * (t1 - tc)), file=sys.stderr)
        mc = Mcl(mat)
        n_it = 0
        d2h_mcl = 0
        for r in inflations:
            st = mc.run(r, a.max_iter, a.pruning)
            n_it += st["rounds"]
            fin = mc.result()                               # D2H: final matrix of this inflation
            interpret_result(fin)
            d2h_mcl += fin.nnz * 8 + (n + 1) * 8
        t2 = time.perf_counter()
        if s >= 1:
            e2e_build.append(t1 - t0)
            e2e_mcl.append((t2 - t1, n_it))
            d2h = sum(v.nbytes for v in table.values()) + tot.nbytes + index.nbytes + d2h_mcl
        mc.close()
        mat.close()
        tab.close()
    e2e_pairs = P / float(np.median(e2e_build)) if e2e_build else None          # median over the passes
    e2e_iters = sum(x[1] for x in e2e_mcl) / sum(x[0] for x in e2e_mcl) if e2e_mcl else None

    # ---- the default sweep of `haphic cluster` (20 inflations 1.1 .. 3.0, HapHiC_cluster.py:2139-2155, 2699-2705) ----------
    default_sweep = None
    if not a.no_default_sweep:
        from haphic_b200.mcl import inflation_values
        tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=hint)
        tab.add(rec, asynchronous=True)
        tab.finish()
        index, _ = tab.linked_index(keep)
        mat = tab.to_matrix(keep, np.nonzero(index < 0)[0].astype(np.int32))
        e0, e1 = ev(), ev()
        e0.record(stream)
        mc = Mcl(mat)
        rounds = []
        for r in inflation_values(1.1, 3.0, 0.1):
            st = mc.run(float(r), a.max_iter, a.pruning)
            rounds.append(st["rounds"])
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        default_sweep = {"inflations": 20, "iterations": int(sum(rounds)), "rounds": rounds, "ms": ms,
                         "value": sum(rounds) / (ms / 1000.0), "unit": "iter/s",
                         "note": "normalise + pre-expansion + 20 mcl() calls, device time (the reference's MCL total, 2951-2953)"}
        mc.close()
        mat.close()
        tab.close()

    # ---- CPU baseline on this box's host cores (bounded samples) ------------------------------------
    cpu = None
    mcl_cpu = None
    if not a.no_cpu_baseline:
        from oracle import refimpl
        cpu = cpu_baseline_block(a, asm, rank, in_nx, rec)
        mcl_cpu = ref_mcl_small(a, inflations) if refimpl.available() else {"unavailable": REF_MISSING}
        # the C3 matrix itself is beyond the reference's reach (10 GB dense intermediate, hours of SpGEMM): one iteration
        # of the CPU port on a sample of columns of iterate M_1, extrapolated
        tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=hint)
        tab.add(rec, asynchronous=True)
        tab.finish()
        index, _ = tab.linked_index(keep)
        mat = tab.to_matrix(keep, np.nonzero(index < 0)[0].astype(np.int32))
        mc = Mcl(mat)
        mc.run(inflations[len(inflations) // 2], 1, a.pruning)
        m_iter1 = mc.result()
        ips, dt, ncols = cpu_mcl_iter_per_sec(m_iter1, a.cpu_sample_cols, inflations[len(inflations) // 2], a.pruning)
        mcl_cpu["port_extrapolated"] = {
            "value": ips, "unit": "iter/s", "cores": 1, "kind": "port",
            "sample": "iteration 1 (expand+inflate+prune) of inflation {} on {} of {} columns of the benchmark's own matrix, {:.1f} s, "
                      "scaled by n/cols; scipy SpGEMM stands in for MKL".format(inflations[len(inflations) // 2], ncols, n, dt)}
        mc.close()
        mat.close()
        tab.close()
    ingest = None
    if not a.no_cpu_baseline and a.ingest_lines > 0:
        ingest = ingest_rate(asm, rec[: a.ingest_lines].cpu().numpy())

    line = {
        "metric": "hic_pairs_per_sec_matrix_build", "value": pairs_per_s, "unit": "pairs/s", "n_gpus": 1,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1000.0 * t_wall / a.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int32 counts / fp32 matrix", "data": "synthetic",
        "config": {"workload": workload_name(a), "inflations": inflations, "max_iter": a.max_iter, "pruning": a.pruning,
                   "cache": "inputs (16 B x pairs = {:.1f} GB) and the dense pre-expanded matrix exceed the 126 MB L2".format(
                       16 * P / 1e9),
                   "step": "link build + index + CSC + normalise + pre-expansion + MCL sweep"},
        "stage_ms": {"link_build": build_ms, "matrix": matrix_ms, "mcl_sweep": mcl_ms},
        "mcl": {"metric": "mcl_iterations_per_sec", "value": iters_per_s, "unit": "iter/s", "iterations": s0["iters"],
                "products": s0["products"], "preexp_ms": s0["preexp_ms"], "normalize_ms": s0["normalize_ms"],
                "preexp": s0["preexp"], "per_inflation": s0["per_inflation"], "e2e": {"value": e2e_iters, "unit": "iter/s"},
                "default_sweep": default_sweep, "cpu_baseline": mcl_cpu},
        "links": {"pairs": P, "used": s0["n_used"], "nnz_full": s0["nnz_full"], "nnz_flank": s0["nnz_flank"],
                  "n_matrix": s0["n_matrix"], "nnz_m0": s0["nnz_m0"]},
        "e2e": {"value": e2e_pairs, "unit": "pairs/s", "h2d_bytes_per_step": 16 * P + 13 * n, "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": preexp_roofline(s0["preexp"], s0["n_matrix"], s0["nnz_m0"], s0["n_matrix"], traffic),
        "roofline_mcl": {"kernel": "all hh_k_col / hh_k_col_win / hh_k_col_small launches of the sweep", "bound": "hbm",
                         "achieved": mcl_achieved, "peak": peak, "unit": "GB/s", "frac": mcl_achieved / peak,
                         "algorithmic_bytes": mcl_bytes, "kernel_ms": s0["kernel_ms"]},
        "roofline_build": {"kernel": "hh_k_part_scatter + 513 x hh_k_part_step (partition, then aggregate in L2-resident scratch tables)",
                           "bound": "hbm", "achieved": build_achieved, "peak": peak, "unit": "GB/s", "frac": build_achieved / peak,
                           "traffic": traffic.get("hh_k_links_partitioned"), "algorithmic_bytes": build_bytes,
                           "note": traffic.get("hh_k_links_partitioned_note")},
        "cpu_baseline": cpu,
        "ingest": ingest,
    }
    print(json.dumps(line))
    ctx.close()


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
