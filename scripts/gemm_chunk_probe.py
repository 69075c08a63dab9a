"""Pre-expansion GEMM at C3 under different drain periods / encodings (env switches of csrc/hh_gemm.cu): one link matrix,
one `Mcl(...)` per variant, prints the engine's own timings.  Usage: python scripts/gemm_chunk_probe.py [variant ...] with
variant = FMT:CHUNK (e.g. f16:3 f16:8 bf16:2)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from haphic_b200 import synth
from haphic_b200._lib import Context
from haphic_b200.links import LinkTable, name_rank
from haphic_b200.mcl import Mcl

variants = sys.argv[1:] or ["f16:3", "f16:4", "f16:6", "f16:8", "f16:12", "bf16:2"]
pairs = int(os.environ.get("PAIRS", "200000000"))
asm = synth.make_assembly(24, 50000, 20000, seed=12345)
rank = name_rank(asm.names)
in_nx = np.ones(asm.n, np.uint8)
rec = synth.make_pairs_range(asm, 0, pairs, seed=12346, device="cuda")
ctx = Context(0)
tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=int(0.45 * pairs))
tab.add(rec, asynchronous=True)
tab.finish()
del rec
keep = np.ones(asm.n, np.uint8)
index, _ = tab.linked_index(keep)
mat = tab.to_matrix(keep, np.nonzero(index < 0)[0].astype(np.int32))
NC = 512                                    # columns of the accuracy check: exact fp64 product of the fp32 M0
exact = None
for v in variants:
    fmt, chunk = v.split(":")
    os.environ["HH_GEMM_FMT"] = fmt
    os.environ["HH_GEMM_CHUNK"] = chunk
    mc = Mcl(mat, preexp="dense")
    mc2 = Mcl(mat, preexp="dense")          # second construction: warm allocator
    p = mc2.preexp
    out = {"variant": v, "gemm_ms": round(p["gemm_ms"], 2), "densify_ms": round(p["densify_ms"], 2), "clip_ms": round(p["clip_ms"], 2),
           "passes": p["passes"], "stages": p["stages"], "tflops": round(p["flops"] / p["gemm_ms"] / 1e9, 1)}
    if exact is None:
        m0 = mc2.m0().astype(np.float64)
        exact = np.asarray((m0 @ m0[:, :NC]).todense())
    mc.close()
    mc2.close()
    part = Mcl(mat, col_lo=0, col_hi=NC, preexp="dense")
    blk = part.m1().astype(np.float64)
    part.close()
    nz = exact != 0
    rel = (blk[nz] - exact[nz]) / exact[nz]
    out["pattern_equal"] = bool(np.array_equal(blk != 0, nz))
    out["max_rel"] = float(np.abs(rel).max())
    out["mean_rel"] = float(rel.mean())
    print("PROBE " + json.dumps(out), flush=True)
