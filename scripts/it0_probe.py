"""Iteration 0 (hh_k_iter0: stream of the dense pre-expanded matrix) at C3: device time of the kernel and the number of
surviving entries per inflation."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from haphic_b200 import synth
from haphic_b200._lib import Context
from haphic_b200.links import LinkTable, name_rank
from haphic_b200.mcl import Mcl

pairs = int(os.environ.get("PAIRS", "200000000"))
asm = synth.make_assembly(24, 50000, 20000, seed=12345)
rec = synth.make_pairs_range(asm, 0, pairs, seed=12346, device="cuda")
ctx = Context(0)
tab = LinkTable(ctx, asm.lengths, name_rank(asm.names), np.ones(asm.n, np.uint8), 500000, capacity_hint=int(0.45 * pairs))
tab.add(rec, asynchronous=True)
tab.finish()
del rec
keep = np.ones(asm.n, np.uint8)
index, _ = tab.linked_index(keep)
mat = tab.to_matrix(keep, np.nonzero(index < 0)[0].astype(np.int32))
mc = Mcl(mat, preexp="dense")
out = {}
for r in (2.0, 1.5, 3.0, 1.7):
    best, nnz = 1e9, None
    for _ in range(3):
        st = mc.run(r, 1, 1e-4)
        best = min(best, float(st["iter_ms"][0]))
        nnz = int(st["iter_nnz"][0])
    out["r{}".format(r)] = {"ms": round(best, 3), "nnz": nnz}
print("IT0 " + json.dumps(out), flush=True)
