"""Link-counting probe at C3 (50k contigs / 200M pairs): wall / device time of add and finish for the direct and the
partitioned engines.  PROFILE=1 adds one partitioned pass (count + index + matrix) under torch.profiler and prints its
per-kernel device times."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from haphic_b200 import synth
from haphic_b200._lib import Context
from haphic_b200.links import LinkTable, name_rank

pairs = int(os.environ.get("PAIRS", "200000000"))
asm = synth.make_assembly(24, 50000, 20000, seed=12345)
rank = name_rank(asm.names)
in_nx = np.ones(asm.n, np.uint8)
rec = synth.make_pairs_range(asm, 0, pairs, seed=12346, device="cuda")
ctx = Context(0)
for mode in os.environ.get("MODES", "0,1").split(","):
    os.environ["HH_LINKS_PARTITION"] = mode
    for rep in range(int(os.environ.get("REPS", "3"))):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=int(0.45 * pairs))
        tab.add(rec, asynchronous=True)
        ctx.sync()
        t1 = time.perf_counter()
        info = tab.finish()
        ctx.sync()
        t2 = time.perf_counter()
        keep = np.ones(asm.n, np.uint8)
        index, _ = tab.linked_index(keep)
        mat = tab.to_matrix(keep, np.nonzero(index < 0)[0].astype(np.int32))
        ctx.sync()
        t3 = time.perf_counter()
        print("mode", mode, "rep", rep, "add ms", round(1e3 * (t1 - t0), 2), "finish ms", round(1e3 * (t2 - t1), 2), "index+matrix ms",
              round(1e3 * (t3 - t2), 2), "nnz", info.nnz_full, "slots", info.table_slots, flush=True)
        mat.close()
        tab.close()

if os.environ.get("PROFILE"):
    from torch.profiler import ProfilerActivity, profile
    os.environ["HH_LINKS_PARTITION"] = "1"
    keep = np.ones(asm.n, np.uint8)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        tab = LinkTable(ctx, asm.lengths, rank, in_nx, 500000, capacity_hint=int(0.45 * pairs))
        tab.add(rec, asynchronous=True)
        tab.finish()
        index, _ = tab.linked_index(keep)
        mat = tab.to_matrix(keep, np.nonzero(index < 0)[0].astype(np.int32))
        ctx.sync()
    print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30, max_name_column_width=60), flush=True)
    mat.close()
    tab.close()
