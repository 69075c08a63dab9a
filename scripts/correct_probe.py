"""Assembly-correction probe at C3 shape (50k contigs, 200M pairs on the device, about 1 % of the contigs in misjoined
groups): device time of each stage from CUDA events on the library's stream, printed as one JSON line with the GPU name
and its power limit.  Stages: coverage (hh_correct_add of all records), detect (round 1, including the scan of the
difference array), split (round 1 of a 2-round run), remap (the second pass over all records)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from haphic_b200 import correct, synth
from haphic_b200._lib import Context

pairs = int(os.environ.get("PAIRS", "200000000"))
asm = synth.make_assembly(24, 50000, 20000, seed=2024)
mis = synth.make_misjoined(asm, synth.make_pairs(asm, pairs, seed=2025, device="cuda").cpu().numpy(), frac=0.004, seed=2026)
rec = torch.from_numpy(mis.pairs).cuda()
ctx = Context(0)
stream = torch.cuda.ExternalStream(ctx.stream)
times = {}


def timed(name, fn, *a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    out = fn(*a)
    e1.record(stream)
    e1.synchronize()
    times.setdefault(name, []).append(e0.elapsed_time(e1))
    return out


args = argparse.Namespace(correct_resolution=500, median_cov_ratio=0.2, region_len_ratio=0.1, min_region_cutoff=5000,
                          RE="GATC", correct_nrounds=2)
reps = int(os.environ.get("REPS", "3"))
for rep in range(reps + 1):                     # the first repetition warms up
    fa = {n: ["", int(L), 1] for n, L in zip(mis.asm.names, mis.asm.lengths.tolist())}
    corr = correct.Corrector(ctx, mis.asm.lengths, 500)
    timed("coverage", corr.add, rec)
    det, spl = corr.detect, corr.split
    corr.detect = lambda *a: timed("detect", det, *a)
    corr.split = lambda *a: timed("split", spl, *a)
    with tempfile.TemporaryDirectory() as tmp:
        cwd = os.getcwd()
        os.chdir(tmp)
        nb, fpos, ffrag = correct.correct_assembly(fa, corr, args)
        os.chdir(cwd)
    corr.set_pieces(*correct.piece_table(mis.asm.names, fa, fpos, ffrag))
    out = rec.clone()
    timed("remap", corr.remap, out)
    corr.close()
    if rep == 0:
        times = {}
gpu = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
except Exception:
    power = "unknown"
print(json.dumps({"gpu": gpu, "power_limit": power, "pairs": pairs, "contigs": mis.asm.n, "broken_round1": nb,
                  "bins": int((mis.asm.lengths // 500 + 1).sum()),
                  "ms": {k: [round(v, 3) for v in vs] for k, vs in times.items()}}))
ctx.close()
