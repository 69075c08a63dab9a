"""bench.py's JSON contract: the reference arm (`--impl reference`) runs without a GPU and must print ONE line with the keys
its readers use; on a GPU, `--dump-outputs` writes what the timed path computed."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
           "--contigs", "2000", "--nchr", "4", "--pairs", "1000000", "--cpu-sample-pairs", "200000"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "hic_pairs_per_sec_matrix_build" and d["unit"] == "pairs/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["mcl"]["unit"] == "iter/s" and d["mcl"]["value"] > 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, cwd=REPO, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_step_counts_and_dump_arguments_are_checked():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=120, cwd=REPO)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-500:])


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """Two runs with the same arguments dump the same arrays; at this size nothing is sampled, so the link table, the matrix
    and the clusters of every inflation are those the oracle computes from the same seeded stream."""
    import scipy.sparse as sp
    from haphic_b200 import synth
    from haphic_b200.links import name_rank
    from oracle import haphic_oracle as orc
    nchr, n_contigs, mean_len, n_pairs, seed, inflations = 4, 600, 20000, 300_000, 7, (2.0, 3.0)
    args = ["--steps", "2", "--warmup", "1", "--contigs", str(n_contigs), "--nchr", str(nchr), "--mean-len", str(mean_len),
            "--pairs", str(n_pairs), "--seed", str(seed), "--inflations", ",".join(map(str, inflations)),
            "--no-cpu-baseline", "--no-default-sweep", "--e2e-steps", "0"]
    dumps = []
    for k in range(2):
        out = tmp_path / str(k)
        r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py")] + args + ["--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=REPO)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2 and line["warmup"] == 1
        dumps.append({f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))})
    got, again = dumps
    assert sorted(got) == sorted(again) and all(np.array_equal(got[k], again[k]) for k in got)
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 << 20

    asm = synth.make_assembly(nchr, n_contigs, mean_len, seed=seed)
    rec = synth.make_pairs_range(asm, 0, n_pairs, seed=seed + 1, device="cuda").cpu().numpy()
    keep = np.ones(asm.n, np.uint8)
    ref = orc.count_links_numpy(rec, asm.lengths, name_rank(asm.names), keep, 500000, with_clm=False)
    links = got["links"]
    assert np.array_equal(links[:, 0:2], ref["full_keys"]) and np.array_equal(links[:, 2], ref["full_vals"])
    assert np.array_equal(got["ctg_links"], ref["ctg_link_total"])
    index = got["matrix_index"].astype(np.int64)
    tail = np.nonzero(index < 0)[0].tolist()
    want_m, want_index = orc.dict_to_matrix(ref["flank_keys"], ref["flank_vals"], keep, tail_order=tail)
    assert np.array_equal(np.where(index >= 0, index, want_index), want_index)
    m = got["matrix"]
    mat = sp.csc_matrix((m[:, 2], (m[:, 0].astype(np.int64), m[:, 1].astype(np.int64))), shape=want_m.shape)
    assert len(m) == want_m.nnz and abs(mat - want_m).max() == 0
    summary = got["mcl_summary"]
    assert summary[:, 0].tolist() == list(inflations) and (summary[:, 2] == 1).all()
    for r, rounds, _conv, nnz in summary.tolist():
        fin = got["mcl_inflation_{}".format(r)]
        assert len(fin) == nnz and len(got["mcl_inflation_{}_iterations".format(r)]) == rounds
        fin = sp.csc_matrix((fin[:, 2], (fin[:, 0].astype(np.int64), fin[:, 1].astype(np.int64))), shape=want_m.shape)
        assert abs(np.asarray(fin.sum(axis=0)).ravel() - 1.0).max() < 1e-6
        assert orc.interpret_result(fin) is not None
