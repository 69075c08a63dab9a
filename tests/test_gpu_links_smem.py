"""GPU: the two-level partitioned link counting (shared-memory tables per sub-partition, with the global scratch-table
fallback for sub-partitions whose keys do not fit), compared bit-exactly with the direct engine on the same records; and the
matrix stage's reuse of the first-seen index and its radix-sort rank."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SUB_SLOTS = 2048          # keys a shared-memory sub-partition table holds (HH_SUB_SLOTS in hh_links.cu)


@pytest.fixture(scope="module")
def ctx():
    from haphic_b200._lib import Context
    c = Context(0)
    yield c
    c.close()


def mix64(k):
    """hh_mix64 of hh_links.cu on a uint64 array (the hash whose top bits pick partition and sub-partition)."""
    k = k.astype(np.uint64)
    with np.errstate(over="ignore"):
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xff51afd7ed558ccd)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xc4ceb9fe1a85ec53)
        k ^= k >> np.uint64(33)
    return k


def count(ctx, monkeypatch, lengths, rank, rec, env):
    """Count `rec` with the engine `env` selects; returns (info fields, fetched arrays, per-fragment totals, launches of finish)."""
    from haphic_b200.links import LinkTable
    for k in ("HH_LINKS_PARTITION", "HH_LINKS_NPART_LOG", "HH_LINKS_SUB_LOG_MAX"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    tab = LinkTable(ctx, lengths, rank, np.ones(len(lengths), np.uint8), 500000)
    tab.add(rec)
    l0 = ctx.launches
    info = tab.finish()
    launches = ctx.launches - l0
    got = tab.fetch()
    tot = tab.fetch_ctg()
    tab.close()
    return (info.n_records, info.n_used, info.nnz_full, info.nnz_flank), got, tot, launches


def check_same(ctx, monkeypatch, lengths, rank, rec, env):
    """Partitioned counting under `env` equals the direct engine; returns the number of fallback sub-partitions."""
    want = count(ctx, monkeypatch, lengths, rank, rec, {"HH_LINKS_PARTITION": 0})
    got = count(ctx, monkeypatch, lengths, rank, rec, dict(env, HH_LINKS_PARTITION=1))
    assert got[0] == want[0]
    for k in want[1]:
        assert np.array_equal(got[1][k], want[1][k]), k
    assert np.array_equal(got[2], want[2])
    # one set of partition regions: level-2 histogram, offsets, scatter and the shared-memory count are 4 launches; a
    # fallback adds the two scratch-table initialisations and one launch per fallback sub-partition plus the last emit
    return 0 if got[3] == 4 else got[3] - 7


def synth_stream(n_contigs, n_pairs, seed):
    from haphic_b200 import synth
    from haphic_b200.links import name_rank
    asm = synth.make_assembly(8, n_contigs, 30000, seed=seed)
    rec = synth.make_pairs(asm, n_pairs, seed=seed + 1).numpy()
    return np.asarray(asm.lengths, np.int64), name_rank(asm.names), np.ascontiguousarray(rec)


def crafted_stream(per_sub, seed):
    """Records whose keys are chosen by hash: sub-partition s of the 2 + 2 top hash bits gets per_sub[s] distinct contig
    pairs, each seen three times at random positions, in random order."""
    rng = np.random.default_rng(seed)
    n = 4000
    i = rng.integers(0, n, 400_000)
    j = rng.integers(0, n, 400_000)
    i, j = np.minimum(i, j), np.maximum(i, j)
    keys = np.unique((i[i != j].astype(np.uint64) << np.uint64(32)) | j[i != j].astype(np.uint64))
    sub = (mix64(keys) >> np.uint64(60)).astype(np.int64)
    chosen = np.concatenate([keys[sub == s][:per_sub[s]] for s in range(16)])
    for s in range(16):
        assert (sub == s).sum() >= per_sub[s]
    kk = np.repeat(chosen, 3)
    a = (kk >> np.uint64(32)).astype(np.int32)
    b = (kk & np.uint64(0xFFFFFFFF)).astype(np.int32)
    swap = rng.random(len(kk)) < 0.5
    a, b = np.where(swap, b, a), np.where(swap, a, b)
    lengths = np.full(n, 2_000_000, np.int64)
    rec = np.stack([a, rng.integers(0, 2_000_000, len(kk)), b, rng.integers(0, 2_000_000, len(kk))], 1).astype(np.int32)
    return lengths, np.arange(n, dtype=np.int32), np.ascontiguousarray(rec[rng.permutation(len(rec))])


def test_smem_path_no_overflow(ctx, monkeypatch):
    lengths, rank, rec = synth_stream(2000, 2_000_000, 21)
    assert check_same(ctx, monkeypatch, lengths, rank, rec, {"HH_LINKS_NPART_LOG": 5}) == 0


def test_smem_and_fallback_mixed(ctx, monkeypatch):
    # 4 partitions x 4 sub-partitions; the even ones hold more distinct keys than a shared table has slots
    per_sub = [3000 if s % 2 == 0 else 300 for s in range(16)]
    lengths, rank, rec = crafted_stream(per_sub, 5)
    env = {"HH_LINKS_NPART_LOG": 2, "HH_LINKS_SUB_LOG_MAX": 2}
    assert check_same(ctx, monkeypatch, lengths, rank, rec, env) == 8


def test_every_sub_partition_falls_back(ctx, monkeypatch):
    # no level-2 split: each of the 4 partitions is one sub-partition with more than SUB_SLOTS distinct keys
    per_sub = [SUB_SLOTS // 2 + 300] * 16
    lengths, rank, rec = crafted_stream(per_sub, 6)
    env = {"HH_LINKS_NPART_LOG": 2, "HH_LINKS_SUB_LOG_MAX": 0}
    assert check_same(ctx, monkeypatch, lengths, rank, rec, env) == 4


def test_hot_pair_spill(ctx, monkeypatch):
    # one contig pair owns 30 % of the records: its level-1 region overflows into the spill list, and its sub-partition
    # holds hundreds of thousands of records of a handful of keys
    lengths, rank, rec = synth_stream(2000, 2_000_000, 31)
    rng = np.random.default_rng(7)
    hot = rng.random(len(rec)) < 0.3
    other = len(lengths) // 2
    rec[hot, 0] = 3
    rec[hot, 2] = other
    rec[hot, 1] = rng.integers(0, lengths[3], hot.sum())
    rec[hot, 3] = rng.integers(0, lengths[other], hot.sum())
    assert check_same(ctx, monkeypatch, lengths, rank, np.ascontiguousarray(rec), {"HH_LINKS_NPART_LOG": 5}) == 0


# ---------------------------------------------------------------------------------------------------------------------
# matrix stage
# ---------------------------------------------------------------------------------------------------------------------

def dense(mat):
    return mat.to_scipy().toarray()


def fresh_matrix(ctx, lengths, rank, parts, keep):
    from haphic_b200.links import LinkTable
    tab = LinkTable(ctx, lengths, rank, np.ones(len(lengths), np.uint8), 500000)
    off = 0
    for p in parts:
        tab.add(p, stream_offset=off)
        off += len(p)
    tab.finish()
    index, _ = tab.linked_index(keep)
    tail = np.nonzero((index < 0) & (keep > 0))[0].astype(np.int32)
    mat = tab.to_matrix(keep, tail)
    out = (index, tail, dense(mat))
    mat.close()
    tab.close()
    return out


def test_matrix_after_index_of_other_keep(ctx):
    from haphic_b200.links import LinkTable
    lengths, rank, rec = synth_stream(300, 200_000, 41)
    rng = np.random.default_rng(2)
    keep1 = (rng.random(len(lengths)) < 0.8).astype(np.uint8)
    keep2 = (rng.random(len(lengths)) < 0.8).astype(np.uint8)
    assert not np.array_equal(keep1, keep2)
    idx2, tail2, want2 = fresh_matrix(ctx, lengths, rank, [rec], keep2)
    idx1, tail1, want1 = fresh_matrix(ctx, lengths, rank, [rec], keep1)
    tab = LinkTable(ctx, lengths, rank, np.ones(len(lengths), np.uint8), 500000)
    tab.add(rec)
    tab.finish()
    index, _ = tab.linked_index(keep1)
    assert np.array_equal(index, idx1)
    for keep, tail, want in ((keep2, tail2, want2), (keep1, tail1, want1), (keep1, tail1, want1)):
        mat = tab.to_matrix(keep, tail)
        assert np.array_equal(dense(mat), want)
        mat.close()
    # the reused index (same mask, nothing changed since): equal to a fresh computation
    index, _ = tab.linked_index(keep2)
    mat = tab.to_matrix(keep2, tail2)
    assert np.array_equal(dense(mat), want2)
    mat.close()
    tab.close()


def test_matrix_after_merge(ctx):
    from haphic_b200.links import LinkTable
    lengths, rank, rec = synth_stream(300, 200_000, 43)
    a, b = rec[:120_000], rec[120_000:]
    keep = np.ones(len(lengths), np.uint8)
    _, tail, want = fresh_matrix(ctx, lengths, rank, [a, b], keep)
    t1 = LinkTable(ctx, lengths, rank, np.ones(len(lengths), np.uint8), 500000)
    t1.add(a)
    t1.finish()
    t1.linked_index(keep)                 # index of the table before the merge
    t2 = LinkTable(ctx, lengths, rank, np.ones(len(lengths), np.uint8), 500000)
    t2.add(b, stream_offset=len(a))
    t1.merge(*t2.export())
    t1.finish()
    mat = t1.to_matrix(keep, tail)
    assert np.array_equal(dense(mat), want)
    mat.close()
    t1.close()
    t2.close()


@pytest.mark.parametrize("n", [1, 1000, 1024, 1025, 5003, 70001])
def test_rank_matches_quadratic_definition(ctx, n):
    """A table built from crafted entries (random first-seen indices), so the touch values are random; the index must be
    index[c] = #{touched d : touch[d] < touch[c]} (the old O(n^2) kernel's definition), -1 for untouched fragments."""
    import torch
    from haphic_b200.links import LinkTable
    rng = np.random.default_rng(n)
    m = 2 * n + 5
    i = rng.integers(0, n, m)
    j = rng.integers(0, n, m)
    ok = i != j
    key = np.unique(np.minimum(i[ok], j[ok]).astype(np.int64) * n + np.maximum(i[ok], j[ok]))
    m = len(key)
    ei, ej = key // n, key % n
    flank = rng.integers(0, 3, m).astype(np.int64)
    full = flank + rng.integers(1, 3, m)
    first_full = rng.permutation(m).astype(np.int64)
    first_flank = np.where(flank > 0, rng.choice(1 << 31, m, replace=False), 0xFFFFFFFF).astype(np.int64)
    ent = np.zeros((m, 9), np.int64)
    ent[:, 0], ent[:, 1], ent[:, 2], ent[:, 3], ent[:, 4], ent[:, 5] = ei, ej, full, flank, first_full, first_flank
    keep = (rng.random(n) < 0.9).astype(np.uint8)
    # touch[c]: earliest flank entry with both ends kept, 2 * first_flank (+1 on the second end)
    touch = np.full(n, np.iinfo(np.int64).max, np.int64)
    sel = (flank > 0) & (keep[ei] > 0) & (keep[ej] > 0)
    np.minimum.at(touch, ei[sel], 2 * first_flank[sel])
    np.minimum.at(touch, ej[sel], 2 * first_flank[sel] + 1)
    touched = touch != np.iinfo(np.int64).max
    if n <= 5003:
        want = np.where(touched, (touch[None, touched] < touch[:, None]).sum(1) if touched.any() else 0, -1)
    else:
        want = np.full(n, -1, np.int64)
        order = np.argsort(touch[touched], kind="stable")
        want[np.nonzero(touched)[0][order]] = np.arange(touched.sum())
    dev = torch.device("cuda", ctx.device)
    tab = LinkTable(ctx, np.full(n, 10_000, np.int64), np.arange(n, dtype=np.int32), np.ones(n, np.uint8), 500000)
    tab.merge(torch.from_numpy(ent.astype(np.uint32).view(np.int32)).to(dev), torch.zeros(n, dtype=torch.int64, device=dev), 0, 0)
    tab.finish()
    index, n_linked = tab.linked_index(keep)
    assert n_linked == int(touched.sum())
    assert np.array_equal(index, want)
    tab.close()
