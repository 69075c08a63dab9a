"""GPU: the tile phases of the level-1 / level-2 partition kernels and the chunked, double-buffered shared-memory count with
its live-slot emit, compared bit-exactly with the direct engine: streams that end inside a tile, sub-partitions at the
record-buffer chunk size, multi-chunk sub-partitions that fit or overflow the table, a table filled exactly, and several
`add` calls that use more than one set of partition regions."""

import numpy as np
import pytest

from tests.test_gpu_links_smem import check_same, mix64, synth_stream

pytestmark = pytest.mark.gpu

SLOTS = 1024              # keys a shared-memory sub-partition table holds (HH_SUB_SLOTS in hh_links.cu)
CHUNK = SLOTS // 2        # records a record buffer of hh_k_sub_count holds (HH_SUB_CHUNK in hh_links.cu)
N_CTG = 4000
ENV = {"HH_LINKS_NPART_LOG": 2, "HH_LINKS_SUB_LOG_MAX": 2}


@pytest.fixture(scope="module")
def ctx():
    from haphic_b200._lib import Context
    c = Context(0)
    yield c
    c.close()


def key_pool(seed):
    """Distinct contig pairs (i < j) of N_CTG contigs, grouped by sub-partition: the top 2 + 2 hash bits."""
    rng = np.random.default_rng(seed)
    i = rng.integers(0, N_CTG, 600_000)
    j = rng.integers(0, N_CTG, 600_000)
    i, j = np.minimum(i, j), np.maximum(i, j)
    keys = np.unique((i[i != j].astype(np.uint64) << np.uint64(32)) | j[i != j].astype(np.uint64))
    keys = keys[rng.permutation(len(keys))]
    sub = (mix64(keys) >> np.uint64(60)).astype(np.int64)
    return [keys[sub == s] for s in range(16)]


def shaped_stream(n_rec, n_keys, seed):
    """Sub-partition s (of 4 partitions x 4) gets exactly n_rec[s] records over exactly n_keys[s] distinct contig pairs,
    ends swapped at random, random positions, in random order."""
    rng = np.random.default_rng(seed)
    pool = key_pool(seed)
    kk = []
    for s in range(16):
        keys = pool[s][:n_keys[s]]
        assert len(keys) == n_keys[s] and n_rec[s] >= n_keys[s]
        kk.append(np.concatenate([keys, rng.choice(keys, n_rec[s] - n_keys[s])]) if n_keys[s] else keys)
    kk = np.concatenate(kk)
    a = (kk >> np.uint64(32)).astype(np.int32)
    b = (kk & np.uint64(0xFFFFFFFF)).astype(np.int32)
    swap = rng.random(len(kk)) < 0.5
    a, b = np.where(swap, b, a), np.where(swap, a, b)
    lengths = np.full(N_CTG, 2_000_000, np.int64)
    rec = np.stack([a, rng.integers(0, 2_000_000, len(kk)), b, rng.integers(0, 2_000_000, len(kk))], 1).astype(np.int32)
    return lengths, np.arange(N_CTG, dtype=np.int32), np.ascontiguousarray(rec[rng.permutation(len(rec))])


def one_big_sub(big_rec, big_keys, seed):
    # sub-partition 0 is the one under test; the other 15 hold 400 records of 150 keys (one chunk each), so that every
    # partition has more than 2 x CHUNK records and the level-2 fan-out is the full 2 bits
    return shaped_stream([big_rec] + [400] * 15, [big_keys] + [150] * 15, seed)


@pytest.mark.parametrize("n", [1, 100, 4095, 4096, 4097, 3 * 4096 + 17])
def test_stream_not_a_multiple_of_the_tile(ctx, monkeypatch, n):
    lengths, rank, rec = synth_stream(2000, n, 50 + n % 97)
    assert check_same(ctx, monkeypatch, lengths, rank, rec, {"HH_LINKS_NPART_LOG": 3}) == 0


@pytest.mark.parametrize("big", [CHUNK - 1, CHUNK, CHUNK + 1])
def test_sub_partition_at_the_chunk_size(ctx, monkeypatch, big):
    lengths, rank, rec = one_big_sub(big, 300, 60 + big % 7)
    assert check_same(ctx, monkeypatch, lengths, rank, rec, ENV) == 0


def test_multi_chunk_sub_partition_fits(ctx, monkeypatch):
    # nine chunks of a sub-partition whose keys all fit the table: counted in shared memory across the chunks
    lengths, rank, rec = one_big_sub(9 * CHUNK - 5, SLOTS - 300, 70)
    assert check_same(ctx, monkeypatch, lengths, rank, rec, ENV) == 0


def test_multi_chunk_sub_partition_overflows_mid_way(ctx, monkeypatch):
    # one record per key: the table fills in the second chunk and overflows in the third, and the sub-partition goes to
    # the scratch-table path; its later chunks are skipped, the other 15 sub-partitions are counted in shared memory
    lengths, rank, rec = one_big_sub(4 * CHUNK, 4 * CHUNK, 71)
    assert check_same(ctx, monkeypatch, lengths, rank, rec, ENV) == 1


@pytest.mark.parametrize("keys, fallbacks", [(SLOTS, 0), (SLOTS + 1, 1)])
def test_table_filled_to_the_threshold(ctx, monkeypatch, keys, fallbacks):
    # exactly as many distinct keys as the table has slots: every slot is live and emitted; one more falls back
    lengths, rank, rec = one_big_sub(keys + 500, keys, 72)
    assert check_same(ctx, monkeypatch, lengths, rank, rec, ENV) == fallbacks


def counted(ctx, monkeypatch, lengths, rank, parts, env):
    from haphic_b200.links import LinkTable
    for k in ("HH_LINKS_PARTITION", "HH_LINKS_NPART_LOG", "HH_LINKS_SUB_LOG_MAX"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    tab = LinkTable(ctx, lengths, rank, np.ones(len(lengths), np.uint8), 500000)
    off = 0
    for p in parts:
        tab.add(p, stream_offset=off)
        off += len(p)
    info = tab.finish()
    got = tab.fetch()
    tot = tab.fetch_ctg()
    tab.close()
    return (info.n_records, info.n_used, info.nnz_full, info.nnz_flank), got, tot


def test_several_adds_several_partition_sets(ctx, monkeypatch):
    # the first add sizes the partition regions; the later, larger ones do not fit them and get region sets of their own
    lengths, rank, rec = synth_stream(2000, 1_500_000, 81)
    parts = [rec[:100_000], rec[100_000:700_000], rec[700_000:701_234], rec[701_234:]]
    want = counted(ctx, monkeypatch, lengths, rank, parts, {"HH_LINKS_PARTITION": 0})
    got = counted(ctx, monkeypatch, lengths, rank, parts, {"HH_LINKS_PARTITION": 1, "HH_LINKS_NPART_LOG": 4})
    assert got[0] == want[0]
    for k in want[1]:
        assert np.array_equal(got[1][k], want[1][k]), k
    assert np.array_equal(got[2], want[2])
