"""CPU checks of the set screen's tile enumeration (gwasdev_set_schedule, host arithmetic): over many set shapes, every wanted
pair lies in exactly one shard's tiles, no listed tile lacks a wanted pair, the pair counts match the closed formula, and the
two-plane list is the whole-table schedule of the sub-table filtered to the tiles that hold a wanted pair."""
import numpy as np
import pytest

import libgwaspp_b200 as gw
from libgwaspp_b200 import build as gwbuild

M_TABLE = 5000


@pytest.fixture(scope="module", autouse=True)
def lib():
    gwbuild.build()
    return gw.load_library()


def segments(a, b):
    """The sub-table's rows as the library orders them: C = A n B, then A \\ B, then B \\ A; c1 = |C|, a1 = |C| + |A \\ B|."""
    b = a if b is None else b
    c = np.intersect1d(a, b)
    rows = np.concatenate([c, np.setdiff1d(a, b), np.setdiff1d(b, a)]).astype(np.int64)
    return rows, len(c), len(c) + len(np.setdiff1d(a, b))


def wanted_matrix(rows, c1, a1):
    """wanted[gi, gj] for sub-table positions, restated from the sets: {rows[gi], rows[gj]} has one SNP in A and one in B."""
    m = len(rows)
    gi, gj = np.meshgrid(np.arange(m), np.arange(m), indexing="ij")
    rule = (gi < gj) & ((gi < c1) | ((gi < a1) & (gj >= a1)))
    return rule


def formula(a, b):
    b = a if b is None else b
    c = len(np.intersect1d(a, b))
    return len(a) * len(b) - c - c * (c - 1) // 2


def set_pairs_brute(a, b):
    """Unordered pairs {i in A, j in B}, i != j, in table indices, as a set of (min, max)."""
    b = a if b is None else b
    out = set()
    for i in a:
        for j in b:
            if i != j:
                out.add((min(i, j), max(i, j)))
    return out


def make_sets(rng, n_a, n_b, n_c, disjoint_ok=True):
    """A and B with |A n B| = n_c, drawn from the table."""
    pool = rng.permutation(M_TABLE)
    c = pool[:n_c]
    a = np.concatenate([c, pool[n_c:n_c + n_a - n_c]])
    b = np.concatenate([c, pool[n_a:n_a + n_b - n_c]])
    return np.sort(a).astype(np.uint32), np.sort(b).astype(np.uint32)


def shapes():
    rng = np.random.default_rng(7)
    out = []
    # within A
    out.append(("within", np.sort(rng.choice(M_TABLE, 700, replace=False)).astype(np.uint32), None))
    # A subset of B, and B = all
    a, b = make_sets(rng, 300, 1500, 300)
    out.append(("a_in_b", a, b))
    out.append(("a_by_all", np.sort(rng.choice(M_TABLE, 90, replace=False)).astype(np.uint32), np.arange(M_TABLE, dtype=np.uint32)))
    # overlapping, disjoint
    a, b = make_sets(rng, 900, 700, 250)
    out.append(("overlap", a, b))
    a, b = make_sets(rng, 600, 800, 0)
    out.append(("disjoint", a, b))
    # |C| at the block edges
    for c in (0, 1, 63, 64, 65, 127, 128, 129):
        a, b = make_sets(rng, c + 70, c + 200, c)
        out.append((f"c{c}", a, b))
    # several bands (8 A-blocks per band at 20 000 samples) and more than 64 tiles per shard
    out.append(("bands", np.sort(rng.choice(M_TABLE, 3000, replace=False)).astype(np.uint32), None))
    return out


SHAPES = shapes()


@pytest.mark.parametrize("tile", [128, 64])
@pytest.mark.parametrize("name,a,b", SHAPES, ids=[s[0] for s in SHAPES])
def test_set_schedule_partitions_the_wanted_pairs(name, a, b, tile):
    rows, c1, a1 = segments(a, b)
    want = wanted_matrix(rows, c1, a1)
    # the segment rule restates the sets: the wanted pairs map onto the set pairs of the table one to one
    gi, gj = np.nonzero(want)
    ti, tj = rows[gi], rows[gj]
    mapped = set(zip(np.minimum(ti, tj).tolist(), np.maximum(ti, tj).tolist()))
    assert len(mapped) == len(gi) == formula(a, b)
    if len(a) * (len(a) if b is None else len(b)) <= 200_000:
        assert mapped == set_pairs_brute(a.tolist(), None if b is None else b.tolist())
    n_samples = 20_000
    for n_shards in (1, 2, 3):
        cover = np.zeros(want.shape, np.int32)
        total = 0
        for shard in range(n_shards):
            tiles, pairs = gw.set_schedule(M_TABLE, a, b, shard, n_shards, tile, n_samples)
            got = 0
            for I, J in tiles.tolist():
                assert I <= J
                blk = want[I * tile:(I + 1) * tile, J * tile:(J + 1) * tile]
                assert blk.any(), f"tile ({I}, {J}) holds no wanted pair"
                cover[I * tile:(I + 1) * tile, J * tile:(J + 1) * tile] += blk
                got += int(blk.sum())
            assert got == pairs
            total += pairs
            if name == "bands" and n_shards == 2:
                assert len(tiles) > 64
        assert total == formula(a, b)
        assert np.array_equal(cover, want.astype(np.int32)), "a wanted pair is not covered exactly once"


@pytest.mark.parametrize("name,a,b", SHAPES, ids=[s[0] for s in SHAPES])
def test_set_schedule_keeps_the_whole_table_order(name, a, b):
    """Two-plane tiles: the whole-table schedule of the sub-table (its L2 bands), filtered, dealt in chunks of 64 positions."""
    rows, c1, a1 = segments(a, b)
    want = wanted_matrix(rows, c1, a1)
    n_samples = 20_000
    full, _ = gw.shard_schedule(len(rows), 0, 1, engine=2, n_samples=n_samples)
    keep = [t for t in full.tolist() if want[t[0] * 128:(t[0] + 1) * 128, t[1] * 128:(t[1] + 1) * 128].any()]
    n_shards = 3
    for shard in range(n_shards):
        tiles, _ = gw.set_schedule(M_TABLE, a, b, shard, n_shards, 128, n_samples)
        mine = [t for p, t in enumerate(keep) if (p // 64) % n_shards == shard]
        assert tiles.tolist() == mine


def test_set_schedule_bands_span():
    a = SHAPES[-1][1]
    tiles, _ = gw.set_schedule(M_TABLE, a, None, 0, 1, 128, 20_000)
    assert tiles[:, 0].max() >= 16, "the large shape should span several bands of 8 A-blocks"


def test_set_schedule_refuses_bad_sets():
    for a, b in (([3, 2], None), ([1, 1], None), ([0, M_TABLE], None), ([1, 2], [5, 4]), ([1, 2], [7, 7])):
        with pytest.raises(gw.GwasDevError):
            gw.set_schedule(M_TABLE, np.array(a), None if b is None else np.array(b))
    with pytest.raises(gw.GwasDevError):
        gw.set_schedule(M_TABLE, [1, 2], tile_snps=96)
    with pytest.raises(gw.GwasDevError):
        gw.set_schedule(M_TABLE, np.ones(M_TABLE - 1, bool))


def test_set_schedule_empty_sets():
    for a, b in (([], None), ([5], None), ([], [1, 2, 3]), ([1, 2], [])):
        tiles, pairs = gw.set_schedule(M_TABLE, np.array(a, np.uint32), None if b is None else np.array(b, np.uint32))
        assert len(tiles) == 0 and pairs == 0
