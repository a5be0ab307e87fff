"""GPU tests of the pair screens over chosen SNP sets (GenoStore.pairwise_scan_sets: within a set, set-by-all, set-by-set).

Every record must be bit-identical to the whole-table screen's record of that pair: the set screen's result is the whole-table
hit list filtered to the pairs {i in A, j in B}, i != j, record for record. The cohorts are those of the screen-edge tests (all
four tensor-core modes, partial and overlapping selections) plus a table whose gathered sub-table spans several L2 bands.
"""
import numpy as np
import pytest

import libgwaspp_b200 as gw
from test_gpu_screen_edges import LOW, SELECTION_COHORTS, Ref, check_oracle, overlap_masks, plant, store_of, tie_cohort, top_k_of

pytestmark = pytest.mark.gpu


def in_sets(h, a, b):
    """records of h whose pair has one SNP in A and the other in B (b=None: both in A)"""
    M = int(max(h["i"].max(initial=0), h["j"].max(initial=0))) + 1
    M = max(M, int(np.max(a, initial=0)) + 1, 0 if b is None else int(np.max(b, initial=0)) + 1)
    ia = np.zeros(M, bool); ia[a] = True
    ib = ia if b is None else np.zeros(M, bool)
    if b is not None:
        ib[b] = True
    keep = (ia[h["i"]] & ib[h["j"]]) | (ib[h["i"]] & ia[h["j"]])
    return h[keep]


def formula(a, b):
    b = a if b is None else b
    c = len(np.intersect1d(a, b))
    return len(a) * len(b) - c - c * (c - 1) // 2


def make_sets(rng, M, n_a, n_b, n_c):
    pool = rng.permutation(M)
    c = pool[:n_c]
    a = np.sort(np.concatenate([c, pool[n_c:n_a]]))
    b = np.sort(np.concatenate([c, pool[n_a:n_a + n_b - n_c]]))
    return a.astype(np.uint32), b.astype(np.uint32)


def set_shapes(M, seed):
    rng = np.random.default_rng(seed)
    out = {"within": (np.sort(rng.choice(M, M // 3, replace=False)).astype(np.uint32), None)}
    a, b = make_sets(rng, M, 40, M // 2, 40)
    out["a_in_b"] = (a, b)
    out["a_by_all"] = (np.sort(rng.choice(M, 25, replace=False)).astype(np.uint32), np.ones(M, bool))
    out["overlap"] = make_sets(rng, M, M // 3, M // 4, 30)
    out["disjoint"] = make_sets(rng, M, M // 3, M // 3, 0)
    for c in (1, 64, 129):
        out[f"c{c}"] = make_sets(rng, M, c + 20, c + 45, c)
    return out


def check_shape(st, a, b, full_by_thr, top_ref):
    bb = None if b is None else (np.flatnonzero(b).astype(np.uint32) if b.dtype == bool else b)
    for thr, full in full_by_thr.items():
        want = in_sets(full, a, bb)
        h, s = st.pairwise_scan_sets(a, b, thr)
        assert np.array_equal(h, want), (thr, len(h), len(want))
        assert s.pairs_tested == formula(a, bb) and s.engine == 2
        assert s.total_ms >= s.screen_ms > 0
    for k in (1, 7):
        top, _ = st.pairwise_scan_sets(a, b, LOW, top_k=k)
        assert np.array_equal(top, top_k_of(in_sets(top_ref, a, bb), k)), k
    h, _ = st.pairwise_scan_sets(a, b, 30.0)
    for n in (2, 3):
        parts = [st.pairwise_scan_sets(a, b, 30.0, shard=r, n_shards=n) for r in range(n)]
        merged = np.sort(np.concatenate([p[0] for p in parts]), order=["i", "j"])
        assert len(merged) == len(h) and np.array_equal(merged, h), n      # disjoint shards whose union is the whole
        assert sum(p[1].pairs_tested for p in parts) == formula(a, bb)


@pytest.mark.parametrize("mode", list(SELECTION_COHORTS))
def test_sets_equal_the_filtered_whole_table_screen(orc, mode):
    M, N, (fca, fco, fne), miss = SELECTION_COHORTS[mode]
    rng = np.random.default_rng(len(mode) * 1000 + M)
    codes, _ = orc.simulate(4242 + M, M, N, N // 2, missing_rate=miss)
    if miss:
        codes[:128][codes[:128] == 3] = 0
    pheno = rng.choice([1, 0, 2], size=N, p=[fca, fco, fne]).astype(np.uint8)
    ca, co, eff = overlap_masks(pheno, rng, 23)
    plant(codes, eff == 1, rng, 6)
    rows = orc.pack_codes(codes)
    ref = Ref(orc, rows, N, eff)
    want_lo = ref.screen(LOW)
    with store_of(rows, N, ca, co) as st:
        full = {thr: st.pairwise_scan(thr, capacity=M * M)[0] for thr in (30.0, LOW)}
        check_oracle(full[LOW], want_lo, N)
        for name, (a, b) in set_shapes(M, 11).items():
            check_shape(st, a, b, full, full[LOW])
        # the oracle, filtered the same way
        a, b = set_shapes(M, 11)["overlap"]
        h, _ = st.pairwise_scan_sets(a, b, LOW)
        hi, hj, hs = want_lo
        rec = np.zeros(len(hi), gw.HIT_DTYPE)
        rec["i"], rec["j"], rec["stat"] = hi, hj, hs
        w = in_sets(rec, a, b)
        check_oracle(h, (w["i"], w["j"], w["stat"]), N)


def test_sets_on_a_table_of_several_bands():
    """5 000 SNPs x 2 000 samples, |A| = 3 000: the sub-table spans several L2 bands of the schedule."""
    M, N = 5000, 2000
    with gw.GenoStore(M, N) as st:
        st.simulate(99, missing_rate=0.0)
        st.select_case_control(gw.simulate_phenotype(99, N, 1000))
        rng = np.random.default_rng(3)
        a = np.sort(rng.choice(M, 3000, replace=False)).astype(np.uint32)
        b = np.sort(rng.choice(M, 1200, replace=False)).astype(np.uint32)
        for thr in (12.0, 30.0):
            full, _ = st.pairwise_scan(thr)
            for bb in (None, b):
                h, s = st.pairwise_scan_sets(a, bb, thr)
                assert np.array_equal(h, in_sets(full, a, bb)), (thr, bb is None)
                assert s.pairs_tested == formula(a, bb)
        tiles, _ = gw.set_schedule(M, a, None, n_samples=N)
        assert tiles[:, 0].max() > 16
        full, _ = st.pairwise_scan(12.0)
        top, _ = st.pairwise_scan_sets(a, None, 12.0, top_k=500)
        assert np.array_equal(top, top_k_of(in_sets(full, a, None), 500))
        parts = [st.pairwise_scan_sets(a, None, 12.0, shard=r, n_shards=3)[0] for r in range(3)]
        assert np.array_equal(np.sort(np.concatenate(parts), order=["i", "j"]), in_sets(full, a, None))


def test_sets_topk_ties(orc):
    copies = [10, 70, 130, 200, 250, 319]
    rows, N, pheno = tie_cohort(orc, copies)
    M, thr = rows.shape[0], 2.0
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        full, _ = st.pairwise_scan(thr, capacity=M * M)
        a = np.array(sorted({3, *copies, *range(100, 180)}), np.uint32)
        for b in (None, np.arange(M, dtype=np.uint32)):
            filt = in_sets(full, a, b)
            tied = np.sort(filt["stat"])[::-1]
            ks = [1] + [k for k in range(2, 40) if tied[k - 1] == tied[k]][:3]
            for k in ks:
                top, _ = st.pairwise_scan_sets(a, b, thr, top_k=k)
                assert np.array_equal(top, top_k_of(filt, k)), k


def test_sets_in_realistic_workflows(orc):
    M, N = 600, 3000
    codes, pheno = orc.simulate(777, M, N, 1400)
    rng = np.random.default_rng(777)
    plant(codes, pheno == 1, rng, 5)
    rows = orc.pack_codes(codes)
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        full, _ = st.pairwise_scan(20.0)
        # a pruned set: ld_prune's keep mask passed as is
        keep = st.ld_prune(50, 0.05)
        assert keep.dtype == bool and 0 < keep.sum() < M
        h, s = st.pairwise_scan_sets(keep, None, 20.0)
        idx = np.flatnonzero(keep).astype(np.uint32)
        assert np.array_equal(h, in_sets(full, idx, None)) and s.pairs_tested == formula(idx, None)
        # set-by-all with the most significant SNPs of the marginal scan
        rec, _ = st.marginal_scan_compact()
        top = np.sort(np.argsort(rec["p_genotypic"], kind="stable")[:30]).astype(np.uint32)
        h2, s2 = st.pairwise_scan_sets(top, np.ones(M, bool), 20.0)
        assert np.array_equal(h2, in_sets(full, top, np.arange(M))) and len(h2) > 0
        assert s2.pairs_tested == formula(top, np.arange(M))
        stat, z = st.gtest(h2["i"], h2["j"])
        assert len(stat) == len(h2) and np.all(np.isfinite(z))


def test_sets_leave_the_parent_store_alone(orc):
    M, N = 300, 1500
    codes, pheno = orc.simulate(31337, M, N, 700, missing_rate=0.01)
    rows = orc.pack_codes(codes)
    a = np.arange(0, M, 3, dtype=np.uint32)
    with store_of(rows, N) as fresh, store_of(rows, N) as other:
        fresh.select_case_control(pheno)
        other.select_case_control(pheno)
        first, _ = fresh.pairwise_scan_sets(a, None, 10.0)     # a set screen as the first screen of a store
        before, _ = other.pairwise_scan(10.0)
        assert np.array_equal(first, in_sets(before, a, None))
        other.pairwise_scan_sets(a, np.ones(M, bool), 10.0)
        after, _ = other.pairwise_scan(10.0)
        assert np.array_equal(after, before)
        assert np.array_equal(fresh.pairwise_scan(10.0)[0], before)


def test_sets_errors(orc):
    M, N = 200, 800
    codes, pheno = orc.simulate(5, M, N, 400)
    rows = orc.pack_codes(codes)
    with store_of(rows, N) as st:
        with pytest.raises(gw.GwasDevError):
            st.pairwise_scan_sets([1, 2, 3])                      # no selection
        st.select_case_control(pheno)
        for a, b in (([3, 2], None), ([1, 1, 4], None), ([1, M], None), ([1, 2], [9, 8]), ([1, 2], [5, 5])):
            with pytest.raises(gw.GwasDevError):
                st.pairwise_scan_sets(np.array(a), None if b is None else np.array(b))
        st.set_pair_engine(1)
        with pytest.raises(gw.GwasDevError, match="tensor-core"):
            st.pairwise_scan_sets([1, 2, 3])
        st.set_pair_engine(0)
        h, s = st.pairwise_scan_sets(np.array([], np.uint32))
        assert len(h) == 0 and s.pairs_tested == 0
        h, _ = st.pairwise_scan_sets([1, 2, 3], np.array([], np.uint32))
        assert len(h) == 0
