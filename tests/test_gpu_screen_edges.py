"""GPU tests of the exhaustive pair screen at the edges of its dispatch and arithmetic.

One pair-screen call runs one of five kernels (two-plane tensor cores, the four-plane kernel in its missing-call, split-class
and two-accumulator modes, AND+POPC), and the two-plane kernel chooses per SNP which genotype classes go on the tensor cores and
drops pairs with an fp32 upper bound whose constant depends on the case fraction. The cohorts here are built to reach what
HWE-simulated 0/1 phenotypes do not: samples outside both classes or flagged in both masks, class sizes at the packed
accumulator's limits, extreme case fractions, degenerate SNPs at block edges, and exact ties at the k-th place of top-k.

The reference is always the C oracle (oracle/gwas_oracle.c); the AND+POPC engine is a cross-check only. Bars as everywhere:
records, counts and tables bit-exact, fp64 statistics within 1e-12 relative (of N ln N for statistics smaller than that:
see check_oracle), NaN patterns equal.
"""
import numpy as np
import pytest

import libgwaspp_b200 as gw
from helpers import rel_close

pytestmark = pytest.mark.gpu
REL_F64 = 1e-12
LOW = -1e9                 # every pair with a finite statistic


# ------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------
def n_gpus():
    return int(gw.load_library().gwasdev_device_count())


def top_k_of(hits, k):
    """the k largest statistics, ties at the k-th place to the smaller (i, j); returned in (i, j) order"""
    order = np.lexsort((hits["j"], hits["i"], -hits["stat"]))[:k]
    return np.sort(hits[order], order=["i", "j"])


def plant(codes, is_case, rng, n_pairs, first=0):
    """case-only dependencies between common SNPs (rows >= first), so that a threshold of 30 has hits"""
    N = codes.shape[1]
    cand = [r for r in range(first, codes.shape[0]) if (codes[r] == 2).sum() > 0.04 * N]
    rng.shuffle(cand)
    for k in range(n_pairs):
        i, j = sorted((cand[2 * k], cand[2 * k + 1]))
        src = codes[i].copy()
        src[src == 3] = 0
        codes[j, is_case] = src[is_case]


def overlap_masks(pheno, rng, n_both):
    """class masks of pheno with n_both extra samples flagged in both; the effective labels (both -> case)"""
    ca, co = gw.stream_masks(pheno)
    eff = pheno.copy()
    for c in rng.choice(len(pheno), n_both, replace=False):
        ca[c >> 4] |= np.uint16(1 << (c & 15))
        co[c >> 4] |= np.uint16(1 << (c & 15))
        eff[c] = 1
    return ca, co, eff


def store_of(rows, N, ca=None, co=None, *, eager=False, device=0):
    st = gw.GenoStore(rows.shape[0], N, device=device)
    if eager:
        st.set_select_mode(True)
    st.put_rows(rows)
    if ca is not None:
        st.select_case_control(case_mask=ca, ctrl_mask=co)
    return st


class Ref:
    """the oracle's view of one selection: compacted rows, margins, and its screen"""

    def __init__(self, orc, rows, N, eff):
        self.orc = orc
        self.sel, self.nca, self.nco = orc.select(rows, N, eff)
        self.mar = orc.margins(self.sel, self.nca, self.nco)

    def screen(self, thr):
        hi, hj, hs, _ = self.orc.boost_screen(self.sel, self.mar, self.nca, self.nco, thr, cap=1 << 22)
        return hi, hj, hs

    def ksa(self, i, j):
        ca, co = self.orc.pair_table(3, i, j, sel=self.sel, nca=self.nca, nco=self.nco, mar=self.mar)
        return self.orc.ksa(ca, co, self.mar[i], self.mar[j], self.nca + self.nco)


def check_oracle(h, want, N):
    """records equal the oracle's: (i, j) exactly, statistics within 1e-12 relative -- or within 1e-12 N ln N where the statistic
    is smaller than that: it is a sum of terms of magnitude up to N ln N that cancel for pairs near independence, so the fp64
    rounding of those terms, not the size of the result, bounds the agreement of two implementations there"""
    hi, hj, hs = want
    assert len(h) == len(hi) and np.array_equal(h["i"], hi) and np.array_equal(h["j"], hj), (len(h), len(hi))
    scale = np.maximum(np.abs(hs), N * np.log(N))
    err = np.abs(h["stat"] - hs) / scale
    assert np.all(err <= REL_F64), float(np.max(err))


def gap_threshold(stats, n_above):
    """a threshold with about n_above statistics above it, halfway between two neighbours far enough apart that no rounding
    difference between implementations moves a pair across it"""
    s = np.sort(stats[np.isfinite(stats)])[::-1]
    k = n_above
    while s[k - 1] - s[k] <= 1e-5 * max(1.0, abs(s[k])):
        k += 1
    return float((s[k - 1] + s[k]) / 2)


def above(ref_hits, thr):
    hi, hj, hs = ref_hits
    k = hs > thr
    return hi[k], hj[k], hs[k]


def expected_tile(st, M, I, J):
    """[64, 128, 2, 4] corner counts from the per-call margins-overload tables (zero outside the table)"""
    A, B = np.meshgrid(np.arange(64 * I, 64 * I + 64), np.arange(128 * J, 128 * J + 128), indexing="ij")
    ok = (A < M) & (B < M)
    t = st.pair_tables(A[ok], B[ok], mode=3).reshape(-1, 2, 16)
    exp = np.zeros((64, 128, 2, 4), np.uint32)
    exp[ok] = t[:, :, [0, 2, 8, 10]]          # AA_BB, AA_bb, aa_BB, aa_bb of the 4x4 table
    return exp


def relabel_homozygotes(row, P):
    """the same SNP with its two homozygote classes swapped in the packed row: codes 1 (plane 1) <-> 3 (both planes)"""
    out = row.copy()
    out[1 + P:1 + 2 * P] ^= out[1:1 + P]
    return out


def merged_shards(st, thr, n):
    parts = [st.pairwise_scan(thr, shard=k, n_shards=n) for k in range(n)]
    return np.sort(np.concatenate([p[0] for p in parts]), order=["i", "j"]), sum(p[1].pairs_tested for p in parts)


# ------------------------------------------------------------------------------------------------------
# A. partial and overlapping selections in every screen mode
# ------------------------------------------------------------------------------------------------------
# (mode, M, N, case / control / neither fractions, missing rate); modes 1 and 2 need n_case >= 16384
SELECTION_COHORTS = {
    "two_plane": (300, 1500, (0.40, 0.45, 0.15), 0.0),
    "four_plane_missing": (300, 1500, (0.40, 0.45, 0.15), 0.01),
    "split_classes": (200, 40000, (0.50, 0.35, 0.15), 0.0),
    "two_accumulators": (200, 40000, (0.50, 0.35, 0.15), 0.003),
}


@pytest.mark.parametrize("mode", list(SELECTION_COHORTS))
def test_partial_and_overlapping_selections(orc, mode):
    """Phenotypes 0 / 1 / 2 (2 = neither class) plus samples flagged in both masks (effective label: case). The tensor-core
    operands are built from the raw rows and the selection's class masks, so a mask mistake counts samples that are in neither
    class; the lazy store (masks on the raw rows) and an eager one (compacted rows) must both give the oracle's records."""
    M, N, (fca, fco, fne), miss = SELECTION_COHORTS[mode]
    rng = np.random.default_rng(len(mode) * 1000 + M)
    codes, _ = orc.simulate(4242 + M, M, N, N // 2, missing_rate=miss)
    if miss:
        codes[:128][codes[:128] == 3] = 0                      # two complete 64-SNP blocks: mixed tiles
    pheno = rng.choice([1, 0, 2], size=N, p=[fca, fco, fne]).astype(np.uint8)
    ca, co, eff = overlap_masks(pheno, rng, 23)
    plant(codes, eff == 1, rng, 6)
    rows = orc.pack_codes(codes)
    ref = Ref(orc, rows, N, eff)
    big = ref.nca >= 16384
    assert big == mode.startswith(("split", "two_acc"))
    with store_of(rows, N, ca, co) as st, store_of(rows, N, ca, co, eager=True) as ev:
        assert (st.n_case, st.n_ctrl) == (ev.n_case, ev.n_ctrl) == (ref.nca, ref.nco)
        assert not st.is_compacted() and ev.is_compacted()
        # the selection's tables against the oracle's for a sample of pairs
        pi, pj = rng.integers(0, M, 40), rng.integers(0, M, 40)
        t = st.pair_tables(pi, pj, mode=3)
        for q in range(40):
            w_ca, w_co = orc.pair_table(3, int(pi[q]), int(pj[q]), sel=ref.sel, nca=ref.nca, nco=ref.nco, mar=ref.mar)
            assert np.array_equal(t[q, :16], w_ca) and np.array_equal(t[q, 16:], w_co)
        want_hi, want_lo = ref.screen(30.0), ref.screen(LOW)
        assert len(want_hi[0]) >= 3 and len(want_lo[0]) > 100 * len(want_hi[0])
        got = {}
        for thr, want in ((30.0, want_hi), (LOW, want_lo)):
            h, s = st.pairwise_scan(thr, capacity=M * M)
            assert s.engine == 2 and s.pairs_tested == M * (M - 1) // 2
            assert (s.tiles_nine_cell > 0) == (miss > 0)
            assert s.candidates >= len(h) > 0                   # candidates went through the fp32 epilogue
            check_oracle(h, want, N)
            he, _ = ev.pairwise_scan(thr, capacity=M * M)
            assert np.array_equal(he, h), thr
            st.set_pair_engine(1)                               # every class here is below 65536
            h1, s1 = st.pairwise_scan(thr, capacity=M * M)
            st.set_pair_engine(0)
            assert s1.engine == 1 and np.array_equal(h1, h), thr
            got[thr] = h
        h = got[30.0]
        if not big:                                             # the two-plane kernel's corner counts of one tile
            for I, J in ((1, 0), (4, 2)):
                assert np.array_equal(st.mma_tile_counts(I, J), expected_tile(st, M, I, J)), (I, J)
        k1, k2 = st.ksa(h["i"], h["j"]), ev.ksa(h["i"], h["j"])
        assert np.array_equal(k1, k2) and np.array_equal(k1, h["stat"])
        g1, g2 = st.gtest(h["i"], h["j"]), ev.gtest(h["i"], h["j"])
        assert np.array_equal(g1[0], g2[0]) and np.array_equal(g1[1], g2[1], equal_nan=True)
        merged, pairs = merged_shards(st, 30.0, 3)
        assert pairs == M * (M - 1) // 2 and np.array_equal(merged, h)
        # another selection, then back: operands, plane choice and bound constants must follow the selection
        pheno2 = rng.choice([1, 0, 2], size=N, p=[fco, fca, fne]).astype(np.uint8)
        ca2, co2, eff2 = overlap_masks(pheno2, rng, 11)
        ref2 = Ref(orc, rows, N, eff2)
        st.select_case_control(case_mask=ca2, ctrl_mask=co2)
        want2 = ref2.screen(LOW)
        thr2 = gap_threshold(want2[2], 300)                     # the planted pairs need not stand out in this selection
        h2, _ = st.pairwise_scan(thr2)
        assert len(h2) >= 300
        check_oracle(h2, above(want2, thr2), N)
        check_oracle(st.pairwise_scan(LOW, capacity=M * M)[0], want2, N)
        if ref2.nca < 16384 and ref2.nco < 131072:
            assert np.array_equal(st.mma_tile_counts(1, 0), expected_tile(st, M, 1, 0))
        st.select_case_control(case_mask=ca, ctrl_mask=co)
        again, _ = st.pairwise_scan(30.0)
        assert np.array_equal(again, h)
        lo_again, _ = st.pairwise_scan(LOW, capacity=M * M)
        assert np.array_equal(lo_again, got[LOW])
        if not big:
            assert np.array_equal(st.mma_tile_counts(4, 2), expected_tile(st, M, 4, 2))


# ------------------------------------------------------------------------------------------------------
# B. dispatch and the packed accumulator's limits
# ------------------------------------------------------------------------------------------------------
def expected_dispatch(nca, nco, missing, four_plane, engine):
    """gwasdev_set_pair_engine's table: (stats.engine, tile with missing calls on a 9-cell kernel?) or None (the call needs
    the AND+POPC kernels with a class of 65536 or more and must fail)"""
    popc_ok = nca < 65536 and nco < 65536
    if engine == 1:
        return (1, missing) if popc_ok else None
    if nca < 16384 and nco < 131072:                   # two-plane kernel for the complete tiles
        if missing and four_plane and not popc_ok:      # FOUR_PLANE = 1: tiles with missing calls stay on AND+POPC
            return None
        return 2, missing
    if not four_plane:                                  # split classes (complete) / two accumulators (missing calls)
        return 2, missing
    return (1, missing) if popc_ok else None            # FOUR_PLANE = 1 also turns the per-class modes off


@pytest.mark.parametrize("nca,nco,M", [(16383, 131071, 250), (16384, 1000, 230), (1000, 131072, 210), (2000, 70000, 260)])
def test_dispatch_and_accumulator_limits(orc, nca, nco, M):
    """The largest two-plane cohort, the first split cohorts on either side, and a two-plane cohort beyond what the AND+POPC
    engine accepts; each complete and with missing calls, with GWASDEV_OPT_FOUR_PLANE 0 and 1 and both engine settings."""
    N = nca + nco
    rng = np.random.default_rng(nca ^ nco)
    codes, _ = orc.simulate(977 + M, M, N, nca)
    pheno = np.zeros(N, np.uint8)
    pheno[rng.choice(N, nca, replace=False)] = 1
    plant(codes, pheno == 1, rng, 4, first=8)
    mono = [1, 2, 3]                                   # monomorphic over all samples (two AA, one BB)
    codes[1] = codes[2] = 0
    codes[3] = 2
    near = [5, 6]                                      # monomorphic except for a handful of samples of both classes
    for r in near:
        codes[r] = 0
        odd = np.concatenate([rng.choice(np.flatnonzero(pheno == 1), 4, replace=False),
                              rng.choice(np.flatnonzero(pheno == 0), 5, replace=False)])
        codes[r, odd] = rng.integers(1, 3, len(odd))
    two_plane = nca < 16384 and nco < 131072
    for missing in (False, True):
        cm = codes.copy()
        if missing:                                    # rows 0..127 stay complete: mixed tiles
            tail = cm[128:]
            tail[rng.random(tail.shape) < 0.002] = 3
        rows = orc.pack_codes(cm)
        ref = Ref(orc, rows, N, pheno)
        assert (ref.nca, ref.nco) == (nca, nco)
        want_lo = ref.screen(LOW)
        want_hi = above(want_lo, 30.0)
        thr_q = gap_threshold(want_lo[2], 300)         # 300 pairs above: many near it, where a wrong fp32 value shows
        want_q = above(want_lo, thr_q)
        assert len(want_hi[0]) >= 3 and len(want_lo[0]) > 0.9 * M * (M - 1) // 2 - 3 * M
        with store_of(rows, N) as st:
            st.select_case_control(pheno)
            for engine, fp in ((0, 0), (0, 1), (1, 0)):
                st.set_pair_engine(engine)
                st.set_option(gw.OPT_FOUR_PLANE, fp)
                exp = expected_dispatch(nca, nco, missing, fp, engine)
                if exp is None:
                    with pytest.raises(gw.GwasDevError, match="65535"):
                        st.pairwise_scan(30.0)
                    continue
                for thr, want in ((30.0, want_hi), (thr_q, want_q), (LOW, want_lo)):
                    h, s = st.pairwise_scan(thr, capacity=M * M)
                    assert (s.engine, s.tiles_nine_cell > 0) == exp, (engine, fp, thr)
                    assert s.pairs_tested == M * (M - 1) // 2
                    check_oracle(h, want, N)
            st.set_pair_engine(0)
            st.set_option(gw.OPT_FOUR_PLANE, 0)
            if not two_plane:
                for probe in (lambda: st.mma_tile_counts(0, 0), lambda: st.ksa_screen_mma_f32([0], [1])):
                    with pytest.raises(gw.GwasDevError, match="outside the tensor-core engine's range"):
                        probe()
            elif not missing:
                for I, J in ((0, 0), ((M - 1) // 64, (M - 1) // 128)):
                    got = st.mma_tile_counts(I, J)
                    assert np.array_equal(got, expected_tile(st, M, I, J)), (I, J)
                    if (I, J) == (0, 0):
                        corners = [tuple(int(v) for v in got[1, 2, :, c]) for c in range(4)]
                        assert (nca, nco) in corners    # every sample in one corner of two monomorphic SNPs
                        if (nca, nco) == (16383, 131071):
                            assert nca + (nco << 14) == 2 ** 31 - 1
            # near-monomorphic pairs: finite statistics equal to the oracle's
            pairs = [(1, 5), (5, 6), (3, 6)] + [(r, 9 + r) for r in near]
            got = st.ksa([p[0] for p in pairs], [p[1] for p in pairs])
            for (i, j), v in zip(pairs, got):
                w = ref.ksa(i, j)
                assert np.isfinite(w) and rel_close([v], [w], REL_F64), (i, j, v, w)
            lo = {(int(a), int(b)) for a, b in zip(want_lo[0], want_lo[1])}
            assert all(p in lo for p in pairs)
            assert not any((a, b) in lo for a in mono for b in mono if a < b)   # no statistic between monomorphic SNPs


# ------------------------------------------------------------------------------------------------------
# C. class imbalance and the bound pre-filter
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,nca", [(4000, 1), (20000, 200), (10000, 500), (4000, 800), (10000, 8000), (16000, 15200)])
def test_bound_prefilter_at_skewed_case_fractions(orc, N, nca):
    """qc of the upper bound grows like 1/x0 at a small case fraction x0, where qc Q - q0 cancels in fp32. Over all ~2e6 pairs of
    2 000 SNPs the bound may fall below the fp64 statistic by fp32 rounding only, inside half the screening margin; end to end,
    at a threshold with hundreds of pairs within the margin of it, both engines must report the oracle's records."""
    M = 2000
    rng = np.random.default_rng(N + nca)
    pheno = np.zeros(N, np.uint8)
    pheno[rng.choice(N, nca, replace=False)] = 1
    margin = max(0.5, 1e-4 * N)
    pi, pj = np.triu_indices(M, 1)
    with gw.GenoStore(M, N) as st:
        st.simulate(31337 + N + nca)
        st.select_case_control(pheno)
        assert (st.n_case, st.n_ctrl) == (nca, N - nca)
        f64_all = np.empty(len(pi))
        worst_ub, worst_f32 = np.inf, 0.0
        for b in range(0, len(pi), 1_000_000):
            a, c = pi[b:b + 1_000_000], pj[b:b + 1_000_000]
            both, f64 = st.ksa_screen_mma_f32(a, c), st.ksa(a, c)
            f32, ub = both[:, 0].astype(np.float64), both[:, 1].astype(np.float64)
            ok = ~np.isnan(f64)
            assert np.array_equal(np.isnan(ub), ~ok) and np.array_equal(np.isnan(f32), ~ok)
            if ok.any():
                worst_ub = min(worst_ub, float(np.min(ub[ok] - f64[ok])))
                worst_f32 = max(worst_f32, float(np.max(np.abs(f32[ok] - f64[ok]))))
            f64_all[b:b + len(a)] = f64
        print(f"N={N} n_case={nca}: {len(pi)} pairs ({int(np.isnan(f64_all).sum())} NaN), "
              f"min(ub - f64) = {worst_ub:.4f}, max|f32 - f64| = {worst_f32:.4f}, margin {margin}")
        assert worst_ub >= -margin / 2, (worst_ub, margin)
        assert worst_f32 <= margin / 2, (worst_f32, margin)
        # end to end on the first Me SNPs (the oracle's screen costs pairs x samples)
        Me = min(M, int(np.sqrt(6e9 / N)))
        rows = st.get_rows(0, Me)
    sub = (pi < Me) & (pj < Me)
    f = f64_all[sub]
    f = np.sort(f[np.isfinite(f)])
    thr = gap_threshold(f, 300)
    assert np.sum(np.abs(f - thr) <= margin) >= 100, "threshold without pairs near it"
    ref = Ref(orc, rows, N, pheno)
    want = ref.screen(thr)
    assert len(want[0]) >= 250
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        h2, s2 = st.pairwise_scan(thr)
        assert s2.engine == 2 and s2.candidates > len(h2)        # pairs inside the margin went through the fp32 epilogue
        st.set_pair_engine(1)
        h1, s1 = st.pairwise_scan(thr)
        assert s1.engine == 1
    assert np.array_equal(h2, h1)
    check_oracle(h2, want, N)


# ------------------------------------------------------------------------------------------------------
# D. degenerate SNPs and plane roles
# ------------------------------------------------------------------------------------------------------
def degenerate_cohort(orc, missing, seed=606):
    """260 SNPs x 1 200 samples (1 080 selected: 500 cases, 580 controls, 120 in neither class): simulated rows with planted
    pairs, and hand-made rows at the 64- and 128-SNP block edges (rows 0, 63, 64, 127, 128, 259 first), so that they take
    the A role and the B role of tiles. Class counts of the tie rows are counted over the selected samples."""
    M, N = 260, 1200
    rng = np.random.default_rng(seed + missing)
    codes, _ = orc.simulate(seed, M, N, 500, missing_rate=0.01 if missing else 0.0)
    pheno = np.full(N, 2, np.uint8)
    sel = rng.permutation(N)[:1080]
    pheno[sel[:500]] = 1
    pheno[sel[500:]] = 0
    plant(codes, pheno == 1, rng, 5, first=10)

    def classes(counts):                                # exact class counts over the selected samples, random elsewhere
        r = rng.integers(0, 3, N).astype(np.uint8)
        r[rng.permutation(sel)] = np.repeat(np.arange(3, dtype=np.uint8), counts)
        return r
    made = {
        "mono_aa": np.zeros(N, np.uint8), "mono_ab": np.ones(N, np.uint8),
        "aa_bb_only": rng.choice([0, 2], N).astype(np.uint8), "aa_ab_only": rng.choice([0, 1], N, p=[0.7, 0.3]).astype(np.uint8),
        "het_rarest": classes((560, 40, 480)),
        "tie_a_b_over_h": classes((420, 240, 420)), "tie_a_h_over_b": classes((420, 420, 240)), "tie_all": classes((360, 360, 360)),
    }
    if missing:
        made["all_missing"] = np.full(N, 3, np.uint8)
        made["called_in_cases_only"] = np.where(pheno == 1, codes[20], 3).astype(np.uint8)
        made["called_in_controls_only"] = np.where(pheno == 0, codes[21], 3).astype(np.uint8)
    # homozygote-relabelled copies (packed rows: the label machine would give a relabelled code sequence the same planes)
    copies = {"mono_bb": "mono_aa", "tie_h_b_over_a": "tie_a_h_over_b", "het_rarest_relabelled": "het_rarest", "simulated_relabelled": None}
    slots = [0, 63, 64, 127, 128, M - 1, 1, 62, 65, 126, 129, M - 2, 191, 192, 2, 61]
    names = list(made) + list(copies)
    assert len(names) <= len(slots)
    at = dict(zip(names, slots))
    for name, row in made.items():
        codes[at[name]] = row
    rows = orc.pack_codes(codes)
    P = (rows.shape[1] - 1) // 2
    for name, src in copies.items():
        rows[at[name]] = relabel_homozygotes(rows[at[src] if src else 100], P)
    return rows, N, pheno, at


@pytest.mark.parametrize("missing", [False, True])
def test_degenerate_snps_and_plane_roles(orc, missing):
    rows, N, pheno, at = degenerate_cohort(orc, missing)
    M = rows.shape[0]
    ref = Ref(orc, rows, N, pheno)
    m = ref.mar["margins"]
    # the hand-made class counts are what the tie rules see
    for name, (x, y, z) in (("tie_a_b_over_h", (420, 240, 420)), ("tie_all", (360, 360, 360))):
        assert tuple(int(v) for v in m[at[name]][:3]) == (x, y, z), name
    for name in ("tie_a_h_over_b", "tie_h_b_over_a"):
        assert sorted(int(v) for v in m[at[name]][:3]) == [240, 420, 420] and int(m[at[name]][1]) == 420, name
    assert int(m[at["het_rarest"]][1]) == 40 and int(m[at["mono_ab"]][1]) == 1080
    want = {thr: ref.screen(thr) for thr in (30.0, LOW)}
    assert len(want[30.0][0]) >= 3 and len(want[LOW][0]) > 100 * len(want[30.0][0])
    deg = [at[k] for k in ("mono_aa", "mono_ab", "mono_bb", "aa_bb_only", "aa_ab_only")]
    lo = set(zip(want[LOW][0].tolist(), want[LOW][1].tolist()))
    assert all(any(r in p for p in lo) for r in deg) and any(at["het_rarest"] in p for p in lo) and any(at["tie_all"] in p for p in lo)
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        results = {}
        for classic in (0, 1, 0):
            st.set_option(gw.OPT_CLASSIC_PLANES, classic)
            if not missing:                                   # the corner-count probe right after a plane-choice switch
                for I, J in ((0, 0), (1, 1), (4, 2)):
                    assert np.array_equal(st.mma_tile_counts(I, J), expected_tile(st, M, I, J)), (classic, I, J)
            for thr in (30.0, LOW):
                got, s = st.pairwise_scan(thr, capacity=M * M)
                assert s.engine == 2 and (s.tiles_nine_cell > 0) == missing
                check_oracle(got, want[thr], N)
                results.setdefault(thr, got)
                assert np.array_equal(got, results[thr]), (classic, thr)
        st.set_pair_engine(1)
        for thr in (30.0, LOW):
            assert np.array_equal(st.pairwise_scan(thr, capacity=M * M)[0], results[thr])
        st.set_pair_engine(0)
        if not missing:
            # the epilogue's fp32 value and bound on every pair of a hand-made SNP: NaN exactly where the statistic is NaN
            special = sorted(at.values())
            pi = np.concatenate([np.full(M, r) for r in special])
            pj = np.tile(np.arange(M), len(special))
            keep = pi != pj
            pi, pj = np.minimum(pi, pj)[keep], np.maximum(pi, pj)[keep]
            both, f64 = st.ksa_screen_mma_f32(pi, pj), st.ksa(pi, pj)
            ok = ~np.isnan(f64)
            assert np.array_equal(np.isnan(both[:, 0]), ~ok) and np.array_equal(np.isnan(both[:, 1]), ~ok)
            assert 0 < ok.sum() < len(ok)
            margin = max(0.5, 1e-4 * N)
            f32, ub = both[ok, 0].astype(np.float64), both[ok, 1].astype(np.float64)
            assert np.min(ub - f64[ok]) >= -margin / 2 and np.max(np.abs(f32 - f64[ok])) <= margin / 2
            for q in range(0, len(pi), 97):                     # and the fp64 statistic is the oracle's
                assert rel_close([f64[q]], [ref.ksa(int(pi[q]), int(pj[q]))], REL_F64), (pi[q], pj[q])


# ------------------------------------------------------------------------------------------------------
# E. exact ties in top-k
# ------------------------------------------------------------------------------------------------------
def tie_cohort(orc, copies, M=320, N=1000, seed=5150):
    """a strong planted pair (3, s) and `copies` identical rows of s: the pairs (3, copy) tie bit for bit"""
    rng = np.random.default_rng(seed)
    codes, pheno = orc.simulate(seed, M, N, 480)
    p = next(r for r in range(3, M) if 0.15 * N < (codes[r] == 2).sum() < 0.4 * N)
    codes[[3, p]] = codes[[p, 3]]
    s = copies[0]
    src = codes[3].copy()
    codes[s, pheno == 1] = src[pheno == 1]
    codes[copies] = codes[s]
    plant(codes, pheno == 1, rng, 2, first=4)
    return orc.pack_codes(codes), N, pheno


def tie_group(full, i, j):
    """(pairs with a larger statistic, size of the group tied with (i, j))"""
    v = full["stat"][(full["i"] == i) & (full["j"] == j)]
    assert len(v) == 1
    return int((full["stat"] > v[0]).sum()), int((full["stat"] == v[0]).sum())


def test_topk_ties_at_the_kth_place(orc):
    copies = [10, 70, 130, 200, 250, 319]
    rows, N, pheno = tie_cohort(orc, copies)
    M, thr = rows.shape[0], 2.0
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        full, _ = st.pairwise_scan(thr, capacity=M * M)
        assert len(full) > 0.3 * M * (M - 1) // 2
        ref = Ref(orc, rows, N, pheno)
        check_oracle(full, ref.screen(thr), N)
        start, size = tie_group(full, 3, copies[0])
        assert size >= len(copies)
        order = np.sort(full["stat"])[::-1]
        ks = [1, start + size - 1, start + size, start + size + 1]
        assert order[ks[1] - 1] == order[ks[1]]                # k = size - 1 cuts through the group
        for cap in (0, 4096):
            st.set_option(gw.OPT_CAND_CAPACITY, cap)
            for engine in (0, 1):
                st.set_pair_engine(engine)
                for k in ks:
                    top, s = st.pairwise_topk(k, thr)
                    assert np.array_equal(top, top_k_of(full, k)), (cap, engine, k)
                    parts = [st.pairwise_topk(k, thr, shard=r, n_shards=3)[0] for r in range(3)]
                    assert np.array_equal(top_k_of(np.concatenate(parts), k), top_k_of(full, k)), (cap, engine, k)
            if cap:
                assert s.candidates < len(full)                 # the device-wide threshold rose while the kernel ran
        st.set_option(gw.OPT_CAND_CAPACITY, 0)
        st.set_pair_engine(0)
        if n_gpus() >= 2:
            others = [st.replicate(d) for d in range(1, min(n_gpus(), 4))]
            try:
                for k in ks:
                    many, _ = gw.pairwise_scan_multi([st] + others, thr, top_k=k)
                    assert np.array_equal(many, top_k_of(full, k)), k
            finally:
                for o in others:
                    o.close()


def test_topk_tie_group_larger_than_the_candidate_buffer(orc):
    """150 identical rows: a group of 150 tied pairs at the top against a buffer of 64 candidates. The call returns the exact
    answer or reports that the buffer is too small; it never returns another list."""
    copies = list(range(100, 250))
    rows, N, pheno = tie_cohort(orc, copies, seed=5151)
    M, thr = rows.shape[0], 2.0
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        full, _ = st.pairwise_scan(thr, capacity=M * M)
        start, size = tie_group(full, 3, copies[0])
        assert size >= len(copies) > 64
        st.set_option(gw.OPT_CAND_CAPACITY, 64)
        outcomes = []
        for engine in (0, 1):
            st.set_pair_engine(engine)
            for k in (start + 20, start + size - 1):
                try:
                    top, _ = st.pairwise_topk(k, thr)
                except gw.GwasDevError as e:
                    assert "raise GWASDEV_OPT_CAND_CAPACITY" in str(e), str(e)
                    outcomes.append("refused")
                    continue
                assert np.array_equal(top, top_k_of(full, k)), (engine, k)
                outcomes.append("exact")
        print("tie group of", size, "against 64 candidates:", outcomes)
