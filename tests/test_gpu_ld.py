"""GPU tests of windowed linkage disequilibrium (gwasdev_ld_window, gwasdev_ld_pairs, GenoStore.ld_prune) against a numpy
restatement of the contract in include/gwasdev.h, on tables with real LD built in numpy and loaded with put_bed."""
import ctypes as C

import numpy as np
import pytest

import libgwaspp_b200 as gw
from helpers import band_of, decoded, ld_reference, list_of

pytestmark = pytest.mark.gpu


# ---- tables ---------------------------------------------------------------------------------------------------------------
def ld_table(M, N, seed, missing=0.0, founders=6, switch=0.02):
    """Genotypes (M, N) in {0, 1, 2, -1 missing}: two haplotypes per sample, each a mosaic of a few founder haplotypes (so r^2
    spans 0 to 1), plus planted duplicates, homozygote-relabelled copies, monomorphic and all-missing rows and rows called in
    only part of the samples."""
    rng = np.random.default_rng(seed)
    freq = rng.uniform(0.05, 0.95, M)
    F = (rng.random((founders, M)) < freq).astype(np.int8)
    def mosaic():
        src = np.zeros((N, M), np.int64)
        src[:, 0] = rng.integers(0, founders, N)
        for m in range(1, M):
            sw = rng.random(N) < switch
            src[:, m] = np.where(sw, rng.integers(0, founders, N), src[:, m - 1])
        return F[src, np.arange(M)[None, :]]
    G = (mosaic() + mosaic()).T.astype(np.int8)          # (M, N)
    if missing:
        G[rng.random((M, N)) < missing] = -1
    if N >= 4:
        for k in range(5, M, 97):                        # exact duplicates: r2 = 1
            G[k] = G[k - 1]
        for k in range(11, M, 89):                       # relabelled copies: first-seen labels flip when the copy's first homozygote differs
            G[k - 1, :2] = (0, 2)
            G[k] = np.where(G[k - 1] < 0, -1, 2 - G[k - 1])
            G[k, 0] = -1
        for k in range(17, M, 131):
            G[k] = 1 if k % 2 else 0                     # monomorphic
        for k in range(23, M, 151):
            G[k] = -1                                    # all missing
        for k in range(29, M, 113):
            G[k, rng.random(N) < 0.5] = -1               # called in part of the samples
    return G


def to_bed(G):
    code = np.array([1, 0, 2, 3], np.uint8)[G.astype(np.int64) + 1]    # -1 missing, 0 hom A1, 1 het, 2 hom A2
    M, N = G.shape
    pad = np.zeros((M, (N + 3) // 4 * 4), np.uint8)
    pad[:, :N] = code
    q = pad.reshape(M, -1, 4)
    return (q[..., 0] | (q[..., 1] << 2) | (q[..., 2] << 4) | (q[..., 3] << 6)).astype(np.uint8)


def load(G):
    M, N = G.shape
    s = gw.GenoStore(M, N)
    s.put_bed(to_bed(G))
    return s


def assert_records_equal(got, want):
    assert len(got) == len(want)
    for f in ("i", "j", "n", "reserved"):
        np.testing.assert_array_equal(got[f], want[f])
    for f in ("r", "r2"):      # bit-equal, NaN included
        np.testing.assert_array_equal(got[f].view(np.uint64), want[f].view(np.uint64))


def assert_band_equal(got, want):
    assert got.shape == want.shape
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
    np.testing.assert_array_equal(np.nan_to_num(got, nan=-7.0).view(np.uint32), np.nan_to_num(want, nan=-7.0).view(np.uint32))


def check_window(s, ref, window, lo=0, hi=None, thr=0.0, mask=None):
    hi = s.n_snps if hi is None else hi
    pairs, band, st = s.ld_window(window, thr, lo, hi, sample_mask=mask, band=True)
    assert_band_equal(band, band_of(ref[2], lo, hi, window))
    assert_records_equal(pairs, list_of(ref, lo, hi, window, thr))
    w1 = min(window, hi - lo - 1)
    assert st.pairs_tested == (hi - lo - w1) * w1 + w1 * (w1 - 1) // 2 and st.pairs_kept == len(pairs)
    return pairs, band, st


# ---- 1. exactness -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [2, 127, 3001, 10000])
@pytest.mark.parametrize("missing", [0.0, 0.02])
def test_window_is_bit_exact(N, missing):
    M = 300 if N < 100 else 700
    G = ld_table(M, N, seed=N + int(missing * 100), missing=missing)
    s = load(G)
    x, c = decoded(s)
    ref = ld_reference(x, c)
    for w in (1, 63, 64, 65, 255, 256, 257, M - 1, M + 40):
        _, _, st = check_window(s, ref, w)
        assert st.rows_per_snp == (1 if c.all() else 3)
    check_window(s, ref, 65, 37, M - 51)          # unaligned SNP ranges
    check_window(s, ref, 257, 300, 611 if M > 611 else M)
    check_window(s, ref, 3, 255, 258)
    if not missing and N > 2:                      # complete rows against np.corrcoef
        clean = np.flatnonzero(c.all(1) & (x.std(1) > 0))[:60]
        cc = np.corrcoef(x[clean].astype(np.float64))
        np.testing.assert_allclose(ref[1][np.ix_(clean, clean)], cc, rtol=0, atol=1e-12)


def test_window_without_missing_calls_uses_one_row_per_snp():
    G = ld_table(600, 3001, seed=3, missing=0.0)
    G[G < 0] = 0
    s = load(G)
    x, c = decoded(s)
    assert c.all()
    ref = ld_reference(x, c)
    for w in (1, 64, 257, 599):
        _, _, st = check_window(s, ref, w)
        assert st.rows_per_snp == 1
    pairs, _, _ = s.ld_window(64, 1.0)
    assert {(k - 1, k) for k in range(5, 600, 97) if ref[2][k - 1, k] == 1.0} <= set(zip(pairs["i"].tolist(), pairs["j"].tolist()))


# ---- 2. band and list -------------------------------------------------------------------------------------------------------
def test_band_list_thresholds_and_overflow():
    M, N = 700, 3001
    G = ld_table(M, N, seed=7, missing=0.01)
    s = load(G)
    x, c = decoded(s)
    ref = ld_reference(x, c)
    W = 100
    for thr in (0.0, 0.3, 0.8, 1.0, 1.5):
        pairs, band, st = check_window(s, ref, W, thr=thr)
        I, J = np.nonzero(~np.isnan(band))
        r2b = ref[2][I, I + J + 1]
        keep = r2b >= thr
        np.testing.assert_array_equal(pairs["i"], I[keep])
        np.testing.assert_array_equal(pairs["j"], I[keep] + J[keep] + 1)
        if thr == 0.0:
            assert len(pairs) == int((~np.isnan(band)).sum())
        if thr == 1.0:
            planted = [(k - 1, k) for k in list(range(5, M, 97)) + list(range(11, M, 89))]
            assert sum(ref[2][p] == 1.0 for p in planted) >= 10
            assert {p for p in planted if ref[2][p] == 1.0} <= set(zip(pairs["i"].tolist(), pairs["j"].tolist()))
        if thr > 1.0:
            assert len(pairs) == 0
    # r = -1 for the relabelled copies
    for k in range(11, M, 89):
        assert ref[1][k - 1, k] == -1.0
    # too small a capacity: GWASDEV_EOVERFLOW with the exact count, then the retry succeeds
    want = list_of(ref, 0, M, W, 0.3)
    buf = np.zeros(5, gw.LD_PAIR_DTYPE)
    got = C.c_uint64()
    rc = s.L.gwasdev_ld_window(s.h, 0, M, W, None, 0.3, gw._ptr(buf), 5, C.byref(got), None, None, 0)
    assert rc == 4 and got.value == len(want)
    buf = np.zeros(got.value, gw.LD_PAIR_DTYPE)
    assert s.L.gwasdev_ld_window(s.h, 0, M, W, None, 0.3, gw._ptr(buf), len(buf), C.byref(got), None, None, 0) == 0
    assert_records_equal(buf, want)
    pairs, _, _ = s.ld_window(W, 0.3, capacity=3)            # the Python wrapper grows the buffer itself
    assert_records_equal(pairs, want)
    # band only, and list only
    p2, b2, _ = s.ld_window(W, 0.3, band=True, pairs=False)
    assert p2 is None
    assert_band_equal(b2, band_of(ref[2], 0, M, W))


# ---- 3. sample masks --------------------------------------------------------------------------------------------------------
def test_sample_masks():
    M, N = 520, 3001
    G = ld_table(M, N, seed=11, missing=0.0)
    s = load(G)
    x, c = decoded(s)
    ones = np.ones(N, bool)
    a = s.ld_window(200, 0.0, band=True)
    b = s.ld_window(200, 0.0, band=True, sample_mask=ones)
    assert_records_equal(a[0], b[0])
    assert_band_equal(a[1], b[1])
    rng = np.random.default_rng(5)
    mask = rng.random(N) < 0.6
    ref = ld_reference(x, c, mask)
    pm, bm, _ = check_window(s, ref, 200, mask=mask)
    sub = load(G[:, mask])                                   # the same samples as a table of their own
    ps, bs, _ = sub.ld_window(200, 0.0, band=True)
    assert_band_equal(bm, bs)
    for f in ("i", "j", "n"):
        np.testing.assert_array_equal(pm[f], ps[f])
    np.testing.assert_array_equal(pm["r2"].view(np.uint64), ps["r2"].view(np.uint64))
    # r is bit-equal up to the sign the first-seen labels give each table
    np.testing.assert_array_equal(np.abs(pm["r"]).view(np.uint64), np.abs(ps["r"]).view(np.uint64))
    xs, cs = decoded(sub)
    assert_records_equal(ps, list_of(ld_reference(xs, cs), 0, M, 200, 0.0))
    # missing calls only in samples 0..9: the full set takes the three-row path, a mask without them the one-row path
    G2 = ld_table(400, 2000, seed=12)
    G2[G2 < 0] = 0
    G2[:, :10][rng.random((400, 10)) < 0.3] = -1
    s2 = load(G2)
    x2, c2 = decoded(s2)
    m2 = np.ones(2000, bool)
    m2[:10] = False
    _, _, st = check_window(s2, ld_reference(x2, c2), 70)
    assert st.rows_per_snp == 3
    _, _, st = check_window(s2, ld_reference(x2, c2, m2), 70, mask=m2)
    assert st.rows_per_snp == 1
    _, _, st = check_window(s2, ld_reference(x2, c2, ~m2), 70, mask=~m2)
    assert st.rows_per_snp == 3


# ---- 4. ld_pairs ------------------------------------------------------------------------------------------------------------
def test_ld_pairs_matches_the_window_and_the_reference():
    M, N = 700, 3001
    G = ld_table(M, N, seed=21, missing=0.02)
    s = load(G)
    x, c = decoded(s)
    ref = ld_reference(x, c)
    win, _, _ = s.ld_window(120, 0.0)
    rng = np.random.default_rng(0)
    pick = win[rng.choice(len(win), 3000, replace=False)]
    flip = rng.random(len(pick)) < 0.5
    pi, pj = np.where(flip, pick["j"], pick["i"]), np.where(flip, pick["i"], pick["j"])
    assert_records_equal(s.ld_pairs(pi, pj), pick)
    # pairs with r2 NaN are in no list: check them and far pairs against the reference
    I, J = rng.integers(0, M, 4000), rng.integers(0, M, 4000)
    ok = I != J
    I, J = I[ok], J[ok]
    got = s.ld_pairs(I, J)
    lo, hi = np.minimum(I, J), np.maximum(I, J)
    want = np.zeros(len(I), gw.LD_PAIR_DTYPE)
    want["i"], want["j"], want["n"], want["r"], want["r2"] = lo, hi, ref[0][lo, hi], ref[1][lo, hi], ref[2][lo, hi]
    assert_records_equal(got, want)
    mask = rng.random(N) < 0.5
    refm = ld_reference(x, c, mask)
    got = s.ld_pairs(I, J, sample_mask=mask)
    want["n"], want["r"], want["r2"] = refm[0][lo, hi], refm[1][lo, hi], refm[2][lo, hi]
    assert_records_equal(got, want)


def test_ld_pairs_on_pair_screen_hits():
    M, N = 1000, 4000
    G = ld_table(M, N, seed=31, missing=0.0)
    G[G < 0] = 0
    s = load(G)
    rng = np.random.default_rng(1)
    s.select_case_control((rng.random(N) < 0.4).astype(np.uint8))
    hits, _ = s.pairwise_scan(threshold=8.0)
    assert len(hits) > 100
    x, c = decoded(s)
    ref = ld_reference(x, c)
    got = s.ld_pairs(hits["i"], hits["j"])
    want = np.zeros(len(hits), gw.LD_PAIR_DTYPE)
    I, J = hits["i"].astype(np.int64), hits["j"].astype(np.int64)
    want["i"], want["j"], want["n"], want["r"], want["r2"] = I, J, ref[0][I, J], ref[1][I, J], ref[2][I, J]
    assert_records_equal(got, want)
    assert (J - I).max() > 300


# ---- 5. operand lifetime ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("missing", [0.0, 0.02])
def test_operand_lifetime_and_chunks(missing):
    M, N = 1500, 1000
    G = ld_table(M, N, seed=41, missing=missing)
    if not missing:
        G[G < 0] = 0
    s = load(G)
    x, c = decoded(s)
    ref = ld_reference(x, c)
    _, _, st = s.ld_window(64, 0.5)
    assert st.built_operand == 1
    _, _, st = s.ld_window(300, 0.2, 100, 1400)
    assert st.built_operand == 0
    mask = np.ones(N, bool)
    mask[::3] = False
    _, _, st = s.ld_window(64, 0.5, sample_mask=mask)
    assert st.built_operand == 1
    _, _, st = s.ld_window(64, 0.5, sample_mask=mask)
    assert st.built_operand == 0
    _, _, st = s.ld_window(64, 0.5)
    assert st.built_operand == 1
    s.put_bed(to_bed(G[:10]), first_row=0)
    _, _, st = s.ld_window(64, 0.5)
    assert st.built_operand == 1
    full = {w: s.ld_window(w, 0.0, band=True) for w in (63, 257, 700)}
    # a budget far below the table: chunks of 256-SNP blocks whose windows cross the chunk edges
    rows = full[63][2].rows_per_snp
    for budget_snps in (300, 900):
        s.set_option(gw.OPT_LD_OPERAND_BYTES, budget_snps * rows * 32 * s.P // 2)
        for w, (p0, b0, _) in full.items():
            p1, b1, st = s.ld_window(w, 0.0, band=True)
            assert st.built_operand == 1
            assert_records_equal(p1, p0)
            assert_band_equal(b1, b0)
        _, _, st = check_window(s, ref, 257, 123, 1333)
    s.set_option(gw.OPT_LD_OPERAND_BYTES, 0)
    _, _, st = s.ld_window(63, 0.0)
    assert st.built_operand == 1


# ---- 6. pruning end to end --------------------------------------------------------------------------------------------------
def prune_restated(r2, lo, hi, window, thr):
    keep = np.zeros(hi - lo, bool)
    for i in range(lo, hi):
        keep[i - lo] = not any(keep[k - lo] and r2[k, i] >= thr for k in range(max(lo, i - window), i))
    return keep


def test_prune_end_to_end():
    M, N = 900, 3001
    G = ld_table(M, N, seed=51, missing=0.01)
    s = load(G)
    x, c = decoded(s)
    ref = ld_reference(x, c)
    for w, thr, lo, hi in ((50, 0.5, 0, M), (200, 0.2, 77, 850), (1, 0.9, 0, M)):
        keep = s.ld_prune(w, thr, lo, hi)
        # the restatement reads the band's fp64 values (the window is bit-equal to ref, checked above)
        _, band, _ = s.ld_window(w, 0.0, lo, hi, band=True)
        assert_band_equal(band, band_of(ref[2], lo, hi, w))
        with np.errstate(invalid="ignore"):
            np.testing.assert_array_equal(keep, prune_restated(ref[2], lo, hi, w, thr))
        assert 0 < keep.sum() < hi - lo


# ---- 7. errors --------------------------------------------------------------------------------------------------------------
def test_errors():
    G = ld_table(300, 100, seed=61)
    s = load(G)
    with pytest.raises(gw.GwasDevError, match="window"):
        s.ld_window(0)
    for lo, hi in ((10, 5), (0, 301)):
        with pytest.raises(gw.GwasDevError, match="range"):
            s.ld_window(10, 0.5, lo, hi)
    bad = np.zeros(s.P, np.uint16)
    bad[100 // 16] = 1 << (100 % 16)                            # sample 100 of 100
    with pytest.raises(gw.GwasDevError, match="sample_mask"):
        s.ld_window(10, 0.5, sample_mask=bad)
    with pytest.raises(gw.GwasDevError, match="sample_mask"):
        s.ld_pairs([0], [1], sample_mask=bad)
    with pytest.raises(gw.GwasDevError):
        s.ld_pairs([3], [3])
    with pytest.raises(gw.GwasDevError):
        s.ld_pairs([0], [300])
    import torch
    pi = torch.zeros(4, dtype=torch.int32, device="cuda")
    pj = torch.ones(4, dtype=torch.int32, device="cuda")
    out = torch.zeros(4 * 32, dtype=torch.uint8, device="cuda")
    assert s.L.gwasdev_ld_pairs(s.h, 4, gw._ptr(pi), gw._ptr(pj), None, gw._ptr(out)) == 1
    assert "host" in s.L.gwasdev_last_error().decode()
    band = torch.zeros(300 * 10, dtype=torch.float32, device="cuda")
    assert s.L.gwasdev_ld_window(s.h, 0, 300, 10, None, 0.5, None, 0, None, gw._ptr(band), None, 0) == 1
    # the same band as a device buffer with on_device = 1
    assert s.L.gwasdev_ld_window(s.h, 0, 300, 10, None, 0.5, None, 0, None, gw._ptr(band), None, 1) == 0
    _, want, _ = s.ld_window(10, 0.5, band=True, pairs=False)
    assert_band_equal(band.cpu().numpy().reshape(300, 10), want)
    # on the device, the list as well
    lst = torch.zeros(5000 * 32, dtype=torch.uint8, device="cuda")
    got = C.c_uint64()
    assert s.L.gwasdev_ld_window(s.h, 0, 300, 10, None, 0.1, gw._ptr(lst), 5000, C.byref(got), None, None, 1) == 0
    torch.cuda.synchronize()
    host, _, _ = s.ld_window(10, 0.1)
    assert_records_equal(lst.cpu().numpy()[: got.value * 32].view(gw.LD_PAIR_DTYPE), host)
