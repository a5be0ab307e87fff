"""GPU tests of the label-permutation test of the marginal scan (gwasdev_marginal_permute)."""
import numpy as np
import pytest

import libgwaspp_b200 as gw

pytestmark = pytest.mark.gpu


def make_store(M, N, seed, missing, pheno):
    s = gw.GenoStore(M, N)
    s.simulate(seed, missing_rate=missing)
    s.select_case_control(pheno)
    return s


def pheno_of(N, seed, frac=0.4, neither=0.0):
    rng = np.random.default_rng(seed)
    p = (rng.random(N) < frac).astype(np.uint8)
    p[rng.random(N) < neither] = 2
    return p


def scan_with_case_mask(s, case_mask, sel_case, sel_ctrl):
    """gwasdev_marginal_scan after re-selecting (case_mask, selection minus case_mask); restores the selection."""
    sel = sel_case | sel_ctrl
    s.select_case_control(case_mask=case_mask, ctrl_mask=sel & ~case_mask)
    st = s.marginal_scan(counts=False, mi=False)["stats"]
    s.select_case_control(case_mask=sel_case, ctrl_mask=sel_ctrl)
    return st


def bits_of(blocks, n):
    return np.unpackbits(np.ascontiguousarray(blocks, np.uint16).view(np.uint8), axis=-1, bitorder="little")[..., :n].astype(bool)


def perm_df(s, masks, sel_ca, sel_co):
    """Genotypic df of every (permutation, SNP) element, from the raw rows and the permuted case masks: the number of genotype
    columns the selection calls, minus 1, when both classes have called samples (else 0)."""
    N, P = s.n_samples, s.P
    rows = s.get_rows()
    sel = bits_of(sel_ca | sel_co, N)
    case = bits_of(masks, N).astype(np.float32)                                  # (n_perm, N); counts stay exact in fp32
    out = []
    for r0 in range(0, rows.shape[0], 2048):
        p1, p2 = bits_of(rows[r0:r0 + 2048, 1:1 + P], N), bits_of(rows[r0:r0 + 2048, 1 + P:], N)
        geno = [(p1 & ~p2) & sel, (p2 & ~p1) & sel, (p1 & p2) & sel]          # aa, ab, bb of the selection: (rows, N)
        pooled = np.stack([g.sum(1) for g in geno])                              # (3, rows)
        called_case = sum(case @ g.T.astype(np.float32) for g in geno)          # (n_perm, rows)
        called_ctrl = pooled.sum(0)[None] - called_case
        cols = (pooled > 0).sum(0)[None]
        out.append(np.where((called_case > 0) & (called_ctrl > 0) & (cols > 1), cols - 1, 0))
    return np.concatenate(out, axis=1)


def check_reductions(out, obs, df=None):
    ps = out["perm_stats"]
    np.testing.assert_array_equal(out["exceed"][:, 0], (ps[:, :, 0] >= obs["chi2_allelic"][None]).sum(0))
    np.testing.assert_array_equal(out["exceed"][:, 1], (ps[:, :, 1] >= obs["chi2_genotypic"][None]).sum(0))
    np.testing.assert_array_equal(out["perm_max"][:, 0], ps[:, :, 0].max(1))
    if df is not None:   # the genotypic maxima split by the element's df (0 when a permutation has no such element)
        for d in (1, 2):
            np.testing.assert_array_equal(out["perm_max"][:, d], np.where(df == d, ps[:, :, 1], 0.0).max(1))


@pytest.mark.parametrize("N, M, P, missing", [(2, 70, 1, 0.0), (127, 130, 255, 0.02), (3001, 200, 257, 0.0), (10000, 65, 1000, 0.02)])
def test_bit_identity_against_reselected_scans(orc, N, M, P, missing):
    pheno = pheno_of(N, N, neither=0.1 if N > 2 else 0.0)
    if N == 2:
        pheno = np.array([1, 0], np.uint8)
    s = make_store(M, N, 11 + N, missing, pheno)
    ca, co = gw.stream_masks(pheno)
    obs = s.marginal_scan(counts=False, mi=False)["stats"]
    out = s.marginal_permute(P, seed=5, perm_stats=True)
    assert out["stats"].planes == (3 if missing else 2) and out["stats"].n_perm == P
    masks = gw.permutation_masks(N, ca, co, 5, 0, P)
    check_reductions(out, obs, perm_df(s, masks, ca, co))
    # explicit masks give the same outputs as the device draws
    ex = s.marginal_permute(P, case_masks=masks, perm_stats=True)
    for key in ("exceed", "perm_max", "perm_stats"):
        np.testing.assert_array_equal(ex[key], out[key])
    # byte for byte against the scan of the re-selected cohort, for a sample of permutations
    for k in sorted({0, P // 2, P - 1}):
        st = scan_with_case_mask(s, masks[k], ca, co)
        np.testing.assert_array_equal(out["perm_stats"][k, :, 0], st["chi2_allelic"])
        np.testing.assert_array_equal(out["perm_stats"][k, :, 1], st["chi2_genotypic"])
        # and the oracle, per element
        counts = None
        for i in range(0, M, max(1, M // 7)):
            if counts is None:
                s.select_case_control(case_mask=masks[k], ctrl_mask=(ca | co) & ~masks[k])
                counts = s.marginal_scan(mi=False, stats=False)["counts"]
                s.select_case_control(case_mask=ca, ctrl_mask=co)
            xa, _ = orc.chi2_allelic(counts[i, :4], counts[i, 4:])
            xg, _, _ = orc.chi2_genotypic(counts[i, :4], counts[i, 4:])
            assert abs(out["perm_stats"][k, i, 0] - xa) <= 1e-12 * max(1.0, abs(xa))
            assert abs(out["perm_stats"][k, i, 1] - xg) <= 1e-12 * max(1.0, abs(xg))
    s.close()


def test_identity_permutation_and_awkward_cohort():
    N, M = 500, 190
    pheno = pheno_of(N, 3, neither=0.1)
    s = gw.GenoStore(M, N)
    s.simulate(8, missing_rate=0.02)
    rows = s.get_rows()
    P = s.P
    rows[0, 1:] = 0                                    # all missing
    called = np.zeros(16 * P, bool)
    called[:N] = True
    rows[1, 1:] = 0
    rows[1, 1:1 + P] = np.packbits(called, bitorder="little").view(np.uint16)   # monomorphic: every sample the first homozygote
    s.put_rows(rows)
    ca, co = gw.stream_masks(pheno)
    both = np.zeros_like(ca)
    both[3] = 0x00F0                                   # samples in both masks count as cases
    s.select_case_control(case_mask=ca | both, ctrl_mask=co | both)
    sel_ca, sel_co = ca | both, (co | both) & ~(ca | both)
    obs = s.marginal_scan(counts=False, mi=False)["stats"]
    assert {0, 1, 2} <= set(obs["df_genotypic"].astype(int))
    ident = s.marginal_permute(1, case_masks=sel_ca[None], perm_stats=True)
    np.testing.assert_array_equal(ident["perm_stats"][0, :, 0], obs["chi2_allelic"])
    np.testing.assert_array_equal(ident["perm_stats"][0, :, 1], obs["chi2_genotypic"])
    assert (ident["exceed"] >= 1).all()
    # a single case
    first = np.zeros(16 * P, bool)
    first[np.flatnonzero(np.unpackbits(sel_co.view(np.uint8), bitorder="little"))[0]] = True
    one = np.packbits(first, bitorder="little").view(np.uint16)
    single = s.marginal_permute(1, case_masks=one[None], perm_stats=True)
    st = scan_with_case_mask(s, one, sel_ca, sel_co)
    np.testing.assert_array_equal(single["perm_stats"][0, :, 1], st["chi2_genotypic"])
    # caller masks with different case counts per mask (several traits) against per-mask scans
    rng = np.random.default_rng(4)
    sel_bits = np.unpackbits((sel_ca | sel_co).view(np.uint8), bitorder="little").astype(bool)
    masks = []
    for frac in (0.05, 0.3, 0.7):
        b = sel_bits & (rng.random(sel_bits.size) < frac)
        masks.append(np.packbits(b, bitorder="little").view(np.uint16))
    masks = np.stack(masks)
    multi = s.marginal_permute(3, case_masks=masks, perm_stats=True)
    df = perm_df(s, masks, sel_ca, sel_co)
    assert {0, 1, 2} <= set(np.unique(df))
    check_reductions(multi, obs, df)
    for k in range(3):
        st = scan_with_case_mask(s, masks[k], sel_ca, sel_co)
        np.testing.assert_array_equal(multi["perm_stats"][k, :, 0], st["chi2_allelic"])
        np.testing.assert_array_equal(multi["perm_stats"][k, :, 1], st["chi2_genotypic"])
    # device draws over a selection with samples in both masks and in neither: the host restatement's masks, all three maxima
    drawn = s.marginal_permute(300, seed=17, perm_stats=True)
    dmasks = gw.permutation_masks(N, ca | both, co | both, 17, 0, 300)
    assert not (bits_of(dmasks, N) & ~bits_of(sel_ca | sel_co, N)).any()
    explicit = s.marginal_permute(300, case_masks=dmasks, perm_stats=True)
    for key in ("exceed", "perm_max", "perm_stats"):
        np.testing.assert_array_equal(drawn[key], explicit[key])
    check_reductions(drawn, obs, perm_df(s, dmasks, sel_ca, sel_co))
    s.close()


def test_more_permutations_than_one_operand_batch():
    N, M, P = 200, 70, 16384 + 300                     # two A-operand batches of the device draws
    pheno = pheno_of(N, 12)
    s = make_store(M, N, 41, 0.02, pheno)
    ca, co = gw.stream_masks(pheno)
    obs = s.marginal_scan(counts=False, mi=False)["stats"]
    out = s.marginal_permute(P, seed=23, perm_stats=True)
    masks = gw.permutation_masks(N, ca, co, 23, 0, P)
    check_reductions(out, obs, perm_df(s, masks, ca, co))
    lo = s.marginal_permute(16384, seed=23, perm_stats=True)
    hi = s.marginal_permute(300, seed=23, first_perm=16384, perm_stats=True)
    np.testing.assert_array_equal(np.concatenate([lo["perm_stats"], hi["perm_stats"]]), out["perm_stats"])
    np.testing.assert_array_equal(lo["exceed"] + hi["exceed"], out["exceed"])
    st = scan_with_case_mask(s, masks[P - 1], ca, co)
    np.testing.assert_array_equal(out["perm_stats"][P - 1, :, 1], st["chi2_genotypic"])
    s.close()


def test_additivity_ranges_chunking_and_lifetime():
    N, M = 2000, 300
    pheno = pheno_of(N, 9)
    s = make_store(M, N, 21, 0.01, pheno)
    whole = s.marginal_permute(500, seed=3)
    assert whole["stats"].built_operand == 1
    a = s.marginal_permute(300, seed=3)
    assert a["stats"].built_operand == 0
    b = s.marginal_permute(200, seed=3, first_perm=300)
    np.testing.assert_array_equal(a["exceed"] + b["exceed"], whole["exceed"])
    np.testing.assert_array_equal(np.concatenate([a["perm_max"], b["perm_max"]]), whole["perm_max"])
    full = s.marginal_permute(64, seed=1, perm_stats=True)
    part = s.marginal_permute(64, seed=1, snp_begin=37, snp_end=230, perm_stats=True)
    np.testing.assert_array_equal(part["perm_stats"], full["perm_stats"][:, 37:230])
    np.testing.assert_array_equal(part["exceed"], full["exceed"][37:230])
    # chunked B operand: same results
    s.set_option(gw.OPT_PERM_OPERAND_BYTES, 3 * 64 * 32 * (s.P // 2 + 4) * 2)
    chunked = s.marginal_permute(64, seed=1, perm_stats=True)
    assert chunked["stats"].built_operand == 1
    for key in ("exceed", "perm_max", "perm_stats"):
        np.testing.assert_array_equal(chunked[key], full[key])
    s.set_option(gw.OPT_PERM_OPERAND_BYTES, 0)
    # re-selection keeps the SNP planes; the results follow the new selection
    again = s.marginal_permute(64, seed=1)
    assert again["stats"].built_operand == 1            # rebuilt after the chunked call
    s.select_case_control(pheno_of(N, 10))
    re = s.marginal_permute(64, seed=1, perm_stats=True)
    assert re["stats"].built_operand == 0
    check_reductions(re, s.marginal_scan(counts=False, mi=False)["stats"])
    # put_rows rebuilds them, and the results follow the new rows
    rows = s.get_rows()
    rows[5:20] = rows[100:115]
    s.put_rows(rows)
    s.select_case_control(pheno_of(N, 10))
    after = s.marginal_permute(64, seed=1, perm_stats=True)
    assert after["stats"].built_operand == 1
    np.testing.assert_array_equal(after["perm_stats"][:, 5:20], re["perm_stats"][:, 100:115])
    s.close()


def test_errors_and_noop():
    N, M = 300, 80
    s = gw.GenoStore(M, N)
    s.simulate(2)
    with pytest.raises(gw.GwasDevError):
        s.marginal_permute(4)                           # no selection
    pheno = pheno_of(N, 1, neither=0.2)
    s.select_case_control(pheno)
    ca, co = gw.stream_masks(pheno)
    outside = ca.copy()
    outside[0] |= ~(ca[0] | co[0]) & 0xFFFF
    if outside[0] != ca[0]:
        with pytest.raises(gw.GwasDevError):
            s.marginal_permute(1, case_masks=outside[None])
    with pytest.raises(gw.GwasDevError):
        s.marginal_permute(1, case_masks=np.zeros((1, s.P), np.uint16))      # empty case class
    with pytest.raises(gw.GwasDevError):
        s.marginal_permute(1, case_masks=(ca | co)[None])                    # empty control class
    s.select_case_control(np.ones(N, np.uint8))
    with pytest.raises(gw.GwasDevError):
        s.marginal_permute(4)                           # no controls to permute against
    s.select_case_control(pheno)
    out = s.marginal_permute(0)
    assert out["stats"].n_perm == 0 and out["perm_max"].shape == (0, 3)
    s.close()


def test_mid_size_run():
    N, M, P = 10000, 50000, 512
    pheno = pheno_of(N, 77, frac=0.5)
    s = make_store(M, N, 31, 0.0, pheno)
    ca, co = gw.stream_masks(pheno)
    obs = s.marginal_scan(counts=False, mi=False)["stats"]
    out = s.marginal_permute(P, seed=99, perm_stats=True)
    masks = gw.permutation_masks(N, ca, co, 99, 0, P)
    check_reductions(out, obs, perm_df(s, masks, ca, co))
    for k in (0, 311):
        st = scan_with_case_mask(s, masks[k], ca, co)
        np.testing.assert_array_equal(out["perm_stats"][k, :, 0], st["chi2_allelic"])
        np.testing.assert_array_equal(out["perm_stats"][k, :, 1], st["chi2_genotypic"])
    emp1, emp2 = gw.permutation_pvalues(obs, out["exceed"], out["perm_max"])
    assert (emp2[:, 0] >= emp1[:, 0]).all()             # max(T) is never below the pointwise p-value
    s.close()
