"""Pins the CPU oracle (oracle/gwas_oracle.c) to the reference BEFORE it is trusted as the checker.

Three independent anchors (SURVEY.md section 8c):
  1. golden vectors captured from the unmodified reference (tests/golden/*.npz, made by make_golden.py);
  2. the reference's own fixture generator scripts/perl/genotype_set_builder.pl (expected xx/aa/ab/bb
     per marker, equal up to the aa<->bb swap its comparer tolerates, contin_output_comparer.pl:119-162);
  3. the five literature tables of src/test/pairwise.c:19-37.
"""
import os

import numpy as np
import pytest


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


COHORTS = ["cohort_missing", "cohort_complete"]


@pytest.mark.parametrize("name", COHORTS)
def test_layout_and_counts_match_reference_golden(orc, golden_dir, name):
    g = load(golden_dir, name)
    codes, pheno = g["codes"], g["pheno"]
    M, N = codes.shape
    rows = orc.pack_codes(codes)
    assert np.array_equal(rows, g["raw_rows"])                       # a5/a6 + first-seen headers (a4)
    sel, nca, nco = orc.select(rows, N, pheno)
    assert (nca, nco) == (int(g["n_case"]), int(g["n_ctrl"]))
    assert np.array_equal(sel, g["sel_rows"])                        # a8
    assert np.array_equal(orc.counts_whole(rows, N), g["whole"])     # a21 (xx incl. padding, defect D5)
    assert np.array_equal(orc.cc_counts_masked(rows, N, pheno), g["cc_masked"])
    assert np.array_equal(orc.cc_counts_selected(sel, nca, nco), g["cc_selected"])   # a9
    mar = orc.margins(sel, nca, nco)
    assert mar.tobytes() == g["margins"].tobytes()                   # a10, bit-exact doubles


@pytest.mark.parametrize("name", COHORTS)
def test_pair_tables_match_reference_golden(orc, golden_dir, name):
    g = load(golden_dir, name)
    codes, pheno = g["codes"], g["pheno"]
    N = codes.shape[1]
    rows = orc.pack_codes(codes)
    sel, nca, nco = orc.select(rows, N, pheno)
    mar = orc.margins(sel, nca, nco)
    for mode in (0, 1, 2, 3):
        for k, (i, j) in enumerate(g["pairs"]):
            ca, co = orc.pair_table(mode, int(i), int(j), rows=rows, sel=sel, n_samples=N, pheno=pheno,
                                    nca=nca, nco=nco, mar=mar)
            assert np.array_equal(np.concatenate([ca, co]), g[f"tables_mode{mode}"][k]), (mode, i, j)


@pytest.mark.parametrize("name", COHORTS)
def test_boost_screen_and_gtest_match_reference_golden(orc, golden_dir, name):
    g = load(golden_dir, name)
    codes, pheno = g["codes"], g["pheno"]
    N = codes.shape[1]
    rows = orc.pack_codes(codes)
    sel, nca, nco = orc.select(rows, N, pheno)
    mar = orc.margins(sel, nca, nco)
    hi, hj, hs, st = orc.boost_screen(sel, mar, nca, nco, threshold=30.0)
    assert len(hi) == int(g["boost_located"])                        # "Located N potential interactions"
    # exact G-test + z for every screened pair, then the reference prints those with exact stat > 30
    exact = [orc.gtest(*orc.pair_table(3, int(i), int(j), sel=sel, nca=nca, nco=nco, mar=mar),
                       mar[int(i)], mar[int(j)], nca + nco) for i, j in zip(hi, hj)]
    kept = [(int(i), int(j), e[0], e[1]) for i, j, e in zip(hi, hj, exact) if e[0] > 30.0]
    assert [(a, b) for a, b, _, _ in kept] == [tuple(x) for x in g["boost_hits"].tolist()]
    # the reference prints with "%f" (6 decimals): compare at that resolution ...
    assert np.allclose([k[2] for k in kept], g["boost_exact"], rtol=0, atol=5.1e-7)
    assert np.allclose([k[3] for k in kept], g["boost_z"], rtol=0, atol=5.1e-7)
    # ... and at full precision through computeGTest's own return values
    for (i, j), s_ref, z_ref in zip(g["gtest_pairs"], g["gtest_stat"], g["gtest_z"]):
        ca, co = orc.pair_table(3, int(i), int(j), sel=sel, nca=nca, nco=nco, mar=mar)
        s, z = orc.gtest(ca, co, mar[int(i)], mar[int(j)], nca + nco)
        assert s == pytest.approx(s_ref, rel=1e-13, abs=1e-10) or (np.isnan(s) and np.isnan(s_ref))
        assert z == pytest.approx(z_ref, rel=1e-13, abs=1e-12) or (np.isnan(z) and np.isnan(z_ref)) \
            or (np.isinf(z) and z == z_ref)


def test_pairwise_c_known_answers(orc, golden_dir):
    k = load(golden_dir, "pairwise_c_kats")
    # frozen literals (SURVEY.md 8c-iii), produced by compiling src/test/pairwise.c itself
    frozen = {"boost0": (5.64124451648526, 0.227590127533315), "boost1": (33.3815424226012, 9.97784906723507e-07),
              "boost2": (30.7156081330587, 3.49877038374422e-06), "biforce1": (39.1623776418192, 6.44864104309708e-08),
              "biforce2": (80.9802754318203, 1.07969600600098e-16)}
    for name, cs, ct, ll, p in zip(k["names"], k["cs"], k["ct"], k["ll"], k["p"]):
        got = orc.pairwise_epi_test(cs, ct)
        assert got == pytest.approx(ll, rel=1e-14)
        assert orc.chisq_upper(got, 4) == pytest.approx(p, rel=1e-13)
        assert got == pytest.approx(frozen[str(name)][0], rel=1e-13)
        assert p == pytest.approx(frozen[str(name)][1], rel=1e-12)


def _read_tped(path):
    lines = []
    with open(path) as f:
        for line in f:
            parts = line.rstrip("\n").split("\t")
            alleles = parts[4:]
            # the TPED reader collapses "A\tC" -> "AC\t" (tped_genotype_file.cpp:127-190)
            lines.append("\t".join(a + b for a, b in zip(alleles[0::2], alleles[1::2])).encode())
    return lines


def _swap_equal(got, want):
    """xx aa ab bb equal up to the aa<->bb relabelling (first-seen vs alphabetical)."""
    got, want = list(map(int, got)), list(map(int, want))
    return got == want or got == [want[0], want[3], want[2], want[1]]


def test_perl_simple_fixture(orc, golden_dir):
    lines = _read_tped(os.path.join(golden_dir, "perl_simple.tped"))
    expected = np.loadtxt(os.path.join(golden_dir, "perl_simple.expected.dist"), dtype=int)
    ref_print = np.loadtxt(os.path.join(golden_dir, "perl_simple.ref_inline_maf_print.txt"), dtype=int)
    n = len(lines[0].split(b"\t"))
    for r, line in enumerate(lines):
        row = orc.pack_text(line, n)
        aa, ab, bb, _ = orc.counts_whole(row[None, :], n)[0]
        mine = [n - (aa + ab + bb), aa, ab, bb]                      # what inline_maf_print prints (maf_func.cpp:332)
        assert mine == list(ref_print[r])                            # exact vs the reference's own output
        assert _swap_equal(mine, expected[r])                        # vs the perl generator's expectation


def test_perl_case_control_fixture(orc, golden_dir):
    lines = _read_tped(os.path.join(golden_dir, "perl_cc.tped"))
    pheno = np.array([int(l.rstrip("\n").split("\t")[5]) for l in open(os.path.join(golden_dir, "perl_cc.tfam"))],
                     np.uint8)
    exp_ca = np.loadtxt(os.path.join(golden_dir, "perl_cc.expected.case.dist"), dtype=int)
    exp_co = np.loadtxt(os.path.join(golden_dir, "perl_cc.expected.control.dist"), dtype=int)
    ref_cc = np.load(os.path.join(golden_dir, "perl_cc.ref_cc_counts.npy"))
    n = len(pheno)
    rows = np.stack([orc.pack_text(line, n) for line in lines])
    sel, nca, nco = orc.select(rows, n, pheno)
    cnt = orc.cc_counts_selected(sel, nca, nco)
    assert np.array_equal(cnt, ref_cc)
    for r in range(len(lines)):
        ca = [cnt[r][3], cnt[r][0], cnt[r][1], cnt[r][2]]
        co = [cnt[r][7], cnt[r][4], cnt[r][5], cnt[r][6]]
        # one relabelling per SNP applies to both classes
        same = list(map(int, ca)) == list(exp_ca[r]) and list(map(int, co)) == list(exp_co[r])
        swapped = list(map(int, ca)) == [exp_ca[r][0], exp_ca[r][3], exp_ca[r][2], exp_ca[r][1]] and \
            list(map(int, co)) == [exp_co[r][0], exp_co[r][3], exp_co[r][2], exp_co[r][1]]
        assert same or swapped


def test_first_seen_labelling_and_abort_cases(orc):
    # het first, then CC, then AA: CC is the first homozygote -> code 1 (plane1), AA -> code 3 (both planes)
    row = orc.pack_text(b"AC\tCC\tAA\t00\tCC", 5)
    assert row[0] == (0x7000 | (5 << 8) | (1 << 4) | 0)
    assert [orc.call_at(row, 5, c) for c in range(5)] == ["AC", "CC", "AA", "00", "CC"]
    # a second heterozygote spelling aborts the reference (compressed_genotype_table5.cpp:325, SURVEY fact 4)
    with pytest.raises(ValueError):
        orc.pack_text(b"AC\tCA\tAA", 3)
    # letters outside ACGT are "unknown" (simulate_data.cpp's 'B' allele problem)
    row = orc.pack_text(b"AB\tBB\tAA", 3)
    assert orc.counts_whole(row[None, :], 3)[0][:3].tolist() == [1, 0, 0]


def test_marginal_information_zero_classes_and_maf(orc):
    m = orc.marginal_information([10, 0, 5, 0], [0, 7, 3, 2], 27)
    assert m["margins"].tolist() == [10, 7, 8, 2]
    assert m["pbc"][1] == 0.0 and m["pca"][1] == 0.0 and m["pbc"][4] == 0.0   # never written by the reference
    assert m["pbc"][0] == 10 / 15 and m["pca"][6] == 3 / 8
    v, tot = orc.maf_reference([10, 5, 1, 3])
    assert tot == 16 and v == pytest.approx(max(25 / 16, 1 - 25 / 16))
    v, _ = orc.maf_reference([1, 2, 9, 0])
    assert v == pytest.approx(1 - 4 / 12)                             # returns max(f, 1-f) (defect D11)


def test_chi_square_spec_against_scipy(orc):
    """Parity-UNPINNED statistics (no reference counterpart): checked against scipy instead."""
    from scipy import stats
    rng = np.random.default_rng(7)
    for _ in range(200):
        ca = rng.integers(0, 400, 4).astype(np.uint32)
        co = rng.integers(0, 400, 4).astype(np.uint32)
        if rng.random() < 0.2:
            ca[rng.integers(0, 3)] = 0
            co[rng.integers(0, 3)] = 0
        x, p = orc.chi2_allelic(ca, co)
        a = np.array([[2.0 * ca[0] + ca[1], 2.0 * ca[2] + ca[1]], [2.0 * co[0] + co[1], 2.0 * co[2] + co[1]]])
        if a.sum(0).min() > 0 and a.sum(1).min() > 0:
            ref = stats.chi2_contingency(a, correction=False)
            assert x == pytest.approx(ref[0], rel=1e-12, abs=1e-12)
            assert p == pytest.approx(ref[1], rel=1e-10, abs=1e-300)
        else:
            assert (x, p) == (0.0, 1.0)
        x, p, df = orc.chi2_genotypic(ca, co)
        g = np.array([ca[:3], co[:3]], float)
        g = g[:, g.sum(0) > 0]
        if g.shape[1] > 1 and g.sum(1).min() > 0:
            ref = stats.chi2_contingency(g, correction=False)
            assert df == ref[2]
            assert x == pytest.approx(ref[0], rel=1e-12, abs=1e-12)
            assert p == pytest.approx(ref[1], rel=1e-10, abs=1e-300)
        else:
            assert (x, p, df) == (0.0, 1.0, 0)
    for df in (1, 2, 4):
        for x in (0.5, 3.84, 30.0, 80.0):
            assert orc.chisq_upper(x, df) == pytest.approx(stats.chi2.sf(x, df), rel=1e-12)


def test_simulator_properties(orc):
    codes, pheno = orc.simulate(20121127, 300, 1000, 480)
    assert pheno.sum() == 480 and set(np.unique(codes)) <= {0, 1, 2}
    minor = (codes == 1).sum(1) + 2 * (codes == 2).sum(1)
    assert minor.max() <= 0.51 * 2000 + 1                              # MAF bins stop at 50.999 %
    assert np.array_equal(codes, orc.simulate(20121127, 300, 1000, 480)[0])   # reproducible
    part, _ = orc.simulate(20121127, 10, 1000, 480, first_snp=100)
    assert np.array_equal(part, codes[100:110])                       # counter-based: any SNP range on its own
    cm, _ = orc.simulate(20121127, 50, 1000, 480, missing_rate=0.05)
    frac = (cm == 3).mean()
    assert 0.03 < frac < 0.07
    assert np.array_equal(cm[cm != 3], codes[:50][cm != 3])
