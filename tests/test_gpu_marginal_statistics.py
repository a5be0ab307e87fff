"""The marginal statistics -- counts, marginal_information, MAFs, the allelic and genotypic chi-square tests and their
p-values -- on constructed genotype counts, against exact rational and 50-digit references, and the marginal scan at the
sample counts where its kernel choice changes, up to 2^23 - 1 samples per class.

Each SNP is a target {aa, ab, bb, xx} per class. Families: dense (Dirichlet-multinomial, with and without missing calls),
structural zeros, exact independence (both statistics exactly 0) and one sample away from it (full cancellation in o - e),
a tail sweep whose statistics land on chosen values (3.84, 30, 700, and ladders across the chi-square values where the
p-value crosses DBL_MIN and 2^-1074 and where it is 0), and relabelled copies whose first called homozygote is bb (the
store's first-seen labels then swap aa and bb). Rows carry exactly the target counts per class, samples shuffled so that
cells span words and blocks; the expected counts are always recounted from the codes.

Bounds, with u = 2^-53 (the operation order is that of csrc/marginal.cu and oracle/gwas_oracle.c):
  dPbc, dPca, maf_pooled    bit-equal to the correctly rounded quotient (one IEEE division of exact integers)
  maf_ref_*                 within 1 ulp of max(m, 1 - m), m = (2 aa + ab) / called (algorithms/maf_func.h:46-54)
  chi2_allelic              relative 8u: d = A_ca B_co - B_ca A_co is exact while the products stay below 2^53
  chi2_genotypic            16u (chi2 + sum |o - e|): the rounding of e, amplified by the subtraction
  entropies                 16u (1 + H)
  p, df 2                   relative 4u of the 50-digit exp(-x/2) at the device's own x
  p, df 1                   relative (x + 16)u of the 50-digit erfc(sqrt(x/2)): the rounding of sqrt(x/2) is amplified by
                            2 (x/2) = x, and the CUDA math library's erfc is accurate to 5 ulp
  below DBL_MIN             2 * 2^-1074 absolute on top (gradual underflow)
"""
import functools
import math
from fractions import Fraction

import mpmath
import numpy as np
import pytest

import libgwaspp_b200 as gw

U = 2.0 ** -53
DBL_MIN = float(np.finfo(np.float64).tiny)
DENORM_MIN = 2.0 ** -1074
CLASS_LIMIT = (1 << 23) - 1
PERM = np.array([2, 1, 0, 3])        # aa <-> bb


# ---- exact and 50-digit references -----------------------------------------------------------------------------------
def q_upper_mp(x, df):
    """50-digit chi-square upper tail at the fp64 value x."""
    if df == 0 or not x > 0:
        return 1.0 if x == x else math.nan
    with mpmath.workdps(50):
        x = mpmath.mpf(float(x))
        return float(mpmath.erfc(mpmath.sqrt(x / 2)) if df == 1 else mpmath.exp(-x / 2))


@functools.lru_cache(maxsize=None)
def tail_crossings(df):
    """The chi-square values where the df-1 / df-2 upper tail equals DBL_MIN and 2^-1074."""
    out = []
    with mpmath.workdps(50):
        for p in (mpmath.mpf(DBL_MIN), mpmath.mpf(2) ** -1074):
            if df == 2:
                out.append(float(-2 * mpmath.log(p)))
            else:
                out.append(float(mpmath.findroot(lambda x: mpmath.log(mpmath.erfc(mpmath.sqrt(x / 2))) - mpmath.log(p), 1400)))
    return tuple(out)


def allelic_exact(ca, co):
    a_ca, b_ca, a_co, b_co = 2 * ca[0] + ca[1], 2 * ca[2] + ca[1], 2 * co[0] + co[1], 2 * co[2] + co[1]
    r1, r2, c1, c2 = a_ca + b_ca, a_co + b_co, a_ca + a_co, b_ca + b_co
    if 0 in (r1, r2, c1, c2):
        return Fraction(0)
    return Fraction((r1 + r2) * (a_ca * b_co - b_ca * a_co) ** 2, r1 * r2 * c1 * c2)


def genotypic_exact(ca, co):
    """(chi2, df, sum |o - e|) of the 2 x 3 Pearson test over the non-empty genotype columns."""
    g1, g2 = sum(ca[:3]), sum(co[:3])
    x, dev, cols = Fraction(0), Fraction(0), 0
    if g1 > 0 and g2 > 0:
        for g in range(3):
            c = ca[g] + co[g]
            if c == 0:
                continue
            cols += 1
            for o, r in ((ca[g], g1), (co[g], g2)):
                e = Fraction(r * c, g1 + g2)
                x += (o - e) ** 2 / e
                dev += abs(o - e)
    df = cols - 1 if cols > 1 else 0
    return (x if df else Fraction(0)), df, dev


def entropy_mp(counts, n):
    with mpmath.workdps(50):
        h = mpmath.mpf(0)
        for c in counts:
            if c > 0:
                t = mpmath.mpf(c) / n
                h -= t * mpmath.log(t)
        return float(h)


def maf_ref_exact(ft):
    tot = ft[0] + ft[1] + ft[2]
    if tot == 0:
        return None
    m = Fraction(2 * ft[0] + ft[1], tot)
    return max(m, 1 - m)


@functools.lru_cache(maxsize=None)
def reference(key):
    """Everything the bounds need for one count vector (8 ints, cases then controls)."""
    ca, co = list(key[:4]), list(key[4:])
    chi_g, df, dev = genotypic_exact(ca, co)
    n = sum(ca) + sum(co)
    mar = [ca[g] + co[g] for g in range(4)]
    called = 2 * (sum(ca[:3]) + sum(co[:3]))
    c1, c2 = 2 * (ca[0] + co[0]) + ca[1] + co[1], 2 * (ca[2] + co[2]) + ca[1] + co[1]
    return dict(chi2_allelic=allelic_exact(ca, co), chi2_genotypic=chi_g, df=df, dev=dev,
                h=entropy_mp(mar, n), hy=entropy_mp(ca + co, n), maf_case=maf_ref_exact(ca), maf_ctrl=maf_ref_exact(co),
                maf_pooled=(np.float64(min(c1, c2)) / np.float64(called)) if called else math.nan)


def _div0(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    with np.errstate(all="ignore"):
        return np.where(a > 0, a / np.where(b > 0, b, 1.0), 0.0)


def check_bounds(counts, mi, stats, what):
    """Every bound of the module docstring for SNPs with these counts. Returns the worst error as a fraction of each bound
    and the per-SNP p-value references."""
    counts = np.asarray(counts, np.int64)
    # the premise of the allelic bound: the products of d = A_ca B_co - B_ca A_co are exact in fp64
    a_ca, b_ca = 2 * counts[:, 0] + counts[:, 1], 2 * counts[:, 2] + counts[:, 1]
    a_co, b_co = 2 * counts[:, 4] + counts[:, 5], 2 * counts[:, 6] + counts[:, 5]
    assert np.all(np.maximum(a_ca * b_co, b_ca * a_co) < 2 ** 53)
    worst = {k: 0.0 for k in ("chi2_allelic", "chi2_genotypic", "entropy", "p_allelic", "p_genotypic", "maf_ref")}

    def ratio(key, err, bound, info):
        assert err <= bound, (what, key, info, float(err), float(bound))
        worst[key] = max(worst[key], float(err / bound) if bound > 0 else 0.0)

    ca, co = counts[:, :4], counts[:, 4:]
    # exact fields: counts, margins, conditional probabilities, pooled MAF, df
    assert np.array_equal(mi["cases"], ca) and np.array_equal(mi["controls"], co), what
    assert np.array_equal(mi["margins"], ca + co), what
    want_pbc = np.concatenate([_div0(ca, ca.sum(1, keepdims=True)), _div0(co, co.sum(1, keepdims=True))], 1)
    want_pca = np.concatenate([_div0(ca, ca + co), _div0(co, ca + co)], 1)
    assert np.array_equal(mi["dPbc"].view(np.uint64), want_pbc.view(np.uint64)), what
    assert np.array_equal(mi["dPca"].view(np.uint64), want_pca.view(np.uint64)), what
    p_ref = np.zeros((len(counts), 2))
    for q, row in enumerate(counts):
        ref = reference(tuple(int(v) for v in row))
        info = (q, row.tolist())
        assert stats["df_genotypic"][q] == ref["df"], info
        mp_ = ref["maf_pooled"]
        assert (math.isnan(mp_) and math.isnan(stats["maf_pooled"][q])) or \
            np.float64(stats["maf_pooled"][q]).view(np.uint64) == np.float64(mp_).view(np.uint64), info
        for f, k in (("maf_ref_case", "maf_case"), ("maf_ref_ctrl", "maf_ctrl")):
            got = stats[f][q]
            if ref[k] is None:
                assert math.isnan(got), info
            else:
                want = float(ref[k])
                ratio("maf_ref", abs(Fraction(float(got)) - ref[k]), Fraction(np.spacing(want)), info)
        # allelic: relative 8u
        x, want = float(stats["chi2_allelic"][q]), ref["chi2_allelic"]
        if want == 0:
            assert x == 0.0, info
        else:
            ratio("chi2_allelic", float(abs(Fraction(x) - want) / want), 8 * U, info)
        # genotypic: conditioning bound
        x, want = float(stats["chi2_genotypic"][q]), ref["chi2_genotypic"]
        bound = 16 * U * float(want + ref["dev"])
        if bound == 0:
            assert x == 0.0, info
        else:
            ratio("chi2_genotypic", float(abs(Fraction(x) - want)), bound, info)
        # entropies
        for f, k in (("dMarginalEntropy", "h"), ("dMarginalEntropy_Y", "hy")):
            ratio("entropy", abs(float(mi[f][q]) - ref[k]), 16 * U * (1 + ref[k]), info)
        # p-values at the device's own statistic
        for j, (fx, fp, df) in enumerate((("chi2_allelic", "p_allelic", 1 if ref["chi2_allelic"] else 0),
                                          ("chi2_genotypic", "p_genotypic", ref["df"]))):
            x, p = float(stats[fx][q]), float(stats[fp][q])
            want = q_upper_mp(x, df)
            p_ref[q, j] = want
            assert math.isnan(p) == math.isnan(want), info
            rel = 4 * U if df == 2 else (x + 16) * U
            bound = rel * want + (2 * DENORM_MIN if want < DBL_MIN else 0.0)
            ratio(fp, abs(p - want), bound, (info, x, df))
    return worst, p_ref


# ---- count families ---------------------------------------------------------------------------------------------------
def _split(rng, n, p):
    return rng.multinomial(n, p).astype(np.int64)


def fam_dense(rng, n1, n2):
    out = []
    for q in range(4):
        miss = 0.0 if q < 2 else 0.05
        p = rng.dirichlet(np.ones(3)) * (1 - miss)
        p = np.append(p, miss)
        p2 = p if q % 2 else np.append(rng.dirichlet(np.ones(3)) * (1 - miss), miss)
        out.append(("dense", _split(rng, n1, p), _split(rng, n2, p2)))
    return out


def fam_structural(n1, n2):
    """Structural zeros for classes of at least 4 samples."""
    def v(*x):
        return np.array(x, np.int64)
    h1, h2 = n1 // 2, n2 // 2
    return [
        ("absent_one_class", v(h1, 0, n1 - h1, 0), v(n2 // 3, n2 // 3, n2 - 2 * (n2 // 3), 0)),
        ("absent_both_df1", v(h1, 0, n1 - h1 - 1, 1), v(n2 // 4, 0, n2 - n2 // 4, 0)),
        ("one_called_genotype", v(n1 - 2, 0, 0, 2), v(n2, 0, 0, 0)),
        ("class_uncalled", v(0, 0, 0, n1), v(h2, n2 - h2, 0, 0)),
        ("all_missing", v(0, 0, 0, n1), v(0, 0, 0, n2)),
        ("heterozygotes_only", v(0, n1, 0, 0), v(0, n2, 0, 0)),
        ("single_minor_allele", v(n1 - 1, 1, 0, 0), v(n2, 0, 0, 0)),
    ]


def fam_independence(rng, n1, n2):
    g = math.gcd(n1, n2)
    out = []
    for q in range(3):
        w = _split(rng, g, np.append(rng.dirichlet(np.ones(3)) * 0.97, 0.03) if q else rng.dirichlet(np.ones(4)))
        ca, co = w * (n1 // g), w * (n2 // g)
        out.append(("independent", ca, co))
        if q < 2:     # one sample moved: a tiny statistic with full cancellation in o - e
            m = ca.copy()
            src = int(np.argmax(m[:3]))
            if m[src] == 0:
                continue
            m[src] -= 1
            m[(src + 1) % 3] += 1
            out.append(("near_independent", m, co.copy()))
    return out


def _sweep_member(kind, n1, n2, k):
    base = []
    for n in (n1, n2):
        if kind == "geno1":
            base.append(np.array([n // 2, 0, n - n // 2, 0], np.int64))
        else:
            base.append(np.array([n // 3, n // 3, n - 2 * (n // 3), 0], np.int64))
    ca, co = base
    ca = ca + np.array([-k, 0, k, 0])
    co = co + np.array([k, 0, -k, 0])
    return ca, co


def _sweep_stat(kind, ca, co):
    ca, co = [int(v) for v in ca], [int(v) for v in co]
    return float(allelic_exact(ca, co) if kind == "allelic" else genotypic_exact(ca, co)[0])


def fam_tail(n1, n2):
    """One-parameter families (k cases aa -> bb, k controls bb -> aa) searched so that the allelic, the genotypic df-2 and the
    genotypic df-1 statistic land on 3.84, 30, 700, on both sides of where p crosses DBL_MIN and 2^-1074, and where p is 0.
    Entries carry the ladder they belong to, in increasing k."""
    out = []
    for kind, df in (("allelic", 1), ("geno2", 2), ("geno1", 1)):
        kmax = min(_sweep_member(kind, n1, n2, 0)[0][0], _sweep_member(kind, n1, n2, 0)[1][2])
        stat = functools.lru_cache(maxsize=None)(lambda k, kind=kind: _sweep_stat(kind, *_sweep_member(kind, n1, n2, k)))

        def first_at_least(t):
            lo, hi = 0, kmax
            if stat(hi) < t:
                return None
            while lo < hi:
                mid = (lo + hi) // 2
                lo, hi = (mid + 1, hi) if stat(mid) < t else (lo, mid)
            return lo
        x_min, x_den = tail_crossings(df)
        ladder = set()
        for t in (3.84, 30.0, 700.0):
            k = first_at_least(t)
            if k is not None:
                ladder.add(k)
        for t in (x_min, x_den):
            k = first_at_least(t)
            if k is not None:
                ladder.update(kk for kk in range(k - 2, k + 2) if 0 <= kk <= kmax)
        for t in (x_den * 1.05, x_den * 2):
            k = first_at_least(t)
            if k is not None:
                ladder.add(k)
        for k in sorted(ladder):
            ca, co = _sweep_member(kind, n1, n2, k)
            out.append(("tail_" + kind, ca, co))
    return out


def families(rng, n1, n2, tail=True):
    """(family, case counts, control counts) for class sizes n1, n2."""
    out = fam_dense(rng, n1, n2)
    if min(n1, n2) >= 4:
        out += fam_structural(n1, n2) + fam_independence(rng, n1, n2)
    if tail and min(n1, n2) >= 2000:
        out += fam_tail(n1, n2)
    return out


def tiny_targets(rng, n1, n2, k):
    """Every lane width and degenerate corner of tiny classes: random compositions, the empty class included."""
    out = []
    for _ in range(k):
        out.append(("tiny", _split(rng, n1, rng.dirichlet(np.full(4, 0.5))), _split(rng, n2, rng.dirichlet(np.full(4, 0.5)))))
    return out


# ---- realised cohorts -------------------------------------------------------------------------------------------------
def first_hom_is_bb(row):
    hom = np.flatnonzero((row == 0) | (row == 2))
    return len(hom) > 0 and row[hom[0]] == 2


def force_bb_first(row, pheno):
    """Swap two samples of one class so that the row's first called homozygote is bb (class counts unchanged)."""
    hom = np.flatnonzero((row == 0) | (row == 2))
    if not len(hom) or row[hom[0]] == 2:
        return len(hom) > 0
    f = hom[0]
    same = np.flatnonzero((row == 2) & (pheno == pheno[f]))
    if len(same):
        row[f], row[same[0]] = 2, row[f]
        return True
    for cls in np.unique(pheno[row == 2]):
        earlier = np.flatnonzero(pheno[:f] == cls)
        if len(earlier):
            g = np.flatnonzero((row == 2) & (pheno == cls))[0]
            row[earlier[0]], row[g] = 2, row[earlier[0]]
            return True
    return False


def recount(codes, pheno):
    """Host recount of the store's counts [K, 8]: per class {aa, ab, bb, xx} under first-seen labels."""
    out = np.zeros((codes.shape[0], 8), np.int64)
    for cls, off in ((1, 0), (0, 4)):
        idx = np.flatnonzero(pheno == cls)
        for r in range(codes.shape[0]):
            out[r, off:off + 4] = np.bincount(codes[r, idx], minlength=4)
    swap = np.array([first_hom_is_bb(codes[r]) for r in range(codes.shape[0])])
    out[swap] = out[swap][:, np.concatenate([PERM, 4 + PERM])]
    return out


class Cohort:
    def __init__(self, entries, n_case, n_ctrl, n_neither, seed, relabel_every=3):
        import oracle
        rng = np.random.default_rng(seed)
        # relabelled copies: the same target again, with its first called homozygote forced to bb
        entries = list(entries)
        self.relabel_of = {}
        for q in range(0, len(entries), relabel_every):
            self.relabel_of[len(entries)] = q
            entries.append((entries[q][0] + "/relabelled",) + tuple(entries[q][1:]))
        self.families = [e[0] for e in entries]
        self.targets = np.array([np.concatenate([e[1], e[2]]) for e in entries], np.int64)
        self.K, self.N = len(entries), n_case + n_ctrl + n_neither
        self.pheno = np.array([1] * n_case + [0] * n_ctrl + [2] * n_neither, np.uint8)
        rng.shuffle(self.pheno)
        self.codes = np.zeros((self.K, self.N), np.uint8)
        idx = [np.flatnonzero(self.pheno == c) for c in (1, 0, 2)]
        for r, t in enumerate(self.targets):
            for c, part in ((0, t[:4]), (1, t[4:])):
                assert part.sum() == len(idx[c])
                self.codes[r, idx[c]] = rng.permutation(np.repeat(np.arange(4, dtype=np.uint8), part))
            self.codes[r, idx[2]] = rng.integers(0, 4, len(idx[2]))
            if r in self.relabel_of:
                force_bb_first(self.codes[r], self.pheno)
        self.rows = oracle.Oracle().pack_codes(self.codes)
        self.n_case, self.n_ctrl = n_case, n_ctrl

    def expected(self, pheno=None):
        return recount(self.codes, self.pheno if pheno is None else pheno)

    def store(self, eager=False):
        st = gw.GenoStore(self.K, self.N)
        st.set_select_mode(eager)
        st.put_rows(self.rows)
        return st


# tier -> (cases, controls, neither)
TIERS = {"2k": (2000, 2000, 300), "45k": (20000, 25000, 0), "200k": (100000, 100000, 0), "660k": (300000, 300000, 60000),
         "1.9M": (1000000, 900000, 0), "2^23": (CLASS_LIMIT, CLASS_LIMIT, 0)}
TINY = [(0, 5, 5), (1, 1, 5), (1, 8, 5), (3, 5, 5), (8, 8, 5), (8, 1, 5)]
SCAN_TIERS = ["tiny"] + list(TIERS)


def _tier_entries(rng, tier):
    n1, n2, _ = TIERS[tier]
    ent = families(rng, n1, n2)
    if tier == "1.9M":          # 63 SNPs with the relabelled copies, for the pair screen: more dense ones
        ent = (fam_dense(rng, n1, n2) + ent)[:56]
    if tier == "2^23":          # 14 SNPs with the copies: one of each kind, 700 and the DBL_MIN crossing of the df-2 ladder, p = 0
        pick = {}
        for e in ent:
            pick.setdefault(e[0], []).append(e)
        tail = pick["tail_geno2"]
        ent = pick["dense"][0:1] + pick["dense"][2:3] + pick["absent_both_df1"] + pick["all_missing"] + pick["independent"][:1] + \
            pick["near_independent"][:1] + tail[2:3] + tail[4:6] + tail[-1:]
    return ent


@functools.lru_cache(maxsize=None)
def cohort(tier, sub=0):
    if tier == "tiny":
        n1, n2, nn = TINY[sub]
        rng = np.random.default_rng(900 + sub)
        return Cohort(tiny_targets(rng, n1, n2, 40) + (fam_structural(n1, n2) if min(n1, n2) >= 4 else []), n1, n2, nn, 950 + sub)
    rng = np.random.default_rng(1000 + list(TIERS).index(tier))
    n1, n2, nn = TIERS[tier]
    return Cohort(_tier_entries(rng, tier), n1, n2, nn, 2000 + list(TIERS).index(tier), relabel_every=8 if tier == "1.9M" else 3)


def cohorts(tier):
    return [cohort("tiny", s) for s in range(len(TINY))] if tier == "tiny" else [cohort(tier)]


@functools.lru_cache(maxsize=None)
def finalize_only():
    """Bare count vectors with class totals up to 2^23 - 1, for gwasdev_marginal_finalize alone."""
    rng = np.random.default_rng(77)
    out = []
    for n1, n2 in ((CLASS_LIMIT, CLASS_LIMIT), (CLASS_LIMIT, 5), (7, CLASS_LIMIT), (4_000_000, 3_000_000), (65_535, 65_536)):
        out += [(f if not f.startswith("tail_") else f"{f}@{n1},{n2}", ca, co) for f, ca, co in families(rng, n1, n2)]
    return np.array([np.concatenate([e[1], e[2]]) for e in out], np.int64), [e[0] for e in out]


# ---- CPU --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tier", ["tiny", "2k", "45k", "200k"])
def test_realiser_builds_the_targets(orc, tier):
    """The oracle's counts of the realised rows are the targets under the store's labels; the relabelled copies do start
    with bb and carry their original's counts with aa and bb swapped."""
    for co_ in cohorts(tier):
        got = orc.cc_counts_masked(co_.rows, co_.N, co_.pheno).astype(np.int64)
        assert np.array_equal(got, co_.expected())
        swap = np.array([first_hom_is_bb(co_.codes[r]) for r in range(co_.K)])
        want = co_.targets.copy()
        want[swap] = want[swap][:, np.concatenate([PERM, 4 + PERM])]
        assert np.array_equal(got, want)
        for r, q in co_.relabel_of.items():
            assert np.array_equal(co_.targets[r], co_.targets[q])
        if tier != "tiny":
            assert sum(swap[r] for r in co_.relabel_of) >= 0.8 * len(co_.relabel_of)


def _oracle_stats(orc, counts):
    n = len(counts)
    from libgwaspp_b200 import MI_DTYPE, STATS_DTYPE
    mi, st = np.zeros(n, MI_DTYPE), np.zeros(n, STATS_DTYPE)
    for q, c in enumerate(counts):
        ca, co = c[:4].astype(np.uint32), c[4:].astype(np.uint32)
        mi[q] = orc.marginal_information(ca, co, int(c.sum()))
        st["maf_ref_case"][q], st["maf_ref_ctrl"][q] = orc.maf_reference(ca)[0], orc.maf_reference(co)[0]
        st["chi2_allelic"][q], st["p_allelic"][q] = orc.chi2_allelic(ca, co)
        st["chi2_genotypic"][q], st["p_genotypic"][q], st["df_genotypic"][q] = orc.chi2_genotypic(ca, co)
        called = 2 * (int(c[:3].sum()) + int(c[4:7].sum()))
        c1 = 2 * (int(c[0]) + int(c[4])) + int(c[1]) + int(c[5])
        st["maf_pooled"][q] = min(c1, called - c1) / called if called else math.nan
    return mi, st


def _count_sets():
    sets = {"finalize_only": finalize_only()}
    for tier in ["tiny", "2k", "45k", "200k"]:
        co_ = cohorts(tier)
        sets[tier] = (np.concatenate([c.expected() for c in co_]), sum((c.families for c in co_), []))
    return sets


@pytest.mark.parametrize("which", ["tiny", "2k", "45k", "200k", "finalize_only"])
def test_oracle_statistics_meet_the_bounds(orc, which):
    """The host oracle's fp64 evaluation, in the device's operation order, meets every bound (so none is too tight), and on
    the near-independence SNPs its genotypic statistic misses a 1e-12 relative bar (so the conditioning bound is needed)."""
    counts, fams = _count_sets()[which]
    mi, st = _oracle_stats(orc, counts)
    worst, _ = check_bounds(counts, mi, st, which)
    print(f"oracle {which}: worst error / bound {worst}")
    if which == "finalize_only":
        near = [q for q, f in enumerate(fams) if f == "near_independent"]
        rel = [abs(Fraction(float(st["chi2_genotypic"][q])) - reference(tuple(int(v) for v in counts[q]))["chi2_genotypic"])
               / reference(tuple(int(v) for v in counts[q]))["chi2_genotypic"] for q in near]
        assert max(rel) > 1e-12, rel


def test_tail_sweep_reaches_its_targets():
    """At 2 000 per class the sweep straddles both underflow crossings of every test kind and reaches p = 0."""
    ent = fam_tail(2000, 2000)
    for kind, df in (("allelic", 1), ("geno2", 2), ("geno1", 1)):
        xs = [_sweep_stat(kind, e[1], e[2]) for e in ent if e[0] == "tail_" + kind]
        assert xs == sorted(xs), (kind, xs)      # increasing along the ladder: the device p-values must not increase
        x_min, x_den = tail_crossings(df)
        for t in (3.84, 30.0, 700.0):
            assert any(t <= x < 1.1 * t for x in xs), (kind, t, xs)
        for t in (x_min, x_den):
            assert any(x < t for x in xs) and any(x >= t for x in xs), (kind, t, xs)
        assert q_upper_mp(xs[-1], df) == 0.0
    assert 1400 < tail_crossings(1)[0] < tail_crossings(2)[0] < 1420 and 1480 < tail_crossings(1)[1] < tail_crossings(2)[1] < 1490


def test_mpmath_restatement_matches_scipy():
    """The references are the textbook tests: scipy's chi2_contingency without continuity correction and chi2.sf, where
    scipy is accurate."""
    scipy_stats = pytest.importorskip("scipy.stats")
    rng = np.random.default_rng(5)
    n = 0
    for name, ca, co in families(rng, 2000, 2500) + families(rng, 37, 41, tail=False):
        ref = reference(tuple(int(v) for v in np.concatenate([ca, co])))
        a = np.array([[2 * ca[0] + ca[1], 2 * ca[2] + ca[1]], [2 * co[0] + co[1], 2 * co[2] + co[1]]])
        if a.sum(0).all() and a.sum(1).all():
            x = scipy_stats.chi2_contingency(a, correction=False)[0]
            assert abs(x - float(ref["chi2_allelic"])) <= 1e-9 * max(x, 1e-3), (name, x)
            n += 1
        g = np.array([ca[:3], co[:3]])
        g = g[:, g.sum(0) > 0]
        if g.shape[1] > 1 and g.sum(1).all():
            x, _, dof, _ = scipy_stats.chi2_contingency(g, correction=False)
            assert dof == ref["df"] and abs(x - float(ref["chi2_genotypic"])) <= 1e-9 * max(x, 1e-3), (name, x)
    assert n > 20
    for x in (0.01, 1.0, 3.84, 30.0, 200.0, 700.0):
        for df in (1, 2):
            want = scipy_stats.chi2.sf(x, df)
            assert abs(q_upper_mp(x, df) - want) <= 1e-13 * want, (x, df)


# ---- GPU --------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _underflow_report(counts, stats, fams):
    """Smallest statistic whose device p-value is subnormal / 0, per test kind."""
    rep = {}
    for f, fp, fx in (("allelic", "p_allelic", "chi2_allelic"), ("geno", "p_genotypic", "chi2_genotypic")):
        for df in ((1,) if f == "allelic" else (1, 2)):
            sel = stats["df_genotypic"] == df if f == "geno" else np.ones(len(stats), bool)
            x, p = stats[fx][sel], stats[fp][sel]
            sub = x[(p < DBL_MIN) & (p > 0)]
            zero = x[p == 0]
            rep[f"{f}_df{df}"] = (float(sub.min()) if len(sub) else None, float(zero.min()) if len(zero) else None)
    return rep


def _check_ladders(stats, fams):
    """p non-increasing along each tail ladder (one per sweep kind and class sizes, in increasing chi-square)."""
    for ladder in set(f for f in fams if f.startswith("tail_") and not f.endswith("/relabelled")):
        q = [i for i, f in enumerate(fams) if f == ladder]
        p = stats["p_allelic" if ladder.startswith("tail_allelic") else "p_genotypic"][q]
        assert len(q) >= 2 and np.all(np.diff(p) <= 0), (ladder, p)


@gpu
@pytest.mark.parametrize("which", ["tiny", "2k", "45k", "200k", "660k", "1.9M", "2^23", "finalize_only"])
def test_finalize_meets_the_bounds(which, record_property):
    if which == "finalize_only":
        counts, fams = finalize_only()
    else:
        co_ = cohorts(which)
        counts, fams = np.concatenate([c.expected() for c in co_]), sum((c.families for c in co_), [])
    mi, st = gw.marginal_finalize(counts.astype(np.uint32))
    worst, _ = check_bounds(counts, mi, st, which)
    _check_ladders(st, fams)
    rep = _underflow_report(counts, st, fams)
    for k, v in worst.items():
        record_property(f"worst_{k}", v)
    print(f"\nfinalize {which}: worst error / bound {worst}; smallest chi2 with subnormal / zero p {rep}")


def _finalize_of(counts):
    return gw.marginal_finalize(np.ascontiguousarray(counts, np.uint32))


def _check_scan(out, want, what, begin=0, end=None):
    end = len(want) if end is None else end
    want = want[begin:end]
    mi, st = _finalize_of(want)
    assert np.array_equal(out["counts"], want), what
    assert out["mi"].tobytes() == mi.tobytes(), what
    assert out["stats"].tobytes() == st.tobytes(), what


def _k0_fits(n_sel_case, n_sel_ctrl):
    return -(-n_sel_case // 128) + -(-n_sel_ctrl // 128) <= 6400


def _scan_paths(co_, pheno, what):
    """Every scan path of one selection: first and later scans, lane widths, the knobs, pieces, unaligned sub-ranges and the
    eager selection; each against the host recount and byte-identical to gwasdev_marginal_finalize of those counts."""
    want = co_.expected(pheno)
    nca, nco = int((pheno == 1).sum()), int((pheno == 0).sum())
    partition = nca + nco == co_.N
    fits = _k0_fits(nca, nco)
    with co_.store() as st:
        st.select_case_control(pheno)
        assert (st.n_case, st.n_ctrl) == (nca, nco)
        _check_scan(st.marginal_scan(), want, (what, "first"))
        assert not st.is_compacted()
        _check_scan(st.marginal_scan(), want, (what, "second"))
        assert st.is_compacted() == (fits and not partition), what
        _check_scan(st.marginal_scan(), want, (what, "third"))
        for b, e in ((1, co_.K - 2), (co_.K - 3, co_.K), (co_.K // 2, co_.K // 2 + 1)):
            if 0 <= b < e <= co_.K:
                _check_scan(st.marginal_scan(b, e), want, (what, "range", b, e), b, e)
        for opt, vals in ((gw.OPT_LANES_PER_ROW, (8, 16, 32)), (gw.OPT_MASKED_SCAN, (1,)), (gw.OPT_ROW_TOTALS, (1,)), (gw.OPT_SCAN_PIECES, (8,))):
            for v in vals:
                st.set_option(opt, v)
                st.select_case_control(pheno)
                for k in range(2):
                    _check_scan(st.marginal_scan(), want, (what, opt, v, k))
                _check_scan(st.marginal_scan(1, co_.K - 1), want, (what, opt, v, "range"), 1, co_.K - 1)
                st.set_option(opt, 0)
        acc = np.zeros((co_.K, 8), np.uint32)
        st.marginal_accumulate(acc)
        assert np.array_equal(acc, want), what
    if fits:
        with co_.store(eager=True) as st:
            st.select_case_control(pheno)
            assert st.is_compacted()
            _check_scan(st.marginal_scan(), want, (what, "eager"))
    return want


@gpu
@pytest.mark.parametrize("tier", SCAN_TIERS)
def test_scan_paths(tier):
    for co_ in cohorts(tier):
        _scan_paths(co_, co_.pheno, tier)
    if tier in ("660k", "1.9M"):
        co_ = cohort(tier)
        if tier == "660k":     # the same table re-selected as a partition: the samples in neither class become controls
            p2 = np.where(co_.pheno == 2, 0, co_.pheno).astype(np.uint8)
        else:                  # 1 000 controls moved out of both classes: two masks of 237 KB, no K0
            p2 = co_.pheno.copy()
            p2[np.flatnonzero(p2 == 0)[:1000]] = 2
        _scan_paths(co_, p2, tier + " reselected")


@gpu
@pytest.mark.parametrize("tier", ["tiny", "2k", "45k"])
def test_scan_compact(tier):
    """32-byte records are the float32 of the fp64 statistics, the tail extremes included; the significant list is exactly
    the SNPs with min(p_allelic, p_genotypic) < threshold (strict), with fp64 statistics equal to the plain scan's."""
    for co_ in cohorts(tier):
        with co_.store() as st:
            st.select_case_control(co_.pheno)
            plain = st.marginal_scan()
            s = plain["stats"]
            for k in range(2):      # first (masked) and later scans
                rec, _ = st.marginal_scan_compact()
                assert np.array_equal(rec["cases"], plain["counts"][:, :4]) and np.array_equal(rec["controls"], plain["counts"][:, 4:])
                for f in ("chi2_allelic", "p_allelic", "chi2_genotypic", "p_genotypic"):
                    assert np.array_equal(rec[f].view(np.uint32), s[f].astype(np.float32).view(np.uint32)), (tier, f, k)
            pmin = np.minimum(s["p_allelic"], s["p_genotypic"])
            present = np.unique(pmin[(pmin > 0) & (pmin < 1)])
            thresholds = [1e-300, DBL_MIN, DENORM_MIN] + ([present[0], present[len(present) // 2], present[-1]] if len(present) else [])
            for thr in thresholds:
                rec, sig = st.marginal_scan_compact(p_threshold=float(thr))
                want = np.flatnonzero(pmin < thr)
                assert np.array_equal(sig["snp"], want), (tier, thr)
                for f in ("maf_pooled", "chi2_allelic", "p_allelic", "chi2_genotypic", "p_genotypic"):
                    assert np.array_equal(sig[f].view(np.uint64), s[f][want].view(np.uint64)), (tier, thr, f)
                assert np.array_equal(sig["df_genotypic"], s["df_genotypic"][want].astype(np.uint32))
            if tier != "tiny":
                assert (pmin == 0).sum() >= 3 and (pmin[pmin > 0] < DBL_MIN).sum() >= 3


@gpu
def test_scan_compact_refuses_records_at_200k():
    co_ = cohort("200k")
    with co_.store() as st:
        st.select_case_control(co_.pheno)
        with pytest.raises(gw.GwasDevError, match="65 536"):
            st.marginal_scan_compact()
        _, sig = st.marginal_scan_compact(records=False, p_threshold=DBL_MIN)
        s = st.marginal_scan()["stats"]
        assert np.array_equal(sig["snp"], np.flatnonzero(np.minimum(s["p_allelic"], s["p_genotypic"]) < DBL_MIN))
        assert len(sig) >= 3


def _caller_masks(rng, co_, sizes):
    sel = np.flatnonzero(co_.pheno != 2)
    masks, phenos = [], []
    for m in sizes:
        p = np.where(co_.pheno == 2, 2, 0).astype(np.uint8)
        p[rng.choice(sel, m, replace=False)] = 1
        phenos.append(p)
        masks.append(gw.stream_masks(p)[0])
    return np.array(masks), phenos


def _check_permute(co_, sizes, seed, what):
    masks, phenos = _caller_masks(np.random.default_rng(seed), co_, sizes)
    with co_.store() as st:
        st.select_case_control(co_.pheno)
        out = st.marginal_permute(len(sizes), case_masks=masks, perm_stats=True)
    worst = {}
    for k, p in enumerate(phenos):
        want = co_.expected(p)
        mi, s = _finalize_of(want)
        ps = out["perm_stats"][k]
        assert np.array_equal(ps[:, 0].view(np.uint64), s["chi2_allelic"].view(np.uint64)), (what, k)
        assert np.array_equal(ps[:, 1].view(np.uint64), s["chi2_genotypic"].view(np.uint64)), (what, k)
        w, _ = check_bounds(want, mi, s, (what, k))
        worst = {key: max(worst.get(key, 0), v) for key, v in w.items()}
    return worst


@gpu
def test_permute_caller_masks_200k():
    """Each perm_stats row is byte-identical to gwasdev_marginal_finalize of the counts recounted under its case mask."""
    n = cohort("200k").N
    worst = _check_permute(cohort("200k"), [n // 2, n // 3, 1, n - 1, 12345, n // 2 + 7, 99_999, 150_000], 31, "200k")
    print(f"\npermute 200k: worst error / bound {worst}")


@gpu
def test_permute_observed_scan_1_9m():
    """The permutation test's observed scan runs on a cohort that K0 cannot compact."""
    n = cohort("1.9M").N
    _check_permute(cohort("1.9M"), [n // 2, 1_000_000], 32, "1.9M")


@gpu
def test_pair_screen_1_9m(orc):
    """The pair screen (four-plane tensor-core kernel, one pair of planes per class) on the 1.9M tier's SNPs without missing
    calls, 1 000 000 cases and 900 000 controls, whose margins come from a scan that K0 cannot compact: every pair with a
    statistic, equal to the oracle. The whole tier, with missing calls, takes the two-accumulator mode, which needs the
    compacted rows: refused with K0's message."""
    co_ = cohort("1.9M")
    keep = np.flatnonzero(~(co_.codes == 3).any(1))
    assert len(keep) >= 30
    rows = co_.rows[keep]
    sel, nca, nco = orc.select(rows, co_.N, co_.pheno)
    mar = orc.margins(sel, nca, nco)
    hi, hj, hs, _ = orc.boost_screen(sel, mar, nca, nco, -1e9)
    with gw.GenoStore(len(keep), co_.N) as st:
        st.put_rows(rows)
        st.select_case_control(co_.pheno)
        hits, stats = st.pairwise_scan(-1e9)
        assert not st.is_compacted()
    assert stats.pairs_tested == len(keep) * (len(keep) - 1) // 2
    assert len(hi) > 0.5 * stats.pairs_tested
    assert np.array_equal(hits["i"], hi) and np.array_equal(hits["j"], hj)
    # the KSA statistic cancels near independence: the conditioning bound of test_gpu_pair_statistics, 2n 16u S
    from test_gpu_pair_statistics import ULPS, ksa_mp
    n = nca + nco
    S = np.array([ksa_mp(*orc.pair_table(3, int(i), int(j), sel=sel, nca=nca, nco=nco, mar=mar), mar[i], mar[j], n)[1]
                  for i, j in zip(hi, hj)])
    assert np.all(np.abs(hits["stat"] - hs) <= 2 * n * ULPS * U * S)
    with co_.store() as st:
        st.select_case_control(co_.pheno)
        with pytest.raises(gw.GwasDevError, match="row buffer"):
            st.pairwise_scan(-1e9)


@gpu
def test_compacted_layout_refused_above_k0_limit():
    """Above K0's row buffer, what needs the compacted layout (eager select, gwasdev_get_selected_rows, gwasdev_counts mode 2,
    gwasdev_pair_tables mode 2) is refused with its message; the mask-on-the-fly counts and pair tables still work."""
    co_ = cohort("1.9M")
    with co_.store(eager=True) as st:
        with pytest.raises(gw.GwasDevError, match="row buffer"):
            st.select_case_control(co_.pheno)
    with co_.store() as st:
        st.select_case_control(co_.pheno)
        for call in (lambda: st.get_selected_rows(0, 1), lambda: st.counts(2), lambda: st.pair_tables([0], [1], 2)):
            with pytest.raises(gw.GwasDevError, match="row buffer"):
                call()
        assert np.array_equal(st.counts(1), co_.expected())
        assert st.pair_tables([0], [1], 1).shape == (1, 32)
        _check_scan(st.marginal_scan(), co_.expected(), "1.9M after refusals")
