"""Shared test helpers (test infrastructure)."""
import os

import numpy as np

import libgwaspp_b200 as gw

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def planted_cohort(orc, seed, M, N, n_case, missing, n_planted):
    """Seeded synthetic cohort with a few case-only SNP-SNP dependencies so that the KSA screen crosses 30
    (same construction as tests/golden/make_golden.py)."""
    codes, pheno = orc.simulate(seed, M, N, n_case, missing_rate=missing)
    rng = np.random.default_rng(seed)
    cand = [r for r in range(M) if (codes[r] == 2).sum() > 0.04 * N]
    rng.shuffle(cand)
    for k in range(n_planted):
        i, j = sorted((cand[2 * k], cand[2 * k + 1]))
        src = codes[i].copy()
        src[src == 3] = 0
        codes[j, pheno == 1] = src[pheno == 1]
    return codes, pheno


def rel_close(a, b, rel):
    """element-wise |a-b| <= rel*|b|, NaN == NaN, inf == inf."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    same_nan = np.isnan(a) & np.isnan(b)
    same_inf = np.isinf(a) & np.isinf(b) & (np.sign(a) == np.sign(b))
    with np.errstate(invalid="ignore"):
        ok = np.abs(a - b) <= rel * np.abs(b)
    return bool(np.all(ok | same_nan | same_inf))


# ---- linkage disequilibrium: the contract of include/gwasdev.h restated in numpy ---------------------------------------------
def bits_of(blocks, n):
    return np.unpackbits(np.ascontiguousarray(blocks, np.uint16).view(np.uint8), axis=-1, bitorder="little")[..., :n].astype(bool)


def decoded(s):
    """(x, called) under the store's own labels, from the raw planes: aa 0, ab 1, bb 2."""
    rows = s.get_rows()
    P, N = s.P, s.n_samples
    p1, p2 = bits_of(rows[:, 1:1 + P], N), bits_of(rows[:, 1 + P:], N)
    return (p2 & ~p1).astype(np.int64) + 2 * (p1 & p2), p1 | p2


def ld_reference(x, c, mask=None):
    """Every pair's (n, r, r2) as (M, M) matrices: the contract's integer sums and IEEE fp64 steps, restated in numpy."""
    cm = c & (True if mask is None else mask[None, :])
    X, Cf = np.where(cm, x, 0).astype(np.float64), cm.astype(np.float64)
    mm = lambda a, b: np.rint(a @ b.T).astype(np.int64)                   # exact: every sum is far below 2^53
    n, sx, sxx, sxy = mm(Cf, Cf), mm(X, Cf), mm(X * X, Cf), mm(X, X)
    sy, syy = sx.T, sxx.T
    num, vx, vy = n * sxy - sx * sy, n * sxx - sx * sx, n * syy - sy * sy
    with np.errstate(invalid="ignore", divide="ignore"):
        v = vx.astype(np.float64) * vy.astype(np.float64)
        r2 = (num.astype(np.float64) * num.astype(np.float64)) / v
        r = num.astype(np.float64) / np.sqrt(v)
    undef = (vx == 0) | (vy == 0)
    r2[undef] = np.nan
    r[undef] = np.nan
    return n, r, r2


def band_of(ref_r2, lo, hi, window):
    b = np.full((hi - lo, window), np.nan, np.float32)
    for i in range(lo, hi):
        j = np.arange(i + 1, min(hi, i + window + 1))
        b[i - lo, j - i - 1] = ref_r2[i, j].astype(np.float32)
    return b


def list_of(ref, lo, hi, window, thr):
    n, r, r2 = ref
    I, J = np.triu_indices(n.shape[0], 1)
    sel = (I >= lo) & (J < hi) & (J - I <= window)
    I, J = I[sel], J[sel]
    with np.errstate(invalid="ignore"):
        k = r2[I, J] >= thr
    out = np.zeros(int(k.sum()), gw.LD_PAIR_DTYPE)
    out["i"], out["j"], out["n"], out["r"], out["r2"] = I[k], J[k], n[I[k], J[k]], r[I[k], J[k]], r2[I[k], J[k]]
    return out
