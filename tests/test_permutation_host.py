"""Host arithmetic of the permutation test: the permutation draws and the empirical p-values (no device needed)."""
import math

import numpy as np
import pytest

import libgwaspp_b200 as gw

M64 = (1 << 64) - 1


def sim_hash(seed, a, b):
    z = (seed + 0x9E3779B97F4A7C15 * (a + 1) + 0xD1B54A32D192ED03 * (b + 1)) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def ref_masks(pheno_case, pheno_ctrl, seed, first_perm, n_perm):
    """Knuth's selection sampling over the selected samples in increasing position (include/gwasdev.h)."""
    n = len(pheno_case)
    sel = np.flatnonzero(pheno_case | pheno_ctrl)
    n_case = int(pheno_case.sum())
    out = np.zeros((n_perm, n), bool)
    for k in range(n_perm):
        need = n_case
        for rank, c in enumerate(sel):
            left = len(sel) - rank
            u = sim_hash(seed, first_perm + k, rank) >> 32
            if (u * left) >> 32 < need:
                out[k, c] = True
                need -= 1
    return out


def to_bits(masks, n):
    bits = np.unpackbits(masks.view(np.uint8), axis=-1, bitorder="little").astype(bool)
    return bits[..., :n]


@pytest.mark.parametrize("n, seed, first_perm", [(37, 1, 0), (300, 7, 5), (1001, 12345, 1 << 33)])
def test_masks_match_the_restatement(n, seed, first_perm):
    rng = np.random.default_rng(n)
    pheno = rng.integers(0, 4, n)                     # 1 case, 0 control, 2 neither, 3 both masks
    ca, co = pheno % 2 == 1, (pheno == 0) | (pheno == 3)
    case_mask, _ = gw.stream_masks(ca.astype(np.uint8))
    ctrl_mask, _ = gw.stream_masks(co.astype(np.uint8))
    n_perm = 9
    got = gw.permutation_masks(n, case_mask, ctrl_mask, seed, first_perm, n_perm)
    bits = to_bits(got, n)
    np.testing.assert_array_equal(bits, ref_masks(ca, co, seed, first_perm, n_perm))
    assert (bits.sum(1) == ca.sum()).all()                      # exactly n_case cases
    assert not (bits & ~(ca | co)).any()                        # never outside the selection
    # offsets restate: permutations 3.. of the same call
    np.testing.assert_array_equal(gw.permutation_masks(n, case_mask, ctrl_mask, seed, first_perm + 3, 4), got[3:7])
    # bits beyond the sample count stay clear
    assert not to_bits(got, 16 * got.shape[1])[:, n:].any()


def chisq_q(x, df):
    if not x > 0:
        return 1.0
    return math.erfc(math.sqrt(0.5 * x)) if df == 1 else math.exp(-0.5 * x)


def ref_pvalues(obs, exceed, perm_max):
    P = perm_max.shape[0]
    emp1 = (exceed + 1.0) / (P + 1)
    emp2 = np.zeros_like(emp1)
    minp = np.array([min(chisq_q(a, 1), chisq_q(b, 2)) for a, b in perm_max[:, 1:]])
    for i, o in enumerate(obs):
        emp2[i, 0] = (1 + (perm_max[:, 0] >= o["chi2_allelic"]).sum()) / (P + 1)
        df = int(o["df_genotypic"])
        emp2[i, 1] = 1.0 if df == 0 else (1 + (minp <= chisq_q(o["chi2_genotypic"], df)).sum()) / (P + 1)
    return emp1, emp2


@pytest.mark.parametrize("P", [1, 2, 50])
def test_pvalues_match_numpy(P):
    rng = np.random.default_rng(P)
    n = 40
    obs = np.zeros(n, gw.STATS_DTYPE)
    obs["chi2_allelic"] = rng.choice([0.0, 0.5, 2.0, 3.841, 10.0], n)
    obs["chi2_genotypic"] = rng.choice([0.0, 1.0, 4.0, 5.99, 12.0], n)
    obs["df_genotypic"] = rng.choice([0, 1, 2], n)
    perm_max = rng.choice([0.0, 0.5, 2.0, 3.841, 4.0, 5.99, 10.0], (P, 3))    # ties at equality with the observed values
    exceed = rng.integers(0, P + 1, (n, 2)).astype(np.uint32)
    emp1, emp2 = gw.permutation_pvalues(obs, exceed, perm_max)
    r1, r2 = ref_pvalues(obs, exceed.astype(float), perm_max)
    np.testing.assert_array_equal(emp1, r1)
    np.testing.assert_array_equal(emp2, r2)
    assert (emp2[obs["df_genotypic"] == 0, 1] == 1.0).all()
