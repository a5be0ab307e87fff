"""CPU checks of the LD surface: gwasdev_ld_prune (host arithmetic) against a restatement of its rule, and the record layouts."""
import ctypes as C

import numpy as np
import pytest

import libgwaspp_b200 as gw
import libgwaspp_b200.build as gwbuild


@pytest.fixture(scope="module", autouse=True)
def lib():
    gwbuild.build()
    return gw.load_library()


def prune_restated(pairs, window, thr, lo, hi):
    """Walk i upwards: i is kept unless a kept k in [max(lo, i - window), i) has r2(k, i) >= thr."""
    r2 = {(int(p["i"]), int(p["j"])): float(p["r2"]) for p in pairs}
    keep = np.zeros(hi - lo, bool)
    for i in range(lo, hi):
        keep[i - lo] = not any(keep[k - lo] and r2.get((k, i), np.nan) >= thr for k in range(max(lo, i - window), i))
    return keep


def random_pairs(rng, lo, hi, window, density):
    pairs = [(i, j) for i in range(lo, hi) for j in range(i + 1, min(hi, i + window + 1)) if rng.random() < density]
    out = np.zeros(len(pairs), gw.LD_PAIR_DTYPE)
    if pairs:
        out["i"], out["j"] = np.array(pairs).T
    out["r2"] = rng.random(len(pairs))
    out["r2"][rng.random(len(pairs)) < 0.05] = np.nan
    out["r"] = np.sqrt(out["r2"])
    return out


def test_layouts():
    assert gw.LD_PAIR_DTYPE.itemsize == 32 and C.sizeof(gw.LdStats) == 40
    assert gw.OPT_LD_OPERAND_BYTES == 11


@pytest.mark.parametrize("seed", range(8))
def test_prune_matches_the_rule_and_its_two_properties(seed):
    rng = np.random.default_rng(seed)
    lo = int(rng.integers(0, 20))
    hi = lo + int(rng.integers(1, 160))
    window = int(rng.integers(1, 40))
    thr = float(rng.choice([0.0, 0.2, 0.5, 0.9, 1.0]))
    pairs = random_pairs(rng, lo, hi, window, float(rng.choice([0.02, 0.2, 0.7])))
    keep = gw.ld_prune(pairs, window, thr, lo, hi)
    np.testing.assert_array_equal(keep, prune_restated(pairs, window, thr, lo, hi))
    hit = {(int(p["i"]), int(p["j"])) for p in pairs if p["r2"] >= thr}
    kept = [i for i in range(lo, hi) if keep[i - lo]]
    # no two kept SNPs within the window reach the threshold
    assert not any((a, b) in hit for a in kept for b in kept if a < b <= a + window)
    # every dropped SNP has a kept SNP before it, within the window, that does
    for i in range(lo, hi):
        if not keep[i - lo]:
            assert any(keep[k - lo] and (k, i) in hit for k in range(max(lo, i - window), i))


def test_prune_of_a_chain():
    # 0-1, 1-2 and 2-3 in LD: 0 is kept, 1 dropped by 0, 2 kept (its only partner before it, 1, is dropped), 3 dropped by 2
    pairs = np.zeros(3, gw.LD_PAIR_DTYPE)
    pairs["i"], pairs["j"], pairs["r2"] = [0, 1, 2], [1, 2, 3], 0.9
    np.testing.assert_array_equal(gw.ld_prune(pairs, 1, 0.8, 0, 4), [True, False, True, False])
    np.testing.assert_array_equal(gw.ld_prune(pairs, 1, 0.95, 0, 4), [True] * 4)
    np.testing.assert_array_equal(gw.ld_prune(pairs[:0], 3, 0.5, 5, 9), [True] * 4)


def test_prune_refuses_malformed_lists():
    pairs = np.zeros(3, gw.LD_PAIR_DTYPE)
    pairs["i"], pairs["j"], pairs["r2"] = [0, 1, 2], [1, 3, 3], 0.5
    gw.ld_prune(pairs, 2, 0.4, 0, 4)
    bad = [pairs[[1, 0, 2]],                                    # unsorted
           np.concatenate([pairs, pairs[-1:]]),                 # duplicate
           pairs.copy(), pairs.copy(), pairs.copy()]
    bad[2]["j"][2] = 4          # j beyond the range
    bad[3]["i"][0], bad[3]["j"][0] = 1, 1   # i == j
    bad[4]["j"][0] = 3          # j - i beyond the window of 2 ... and (0, 3) before (1, 3) is still sorted
    for b in bad:
        with pytest.raises(gw.GwasDevError):
            gw.ld_prune(b, 2, 0.4, 0, 4)
    with pytest.raises(gw.GwasDevError):
        gw.ld_prune(pairs, 2, 0.4, 1, 4)     # i below the range
    with pytest.raises(gw.GwasDevError):
        gw.ld_prune(pairs, 0, 0.4, 0, 4)     # window 0
    with pytest.raises(gw.GwasDevError):
        gw.ld_prune(pairs, 2, 0.4, 4, 0)     # bad range
