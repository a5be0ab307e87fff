"""Windowed LD, the permutation GEMM and the set screens at sizes where every CTA pair runs many tiles.

ld_gemm_kernel<1|3>, perm_gemm_kernel<2|3> and the SETS instantiations of pair_screen_mma_kernel / pair_screen_mma4_kernel<0|1|2>
run on the CTA-pair pipeline of mma_common.cuh: a CTA pair draws tiles from a device counter until the list runs out, and the
operand ring's stage parity, the double-buffered TMEM accumulator with its tfull / tempty phases and the 4-slot schedule ring
carry from one tile to the next. Those paths only run once a pair has computed its third, fifth and ninth tile, so every case
here asserts (tile_guard) that each launch has at least 8 tiles per CTA pair of this device, from the host code's own geometry,
and compares every output element with an exact, independent reference:
  - LD: the contract's integer sums, as exact float64 products per 256-SNP A-block against its window, and its int64 / fp64
    steps (ld_reference's arithmetic); band bits, list records and ld_pairs records bit-equal, NaN included.
  - permutations: the case counts of every (permutation, SNP) per genotype class, as exact float64 products of the permuted
    case masks with one-hot class planes, through gwasdev_marginal_finalize; perm_stats bit-equal to its statistics.
  - set screens: the whole-table screen (tensor cores and AND+POPC, which must agree) filtered to the wanted pairs, record for
    record.
The CPU tests at the end check the two counting references against full-matrix and brute-force restatements.
"""
from fractions import Fraction

import numpy as np
import pytest

import libgwaspp_b200 as gw
from helpers import bits_of, ld_reference, planted_cohort
from test_gpu_ld import assert_band_equal, assert_records_equal, ld_table, to_bed
from test_gpu_pair_sets import formula, in_sets
from test_gpu_permutation import check_reductions, make_store, perm_df, pheno_of
from test_gpu_screen_edges import LOW, store_of, top_k_of

gpu = pytest.mark.gpu


# ---- regime guard -----------------------------------------------------------------------------------------------------------
LD_A = 256                      # A-SNPs per LD tile
PERM_BLK, PSNP_BLK, PERM_BATCH = 256, 64, 16384


def cta_pairs():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count // 2


def tile_guard(tiles, what, per_pair=8):
    """every launch in `tiles` hands each CTA pair of this device at least `per_pair` tiles"""
    pairs = cta_pairs()
    print(f"{what}: tiles per launch {list(tiles)}, {pairs} CTA pairs")
    assert min(tiles) >= per_pair * pairs, (what, list(tiles), pairs)


def row_words(n_samples):
    """32-bit words per raw plane on the device (gwasdev_create: Wr = round_up(P / 2, 4))"""
    return -(-(gw.plane_blocks(n_samples) // 2) // 4) * 4


def ld_launch_tiles(n_snps, lo, hi, window, rows_per_snp, snp_bytes=0, budget=0):
    """tiles of each ld_gemm_kernel launch of gwasdev_ld_window over [lo, hi) (launch_ld / ld_window_body): one launch over
    the resident operand (budget 0), else one per chunk of whole A-blocks"""
    NB = 256 if rows_per_snp == 1 else 32
    w_eff = min(window, hi - lo)

    def tiles(a0, a_end, op0, op_snps):
        I0 = (a0 - op0) // LD_A
        nI = (a_end - 1 - op0) // LD_A - I0 + 1
        nb = -(-min(op_snps, hi - op0) // NB)
        return nI * min((LD_A - 1 + w_eff) // NB + 1, nb)
    if not budget:
        return [tiles(lo // LD_A * LD_A, hi, 0, n_snps)]
    fit = budget // snp_bytes
    chunk = max(LD_A, (fit - w_eff) // LD_A * LD_A if fit > w_eff + LD_A else LD_A)
    return [tiles(a0, min(a0 + chunk, hi), a0, min(min(a0 + chunk, hi) + w_eff, hi) - a0) for a0 in range(lo, hi, chunk)]


def perm_launch_tiles(n_snps, n_perm, snp_bytes=0, budget=0):
    """tiles of each perm_gemm_kernel launch of gwasdev_marginal_permute (permute_body): ceil(P / 256) x ceil(M / 64) per
    SNP chunk and permutation batch"""
    chunk = max(PSNP_BLK, budget // snp_bytes // PSNP_BLK * PSNP_BLK) if budget else n_snps
    out = []
    for c0 in range(0, n_snps, chunk):
        for b0 in range(0, n_perm, PERM_BATCH):
            nb = min(PERM_BATCH, n_perm - b0)
            out.append(-(-nb // PERM_BLK) * -(-min(chunk, n_snps - c0) // PSNP_BLK))
    return out


# ---- exact integer products -------------------------------------------------------------------------------------------------
def _device():
    import torch
    return torch.cuda.is_available()


def f64(a):
    """a as float64 operand of exact_mm: a torch tensor on the device when there is one, else a numpy array"""
    if _device():
        import torch
        return torch.from_numpy(np.ascontiguousarray(a)).cuda().double()
    return np.asarray(a, np.float64)


def exact_mm(a, b):
    """a @ b.T of integer-valued float64 operands, as int64. Exact while every partial sum stays below 2^53, in any summation
    order: cuBLAS DGEMM on the device (no reduced-precision mode applies to float64), numpy on the host."""
    if not isinstance(a, np.ndarray):
        a = (a @ b.T).cpu().numpy()
    else:
        a = a @ b.T
    return np.rint(a).astype(np.int64)


# ---- LD reference -----------------------------------------------------------------------------------------------------------
def decode(s, chunk_bytes=1 << 25):
    """(x int8, called bool), (M, N) under the store's own labels (aa 0, ab 1, bb 2; x = 0 where not called): test_gpu_ld's
    decoded, in row chunks and without its int64 arrays"""
    M, N, P = s.n_snps, s.n_samples, s.P
    x, c = np.empty((M, N), np.int8), np.empty((M, N), bool)
    step = max(1, chunk_bytes // (16 * P))
    for r0 in range(0, M, step):
        rows = s.get_rows(r0, min(step, M - r0))
        p1, p2 = bits_of(rows[:, 1:1 + P], N), bits_of(rows[:, 1 + P:], N)
        x[r0:r0 + len(rows)] = (p2 & ~p1).astype(np.int8) + 2 * (p1 & p2).astype(np.int8)
        c[r0:r0 + len(rows)] = p1 | p2
    return x, c


class LdBand:
    """The contract's (n, r, r2) of the band pairs of one block of A-SNPs: the six integer sums as exact float64 products of
    the rows X (allele count where called), C (called) and Q = X^2, then ld_reference's int64 and fp64 steps."""

    def __init__(self, x, c):
        X = np.where(c, x, 0).astype(np.int8)
        self.X, self.C, self.Q = f64(X), f64(c.astype(np.int8)), f64(X * X)

    def block(self, a0, a1, hi, window):
        """pairs (i, j = i + d + 1), a0 <= i < a1, 0 <= d < window, j < hi as (a1 - a0, window) arrays n, r, r2 (n 0 and
        NaN outside the band), the valid mask and the sums of the valid pairs"""
        b0, b1 = a0 + 1, min(hi, a1 + window)
        na = a1 - a0
        I = np.arange(a0, a1)[:, None]
        J = I + np.arange(window)[None, :] + 1
        valid = J < hi
        n_out = np.zeros((na, window), np.int64)
        r_out, r2_out = np.full((na, window), np.nan), np.full((na, window), np.nan)
        sums = {}
        if b1 <= b0:
            return n_out, r_out, r2_out, valid, sums
        Xa, Ca, Qa, Xb, Cb, Qb = self.X[a0:a1], self.C[a0:a1], self.Q[a0:a1], self.X[b0:b1], self.C[b0:b1], self.Q[b0:b1]
        n, sx, sy, sxx, syy, sxy = (exact_mm(Ca, Cb), exact_mm(Xa, Cb), exact_mm(Ca, Xb), exact_mm(Qa, Cb), exact_mm(Ca, Qb),
                                    exact_mm(Xa, Xb))
        num, vx, vy = n * sxy - sx * sy, n * sxx - sx * sx, n * syy - sy * sy
        with np.errstate(invalid="ignore", divide="ignore"):
            v = vx.astype(np.float64) * vy.astype(np.float64)
            r2 = (num.astype(np.float64) * num.astype(np.float64)) / v
            r = num.astype(np.float64) / np.sqrt(v)
        undef = (vx == 0) | (vy == 0)
        r2[undef] = np.nan
        r[undef] = np.nan
        col = np.where(valid, J - b0, 0)
        pick = lambda m: np.take_along_axis(m, col, axis=1)[valid]
        n_out[valid], r_out[valid], r2_out[valid] = pick(n), pick(r), pick(r2)
        sums = {"n": pick(n), "sxx": pick(sxx), "sxy": pick(sxy)}
        return n_out, r_out, r2_out, valid, sums


def band_reference(x, c, lo, hi, window, blk=LD_A):
    """(n, r, r2) of every band pair of [lo, hi) as (hi - lo, window) arrays, block by block (the CPU tests' entry point)"""
    ref = LdBand(x, c)
    parts = [ref.block(a0, min(a0 + blk, hi), hi, window)[:3] for a0 in range(lo, hi, blk)]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def records(i, j, n, r, r2):
    out = np.zeros(len(i), gw.LD_PAIR_DTYPE)
    out["i"], out["j"], out["n"], out["r"], out["r2"] = i, j, n, r, r2
    return out


def check_ld(s, ref, lo, hi, window, rows_per_snp, n_kept=300_000, n_probe=100_000, seed=0, keep=None):
    """gwasdev_ld_window over [lo, hi) (band, and the list at a threshold that keeps about n_kept pairs) and gwasdev_ld_pairs
    on n_probe random band pairs against the block reference, block by block. Returns the outputs for later comparisons."""
    _, band, st = s.ld_window(window, 0.0, lo, hi, band=True, pairs=False)
    w1 = min(window, hi - lo - 1)
    n_band = (hi - lo - w1) * w1 + w1 * (w1 - 1) // 2
    assert st.pairs_tested == n_band and st.rows_per_snp == rows_per_snp
    vals = band[~np.isnan(band)]
    thr = 0.0 if len(vals) <= n_kept else float(np.partition(vals, len(vals) - n_kept)[len(vals) - n_kept])
    pairs, _, st = s.ld_window(window, thr, lo, hi)
    assert st.pairs_tested == n_band and st.pairs_kept == len(pairs) and st.rows_per_snp == rows_per_snp
    # random band pairs, either order
    rng = np.random.default_rng(seed)
    n_probe = min(n_probe, n_band)
    pi = rng.integers(lo, hi - 1, n_probe)
    pj = pi + 1 + (rng.random(n_probe) * np.minimum(window, hi - 1 - pi)).astype(np.int64)
    flip = rng.random(n_probe) < 0.5
    got_probe = s.ld_pairs(np.where(flip, pj, pi), np.where(flip, pi, pj))
    want_probe = records(pi, pj, 0, np.nan, np.nan)
    want_list = []
    for a0 in range(lo, hi, LD_A):
        a1 = min(a0 + LD_A, hi)
        n, r, r2, valid, _ = ref.block(a0, a1, hi, window)
        assert_band_equal(band[a0 - lo:a1 - lo], np.where(valid, r2, np.nan).astype(np.float32))
        with np.errstate(invalid="ignore"):
            I, D = np.nonzero(valid & (r2 >= thr))
        want_list.append(records(a0 + I, a0 + I + D + 1, n[I, D], r[I, D], r2[I, D]))
        k = (pi >= a0) & (pi < a1)
        d = pj[k] - pi[k] - 1
        want_probe["n"][k], want_probe["r"][k], want_probe["r2"][k] = n[pi[k] - a0, d], r[pi[k] - a0, d], r2[pi[k] - a0, d]
    want_list = np.concatenate(want_list)
    if len(vals) > n_kept:
        assert n_kept // 3 <= len(want_list) <= 3 * n_kept, len(want_list)
    assert_records_equal(pairs, want_list)
    assert_records_equal(got_probe, want_probe)
    return band, pairs, thr


# ---- 1. windowed LD at scale ------------------------------------------------------------------------------------------------
def load_ld(G):
    s = gw.GenoStore(*G.shape)
    s.put_bed(to_bed(G))
    return s


@gpu
def test_ld_one_row_per_snp_at_scale():
    """complete data (ld_gemm_kernel<1>, 256 x 256 tiles): 12 000 SNPs x 3 001 samples (padding bits in the last word),
    window 4 000, whole and an unaligned sub-range"""
    M, N, W = 12_000, 3001, 4000
    G = ld_table(M, N, seed=1201)
    G[G < 0] = 0
    with load_ld(G) as s:
        x, c = decode(s)
        assert c.all()
        ref = LdBand(x, c)
        for lo, hi in ((0, M), (37, M - 51)):
            tile_guard(ld_launch_tiles(M, lo, hi, W, 1), f"ld<1> [{lo}, {hi}) window {W}")
            check_ld(s, ref, lo, hi, W, 1, seed=lo)


@gpu
def test_ld_three_rows_per_snp_at_scale():
    """2 % missing calls plus ld_table's duplicates, relabelled copies, monomorphic, all-missing and half-called rows
    (ld_gemm_kernel<3>, 256 x 32 tiles): 6 000 SNPs x 3 001 samples, window 1 000"""
    M, N, W = 6000, 3001, 1000
    with load_ld(ld_table(M, N, seed=603, missing=0.02)) as s:
        x, c = decode(s)
        tile_guard(ld_launch_tiles(M, 0, M, W, 3), f"ld<3> window {W}")
        _, pairs, _ = check_ld(s, LdBand(x, c), 0, M, W, 3)
        assert (pairs["r2"] == 1.0).any() and (pairs["r"] == -1.0).any()      # duplicates and relabelled copies are in the list


@gpu
def test_ld_chunked_operand_at_scale():
    """three rows per SNP, 12 000 SNPs, window 1 000, with GWASDEV_OPT_LD_OPERAND_BYTES at 3 chunks of at least 600 tiles each:
    the same band and list as the resident operand, which equal the reference"""
    M, N, W = 12_000, 3001, 1000
    with load_ld(ld_table(M, N, seed=1207, missing=0.02)) as s:
        x, c = decode(s)
        tile_guard(ld_launch_tiles(M, 0, M, W, 3), f"ld<3> resident window {W}")
        band, pairs, thr = check_ld(s, LdBand(x, c), 0, M, W, 3)
        snp_bytes = 3 * 32 * row_words(N)
        budget = (4096 + W + 128) * snp_bytes                 # chunks of 4 096 A-SNPs plus their window
        chunks = ld_launch_tiles(M, 0, M, W, 3, snp_bytes, budget)
        assert len(chunks) >= 3
        tile_guard(chunks, f"ld<3> chunked window {W}")
        s.set_option(gw.OPT_LD_OPERAND_BYTES, budget)
        p1, b1, st = s.ld_window(W, thr, band=True)
        assert st.built_operand == 1 and st.rows_per_snp == 3
        assert_band_equal(b1, band)
        assert_records_equal(p1, pairs)
        s.set_option(gw.OPT_LD_OPERAND_BYTES, 0)


def deep_table(M, N, seed):
    """(M, N) genotypes in {0, 1, 2, -1 missing} without ld_table's (N, M) int64 mosaic: independent rows at allele
    frequencies from 0.02 to 0.995, exact, noisy (a growing share of samples redrawn) and homozygote-relabelled copies, so that
    r^2 spans 0 to 1, 2 % missing calls, and all-missing, monomorphic and half-called rows"""
    rng = np.random.default_rng(seed)
    G = np.empty((M, N), np.int8)
    for m in range(M):
        p = 0.995 if m % 40 == 0 else rng.uniform(0.02, 0.98)
        kind = m % 5
        if kind == 1:
            G[m] = G[m - 1]                                   # exact copy
        elif kind == 2:
            redraw = rng.random(N) < (m % 97) / 97
            G[m] = np.where(redraw, (rng.random(N) < p).astype(np.int8) + (rng.random(N) < p), G[m - 2])   # noisy copy
        elif kind == 3:
            G[m] = 2 - G[m - 3]                               # relabelled copy: r = -1
        else:
            G[m] = (rng.random(N) < p).astype(np.int8) + (rng.random(N) < p)
    for m in range(M):
        if m % 40 >= 2:                                       # rows 40k, 40k + 1 (mostly bb, and its copy) stay fully called: Sxy near 4 N
            G[m, rng.random(N) < 0.02] = -1
        else:
            G[m, 0] = 0                                       # first homozygote aa, so the store's first-seen labels keep x = G
    G[7] = -1                                                 # all missing
    G[13] = np.where(G[13] < 0, -1, 0)                        # monomorphic
    G[19] = np.where(G[19] < 0, -1, 2)
    G[29, rng.random(N) < 0.5] = -1                           # half called
    return G


@gpu
def test_ld_deep_sample_dimension():
    """1 000 003 samples x 320 SNPs, three rows per SNP, full window: Sxy approaches 4e6 and n Sxx 4e12 (the sample dimension;
    20 tiles, so exempt from the tile guard)"""
    M, N = 320, 1_000_003
    G = deep_table(M, N, seed=77)
    with gw.GenoStore(M, N) as s:
        for r0 in range(0, M, 32):
            s.put_bed(to_bed(G[r0:r0 + 32]), first_row=r0)
        del G
        x, c = decode(s)
        ref = LdBand(x, c)
        del x, c
        check_ld(s, ref, 0, M, M - 1, 3, n_probe=M * (M - 1) // 2)
        sums = [ref.block(a0, min(a0 + LD_A, M), M, M - 1)[4] for a0 in range(0, M, LD_A)]
        sxy = max(int(b["sxy"].max()) for b in sums)
        nsxx = max(int((b["n"] * b["sxx"]).max()) for b in sums)
        print(f"deep K: max Sxy {sxy}, max n Sxx {nsxx}")
        assert sxy > 3.9e6 and nsxx > 3.9e12


# ---- 2. permutation GEMM at scale -------------------------------------------------------------------------------------------
class PermCounts:
    """Case and control counts per genotype class (aa, ab, bb, xx) of every (permutation, SNP): exact float64 products of the
    permuted case masks with one-hot class planes of the selected samples; controls are the selected class totals minus the
    cases. p1, p2: (M, N) bool raw planes (aa p1 only, ab p2 only, bb both, xx neither); sel: (N,) bool selection."""

    def __init__(self, p1, p2, sel):
        planes = [p1 & ~p2 & sel, p2 & ~p1 & sel, p1 & p2 & sel, ~(p1 | p2) & sel]
        self.totals = np.stack([g.sum(1) for g in planes], -1).astype(np.int64)            # (M, 4)
        self.planes = [f64(g.astype(np.int8)) for g in planes]

    def counts(self, case):
        """case: (n_perm, N) bool masks -> (n_perm, M, 8) uint32 counts in gwasdev_marginal_finalize's layout"""
        A = f64(case.astype(np.int8))
        cases = np.stack([exact_mm(A, g) for g in self.planes], -1)
        return np.concatenate([cases, self.totals[None] - cases], -1).astype(np.uint32)


def planes_of(s):
    N, P = s.n_samples, s.P
    rows = s.get_rows()
    return bits_of(rows[:, 1:1 + P], N), bits_of(rows[:, 1 + P:], N)


def check_perm_stats(s, out, masks, sel_ca, sel_co, orc, seed, slab=128):
    """every element of perm_stats bit-equal to finalize's statistics of the reference counts; a sample against the oracle"""
    N = s.n_samples
    p1, p2 = planes_of(s)
    ref = PermCounts(p1, p2, bits_of(sel_ca | sel_co, N))
    case = bits_of(masks, N)
    ps = out["perm_stats"]
    assert ps.shape == (len(masks), s.n_snps, 2)
    rng = np.random.default_rng(seed)
    spots = 0
    for q0 in range(0, len(masks), slab):
        cnt = ref.counts(case[q0:q0 + slab])
        _, st = gw.marginal_finalize(cnt.reshape(-1, 8))
        for k, key in enumerate(("chi2_allelic", "chi2_genotypic")):
            want = st[key].reshape(cnt.shape[:2])
            np.testing.assert_array_equal(ps[q0:q0 + slab, :, k].view(np.uint64), want.view(np.uint64), err_msg=f"{key} {q0}")
        for _ in range(4):
            q, m = int(rng.integers(len(cnt))), int(rng.integers(s.n_snps))
            xa, _ = orc.chi2_allelic(cnt[q, m, :4], cnt[q, m, 4:])
            xg, _, _ = orc.chi2_genotypic(cnt[q, m, :4], cnt[q, m, 4:])
            for got, w in ((ps[q0 + q, m, 0], xa), (ps[q0 + q, m, 1], xg)):
                assert (np.isnan(got) and np.isnan(w)) or abs(got - w) <= 1e-12 * max(1.0, abs(w)), (q0 + q, m, got, w)
            spots += 1
    assert spots >= 40


@gpu
@pytest.mark.parametrize("missing", [0.01, 0.0], ids=["three_planes", "two_planes"])
def test_permutation_gemm_every_element(orc, missing):
    """6 000 SNPs x 3 001 samples (10 % in neither class), 2 560 device-drawn permutations: every element of perm_stats, the
    reductions, and -- on the three-plane table -- a chunked B operand and 2 048 caller masks with different case counts"""
    M, N, P = 6000, 3001, 2560
    pheno = pheno_of(N, 601, neither=0.1)
    s = make_store(M, N, 602, missing, pheno)
    try:
        ca, co = gw.stream_masks(pheno)
        obs = s.marginal_scan(counts=False, mi=False)["stats"]
        PL = 3 if missing else 2
        tile_guard(perm_launch_tiles(M, P), f"perm<{PL}> {P} permutations")
        out = s.marginal_permute(P, seed=11, perm_stats=True)
        assert out["stats"].planes == PL and out["stats"].n_perm == P
        masks = gw.permutation_masks(N, ca, co, 11, 0, P)
        check_perm_stats(s, out, masks, ca, co, orc, seed=PL)
        check_reductions(out, obs, perm_df(s, masks, ca, co))
        if not missing:
            return
        # chunked B operand: chunks of 2 048 SNPs, each its own launch (at least 4 tiles per CTA pair there)
        snp_bytes = PL * 32 * row_words(N)
        budget = 2048 * snp_bytes + snp_bytes
        chunks = perm_launch_tiles(M, P, snp_bytes, budget)
        assert len(chunks) >= 3
        tile_guard(chunks, f"perm<{PL}> chunked", per_pair=4)
        s.set_option(gw.OPT_PERM_OPERAND_BYTES, budget)
        chunked = s.marginal_permute(P, seed=11, perm_stats=True)
        s.set_option(gw.OPT_PERM_OPERAND_BYTES, 0)
        assert chunked["stats"].built_operand == 1
        for key in ("exceed", "perm_max", "perm_stats"):
            np.testing.assert_array_equal(chunked[key].view(np.uint8), out[key].view(np.uint8), err_msg=key)
        del chunked
        # caller masks, case fractions from 2 % to 98 % of the selection
        Q = 2048
        tile_guard(perm_launch_tiles(M, Q), f"perm<{PL}> {Q} caller masks")
        rng = np.random.default_rng(5)
        sel = bits_of(ca | co, 16 * s.P)
        frac = np.linspace(0.02, 0.98, Q)
        bits = sel[None] & (rng.random((Q, sel.size)) < frac[:, None])
        cmasks = np.packbits(bits, axis=1, bitorder="little").view(np.uint16)
        ncase = bits.sum(1)
        assert ncase.min() > 0 and (sel.sum() - ncase).min() > 0 and len(np.unique(ncase)) > Q // 2
        multi = s.marginal_permute(Q, case_masks=cmasks, perm_stats=True)
        check_perm_stats(s, multi, cmasks, ca, co, orc, seed=9)
        check_reductions(multi, obs, perm_df(s, cmasks, ca, co))
    finally:
        s.close()


# ---- 3. set screens on the four-plane kernel at scale -----------------------------------------------------------------------
def set_shapes(M, seed):
    """within A (|A| 2 400), set-by-all (|A| 1 000) and set-by-set (1 600 x 1 600 sharing 300)"""
    rng = np.random.default_rng(seed)
    pool = rng.permutation(M)
    c = pool[:300]
    a = np.sort(np.concatenate([c, pool[300:1600]])).astype(np.uint32)
    b = np.sort(np.concatenate([c, pool[1600:2900]])).astype(np.uint32)
    return {"within": (np.sort(rng.choice(M, 2400, replace=False)).astype(np.uint32), None),
            "by_all": (np.sort(rng.choice(M, 1000, replace=False)).astype(np.uint32), np.arange(M, dtype=np.uint32)),
            "by_set": (a, b)}


def sub_table(a, b):
    """rows of the gathered sub-table: A n B, then A \\ B, then B \\ A"""
    if b is None:
        return a
    return np.concatenate([np.intersect1d(a, b), np.setdiff1d(a, b), np.setdiff1d(b, a)])


# (M, N, cases, missing rate, kernels): missing calls in half the row runs of the mixed cohort only
SET_COHORTS = {
    "mixed_tiles": (3000, 2000, 900, 0.01),
    "split_classes": (3000, 40000, 20000, 0.0),
    "two_accumulators": (3000, 40000, 20000, 0.003),
}


def assert_hits_equal(got, want, what):
    assert len(got) == len(want), (what, len(got), len(want))
    assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), what       # bits of (i, j, stat)


@gpu
@pytest.mark.parametrize("cohort", list(SET_COHORTS))
def test_set_screens_at_scale(orc, cohort):
    M, N, n_case, miss = SET_COHORTS[cohort]
    codes, pheno = planted_cohort(orc, 9000 + N, M, N, n_case, miss, 12)
    if cohort == "mixed_tiles":
        clean = (np.arange(M) // 320) % 2 == 1                 # runs of 320 rows with and without missing calls
        cc = codes[clean]
        cc[cc == 3] = 0
        codes[clean] = cc
    sel = (pheno == 0) | (pheno == 1)
    row_missing = ((codes == 3) & sel[None]).any(1)
    assert row_missing.any() == (miss > 0)
    rows = orc.pack_codes(codes)
    del codes
    with store_of(rows, N) as st:
        st.select_case_control(pheno)
        assert (st.n_case >= 16384) == (cohort != "mixed_tiles")
        full = {}
        for thr in (30.0, LOW):
            h2, s2 = st.pairwise_scan(thr, capacity=M * M)
            st.set_pair_engine(1)
            h1, s1 = st.pairwise_scan(thr, capacity=M * M)
            st.set_pair_engine(0)
            assert s2.engine == 2 and s1.engine == 1
            assert_hits_equal(h2, h1, f"engines at {thr}")
            full[thr] = h2
        assert len(full[30.0]) >= 3 and len(full[LOW]) > M * (M - 1) // 4
        n_hi = 0
        for name, (a, b) in set_shapes(M, 17).items():
            t64, _ = gw.set_schedule(M, a, b, tile_snps=64, n_samples=N)
            t128, _ = gw.set_schedule(M, a, b, tile_snps=128, n_samples=N)
            tile_guard([len(t64)], f"{cohort} {name}: four-plane set tiles")
            sub_missing = row_missing[sub_table(a, b)]                # 64-SNP blocks of the sub-table with missing calls
            nb = -(-len(sub_missing) // 64)
            flags = np.concatenate([sub_missing, np.zeros(64 * nb - len(sub_missing), bool)]).reshape(nb, 64).any(1)
            nine = int((flags[t64[:, 0]] | flags[t64[:, 1]]).sum())
            for thr in (LOW, 30.0):
                want = in_sets(full[thr], a, b)
                h, s = st.pairwise_scan_sets(a, b, thr, capacity=max(1, len(want)))
                assert_hits_equal(h, want, f"{name} at {thr}")
                assert s.pairs_tested == formula(a, b) and s.engine == 2
                if cohort == "mixed_tiles":     # two-plane kernel on the 128-SNP list, pair_screen_mma4_kernel<0> on the tiles with missing calls
                    assert (s.tiles, s.tiles_nine_cell) == (len(t128), nine) and 0 < nine < len(t64), (s.tiles, s.tiles_nine_cell, nine)
                elif cohort == "split_classes":  # pair_screen_mma4_kernel<1> on every 64-SNP tile
                    assert (s.tiles, s.tiles_nine_cell) == (len(t64), 0)
                else:                            # pair_screen_mma4_kernel<2> on every tile
                    assert (s.tiles, s.tiles_nine_cell) == (len(t64), nine) and nine > 0
            n_hi += len(in_sets(full[30.0], a, b))
            ref_lo = in_sets(full[LOW], a, b)
            for k in (1, 1000):
                top, _ = st.pairwise_scan_sets(a, b, LOW, top_k=k)
                assert_hits_equal(top, top_k_of(ref_lo, k), f"{name} top {k}")
            parts = [st.pairwise_scan_sets(a, b, LOW, shard=r, n_shards=3, capacity=len(ref_lo)) for r in range(3)]
            merged = np.sort(np.concatenate([p[0] for p in parts]), order=["i", "j"])
            assert_hits_equal(merged, ref_lo, f"{name} shards")
            assert sum(p[1].pairs_tested for p in parts) == formula(a, b)
        assert n_hi > 0


# ---- 4. the references on tiny tables (CPU) ---------------------------------------------------------------------------------
@pytest.mark.parametrize("N, missing", [(127, 0.0), (127, 0.02), (501, 0.02)])
def test_band_reference_equals_the_full_matrix_reference(N, missing):
    M = 700
    G = ld_table(M, N, seed=N + int(100 * missing), missing=missing)
    if not missing:
        G[G < 0] = 0
    x = np.where(G < 0, 0, G).astype(np.int8)
    c = G >= 0
    n, r, r2 = ld_reference(x.astype(np.int64), c)
    num_checked = 0
    for lo, hi, w, blk in ((0, M, 63, 256), (0, M, 300, 256), (37, M - 51, 257, 256), (5, 400, M + 40, 64), (255, 258, 3, 256)):
        bn, br, br2 = band_reference(x, c, lo, hi, w, blk)
        I = np.arange(lo, hi)[:, None]
        J = I + np.arange(w)[None, :] + 1
        valid = J < hi
        Jc = np.where(valid, J, 0)
        np.testing.assert_array_equal(bn, np.where(valid, n[I, Jc], 0))
        for got, full in ((br, r), (br2, r2)):
            want = np.where(valid, full[I, Jc], np.nan)
            np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))
        num_checked += int(valid.sum())
    assert num_checked > 100_000
    # r2 within 1 ulp of the exact rational num^2 / (vx vy)
    X, C = np.where(c, x, 0).astype(np.int64), c.astype(np.int64)
    rng = np.random.default_rng(N)
    ok = np.flatnonzero(~np.isnan(r2[np.triu_indices(M, 1)]))
    iu = np.triu_indices(M, 1)
    for k in rng.choice(ok, 400, replace=False):
        i, j = int(iu[0][k]), int(iu[1][k])
        both = (C[i] & C[j]).astype(bool)
        xi, xj = X[i][both], X[j][both]
        nn, sx, sy = int(both.sum()), int(xi.sum()), int(xj.sum())
        num = nn * int((xi * xj).sum()) - sx * sy
        vx, vy = nn * int((xi * xi).sum()) - sx * sx, nn * int((xj * xj).sum()) - sy * sy
        exact = float(Fraction(num * num, vx * vy))
        assert abs(r2[i, j] - exact) <= np.spacing(exact), (i, j, r2[i, j], exact)


def test_permutation_counts_equal_a_brute_force_loop():
    rng = np.random.default_rng(3)
    M, N, Q = 37, 83, 9
    code = rng.integers(0, 4, (M, N))                           # 0 xx, 1 aa, 2 ab, 3 bb
    code[5] = 1                                                 # monomorphic
    code[9] = 0                                                 # all missing
    p1, p2 = (code == 1) | (code == 3), (code == 2) | (code == 3)
    sel = rng.random(N) < 0.85
    case = (rng.random((Q, N)) < rng.uniform(0.1, 0.9, (Q, 1))) & sel
    got = PermCounts(p1, p2, sel).counts(case)
    want = np.zeros((Q, M, 8), np.uint32)
    cls = {1: 0, 2: 1, 3: 2, 0: 3}                              # aa, ab, bb, xx
    for q in range(Q):
        for m in range(M):
            for k in range(N):
                if sel[k]:
                    want[q, m, cls[int(code[m, k])] + (0 if case[q, k] else 4)] += 1
    np.testing.assert_array_equal(got, want)


def test_tile_geometry():
    """the launch geometry the guards use, at the sizes above (host arithmetic)"""
    assert ld_launch_tiles(12_000, 0, 12_000, 4000, 1) == [47 * 17]
    assert ld_launch_tiles(12_000, 37, 11_949, 4000, 1) == [47 * 17]
    assert ld_launch_tiles(6000, 0, 6000, 1000, 3) == [24 * 40]
    assert ld_launch_tiles(320, 0, 320, 319, 3) == [2 * 10]
    sb = 3 * 32 * row_words(3001)
    assert ld_launch_tiles(12_000, 0, 12_000, 1000, 3, sb, (4096 + 1000 + 128) * sb) == [16 * 40, 16 * 40, 15 * 40]
    assert perm_launch_tiles(6000, 2560) == [10 * 94]
    assert perm_launch_tiles(6000, 16384 + 300) == [64 * 94, 2 * 94]
    sb = 3 * 32 * row_words(3001)
    assert perm_launch_tiles(6000, 2560, sb, 2049 * sb) == [10 * 32, 10 * 32, 10 * 30]
