"""GPU tests: everything the resident store caches follows the rows, selection, stream masks and options it was built from.

A store is built once and reused, and more than a dozen derived objects (compacted rows, margins, pair-screen operands, row
totals, permutation planes, the LD operand, ...) are built lazily by the first call that needs them and kept until some call
marks them stale (DESIGN.md section 4 has the table). A stale object fails silently: the kernels are right and the numbers are
plausible, but they come from the old rows or the old selection. So the reference here is a FRESH store, built from scratch
from a host-side shadow of what the reused store should hold (rows, selection, stream masks, options, engine, select mode):
after every step both must give the same bytes on every observer. The fresh store's results are what the rest of the suite
checks against the oracle; each walk also ends with its final state checked against the oracle and the exact integer LD
reference directly.

Two ways of driving it: a scripted matrix with one named case per (cache, mutator) pair, which also checks the
built_operand flags where the contract promises reuse, and seeded random walks over three cohorts. A walk's steps come from
a fixed seed, so a failure names its step and the walk can be replayed on the host.
"""
import ctypes as C
import os

import numpy as np
import pytest

import libgwaspp_b200 as gw
from helpers import band_of, decoded, ld_reference, list_of, planted_cohort

pytestmark = pytest.mark.gpu

EINVAL = 1
THR = 10.0                 # pair-screen threshold: the planted pairs and a few hundred candidates above it
LD_WINDOW, LD_THR = 40, 0.05
N_PERM = 64
# (SNPs, samples, missing-call rate): small tables, so that a fresh store costs milliseconds
COHORTS = {"a": (640, 2003, 0.0), "b": (640, 2003, 0.01), "c": (320, 17000, 0.01)}
WRITE_FIRSTS = (63, 191, 319, 447)    # three rows in the middle of a 128-SNP block, across its 64-SNP edge
# fixed pairs across the 64- and 128-SNP block edges, and through the rows the writes replace
EDGE_PAIRS = [(63, 64), (127, 128), (63, 128), (0, 255), (64, 191), (190, 192), (191, 256), (192, 193), (255, 256),
              (127, 319), (300, 319), (318, 319), (320, 321), (383, 384), (447, 449), (511, 512), (5, 639)]
LONG = ("scan", "scan_sub", "compact", "counts", "selected_rows", "pair_tables", "pair_stats", "tile", "screen", "shards",
        "sets", "perm", "ld_all", "ld_mask", "ld_ones", "ld_pairs")


# ------------------------------------------------------------------------------------------------------
# cohorts and encoders (codes: 0 AA, 1 AC, 2 CC, 3 missing)
# ------------------------------------------------------------------------------------------------------
_COHORT = {}


def cohort(orc, name):
    if name not in _COHORT:
        M, N, missing = COHORTS[name]
        codes, pheno = planted_cohort(orc, 7001 + ord(name), M, N, N // 2, missing, 4)
        _COHORT[name] = (codes, orc.pack_codes(codes), pheno)
    return _COHORT[name]


def bed_of(codes):
    q = np.array([0, 2, 3, 1], np.uint8)[codes]          # .bed: 0 hom A1, 1 missing, 2 het, 3 hom A2
    M, N = codes.shape
    pad = np.zeros((M, (N + 3) // 4 * 4), np.uint8)
    pad[:, :N] = q
    p = pad.reshape(M, -1, 4)
    return (p[..., 0] | (p[..., 1] << 2) | (p[..., 2] << 4) | (p[..., 3] << 6)).astype(np.uint8)


def tped_of(codes, first):
    spell = np.array([b"A A", b"A C", b"C C", b"0 0"])
    return b"".join(b"1 rs%d 0 %d " % (first + r, first + r) + b" ".join(spell[codes[r]]) + b"\n" for r in range(len(codes)))


def masks_of(pheno, rng=None, n_both=0):
    """class masks of pheno (1 case, 0 control, else neither) with n_both samples flagged in both; the effective labels"""
    ca, co = gw.stream_masks(pheno)
    eff = pheno.copy()
    if n_both:
        for c in rng.choice(len(pheno), n_both, replace=False):
            ca[c >> 4] |= np.uint16(1 << (c & 15))
            co[c >> 4] |= np.uint16(1 << (c & 15))
            eff[c] = 1
    return ca, co, eff


def n_gpus():
    return int(gw.load_library().gwasdev_device_count())


# ------------------------------------------------------------------------------------------------------
# observers: fixed inputs, one result per key; an error is its status
# ------------------------------------------------------------------------------------------------------
class Err(tuple):
    pass


def status_of(e):
    return int(str(e).split("status ")[1].split(":")[0])


def selected_rows(st):
    a, b = C.c_uint32(), C.c_uint32()
    gw._check(st.L.gwasdev_case_control_counts(st.h, C.byref(a), C.byref(b)), "gwasdev_case_control_counts")
    st.n_case, st.n_ctrl = a.value, b.value
    return st.get_selected_rows()


def screen_fields(ps):
    """what the pair screen reports and its cached pair / tile counts decide (timings and candidate counts left out)"""
    return np.array([ps.pairs_tested, ps.hits, ps.tiles, ps.tiles_nine_cell, ps.engine], np.uint64)


def observers(w, st, info):
    """name -> {key: thunk}; info receives the live store's built_operand / planes / rows_per_snp per observer"""
    pi, pj = w.pairs

    def perm():
        o = st.marginal_permute(N_PERM, seed=11, perm_stats=True)
        info["perm"] = (o["stats"].built_operand, o["stats"].planes)
        return o["exceed"], o["perm_max"], o["perm_stats"], np.uint32(o["stats"].planes)

    def ld(name, mask):
        def run():
            pairs, band, st_ = st.ld_window(LD_WINDOW, LD_THR, sample_mask=mask, band=True)
            info[name] = (st_.built_operand, st_.rows_per_snp)
            return pairs, band, np.uint32(st_.rows_per_snp)
        return run

    def shards():
        parts = [st.pairwise_scan(THR, shard=k, n_shards=3) for k in range(3)]
        return np.sort(np.concatenate([p[0] for p in parts]), order=["i", "j"]), tuple(screen_fields(p[1]) for p in parts)

    def screen():
        h, ps = st.pairwise_scan(THR)
        return h, screen_fields(ps)

    def sets(b):
        def run():
            h, ps = st.pairwise_scan_sets(w.set_a, None if b is None else b, THR)
            return h, np.uint64(ps.pairs_tested)
        return run

    return {
        "scan": {"full": lambda: tuple(st.marginal_scan().values())},
        "scan_sub": {"sub": lambda: tuple(st.marginal_scan(100, 300).values())},
        "compact": {"compact": lambda: st.marginal_scan_compact(p_threshold=1e-3)},
        "counts": {f"mode{m}": (lambda m=m: st.counts(m)) for m in (0, 1, 2)},
        "selected_rows": {"rows": lambda: selected_rows(st)},
        "pair_tables": {f"mode{m}": (lambda m=m: st.pair_tables(pi, pj, m)) for m in range(4)},
        "pair_stats": {"ksa": lambda: st.ksa(pi, pj), "ksa_mma": lambda: st.ksa_screen_mma_f32(pi, pj),
                       "gtest": lambda: st.gtest(pi, pj), "epi1": lambda: st.epi_pairs(pi, pj, 1)},
        "tile": {"tile": lambda: st.mma_tile_counts(1, 1)},
        "screen": {"scan": screen, "topk": lambda: st.pairwise_topk(50, 0.0)[0]},
        "shards": {"union": shards},
        "sets": {"within": sets(None), "by_all": sets(np.arange(w.M, dtype=np.uint32))},
        "perm": {"perm": perm},
        "ld_all": {"ld": ld("ld_all", None)},
        "ld_mask": {"ld": ld("ld_mask", w.ld_mask)},
        "ld_ones": {"ld": ld("ld_ones", np.ones(w.N, bool))},
        "ld_pairs": {"all": lambda: st.ld_pairs(pi, pj), "mask": lambda: st.ld_pairs(pi, pj, w.ld_mask)},
    }


def canon(v):
    if isinstance(v, np.ndarray):
        return v
    if isinstance(v, (tuple, list)) and not isinstance(v, Err):
        return tuple(canon(x) for x in v)
    if isinstance(v, np.generic):
        return np.asarray(v)
    return v


def run_observers(w, st, names, info=None):
    info = {} if info is None else info
    obs = observers(w, st, info)
    out = {}
    for name in names:
        for key, fn in obs[name].items():
            try:
                out[f"{name}.{key}"] = canon(fn())
            except gw.GwasDevError as e:
                out[f"{name}.{key}"] = Err(("error", status_of(e)))
    return out


def assert_same(got, want, where):
    """bytes equal (so NaN patterns too), arrays in nested tuples; errors by status"""
    for key in want:
        a, b = got[key], want[key]
        if isinstance(b, Err) or isinstance(a, Err):
            assert isinstance(a, Err) and isinstance(b, Err) and a == b, f"{where}: {key}: {a} vs {b}"
            continue
        for k, (x, y) in enumerate(zip(*(_flat(a), _flat(b)))):
            assert x.dtype == y.dtype and x.shape == y.shape, f"{where}: {key}[{k}]: {x.dtype}{x.shape} vs {y.dtype}{y.shape}"
            if x.tobytes() != y.tobytes():
                bx, by = x.reshape(-1).view(np.uint8), y.reshape(-1).view(np.uint8)
                n = min(len(bx), len(by))
                first = int(np.flatnonzero(bx[:n] != by[:n])[0]) // max(1, x.itemsize) if n else 0
                pytest.fail(f"{where}: {key}[{k}] differs first at element {first}")


def _flat(v):
    if v is None:
        return []
    if isinstance(v, np.ndarray):
        return [np.ascontiguousarray(v)]
    out = []
    for x in v:
        out += _flat(x)
    return out


# ------------------------------------------------------------------------------------------------------
# the reused store and its host shadow
# ------------------------------------------------------------------------------------------------------
class Walk:
    def __init__(self, orc, name, tmp_path, st=None):
        self.orc, self.name, self.tmp = orc, name, tmp_path
        self.codes, self.orig, self.pheno = cohort(orc, name)
        self.M, self.N, _ = COHORTS[name]
        self.rows = self.orig.copy()
        self.cur_codes = self.codes.copy()      # codes of the rows written by this walk (None after simulate)
        self.sel = None                         # (case mask, control mask, effective labels)
        self.fly = None                         # stream masks
        self.opts, self.engine, self.eager = {}, 0, False
        self.st = st or gw.GenoStore(self.M, self.N)
        if st is None:
            self.st.put_rows(self.rows)
        self.pairs = np.array([p for p in EDGE_PAIRS if p[1] < self.M], np.uint32).T.copy()
        self.set_a = np.arange(0, self.M, 3, dtype=np.uint32)
        self.ld_mask = np.random.default_rng(5).random(self.N) < 0.7
        self.n_writes = 0

    def close(self):
        self.st.close()

    # -- the reference
    def fresh(self):
        st = gw.GenoStore(self.M, self.N)
        st.put_rows(self.rows)
        for o, v in self.opts.items():
            st.set_option(o, v)
        st.set_pair_engine(self.engine)
        st.set_select_mode(self.eager)
        if self.sel is not None:
            st.select_case_control(case_mask=self.sel[0], ctrl_mask=self.sel[1])
        if self.fly is not None and (self.sel is None or not (np.array_equal(self.fly[0], self.sel[0]) and
                                                              np.array_equal(self.fly[1], self.sel[1]))):
            st.set_stream_masks(case_mask=self.fly[0], ctrl_mask=self.fly[1])
        return st

    def check(self, names, where, expect=None):
        info = {}
        got = run_observers(self, self.st, names, info)
        with self.fresh() as ref:
            want = run_observers(self, ref, names)
        assert_same(got, want, where)
        for key, v in (expect or {}).items():
            name, what = key.split(".")
            assert name in info, f"{where}: {name} failed: {[v for k, v in got.items() if k.startswith(name)]}"
            assert info[name][{"built": 0, "planes": 1, "rows": 1}[what]] == v, f"{where}: {key} = {info[name]}, expected {v}"
        return got

    # -- mutators: the store and the shadow change together
    def select(self, variant, rng):
        ph = self.pheno
        if variant == "pheno":
            ca, co, eff = masks_of(ph)
        elif variant == "shuffle":
            ca, co, eff = masks_of(rng.permutation(ph))
        elif variant.startswith("frac"):
            ca, co, eff = masks_of((rng.random(self.N) < float(variant[4:])).astype(np.uint8))
        elif variant == "neither":
            p = ph.copy()
            p[rng.random(self.N) < 0.1] = 2
            ca, co, eff = masks_of(p)
        elif variant == "both":
            ca, co, eff = masks_of(ph, rng, self.N // 20)
        elif variant.startswith("ncase"):
            p = np.zeros(self.N, np.uint8)
            p[rng.choice(self.N, int(variant[5:]), replace=False)] = 1
            ca, co, eff = masks_of(p)
        else:
            raise ValueError(variant)
        self.st.select_case_control(case_mask=ca, ctrl_mask=co)
        self.sel, self.fly = (ca, co, eff), (ca, co)

    def stream(self, rng):
        ph = rng.integers(0, 3, self.N).astype(np.uint8)        # unrelated to the selection, some samples in neither
        ca, co, _ = masks_of(ph, rng, self.N // 50)
        self.st.set_stream_masks(case_mask=ca, ctrl_mask=co)
        self.fly = (ca, co)

    def option(self, opt, value):
        self.st.set_option(opt, value)
        self.opts[opt] = value

    def set_engine(self, e):
        self.st.set_pair_engine(e)
        self.engine = e

    def set_eager(self, b):
        self.st.set_select_mode(b)
        self.eager = b

    def write(self, how, variant, first=191, rng=None):
        """three rows replaced through one loader: 'missing' gives them missing calls, 'complete' none, 'restore' puts the
        cohort's own rows back"""
        n = 3
        if variant == "restore":
            codes = self.codes[first:first + n].copy()
        else:
            donor = (first + 200 + 7 * self.n_writes) % (self.M - n)
            codes = self.codes[donor:donor + n].copy()
            codes[codes == 3] = 0
            if variant == "missing":
                codes[:, 1::97] = 3
        self.n_writes += 1
        if how == "put_rows":
            self.st.put_rows(self.orc.pack_codes(codes), first)
        elif how == "put_bed":
            self.st.put_bed(bed_of(codes), np.tile(np.array([[2, 3]], np.uint8), (n, 1)), first)
        elif how == "tped_text":
            assert self.st.put_tped_text(tped_of(codes, first), first)[0] == n
        elif how == "load_tped":
            path = os.path.join(self.tmp, f"w{self.n_writes}.tped")
            with open(path, "wb") as f:
                f.write(tped_of(codes, first))
            assert self.st.load_tped(path, first) == n
        else:
            raise ValueError(how)
        self.rows[first:first + n] = self.st.get_rows(first, n)
        if how == "put_rows":
            assert np.array_equal(self.rows[first:first + n], self.orc.pack_codes(codes))
        if self.cur_codes is not None:
            self.cur_codes[first:first + n] = codes
        self.sel = None

    def restore(self):
        self.st.put_rows(self.orig)
        self.rows, self.cur_codes, self.sel = self.orig.copy(), self.codes.copy(), None

    def simulate(self, seed, missing):
        self.st.simulate(seed, missing_rate=missing)
        self.rows, self.cur_codes, self.sel = self.st.get_rows(), None, None

    # -- scripted steps
    def step(self, s, rng):
        kind = s[0]
        if kind == "sel":
            self.select(s[1], rng)
        elif kind == "stream":
            self.stream(rng)
        elif kind == "write":
            self.write(s[1], s[2], *(s[3:4] or (191,)))
        elif kind == "sim":
            self.simulate(s[1], s[2])
        elif kind == "restore":
            self.restore()
        elif kind == "opt":
            self.option(s[1], s[2])
        elif kind == "engine":
            self.set_engine(s[1])
        elif kind == "eager":
            self.set_eager(s[1])
        else:
            raise ValueError(kind)


# ------------------------------------------------------------------------------------------------------
# final-state anchors: the oracle and the exact integer LD reference
# ------------------------------------------------------------------------------------------------------
def anchor(w):
    orc, st = w.orc, w.st
    ca, co, eff = w.sel
    sel, nca, nco = orc.select(w.rows, w.N, eff)
    assert np.array_equal(st.marginal_scan()["counts"], orc.cc_counts_selected(sel, nca, nco)), "counts differ from the oracle"
    # screen hits of the corner i < 128; a pair within rounding of the threshold may fall on either side
    mar = orc.margins(sel, nca, nco)
    hi, hj, hs, _ = orc.boost_screen(sel, mar, nca, nco, THR, 0, 128)
    hits, _ = st.pairwise_scan(THR)
    h = hits[hits["i"] < 128]
    got = {(int(a), int(b)): s for a, b, s in zip(h["i"], h["j"], h["stat"])}
    want = {(int(a), int(b)): s for a, b, s in zip(hi, hj, hs)}
    scale = w.N * np.log(w.N)
    for key in set(got) | set(want):
        if key in got and key in want:
            assert abs(got[key] - want[key]) <= 1e-12 * max(abs(want[key]), scale), (key, got[key], want[key])
        else:
            s = got.get(key, want.get(key))
            assert abs(s - THR) <= 1e-9 * scale, f"pair {key} ({s}) only on one side"
    # LD over every sample and over the mask, against the integer sums
    x, c = decoded(st)
    for mask in (None, w.ld_mask):
        ref = ld_reference(x, c, mask)
        pairs, band, _ = st.ld_window(LD_WINDOW, LD_THR, sample_mask=mask, band=True)
        want_band = band_of(ref[2], 0, w.M, LD_WINDOW)
        assert np.array_equal(np.isnan(band), np.isnan(want_band))
        assert np.array_equal(np.nan_to_num(band, nan=-7).view(np.uint32), np.nan_to_num(want_band, nan=-7).view(np.uint32))
        want_list = list_of(ref, 0, w.M, LD_WINDOW, LD_THR)
        assert len(pairs) == len(want_list)
        for f in ("i", "j", "n"):
            assert np.array_equal(pairs[f], want_list[f])
        for f in ("r", "r2"):
            assert np.array_equal(pairs[f].view(np.uint64), want_list[f].view(np.uint64))


# ------------------------------------------------------------------------------------------------------
# 1. scripted matrix: one case per (cache, mutator) pair
# ------------------------------------------------------------------------------------------------------
SCRIPTS = {
    # per-SNP row totals (tot_valid): rows only; a re-selection reuses them
    "row_totals/row_write": ("a", [("sel", "pheno"), ("obs", ["scan"]), ("obs", ["scan", "counts"]),
                                   ("write", "put_rows", "complete"), ("sel", "pheno"), ("obs", ["scan", "scan_sub", "counts"])]),
    "row_totals/reselection_keeps": ("a", [("sel", "pheno"), ("obs", ["scan"]), ("sel", "shuffle"), ("obs", ["scan", "compact"]),
                                           ("sel", "pheno"), ("obs", ["scan"])]),
    "row_totals/option": ("a", [("sel", "pheno"), ("obs", ["scan"]), ("opt", gw.OPT_ROW_TOTALS, 1), ("sel", "shuffle"),
                                ("obs", ["scan"]), ("opt", gw.OPT_ROW_TOTALS, 0), ("obs", ["scan"]), ("sel", "pheno"), ("obs", ["scan"])]),
    # compacted rows (sel_built, K0)
    "compacted/selection": ("a", [("sel", "neither"), ("obs", ["selected_rows", "counts"]), ("sel", "both"),
                                  ("obs", ["selected_rows", "counts", "pair_tables"]), ("sel", "pheno"), ("obs", ["selected_rows", "scan"])]),
    "compacted/row_write": ("b", [("eager", True), ("sel", "pheno"), ("obs", ["selected_rows"]), ("write", "put_bed", "complete"),
                                  ("sel", "pheno"), ("obs", ["selected_rows", "counts", "scan"])]),
    "compacted/select_kernel": ("b", [("sel", "pheno"), ("opt", gw.OPT_SELECT_KERNEL, 1), ("sel", "neither"), ("obs", ["selected_rows"]),
                                      ("opt", gw.OPT_SELECT_KERNEL, 0), ("sel", "both"), ("obs", ["selected_rows", "scan"])]),
    # margins, per-SNP records, tile-missing flags
    "margins/selection": ("a", [("sel", "pheno"), ("obs", ["screen", "pair_stats"]), ("sel", "neither"), ("obs", ["screen", "pair_stats"]),
                                ("sel", "both"), ("obs", ["screen", "shards"])]),
    "margins/first_missing_call": ("a", [("sel", "pheno"), ("obs", ["screen"]), ("write", "put_rows", "missing"), ("sel", "pheno"),
                                         ("obs", ["screen", "shards", "pair_stats", "sets"])]),
    "margins/last_missing_call_removed": ("a", [("write", "put_rows", "missing"), ("sel", "pheno"), ("obs", ["screen", "shards"]),
                                                ("write", "put_rows", "restore"), ("sel", "pheno"), ("obs", ["screen", "shards", "tile"])]),
    # two-plane tensor-core operands (mm_built, mma_side_valid)
    "mma_planes/classic_planes_toggle": ("a", [("sel", "pheno"), ("obs", ["screen", "pair_stats"]), ("opt", gw.OPT_CLASSIC_PLANES, 1),
                                               ("obs", ["screen", "pair_stats", "tile"]), ("opt", gw.OPT_CLASSIC_PLANES, 0),
                                               ("obs", ["screen", "pair_stats", "sets"])]),
    "mma_planes/selection": ("a", [("sel", "pheno"), ("obs", ["screen"]), ("sel", "shuffle"), ("obs", ["screen", "pair_stats"])]),
    "mma_planes/row_write": ("a", [("sel", "pheno"), ("obs", ["screen"]), ("write", "tped_text", "complete"), ("sel", "pheno"),
                                   ("obs", ["screen", "tile", "pair_stats"])]),
    # four-plane operands (mm4_mode 0 / 1 / 2) across the packed accumulator's limit
    "mm4/accumulator_limit_missing": ("c", [("sel", "ncase16383"), ("obs", ["screen", "pair_stats"]), ("sel", "ncase16384"),
                                            ("obs", ["screen", "pair_stats", "sets"]), ("sel", "ncase16383"), ("obs", ["screen", "shards"])]),
    "mm4/accumulator_limit_complete": ("c", [("sim", 99, 0.0), ("sel", "ncase16383"), ("obs", ["screen"]), ("sel", "ncase16384"),
                                             ("obs", ["screen", "shards"]), ("sel", "ncase16383"), ("obs", ["screen", "pair_stats"])]),
    "mm4/four_plane_option": ("b", [("sel", "pheno"), ("obs", ["screen"]), ("opt", gw.OPT_FOUR_PLANE, 1), ("obs", ["screen", "shards"]),
                                    ("opt", gw.OPT_FOUR_PLANE, 0), ("obs", ["screen", "shards"])]),
    "mm4/row_write": ("b", [("sel", "pheno"), ("obs", ["screen"]), ("write", "load_tped", "missing"), ("sel", "pheno"),
                            ("obs", ["screen", "pair_stats"])]),
    # the bound pre-filter's constants follow the case fraction
    "bound/case_fraction": ("a", [("sel", "pheno"), ("obs", ["pair_stats", "screen"]), ("sel", "frac0.2"), ("obs", ["pair_stats", "screen"]),
                                  ("sel", "frac0.7"), ("obs", ["pair_stats", "screen"])]),
    # cached pair / tile counts of the last screen's shard
    "pair_counts/engine": ("b", [("sel", "pheno"), ("obs", ["screen", "shards"]), ("engine", 1), ("obs", ["screen", "shards"]),
                                 ("engine", 2), ("obs", ["screen"]), ("engine", 0), ("obs", ["screen", "shards"])]),
    "pair_counts/row_write": ("a", [("sel", "pheno"), ("obs", ["shards"]), ("write", "put_rows", "missing"), ("sel", "pheno"),
                                    ("obs", ["shards", "screen"])]),
    "pair_counts/selection": ("c", [("sel", "pheno"), ("obs", ["shards"]), ("sel", "ncase16384"), ("obs", ["shards"])]),
    "candidates/overflow_rerun": ("a", [("sel", "pheno"), ("opt", gw.OPT_CAND_CAPACITY, 16), ("obs", ["screen", "shards", "sets"]),
                                        ("opt", gw.OPT_CAND_CAPACITY, 0), ("obs", ["screen"])]),
    # permutation SNP planes: rows only, they survive re-selection
    "perm_planes/reselection_keeps": ("a", [("sel", "pheno"), ("obs", ["perm"], {"perm.built": 1}), ("sel", "shuffle"),
                                            ("obs", ["perm"], {"perm.built": 0}), ("sel", "neither"), ("obs", ["perm"], {"perm.built": 0})]),
    "perm_planes/row_write": ("a", [("sel", "pheno"), ("obs", ["perm"], {"perm.built": 1, "perm.planes": 2}),
                                    ("write", "put_rows", "missing"), ("sel", "pheno"), ("obs", ["perm"], {"perm.built": 1, "perm.planes": 3}),
                                    ("write", "put_rows", "restore"), ("sel", "pheno"), ("obs", ["perm"], {"perm.built": 1, "perm.planes": 2}),
                                    ("obs", ["perm"], {"perm.built": 0})]),
    "perm_planes/budget": ("b", [("sel", "pheno"), ("obs", ["perm"], {"perm.built": 1}), ("obs", ["perm"], {"perm.built": 0}),
                                 ("opt", gw.OPT_PERM_OPERAND_BYTES, 1), ("obs", ["perm"], {"perm.built": 1}),
                                 ("opt", gw.OPT_PERM_OPERAND_BYTES, 0), ("obs", ["perm"], {"perm.built": 1}), ("obs", ["perm"], {"perm.built": 0})]),
    # LD operand: rows and the sample set S; it survives re-selection
    "ld_operand/sample_set": ("a", [("obs", ["ld_all"], {"ld_all.built": 1}), ("obs", ["ld_all"], {"ld_all.built": 0}),
                                    ("obs", ["ld_mask"], {"ld_mask.built": 1}), ("obs", ["ld_all"], {"ld_all.built": 1}),
                                    ("obs", ["ld_ones", "ld_pairs"]), ("obs", ["ld_mask", "ld_all"])]),
    "ld_operand/row_write": ("a", [("obs", ["ld_all"], {"ld_all.built": 1, "ld_all.rows": 1}), ("write", "put_bed", "missing"),
                                   ("obs", ["ld_all", "ld_pairs"], {"ld_all.built": 1, "ld_all.rows": 3}), ("write", "put_bed", "restore"),
                                   ("obs", ["ld_all"], {"ld_all.built": 1, "ld_all.rows": 1}), ("obs", ["ld_all"], {"ld_all.built": 0})]),
    "ld_operand/budget": ("b", [("obs", ["ld_mask"], {"ld_mask.built": 1}), ("opt", gw.OPT_LD_OPERAND_BYTES, 1),
                                ("obs", ["ld_mask"], {"ld_mask.built": 1}), ("obs", ["ld_mask"], {"ld_mask.built": 1}),
                                ("opt", gw.OPT_LD_OPERAND_BYTES, 0), ("obs", ["ld_mask"], {"ld_mask.built": 1}),
                                ("obs", ["ld_mask"], {"ld_mask.built": 0})]),
    "ld_operand/selection_keeps": ("a", [("obs", ["ld_all"], {"ld_all.built": 1}), ("sel", "pheno"), ("obs", ["ld_all"], {"ld_all.built": 0}),
                                         ("sel", "neither"), ("obs", ["ld_all", "ld_pairs"], {"ld_all.built": 0})]),
    # stream masks (fly_valid): set by a selection and by set_stream_masks, kept by a row write
    "stream_masks/selection_resets": ("a", [("sel", "pheno"), ("stream",), ("obs", ["counts", "pair_tables", "pair_stats"]),
                                            ("sel", "neither"), ("obs", ["counts", "pair_tables"]), ("stream",), ("obs", ["counts"])]),
    "stream_masks/survive_row_write": ("a", [("sel", "pheno"), ("stream",), ("write", "put_rows", "complete"),
                                             ("obs", ["counts", "pair_tables", "pair_stats", "scan"]), ("sel", "both"), ("obs", ["counts"])]),
    # which scan runs: scans since the selection, eager compaction, the scan knobs
    "scan_mode/masked_scan_option": ("a", [("sel", "neither"), ("obs", ["scan", "scan_sub"]), ("obs", ["scan"]),
                                           ("opt", gw.OPT_MASKED_SCAN, 1), ("sel", "neither"), ("obs", ["scan"]),
                                           ("opt", gw.OPT_MASKED_SCAN, 0), ("sel", "both"), ("obs", ["scan", "compact"])]),
    "scan_mode/eager": ("b", [("eager", True), ("sel", "neither"), ("obs", ["scan", "counts"]), ("eager", False), ("sel", "pheno"),
                              ("obs", ["scan", "selected_rows"])]),
    "scan_mode/lanes_and_pieces": ("b", [("sel", "pheno"), ("opt", gw.OPT_LANES_PER_ROW, 8), ("obs", ["scan"]),
                                         ("opt", gw.OPT_SCAN_PIECES, 3), ("obs", ["scan", "compact", "scan_sub"]),
                                         ("opt", gw.OPT_LANES_PER_ROW, 32), ("sel", "neither"), ("obs", ["scan"])]),
    # a whole-table rewrite
    "loaders/simulate": ("b", [("sel", "pheno"), ("obs", ["scan", "perm", "ld_all"]), ("sim", 5, 0.01), ("sel", "pheno"),
                               ("obs", ["scan", "perm", "ld_all", "screen"], {"perm.built": 1, "ld_all.built": 1})]),
}


@pytest.mark.parametrize("case", list(SCRIPTS))
def test_scripted(orc, tmp_path, case):
    name, steps = SCRIPTS[case]
    rng = np.random.default_rng(sum(map(ord, case)))
    w = Walk(orc, name, str(tmp_path))
    try:
        for k, s in enumerate(steps):
            if s[0] == "obs":
                w.check(s[1], f"{case} step {k} {s[1]}", s[2] if len(s) > 2 else None)
            else:
                w.step(s, rng)
    finally:
        w.close()


def test_row_write_drops_the_selection(orc, tmp_path):
    """After a row write, every call on a selection fails with GWASDEV_EINVAL, and the stream-mask calls, the whole-cohort
    counts and LD read the new rows (include/gwasdev.h, gwasdev_put_rows)."""
    w = Walk(orc, "b", str(tmp_path))
    try:
        rng = np.random.default_rng(3)
        w.select("pheno", rng)
        before = w.check(list(LONG), "before")
        w.stream(rng)
        w.write("put_rows", "complete")
        got = w.check(list(LONG), "after the write")
        fails = {k for k, v in got.items() if isinstance(v, Err)}
        assert all(got[k] == ("error", EINVAL) for k in fails)
        ok = {"counts.mode0", "counts.mode1", "pair_tables.mode0", "pair_tables.mode1", "pair_stats.epi1", "ld_all.ld", "ld_mask.ld",
              "ld_ones.ld", "ld_pairs.all", "ld_pairs.mask"}
        assert set(got) - fails == ok, sorted(set(got) - fails)
        assert w.st.L.gwasdev_is_compacted(w.st.h) == -1
        w.select("pheno", rng)
        again = w.check(list(LONG), "re-selected")
        assert {k for k, v in again.items() if isinstance(v, Err)} == {k for k, v in before.items() if isinstance(v, Err)}
    finally:
        w.close()


# ------------------------------------------------------------------------------------------------------
# 2. seeded random walks
# ------------------------------------------------------------------------------------------------------
WALK_OPTIONS = [(gw.OPT_CLASSIC_PLANES, (0, 1)), (gw.OPT_FOUR_PLANE, (0, 1)), (gw.OPT_ROW_TOTALS, (0, 1)), (gw.OPT_MASKED_SCAN, (0, 1)),
                (gw.OPT_LANES_PER_ROW, (0, 8, 16, 32)), (gw.OPT_SCAN_PIECES, (0, 1, 3, 8)), (gw.OPT_SELECT_KERNEL, (0, 1)),
                (gw.OPT_CAND_CAPACITY, (0, 16)), (gw.OPT_PERM_OPERAND_BYTES, (0, 1)), (gw.OPT_LD_OPERAND_BYTES, (0, 1))]
N_STEPS = 40


def random_step(w, rng):
    """one seeded mutator; returns its description"""
    r = rng.random()
    if w.sel is None and r < 0.5:
        r = 0.0                                  # after a row write, mostly select again
    if r < 0.30:
        variants = ["pheno", "shuffle", "frac0.3", "frac0.6", "neither", "both"]
        if w.name == "c":
            variants += ["ncase16383", "ncase16384"] * 2
        s = ("sel", str(rng.choice(variants)))
    elif r < 0.40:
        s = ("stream",)
    elif r < 0.60:
        s = ("write", str(rng.choice(["put_rows", "put_bed", "tped_text", "load_tped"])),
             str(rng.choice(["missing", "complete", "restore"])), int(rng.choice([f for f in WRITE_FIRSTS if f + 3 <= w.M])))
    elif r < 0.63:
        s = ("sim", int(rng.integers(1, 1 << 30)), float(rng.choice([0.0, 0.01])))
    elif r < 0.67:
        s = ("restore",)
    elif r < 0.88:
        opt, vals = WALK_OPTIONS[int(rng.integers(len(WALK_OPTIONS)))]
        s = ("opt", opt, int(rng.choice(vals)))
    elif r < 0.94:
        s = ("engine", int(rng.integers(3)))
    else:
        s = ("eager", bool(rng.integers(2)))
    w.step(s, rng)
    return s


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("name", list(COHORTS))
def test_random_walk(orc, tmp_path, name, seed):
    rng = np.random.default_rng(1000 * seed + ord(name))
    w = Walk(orc, name, str(tmp_path))
    age = {o: 0 for o in LONG}
    try:
        for k in range(N_STEPS):
            s = random_step(w, rng)
            due = [o for o in LONG if age[o] >= 4]
            extra = [str(o) for o in rng.choice(LONG, 3, replace=False)]
            names = [o for o in LONG if o in set(due) | set(extra)]
            w.check(names, f"walk {name}/{seed} step {k} {s}")
            for o in LONG:
                age[o] = 0 if o in names else age[o] + 1
            if k == N_STEPS // 2:              # a replica mid-walk equals the original on every observer
                with w.st.replicate(w.st.device) as rep:
                    got = run_observers(w, rep, LONG)
                want = run_observers(w, w.st, LONG)
                assert_same(got, want, f"walk {name}/{seed} replica after step {k}")
        w.step(("sel", "pheno"), rng)
        w.check(list(LONG), f"walk {name}/{seed} final battery")
        anchor(w)
    finally:
        w.close()


# ------------------------------------------------------------------------------------------------------
# 3. a table sized by the TPED loader, replicas
# ------------------------------------------------------------------------------------------------------
def test_from_tped_store_equals_a_put_rows_store(orc, tmp_path):
    """gwasdev_create_from_tped allocates for the file size and trims M and Mpad to the rows found: every cache sized from the
    table must follow the trimmed geometry."""
    codes, rows, pheno = cohort(orc, "b")
    path = str(tmp_path / "b.tped")
    with open(path, "wb") as f:
        f.write(tped_of(codes, 0))
    st = gw.GenoStore.from_tped(path)
    assert (st.n_snps, st.n_samples) == codes.shape
    assert np.array_equal(st.get_rows(), rows)
    w = Walk(orc, "b", str(tmp_path), st=st)
    try:
        rng = np.random.default_rng(8)
        w.select("pheno", rng)
        w.check(list(LONG), "from_tped")
        w.option(gw.OPT_CLASSIC_PLANES, 1)
        w.write("put_rows", "missing", 447)
        w.select("both", rng)
        w.check(list(LONG), "from_tped after a write")
        w.select("pheno", rng)
        anchor(w)
    finally:
        w.close()


def test_replica_carries_stream_masks_and_options(orc, tmp_path):
    """gwasdev_replicate re-applies options, engine, select mode, the selection and then the stream masks: its mask-on-the-fly
    observers (counts mode 1, pair_tables mode 1, epi_pairs mode 1) answer over the masks of gwasdev_set_stream_masks, as the
    original does -- also after a row write has dropped the selection."""
    w = Walk(orc, "b", str(tmp_path))
    try:
        rng = np.random.default_rng(4)
        w.option(gw.OPT_CLASSIC_PLANES, 1)
        w.option(gw.OPT_LANES_PER_ROW, 16)
        w.option(gw.OPT_LD_OPERAND_BYTES, 1)
        w.set_eager(True)
        w.select("neither", rng)
        w.stream(rng)
        for where in ("after set_stream_masks", "after a row write"):
            if where == "after a row write":
                w.write("put_rows", "missing")
            with w.st.replicate(w.st.device) as rep:
                got = run_observers(w, rep, LONG)
            want = run_observers(w, w.st, LONG)
            assert_same(got, want, f"replica {where}")
            with w.fresh() as ref:            # and both answer over the stream masks, not over the selection
                assert np.array_equal(ref.counts(1), want["counts.mode1"])
                assert np.array_equal(ref.pair_tables(*w.pairs, 1), want["pair_tables.mode1"])
    finally:
        w.close()


@pytest.mark.skipif(n_gpus() < 2, reason="needs two GPUs in this process")
def test_replica_on_another_device(orc, tmp_path):
    w = Walk(orc, "b", str(tmp_path))
    try:
        rng = np.random.default_rng(6)
        w.option(gw.OPT_FOUR_PLANE, 1)
        w.select("both", rng)
        w.stream(rng)
        w.check(["screen"], "warm")
        with w.st.replicate(1) as rep:
            assert_same(run_observers(w, rep, LONG), run_observers(w, w.st, LONG), "replica on device 1")
            hits, _ = gw.pairwise_scan_multi([w.st, rep], THR, gather="peer")
            assert np.array_equal(hits, w.st.pairwise_scan(THR)[0])
            pi, pj = w.pairs
            s, z = gw.gtest_multi([w.st, rep], pi, pj)
            s1, z1 = w.st.gtest(pi, pj)
            assert s.tobytes() == s1.tobytes() and z.tobytes() == z1.tobytes()
    finally:
        w.close()
