"""TEST INFRASTRUCTURE -- NOT PRODUCT CODE.

ctypes front-ends for the two CPU checkers of the association hot path:

* ``Oracle``  -- the plain-C restatement in ``oracle/gwas_oracle.c`` (built to
  ``oracle/libgwas_oracle.so``); every function cites the reference file:line it follows.
* ``Ref``     -- the UNMODIFIED reference compiled from ``/root/reference`` by
  ``oracle/ref_build/Makefile`` into ``oracle/_ref/libgwasref.so`` (git-ignored, travels to the GPU box).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this package.  The product (``libgwaspp_b200``) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "libgwas_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libgwasref.so")
# the same unmodified reference objects with the device table plugged into GeneticData's factory (level 6); see
# oracle/ref_build/Makefile and libgwaspp_b200/binding/device_genotype_table.h
REF_DEV_SO = os.path.join(HERE, "_ref", "libgwasref_dev.so")
REFERENCE_ROOT = "/root/reference"

# genetics/genotype/common_genotype.h:101-106 (192 bytes)
MI_DTYPE = np.dtype(
    [("margins", "<u4", 4), ("cases", "<u4", 4), ("controls", "<u4", 4),
     ("entropy", "<f8"), ("entropy_y", "<f8"), ("pbc", "<f8", 8), ("pca", "<f8", 8)]
)
assert MI_DTYPE.itemsize == 192

# data/maf_spectrum.tab restated as data (no run-time read of /root/reference). The table lives with the
# product's synthetic-cohort generator; the oracle may import product data, never the reverse.
def _load_spectrum():
    ns = {}
    with open(os.path.join(os.path.dirname(HERE), "libgwaspp_b200", "maf_spectrum.py")) as f:
        exec(f.read(), ns)
    return ns["MAF_SPECTRUM"]


MAF_SPECTRUM = _load_spectrum()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def build_oracle(force: bool = False) -> str:
    """gcc the C restatement (seconds)."""
    src = os.path.join(HERE, "gwas_oracle.c")
    if force or not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < max(
            os.path.getmtime(src), os.path.getmtime(os.path.join(HERE, "gwas_oracle.h"))):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c99", "-fno-fast-math",
                               "-ffp-contract=off", "-o", ORACLE_SO, src, "-lm"])
    return ORACLE_SO


def build_ref(force: bool = False) -> str | None:
    """Build oracle/_ref from the reference sources where they lie. No-op when /root/reference is absent
    (the GPU box): the prebuilt .so travels with the snapshot."""
    if not os.path.isdir(REFERENCE_ROOT):
        return REF_SO if os.path.exists(REF_SO) else None
    gwasdev = os.path.join(os.path.dirname(HERE), "libgwaspp_b200", "libgwasdev.so")
    stale = os.path.exists(gwasdev) and (not os.path.exists(REF_DEV_SO) or os.path.getmtime(REF_DEV_SO) < os.path.getmtime(gwasdev))
    if force or not os.path.exists(REF_SO) or stale:
        subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(HERE, "ref_build")],
                              stdout=subprocess.DEVNULL)
    return REF_SO


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def have_ref_dev() -> bool:
    return os.path.exists(REF_DEV_SO)


class Oracle:
    """numpy-level view of gwas_oracle.c."""

    def __init__(self):
        build_oracle()
        L = self.L = C.CDLL(ORACLE_SO)
        L.go_maf_reference.restype = C.c_double
        L.go_ksa.restype = C.c_double
        L.go_pairwise_epi_test.restype = C.c_double
        L.go_chisq_upper.restype = C.c_double
        L.go_chisq_upper.argtypes = [C.c_double, C.c_int]
        L.go_boost_screen.restype = C.c_long
        L.go_boost_screen.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_long, C.c_long,
                                      C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        L.go_compute_margins.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_void_p]
        L.go_sim_hash.restype = C.c_uint64
        L.go_sim_hash.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
        L.go_sim_row_codes.argtypes = [C.c_uint64, C.c_void_p, C.c_long, C.c_int, C.c_uint32, C.c_void_p]
        L.go_sim_phenotype.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_void_p]
        L.go_sim_minor_alleles.restype = C.c_uint64
        L.go_sim_minor_alleles.argtypes = [C.c_uint64, C.c_void_p, C.c_long, C.c_int]
        L.go_pack_row_text.argtypes = [C.c_char_p, C.c_long, C.c_int, C.c_void_p]

    # -- geometry
    def plane_blocks(self, n):
        return int(self.L.go_plane_blocks(int(n)))

    # -- store
    def pack_codes(self, codes):
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        M, N = codes.shape
        P = self.plane_blocks(N)
        rows = np.zeros((M, 2 * P + 1), dtype=np.uint16)
        for r in range(M):
            rc = self.L.go_pack_row_codes(_p(codes[r]), N, _p(rows[r]))
            if rc != 0:
                raise ValueError(f"row {r}: the reference aborts on this genotype sequence")
        return rows

    def pack_text(self, line: bytes, n_samples: int):
        P = self.plane_blocks(n_samples)
        row = np.zeros(2 * P + 1, dtype=np.uint16)
        rc = self.L.go_pack_row_text(line, len(line), n_samples, _p(row))
        if rc != 0:
            raise ValueError("the reference aborts on this genotype sequence")
        return row

    def call_at(self, row, n_samples, col):
        out = C.create_string_buffer(3)
        self.L.go_call_at(_p(row), n_samples, col, out)
        return out.value.decode()

    def masks(self, pheno):
        pheno = np.ascontiguousarray(pheno, dtype=np.uint8)
        P = self.plane_blocks(len(pheno))
        ca = np.zeros(P, np.uint16)
        co = np.zeros(P, np.uint16)
        nca, nco = C.c_int(), C.c_int()
        self.L.go_stream_masks(_p(pheno), len(pheno), _p(ca), _p(co), C.byref(nca), C.byref(nco))
        return ca, co, nca.value, nco.value

    def select(self, rows, n_samples, pheno):
        ca, co, nca, nco = self.masks(pheno)
        S = 2 * (self.plane_blocks(nca) + self.plane_blocks(nco))
        out = np.zeros((rows.shape[0], S), np.uint16)
        for r in range(rows.shape[0]):
            self.L.go_select_row(_p(rows[r]), n_samples, _p(ca), _p(co), nca, nco, _p(out[r]))
        return out, nca, nco

    # -- counts
    def cc_counts_selected(self, sel, nca, nco):
        out = np.zeros((sel.shape[0], 8), np.uint32)
        for r in range(sel.shape[0]):
            self.L.go_cc_counts_selected(_p(sel[r]), nca, nco, _p(out[r]))
        return out

    def cc_counts_masked(self, rows, n_samples, pheno):
        ca, co, nca, nco = self.masks(pheno)
        out = np.zeros((rows.shape[0], 8), np.uint32)
        for r in range(rows.shape[0]):
            self.L.go_cc_counts_masked(_p(rows[r]), n_samples, _p(ca), _p(co), nca, nco, _p(out[r]))
        return out

    def counts_whole(self, rows, n_samples):
        out = np.zeros((rows.shape[0], 4), np.uint32)
        for r in range(rows.shape[0]):
            self.L.go_counts_whole(_p(rows[r]), n_samples, _p(out[r]))
        return out

    def margins(self, sel, nca, nco):
        sel = np.ascontiguousarray(sel)
        out = np.zeros(sel.shape[0], MI_DTYPE)
        self.L.go_compute_margins(_p(sel), sel.shape[0], nca, nco, _p(out))
        return out

    def marginal_information(self, ca, co, n):
        ca = np.ascontiguousarray(ca, np.uint32)
        co = np.ascontiguousarray(co, np.uint32)
        out = np.zeros(1, MI_DTYPE)
        self.L.go_marginal_information_fill(_p(ca), _p(co), C.c_uint32(int(n)), _p(out))
        return out[0]

    def maf_reference(self, ft):
        ft = np.ascontiguousarray(ft, np.uint32)
        tot = C.c_double()
        v = self.L.go_maf_reference(_p(ft), C.byref(tot))
        return v, tot.value

    # -- pair tables
    def pair_table(self, mode, i, j, *, rows=None, sel=None, n_samples=None, pheno=None, nca=None, nco=None, mar=None):
        ca = np.zeros(16, np.uint32)
        co = np.zeros(16, np.uint32)
        if mode == 0:
            self.L.go_pair_table_whole(_p(rows[i]), _p(rows[j]), n_samples, _p(ca))
        elif mode == 1:
            mca, mco, _, _ = self.masks(pheno)
            self.L.go_pair_table_masked(_p(rows[i]), _p(rows[j]), n_samples, _p(mca), _p(mco), _p(ca), _p(co))
        elif mode == 2:
            self.L.go_pair_table_selected(_p(sel[i]), _p(sel[j]), nca, nco, _p(ca), _p(co))
        else:
            self.L.go_pair_table_margins(_p(sel[i]), _p(sel[j]), nca, nco, _p(mar[i:i + 1]), _p(mar[j:j + 1]),
                                         _p(ca), _p(co))
        return ca, co

    def ksa(self, ca, co, m1, m2, n):
        m1 = np.array([m1], MI_DTYPE)
        m2 = np.array([m2], MI_DTYPE)
        return float(self.L.go_ksa(_p(np.ascontiguousarray(ca, np.uint32)), _p(np.ascontiguousarray(co, np.uint32)),
                                   _p(m1), _p(m2), int(n)))

    def gtest(self, ca, co, m1, m2, n):
        m1 = np.array([m1], MI_DTYPE)
        m2 = np.array([m2], MI_DTYPE)
        s, z = C.c_double(), C.c_double()
        self.L.go_gtest(_p(np.ascontiguousarray(ca, np.uint32)), _p(np.ascontiguousarray(co, np.uint32)),
                        _p(m1), _p(m2), C.c_uint32(int(n)), C.byref(s), C.byref(z))
        return s.value, z.value

    def gtest_ex(self, ca, co, m1, m2, n):
        """(stat, z, IPF sweeps, S): go_gtest plus the sweep count and the error scale S of the statistic."""
        m1 = np.array([m1], MI_DTYPE)
        m2 = np.array([m2], MI_DTYPE)
        s, z, sw, S = C.c_double(), C.c_double(), C.c_uint32(), C.c_double()
        self.L.go_gtest_ex(_p(np.ascontiguousarray(ca, np.uint32)), _p(np.ascontiguousarray(co, np.uint32)),
                           _p(m1), _p(m2), C.c_uint32(int(n)), C.byref(s), C.byref(z), C.byref(sw), C.byref(S))
        return s.value, z.value, sw.value, S.value

    def pairwise_epi_test(self, cs, ct):
        cs = np.ascontiguousarray(cs, np.int32).reshape(9)
        ct = np.ascontiguousarray(ct, np.int32).reshape(9)
        return float(self.L.go_pairwise_epi_test(_p(cs), _p(ct)))

    def chisq_upper(self, x, df):
        return float(self.L.go_chisq_upper(float(x), int(df)))

    def chi2_allelic(self, ca, co):
        x, p = C.c_double(), C.c_double()
        self.L.go_chi2_allelic(_p(np.ascontiguousarray(ca, np.uint32)), _p(np.ascontiguousarray(co, np.uint32)),
                               C.byref(x), C.byref(p))
        return x.value, p.value

    def chi2_genotypic(self, ca, co):
        x, p, df = C.c_double(), C.c_double(), C.c_int()
        self.L.go_chi2_genotypic(_p(np.ascontiguousarray(ca, np.uint32)), _p(np.ascontiguousarray(co, np.uint32)),
                                 C.byref(x), C.byref(p), C.byref(df))
        return x.value, p.value, df.value

    def boost_screen(self, sel, mar, nca, nco, threshold=30.0, i0=0, i1=None, cap=1 << 20):
        sel = np.ascontiguousarray(sel)
        M = sel.shape[0]
        i1 = M if i1 is None else i1
        hi = np.zeros(cap, np.uint32)
        hj = np.zeros(cap, np.uint32)
        hs = np.zeros(cap, np.float64)
        st = np.zeros(4, np.float64)
        n = self.L.go_boost_screen(_p(sel), _p(mar), M, nca, nco, i0, i1, threshold, _p(hi), _p(hj), _p(hs), cap, _p(st))
        if n > cap:
            raise RuntimeError("hit capacity exceeded")
        return hi[:n].copy(), hj[:n].copy(), hs[:n].copy(), st

    # -- synthetic cohort
    def simulate(self, seed, n_snps, n_samples, n_case, panel="affy6", missing_rate=0.0, first_snp=0):
        bins = np.asarray(MAF_SPECTRUM[panel], np.uint32)
        q = int(missing_rate * 4294967296.0) & 0xFFFFFFFF
        codes = np.zeros((n_snps, n_samples), np.uint8)
        for r in range(n_snps):
            self.L.go_sim_row_codes(seed, _p(bins), first_snp + r, n_samples, q, _p(codes[r]))
        pheno = np.zeros(n_samples, np.uint8)
        self.L.go_sim_phenotype(seed, n_samples, n_case, _p(pheno))
        return codes, pheno


def _minor_alleles(self, seed, n_snps, n_samples, panel="affy6", first_snp=0):
    bins = np.asarray(MAF_SPECTRUM[panel], np.uint32)
    return np.array([self.L.go_sim_minor_alleles(seed, _p(bins), first_snp + r, n_samples) for r in range(n_snps)],
                    np.uint64)


Oracle.minor_alleles = _minor_alleles


class Ref:
    """The unmodified reference (T3/T4/T5 tables + its own test functions) behind a C-ABI harness."""

    _lib = None
    SO = REF_SO

    @classmethod
    def lib(cls):
        if cls._lib is None:
            if not os.path.exists(cls.SO):
                raise FileNotFoundError(cls.SO)
            L = C.CDLL(cls.SO)
            L.gwasref_create.restype = C.c_void_p
            L.gwasref_load_tplink.restype = C.c_void_p
            L.gwasref_load_tplink.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
            L.gwasref_pairwise_c.restype = C.c_double
            L.gwasref_time_phase.restype = C.c_double
            L.gwasref_add_row_text.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_long]
            L.gwasref_run.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_long]
            assert L.gwasref_sizeof_marginal_information() == MI_DTYPE.itemsize
            cls._lib = L
        return cls._lib

    def __init__(self, n_snps=None, n_samples=None, level=5, *, tped=None, tfam=None):
        L = self.L = self.lib()
        if tped is not None:
            self.h = C.c_void_p(L.gwasref_load_tplink(tped.encode(), tfam.encode(), level))
        else:
            self.h = C.c_void_p(L.gwasref_create(int(n_snps), int(n_samples), int(level)))
        self.n_snps = L.gwasref_n_snps(self.h)
        self.n_samples = L.gwasref_n_samples(self.h)
        self.level = level

    def add_codes(self, codes, first_row=0):
        codes = np.ascontiguousarray(codes, np.uint8)
        self.L.gwasref_add_rows_codes(self.h, first_row, codes.shape[0], _p(codes))

    def add_row_text(self, r, line: bytes):
        self.L.gwasref_add_row_text(self.h, r, line, len(line))

    def set_case_control(self, pheno):
        pheno = np.ascontiguousarray(pheno, np.uint8)
        self.L.gwasref_set_case_control(self.h, _p(pheno))

    @property
    def n_cases(self):
        return self.L.gwasref_n_cases(self.h)

    @property
    def n_controls(self):
        return self.L.gwasref_n_controls(self.h)

    def select(self):
        self.L.gwasref_select(self.h)

    def dist(self, r):
        out = np.zeros(4, np.uint32)
        self.L.gwasref_dist(self.h, r, _p(out))
        return out

    def cc_dist(self, r, mode):
        out = np.zeros(8, np.uint32)
        mi = np.zeros(1, MI_DTYPE)
        self.L.gwasref_cc_dist(self.h, r, mode, _p(out), _p(mi))
        return out, mi[0]

    def margins(self):
        out = np.zeros(self.n_snps, MI_DTYPE)
        self.L.gwasref_margins(self.h, _p(out))
        return out

    def pair_table(self, i, j, mode):
        ca = np.zeros(16, np.uint32)
        co = np.zeros(16, np.uint32)
        self.L.gwasref_pair_table(self.h, i, j, mode, _p(ca), _p(co))
        return ca, co

    def run(self, which, cap=1 << 26):
        names = {"computeBoost": 0, "select_cc_maf": 1, "inline_cc_maf": 2, "inline_maf_print": 3,
                 "genotype_dist_performance": 4, "ContingencyDebug": 5, "EpistasisDebug": 6}
        buf = C.create_string_buffer(cap)
        n = self.L.gwasref_run(self.h, names[which], buf, cap)
        if n >= cap:
            raise RuntimeError("output truncated")
        return buf.value.decode()

    def gtest(self, pi, pj):
        pi = np.ascontiguousarray(pi, np.uint32)
        pj = np.ascontiguousarray(pj, np.uint32)
        s = np.zeros(len(pi))
        z = np.zeros(len(pi))
        self.L.gwasref_gtest(self.h, len(pi), _p(pi), _p(pj), _p(s), _p(z))
        return s, z

    def pairwise_c(self, cs, ct):
        cs = np.ascontiguousarray(cs, np.int32).reshape(9)
        ct = np.ascontiguousarray(ct, np.int32).reshape(9)
        p = C.c_double()
        ll = self.L.gwasref_pairwise_c(_p(cs), _p(ct), C.byref(p))
        return float(ll), p.value

    def raw_row(self, r):
        n = self.L.gwasref_raw_row(self.h, r, None, 0)
        out = np.zeros(n, np.uint16)
        self.L.gwasref_raw_row(self.h, r, _p(out), n)
        return out

    def selected_row(self, r):
        geom = (C.c_int * 4)()
        n = self.L.gwasref_selected_row(self.h, r, None, 0, geom)
        out = np.zeros(n, np.uint16)
        self.L.gwasref_selected_row(self.h, r, _p(out), n, geom)
        return out, list(geom)

    def call_at(self, r, c):
        out = C.create_string_buffer(3)
        self.L.gwasref_call_at(self.h, r, c, out)
        return out.value.decode()

    def time_phase(self, phase, reps=1):
        return float(self.L.gwasref_time_phase(self.h, phase, reps))


class RefDev(Ref):
    """The same harness over the reference build whose GeneticData factory knows the device table: level 6 =
    libgwaspp_b200/binding/DeviceGenotypeTable (needs a GPU); levels 3-5 are the reference's own tables as in Ref."""
    _lib = None
    SO = REF_DEV_SO

    def __init__(self, n_snps=None, n_samples=None, level=6, **kw):
        super().__init__(n_snps, n_samples, level, **kw)


def parse_boost_output(text: str):
    """Parse computeBoost's result lines "%7d\\t%7d\\t%7d\\t%f\\t%f\\t%f\\t%f" (epistasis_func.cpp:497-505)."""
    hits = []
    located = None
    for line in text.splitlines():
        if line.startswith("Located "):
            located = int(line.split()[1])
        parts = line.split("\t")
        if len(parts) == 7:
            try:
                hits.append((int(parts[1]), int(parts[2]), float(parts[5]), float(parts[6])))
            except ValueError:
                pass
    return hits, located
