"""libgwaspp_b200 -- B200-native association hot path of libgwaspp behind a C-ABI.

This package is the thin Python plumbing over ``libgwasdev.so`` (hand-written sm_100a CUDA + the C-ABI
declared in ``include/gwasdev.h``). The product is the shared library; Python only loads it, moves
buffers and, for multi-GPU runs, gathers hits with ``torch.distributed``.

There is no CPU path: without the compiled extension, or without a CUDA device, every compute entry
point raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .maf_spectrum import MAF_SPECTRUM, PANELS  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
# GWASDEV_LIB selects another build of the same library (the -DGWASDEV_SWEEP build the tuning scripts under tools/ use)
LIB_PATH = os.environ.get("GWASDEV_LIB") or os.path.join(HERE, "libgwasdev.so")

# genetics/genotype/common_genotype.h:101-106 of the reference (192 bytes)
MI_DTYPE = np.dtype([("margins", "<u4", 4), ("cases", "<u4", 4), ("controls", "<u4", 4),
                     ("dMarginalEntropy", "<f8"), ("dMarginalEntropy_Y", "<f8"), ("dPbc", "<f8", 8), ("dPca", "<f8", 8)])
STATS_DTYPE = np.dtype([("maf_ref_case", "<f8"), ("maf_ref_ctrl", "<f8"), ("maf_pooled", "<f8"), ("df_genotypic", "<f8"),
                        ("chi2_allelic", "<f8"), ("p_allelic", "<f8"), ("chi2_genotypic", "<f8"), ("p_genotypic", "<f8")])
HIT_DTYPE = np.dtype([("i", "<u4"), ("j", "<u4"), ("stat", "<f8")])
COMPACT_DTYPE = np.dtype([("cases", "<u2", 4), ("controls", "<u2", 4), ("chi2_allelic", "<f4"), ("p_allelic", "<f4"),
                          ("chi2_genotypic", "<f4"), ("p_genotypic", "<f4")])
SIG_DTYPE = np.dtype([("snp", "<u4"), ("df_genotypic", "<u4"), ("maf_pooled", "<f8"), ("chi2_allelic", "<f8"), ("p_allelic", "<f8"),
                      ("chi2_genotypic", "<f8"), ("p_genotypic", "<f8")])
# gwasdev_ld_pair: one SNP pair of the LD calls (i < j), its pairwise-complete sample count and genotypic r, r^2
LD_PAIR_DTYPE = np.dtype([("i", "<u4"), ("j", "<u4"), ("n", "<u4"), ("reserved", "<u4"), ("r", "<f8"), ("r2", "<f8")])
assert LD_PAIR_DTYPE.itemsize == 32
assert MI_DTYPE.itemsize == 192 and STATS_DTYPE.itemsize == 64 and HIT_DTYPE.itemsize == 16
assert COMPACT_DTYPE.itemsize == 32 and SIG_DTYPE.itemsize == 48

# gwasdev_set_option keys (include/gwasdev.h)
OPT_SELECT_KERNEL, OPT_LANES_PER_ROW, OPT_INGEST_CHUNK, OPT_SCAN_PIECES, OPT_MASKED_SCAN, OPT_TRACE, OPT_FOUR_PLANE, \
    OPT_ROW_TOTALS, OPT_CAND_CAPACITY, OPT_CLASSIC_PLANES, OPT_PERM_OPERAND_BYTES, OPT_LD_OPERAND_BYTES = range(12)


class PairStats(C.Structure):
    _fields_ = [("pairs_tested", C.c_uint64), ("candidates", C.c_uint64), ("hits", C.c_uint64),
                ("word_cells", C.c_uint64), ("screen_ms", C.c_double), ("total_ms", C.c_double),
                ("tiles", C.c_uint32), ("tiles_nine_cell", C.c_uint32), ("engine", C.c_uint32), ("reserved", C.c_uint32)]


class PermStats(C.Structure):
    _fields_ = [("n_perm", C.c_uint64), ("snps", C.c_uint64), ("gemm_ms", C.c_double), ("total_ms", C.c_double),
                ("planes", C.c_uint32), ("built_operand", C.c_uint32)]


class LdStats(C.Structure):
    _fields_ = [("pairs_tested", C.c_uint64), ("pairs_kept", C.c_uint64), ("gemm_ms", C.c_double), ("total_ms", C.c_double),
                ("rows_per_snp", C.c_uint32), ("built_operand", C.c_uint32)]


class GwasDevError(RuntimeError):
    pass


_lib = None

# every symbol include/gwasdev.h declares (tests/test_abi.py checks header <-> library <-> this list)
ABI_SYMBOLS = [
    "gwasdev_last_error", "gwasdev_device_count", "gwasdev_create", "gwasdev_destroy", "gwasdev_set_stream",
    "gwasdev_launch_count", "gwasdev_synchronize", "gwasdev_plane_blocks", "gwasdev_pack_row_text",
    "gwasdev_put_rows", "gwasdev_get_rows", "gwasdev_call_at", "gwasdev_simulate", "gwasdev_simulate_phenotype",
    "gwasdev_select_case_control", "gwasdev_case_control_counts", "gwasdev_get_selected_rows",
    "gwasdev_marginal_scan", "gwasdev_last_scan_ms", "gwasdev_counts", "gwasdev_pair_tables",
    "gwasdev_pairwise_scan", "gwasdev_ksa", "gwasdev_ksa_screen_f32", "gwasdev_gtest", "gwasdev_pairwise_epi_test",
    "gwasdev_popc_peak", "gwasdev_hbm_read_peak", "gwasdev_set_pair_engine", "gwasdev_mma_tile_counts",
    "gwasdev_ksa_screen_mma_f32", "gwasdev_pack_row_text_block", "gwasdev_simulate_block", "gwasdev_marginal_accumulate",
    "gwasdev_marginal_finalize", "gwasdev_put_tped_text", "gwasdev_tped_dims", "gwasdev_load_tped", "gwasdev_put_bed",
    "gwasdev_bed_dims", "gwasdev_load_bed", "gwasdev_set_select_mode", "gwasdev_epi_pairs", "gwasdev_create_from_tped",
    "gwasdev_set_option", "gwasdev_set_stream_masks", "gwasdev_marginal_scan_compact", "gwasdev_pairwise_topk",
    "gwasdev_replicate", "gwasdev_pairwise_scan_multi", "gwasdev_shard_schedule", "gwasdev_i8_peak", "gwasdev_l2_read_peak", "gwasdev_gtest_multi", "gwasdev_is_compacted",
    "gwasdev_marginal_permute", "gwasdev_permutation_masks", "gwasdev_permutation_pvalues",
    "gwasdev_ld_window", "gwasdev_ld_pairs", "gwasdev_ld_prune", "gwasdev_fp64_div_probe",
]


def load_library():
    """dlopen libgwasdev.so; fails loudly when it has not been built (python -m libgwaspp_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GwasDevError(f"{LIB_PATH} is missing: build it with `python libgwaspp_b200/build.py` "
                           "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.gwasdev_last_error.restype = C.c_char_p
    L.gwasdev_launch_count.restype = u64
    L.gwasdev_plane_blocks.restype = u32
    L.gwasdev_plane_blocks.argtypes = [u32]
    L.gwasdev_last_scan_ms.restype = C.c_double
    L.gwasdev_last_scan_ms.argtypes = [vp]
    L.gwasdev_create.argtypes = [u64, u32, i32, C.POINTER(vp)]
    L.gwasdev_destroy.argtypes = [vp]
    L.gwasdev_destroy.restype = None
    L.gwasdev_set_stream.argtypes = [vp, vp]
    L.gwasdev_synchronize.argtypes = [vp]
    L.gwasdev_set_option.argtypes = [vp, i32, C.c_longlong]
    L.gwasdev_set_stream_masks.argtypes = [vp, vp, vp]
    L.gwasdev_is_compacted.argtypes = [vp]
    L.gwasdev_marginal_scan_compact.argtypes = [vp, u64, u64, vp, C.c_double, vp, u64, C.POINTER(u64), i32]
    L.gwasdev_pack_row_text.argtypes = [C.c_char_p, C.c_size_t, u32, vp]
    L.gwasdev_put_rows.argtypes = [vp, u64, u64, vp]
    L.gwasdev_get_rows.argtypes = [vp, u64, u64, vp]
    L.gwasdev_call_at.argtypes = [vp, u64, u32, C.c_char_p]
    L.gwasdev_simulate.argtypes = [vp, u64, vp, u32]
    L.gwasdev_simulate_phenotype.argtypes = [u64, u32, u32, vp]
    L.gwasdev_select_case_control.argtypes = [vp, vp, vp]
    L.gwasdev_case_control_counts.argtypes = [vp, C.POINTER(u32), C.POINTER(u32)]
    L.gwasdev_get_selected_rows.argtypes = [vp, u64, u64, vp]
    L.gwasdev_marginal_scan.argtypes = [vp, u64, u64, vp, vp, vp, i32]
    L.gwasdev_counts.argtypes = [vp, u64, u64, i32, vp]
    L.gwasdev_pair_tables.argtypes = [vp, u64, vp, vp, i32, vp]
    L.gwasdev_pairwise_scan.argtypes = [vp, C.c_double, u32, u32, vp, u64, C.POINTER(u64), C.POINTER(PairStats), i32]
    L.gwasdev_pairwise_topk.argtypes = [vp, C.c_double, u64, u32, u32, vp, C.POINTER(u64), C.POINTER(PairStats), i32]
    L.gwasdev_replicate.argtypes = [vp, i32, C.POINTER(vp)]
    L.gwasdev_pairwise_scan_multi.argtypes = [C.POINTER(vp), u32, C.c_double, u64, vp, u64, C.POINTER(u64), C.POINTER(PairStats), i32]
    L.gwasdev_shard_schedule.argtypes = [u64, u64, i32, u32, u32, vp, u64, C.POINTER(u64), C.POINTER(u64)]
    L.gwasdev_ksa.argtypes = [vp, u64, vp, vp, vp]
    L.gwasdev_ksa_screen_f32.argtypes = [vp, u64, vp, vp, vp]
    L.gwasdev_gtest.argtypes = [vp, u64, vp, vp, vp, vp]
    L.gwasdev_pack_row_text_block.argtypes = [C.c_char_p, C.c_size_t, u32, vp, C.POINTER(C.c_uint16)]
    L.gwasdev_simulate_block.argtypes = [vp, u64, vp, u32, u32, u32]
    L.gwasdev_marginal_accumulate.argtypes = [vp, u64, u64, vp, i32]
    L.gwasdev_marginal_finalize.argtypes = [i32, u64, vp, vp, vp, i32]
    L.gwasdev_set_pair_engine.argtypes = [vp, i32]
    L.gwasdev_set_select_mode.argtypes = [vp, i32]
    L.gwasdev_epi_pairs.argtypes = [vp, u64, vp, vp, i32, vp, vp]
    L.gwasdev_put_tped_text.argtypes = [vp, u64, vp, C.c_size_t, C.POINTER(u64), C.POINTER(C.c_size_t)]
    L.gwasdev_tped_dims.argtypes = [C.c_char_p, C.POINTER(u64), C.POINTER(u32)]
    L.gwasdev_load_tped.argtypes = [vp, C.c_char_p, u64, C.POINTER(u64)]
    L.gwasdev_create_from_tped.argtypes = [C.c_char_p, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u32)]
    L.gwasdev_put_bed.argtypes = [vp, u64, u64, vp, vp]
    L.gwasdev_bed_dims.argtypes = [C.c_char_p, u32, C.POINTER(u64)]
    L.gwasdev_load_bed.argtypes = [vp, C.c_char_p, vp, u64, C.POINTER(u64)]
    L.gwasdev_mma_tile_counts.argtypes = [vp, u32, u32, vp]
    L.gwasdev_ksa_screen_mma_f32.argtypes = [vp, u64, vp, vp, vp]
    L.gwasdev_pairwise_epi_test.argtypes = [i32, u64, vp, vp, vp, vp]
    L.gwasdev_popc_peak.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.gwasdev_i8_peak.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.gwasdev_gtest_multi.argtypes = [C.POINTER(vp), u32, u64, vp, vp, vp, vp]
    L.gwasdev_hbm_read_peak.argtypes = [i32, u64, C.POINTER(C.c_double)]
    L.gwasdev_l2_read_peak.argtypes = [i32, u64, u32, C.POINTER(C.c_double)]
    L.gwasdev_marginal_permute.argtypes = [vp, u64, u64, u64, u64, u64, vp, vp, vp, vp, C.POINTER(PermStats), i32]
    L.gwasdev_permutation_masks.argtypes = [u32, vp, vp, u64, u64, u64, vp]
    L.gwasdev_permutation_pvalues.argtypes = [u64, u64, vp, vp, vp, vp, vp]
    L.gwasdev_ld_window.argtypes = [vp, u64, u64, u32, vp, C.c_double, vp, u64, C.POINTER(u64), vp, C.POINTER(LdStats), i32]
    L.gwasdev_ld_pairs.argtypes = [vp, u64, vp, vp, vp, vp]
    L.gwasdev_ld_prune.argtypes = [u64, u64, u32, C.c_double, vp, u64, vp]
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        raise GwasDevError(f"{what}: status {rc}: {load_library().gwasdev_last_error().decode()}")


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if isinstance(a, int):
        return C.c_void_p(a)
    # torch tensor (host pinned or device): plain address
    return C.c_void_p(a.data_ptr())


def plane_blocks(n: int) -> int:
    return int(load_library().gwasdev_plane_blocks(int(n)))


def pack_row_text(line: bytes, n_samples: int) -> np.ndarray:
    """Host-side packer with GenoTable::addGenotypeRow semantics -> [hdr][plane1][plane2] uint16 blocks."""
    row = np.zeros(2 * plane_blocks(n_samples) + 1, np.uint16)
    _check(load_library().gwasdev_pack_row_text(line, len(line), n_samples, _ptr(row)), "gwasdev_pack_row_text")
    return row


def stream_masks(pheno) -> tuple[np.ndarray, np.ndarray]:
    """CaseControlSet stream masks (genetics/analyzable/case_control_set.cpp:77-150): bit c&15 of block c>>4.
    pheno: 1 = case, 0 = control, anything else = neither."""
    pheno = np.asarray(pheno)
    n = len(pheno)
    P = plane_blocks(n)
    bits = np.zeros(P * 16, np.uint8)
    ca, co = bits.copy(), bits.copy()
    ca[:n] = pheno == 1
    co[:n] = pheno == 0
    w = (1 << np.arange(16, dtype=np.uint32)).astype(np.uint32)
    return ((ca.reshape(P, 16) * w).sum(1).astype(np.uint16), (co.reshape(P, 16) * w).sum(1).astype(np.uint16))


def simulate_phenotype(seed: int, n_samples: int, n_case: int) -> np.ndarray:
    out = np.zeros(n_samples, np.uint8)
    _check(load_library().gwasdev_simulate_phenotype(seed, n_samples, n_case, _ptr(out)), "gwasdev_simulate_phenotype")
    return out


def permutation_masks(n_samples: int, case_mask, ctrl_mask, seed: int, first_perm: int, n_perm: int) -> np.ndarray:
    """Case masks (n_perm x P uint16 blocks) of permutations first_perm.. of a selection, as gwasdev_marginal_permute draws
    them on the device (host arithmetic)."""
    case_mask = np.ascontiguousarray(case_mask, np.uint16)
    ctrl_mask = np.ascontiguousarray(ctrl_mask, np.uint16)
    P = plane_blocks(n_samples)
    assert len(case_mask) == P and len(ctrl_mask) == P
    out = np.zeros((n_perm, P), np.uint16)
    _check(load_library().gwasdev_permutation_masks(n_samples, _ptr(case_mask), _ptr(ctrl_mask), seed, first_perm, n_perm, _ptr(out)),
           "gwasdev_permutation_masks")
    return out


def permutation_pvalues(observed, exceed, perm_max) -> tuple[np.ndarray, np.ndarray]:
    """EMP1 and EMP2 (max(T)), each (n_snps, 2) = (allelic, genotypic), from the observed statistics (STATS_DTYPE), the summed
    exceed counts (n_snps, 2) and the concatenated perm_max rows (n_perm, 3) of one or more marginal_permute calls."""
    observed = np.ascontiguousarray(observed, STATS_DTYPE)
    exceed = np.ascontiguousarray(exceed, np.uint32).reshape(-1, 2)
    perm_max = np.ascontiguousarray(perm_max, np.float64).reshape(-1, 3)
    n = len(observed)
    assert exceed.shape[0] == n
    emp1, emp2 = np.zeros((n, 2)), np.zeros((n, 2))
    _check(load_library().gwasdev_permutation_pvalues(n, perm_max.shape[0], _ptr(observed), _ptr(exceed), _ptr(perm_max),
                                                      _ptr(emp1), _ptr(emp2)), "gwasdev_permutation_pvalues")
    return emp1, emp2


def ld_prune(pairs, window: int, r2_threshold: float, snp_begin: int, snp_end: int) -> np.ndarray:
    """Greedy LD pruning of SNPs [snp_begin, snp_end) (host arithmetic, gwasdev_ld_prune): walking upwards, a SNP is kept unless
    an earlier kept SNP within `window` has r2 >= r2_threshold with it. pairs: LD_PAIR_DTYPE records sorted by (i, j), as
    GenoStore.ld_window returns them at a threshold at or below r2_threshold. Returns a bool keep mask over the range."""
    pairs = np.ascontiguousarray(pairs, LD_PAIR_DTYPE)
    keep = np.zeros(max(snp_end - snp_begin, 0), np.uint8)
    _check(load_library().gwasdev_ld_prune(snp_begin, snp_end, window, r2_threshold, _ptr(pairs), len(pairs), _ptr(keep)),
           "gwasdev_ld_prune")
    return keep.astype(bool)


def pack_row_text_block(line: bytes, n_samples: int, label_state: int = 0):
    """One sample block of a text row; returns (row, new label state) -- see gwasdev_pack_row_text_block."""
    P = plane_blocks(n_samples)
    row = np.zeros(2 * P + 1, np.uint16)
    st = C.c_uint16(label_state)
    _check(load_library().gwasdev_pack_row_text_block(line, len(line), n_samples, _ptr(row), C.byref(st)), "gwasdev_pack_row_text_block")
    return row, int(st.value)


def marginal_finalize(counts: np.ndarray, device: int = 0):
    """marginal_information + statistics from summed counts [n, 8] (host arrays)."""
    counts = np.ascontiguousarray(counts, np.uint32)
    n = counts.shape[0]
    mi, stats = np.zeros(n, MI_DTYPE), np.zeros(n, STATS_DTYPE)
    _check(load_library().gwasdev_marginal_finalize(device, n, _ptr(counts), _ptr(mi), _ptr(stats), 0), "gwasdev_marginal_finalize")
    return mi, stats


def popc_peak(device: int = 0) -> tuple[float, float]:
    r, mhz = C.c_double(), C.c_double()
    _check(load_library().gwasdev_popc_peak(device, C.byref(r), C.byref(mhz)), "gwasdev_popc_peak")
    return r.value, mhz.value


def i8_peak(device: int = 0) -> tuple[float, float]:
    """(burst, sustained) int8 tensor-core TOP/s of the screen kernel's own MMA instruction on resident operands."""
    a, b = C.c_double(), C.c_double()
    _check(load_library().gwasdev_i8_peak(device, C.byref(a), C.byref(b)), "gwasdev_i8_peak")
    return a.value, b.value


def l2_read_peak(device: int = 0, nbytes: int = 32 << 20, passes: int = 400) -> float:
    """GB/s the L2 delivers to the SMs: plain 128-bit loads past L1 over an L2-resident buffer, `passes` times in one launch."""
    r = C.c_double()
    _check(load_library().gwasdev_l2_read_peak(device, nbytes, passes, C.byref(r)), "gwasdev_l2_read_peak")
    return r.value


def hbm_read_peak(device: int = 0, nbytes: int = 1 << 31) -> float:
    r = C.c_double()
    _check(load_library().gwasdev_hbm_read_peak(device, nbytes, C.byref(r)), "gwasdev_hbm_read_peak")
    return r.value


def pairwise_epi_test(cs, ct, device: int = 0):
    cs = np.ascontiguousarray(cs, np.int32).reshape(-1, 9)
    ct = np.ascontiguousarray(ct, np.int32).reshape(-1, 9)
    ll = np.zeros(len(cs))
    p = np.zeros(len(cs))
    _check(load_library().gwasdev_pairwise_epi_test(device, len(cs), _ptr(cs), _ptr(ct), _ptr(ll), _ptr(p)),
           "gwasdev_pairwise_epi_test")
    return ll, p


def fp64_div_probe(a, b, device: int = 0):
    """The G-test's branch-free fp64 division next to __ddiv_rn on operand arrays a, b (gwasdev_fp64_div_probe):
    (q_fast, q_rn, bad)."""
    a = np.ascontiguousarray(a, np.float64).ravel()
    b = np.ascontiguousarray(b, np.float64).ravel()
    assert a.shape == b.shape
    q_fast, q_rn, bad = np.zeros(len(a)), np.zeros(len(a)), np.zeros(len(a), np.uint8)
    f = load_library().gwasdev_fp64_div_probe
    f.argtypes = [C.c_int, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    _check(f(device, len(a), _ptr(a), _ptr(b), _ptr(q_fast), _ptr(q_rn), _ptr(bad)), "gwasdev_fp64_div_probe")
    return q_fast, q_rn, bad.astype(bool)


def tped_dims(path: str) -> tuple[int, int]:
    """(non-blank lines, genotype columns of the first line) of a TPED file, plain or .gz."""
    rows, cols = C.c_uint64(), C.c_uint32()
    _check(load_library().gwasdev_tped_dims(os.fsencode(path), C.byref(rows), C.byref(cols)), "gwasdev_tped_dims")
    return int(rows.value), int(cols.value)


def bed_dims(path: str, n_samples: int) -> int:
    rows = C.c_uint64()
    _check(load_library().gwasdev_bed_dims(os.fsencode(path), n_samples, C.byref(rows)), "gwasdev_bed_dims")
    return int(rows.value)


def launch_count() -> int:
    return int(load_library().gwasdev_launch_count())


def gtest_multi(stores, pi, pj):
    """computeGTest on the given pairs, split over the stores' devices (one host thread each inside the library)."""
    L = load_library()
    pi = np.ascontiguousarray(pi, np.uint32).ravel()
    pj = np.ascontiguousarray(pj, np.uint32).ravel()
    s, z = np.zeros(len(pi)), np.zeros(len(pi))
    arr = (C.c_void_p * len(stores))(*[st.h for st in stores])
    _check(L.gwasdev_gtest_multi(arr, len(stores), len(pi), _ptr(pi), _ptr(pj), _ptr(s), _ptr(z)), "gwasdev_gtest_multi")
    return s, z


def shard_schedule(n_snps: int, shard: int, n_shards: int, engine: int = 2, n_samples: int = 10_000):
    """Tile pairs ((I, J) SNP-block indices, [n, 2]) the shard owns in the screen's schedule, and the pairs they cover: the
    library's own enumeration (host arithmetic, no device needed). engine 2: tensor cores (128-SNP blocks; the table's number
    of individuals n_samples decides how many A-blocks form an L2 band), 1: AND+POPC (64-SNP blocks)."""
    L = load_library()
    nt, npairs = C.c_uint64(), C.c_uint64()
    _check(L.gwasdev_shard_schedule(n_snps, n_samples, engine, shard, n_shards, None, 0, C.byref(nt), C.byref(npairs)), "gwasdev_shard_schedule")
    tiles = np.zeros((nt.value, 2), np.uint32)
    _check(L.gwasdev_shard_schedule(n_snps, n_samples, engine, shard, n_shards, _ptr(tiles), nt.value, C.byref(nt), C.byref(npairs)), "gwasdev_shard_schedule")
    return tiles, int(npairs.value)


def pairwise_scan_multi(stores, threshold: float = 30.0, top_k: int = 0, capacity: int = 1 << 20, gather: str = "nccl"):
    """One process, len(stores) devices: every store runs its shard of the tile-pair schedule on its own host thread
    inside the library and the hit records are combined over NVLink (NCCL all-gather, or peer copies with gather="peer").
    Returns (hits[HIT_DTYPE] sorted by (i, j), [PairStats per shard])."""
    L = load_library()
    n = len(stores)
    arr = (C.c_void_p * n)(*[st.h for st in stores])
    stats = (PairStats * n)()
    cap = top_k if top_k else capacity
    hits = np.zeros(cap, HIT_DTYPE)
    got = C.c_uint64()
    rc = L.gwasdev_pairwise_scan_multi(arr, n, threshold, top_k, _ptr(hits), cap, C.byref(got), stats, {"nccl": 0, "peer": 1}[gather])
    if rc == 4 and not top_k:   # GWASDEV_EOVERFLOW: grow and retry once
        return pairwise_scan_multi(stores, threshold, top_k, int(got.value), gather)
    _check(rc, "gwasdev_pairwise_scan_multi")
    return hits[: got.value].copy(), list(stats)


class GenoStore:
    """Device-resident genotype store: the handle behind the reference's GenoTable for this path."""

    def __init__(self, n_snps: int, n_samples: int, device: int = 0):
        self.L = load_library()
        self.h = C.c_void_p()
        _check(self.L.gwasdev_create(n_snps, n_samples, device, C.byref(self.h)), "gwasdev_create")
        self.n_snps, self.n_samples, self.device = n_snps, n_samples, device
        self.P = plane_blocks(n_samples)
        self.n_case = self.n_ctrl = None

    @classmethod
    def from_tped(cls, path: str, device: int = 0) -> "GenoStore":
        """Table sized from and loaded with a TPED file (plain: one pass; .gz: counting pass first), parsed on the device."""
        self = cls.__new__(cls)
        self.L = load_library()
        self.h = C.c_void_p()
        rows, cols = C.c_uint64(), C.c_uint32()
        _check(self.L.gwasdev_create_from_tped(os.fsencode(path), device, C.byref(self.h), C.byref(rows), C.byref(cols)),
               "gwasdev_create_from_tped")
        self.n_snps, self.n_samples, self.device = int(rows.value), int(cols.value), device
        self.P = plane_blocks(self.n_samples)
        self.n_case = self.n_ctrl = None
        return self

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.L.gwasdev_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- loading
    def set_stream(self, cuda_stream: int):
        _check(self.L.gwasdev_set_stream(self.h, C.c_void_p(cuda_stream)), "gwasdev_set_stream")

    def synchronize(self):
        _check(self.L.gwasdev_synchronize(self.h), "gwasdev_synchronize")

    def set_option(self, option: int, value: int):
        """Explicit knob of this store (OPT_* constants; include/gwasdev.h). The library reads no environment variables."""
        _check(self.L.gwasdev_set_option(self.h, option, value), "gwasdev_set_option")

    def put_rows(self, rows: np.ndarray, first_row: int = 0):
        rows = np.ascontiguousarray(rows, np.uint16)
        assert rows.ndim == 2 and rows.shape[1] == 2 * self.P + 1, rows.shape
        _check(self.L.gwasdev_put_rows(self.h, first_row, rows.shape[0], _ptr(rows)), "gwasdev_put_rows")

    def put_text_rows(self, lines, first_row: int = 0):
        self.put_rows(np.stack([pack_row_text(l, self.n_samples) for l in lines]), first_row)

    def put_tped_text(self, text: bytes, first_row: int = 0) -> tuple[int, int]:
        """TPED lines parsed, labelled and packed on the device; returns (rows written, bytes consumed)."""
        rows, used = C.c_uint64(), C.c_size_t()
        buf = np.frombuffer(text, np.uint8) if len(text) else np.zeros(1, np.uint8)
        _check(self.L.gwasdev_put_tped_text(self.h, first_row, _ptr(buf), len(text), C.byref(rows), C.byref(used)), "gwasdev_put_tped_text")
        return int(rows.value), int(used.value)

    def load_tped(self, path: str, first_row: int = 0) -> int:
        rows = C.c_uint64()
        _check(self.L.gwasdev_load_tped(self.h, os.fsencode(path), first_row, C.byref(rows)), "gwasdev_load_tped")
        return int(rows.value)

    def put_bed(self, bed: np.ndarray, alleles: np.ndarray | None = None, first_row: int = 0):
        bed = np.ascontiguousarray(bed, np.uint8)
        assert bed.ndim == 2 and bed.shape[1] == (self.n_samples + 3) // 4, bed.shape
        if alleles is not None:
            alleles = np.ascontiguousarray(alleles, np.uint8)
            assert alleles.shape == (bed.shape[0], 2)
        _check(self.L.gwasdev_put_bed(self.h, first_row, bed.shape[0], _ptr(bed), _ptr(alleles)), "gwasdev_put_bed")

    def load_bed(self, path: str, alleles: np.ndarray | None = None, first_row: int = 0) -> int:
        rows = C.c_uint64()
        if alleles is not None:
            alleles = np.ascontiguousarray(alleles, np.uint8)
        _check(self.L.gwasdev_load_bed(self.h, os.fsencode(path), _ptr(alleles), first_row, C.byref(rows)), "gwasdev_load_bed")
        return int(rows.value)

    def get_rows(self, first_row: int = 0, n_rows: int | None = None) -> np.ndarray:
        n_rows = self.n_snps - first_row if n_rows is None else n_rows
        out = np.zeros((n_rows, 2 * self.P + 1), np.uint16)
        _check(self.L.gwasdev_get_rows(self.h, first_row, n_rows, _ptr(out)), "gwasdev_get_rows")
        return out

    def call_at(self, row: int, col: int) -> str:
        buf = C.create_string_buffer(3)
        _check(self.L.gwasdev_call_at(self.h, row, col, buf), "gwasdev_call_at")
        return buf.value.decode()

    def simulate(self, seed: int, panel: str = "affy6", missing_rate: float = 0.0):
        bins = np.asarray(MAF_SPECTRUM[panel], np.uint32)
        q = int(missing_rate * 4294967296.0) & 0xFFFFFFFF
        _check(self.L.gwasdev_simulate(self.h, seed, _ptr(bins), q), "gwasdev_simulate")

    def simulate_block(self, seed: int, first_sample: int, n_total_samples: int, panel: str = "affy6", missing_rate: float = 0.0):
        """This store = samples [first_sample, first_sample + n_samples) of the whole-cohort table of gwasdev_simulate."""
        bins = np.asarray(MAF_SPECTRUM[panel], np.uint32)
        q = int(missing_rate * 4294967296.0) & 0xFFFFFFFF
        _check(self.L.gwasdev_simulate_block(self.h, seed, _ptr(bins), q, first_sample, n_total_samples), "gwasdev_simulate_block")

    # -- case/control
    def set_select_mode(self, eager: bool):
        """eager: build the compacted rows inside select_case_control; default lazy (see include/gwasdev.h)."""
        _check(self.L.gwasdev_set_select_mode(self.h, int(bool(eager))), "gwasdev_set_select_mode")

    def select_case_control(self, pheno=None, *, case_mask=None, ctrl_mask=None):
        if pheno is not None:
            case_mask, ctrl_mask = stream_masks(pheno)
        case_mask = np.ascontiguousarray(case_mask, np.uint16)
        ctrl_mask = np.ascontiguousarray(ctrl_mask, np.uint16)
        assert len(case_mask) == self.P and len(ctrl_mask) == self.P
        _check(self.L.gwasdev_select_case_control(self.h, _ptr(case_mask), _ptr(ctrl_mask)), "gwasdev_select_case_control")
        a, b = C.c_uint32(), C.c_uint32()
        _check(self.L.gwasdev_case_control_counts(self.h, C.byref(a), C.byref(b)), "gwasdev_case_control_counts")
        self.n_case, self.n_ctrl = a.value, b.value

    def is_compacted(self) -> bool:
        """True when kernel K0 has built the compacted rows of the current selection."""
        return self.L.gwasdev_is_compacted(self.h) == 1

    def set_stream_masks(self, pheno=None, *, case_mask=None, ctrl_mask=None):
        """Masks of the mask-on-the-fly overloads only (counts mode 1, pair_tables mode 1); the selection stays as it is."""
        if pheno is not None:
            case_mask, ctrl_mask = stream_masks(pheno)
        case_mask = np.ascontiguousarray(case_mask, np.uint16)
        ctrl_mask = np.ascontiguousarray(ctrl_mask, np.uint16)
        assert len(case_mask) == self.P and len(ctrl_mask) == self.P
        _check(self.L.gwasdev_set_stream_masks(self.h, _ptr(case_mask), _ptr(ctrl_mask)), "gwasdev_set_stream_masks")

    def get_selected_rows(self, first_row: int = 0, n_rows: int | None = None) -> np.ndarray:
        n_rows = self.n_snps - first_row if n_rows is None else n_rows
        S = 2 * (plane_blocks(self.n_case) + plane_blocks(self.n_ctrl))
        out = np.zeros((n_rows, S), np.uint16)
        _check(self.L.gwasdev_get_selected_rows(self.h, first_row, n_rows, _ptr(out)), "gwasdev_get_selected_rows")
        return out

    # -- marginal scan
    def marginal_scan(self, snp_begin: int = 0, snp_end: int | None = None, *, counts=True, mi=True, stats=True):
        """Host-buffer call (the e2e path): returns dict of numpy arrays."""
        snp_end = self.n_snps if snp_end is None else snp_end
        n = snp_end - snp_begin
        out = {}
        if counts:
            out["counts"] = np.zeros((n, 8), np.uint32)
        if mi:
            out["mi"] = np.zeros(n, MI_DTYPE)
        if stats:
            out["stats"] = np.zeros(n, STATS_DTYPE)
        _check(self.L.gwasdev_marginal_scan(self.h, snp_begin, snp_end, _ptr(out.get("counts")), _ptr(out.get("mi")),
                                            _ptr(out.get("stats")), 0), "gwasdev_marginal_scan")
        return out

    def marginal_permute(self, n_perm: int, seed: int = 0, first_perm: int = 0, case_masks=None, snp_begin: int = 0,
                         snp_end: int | None = None, perm_stats: bool = False):
        """Label-permutation test of the current selection (gwasdev_marginal_permute): dict with exceed (n_snps, 2),
        perm_max (n_perm, 3), perm_stats (n_perm, n_snps, 2) when asked for, and stats (PermStats). case_masks: (n_perm, P)
        uint16 case masks instead of the device draws."""
        snp_end = self.n_snps if snp_end is None else snp_end
        n = snp_end - snp_begin
        if case_masks is not None:
            case_masks = np.ascontiguousarray(case_masks, np.uint16).reshape(n_perm, self.P)
        out = {"exceed": np.zeros((n, 2), np.uint32), "perm_max": np.zeros((n_perm, 3), np.float64)}
        st = PermStats()
        if perm_stats:
            import torch
            dev = torch.empty((n_perm, n, 2), dtype=torch.float64, device=f"cuda:{self.device}")
            ex = torch.empty((n, 2), dtype=torch.int32, device=dev.device)
            pm = torch.empty((n_perm, 3), dtype=torch.float64, device=dev.device)
            _check(self.L.gwasdev_marginal_permute(self.h, snp_begin, snp_end, seed, first_perm, n_perm, _ptr(case_masks),
                                                   _ptr(ex), _ptr(pm), _ptr(dev), C.byref(st), 1), "gwasdev_marginal_permute")
            torch.cuda.synchronize(dev.device)
            out["exceed"], out["perm_max"] = ex.cpu().numpy().view(np.uint32), pm.cpu().numpy()
            out["perm_stats"] = dev.cpu().numpy()
        else:
            _check(self.L.gwasdev_marginal_permute(self.h, snp_begin, snp_end, seed, first_perm, n_perm, _ptr(case_masks),
                                                   _ptr(out["exceed"]), _ptr(out["perm_max"]), None, C.byref(st), 0),
                   "gwasdev_marginal_permute")
        out["stats"] = st
        return out

    def marginal_scan_into(self, snp_begin, snp_end, counts=None, mi=None, stats=None, on_device=True):
        """Raw-pointer call: buffers are torch tensors / numpy arrays / int addresses (device when on_device)."""
        _check(self.L.gwasdev_marginal_scan(self.h, snp_begin, snp_end, _ptr(counts), _ptr(mi), _ptr(stats),
                                            1 if on_device else 0), "gwasdev_marginal_scan")

    def marginal_scan_compact(self, snp_begin: int = 0, snp_end: int | None = None, *, records=True, p_threshold: float = 0.0,
                              sig_capacity: int = 1 << 16):
        """Host-buffer call with compact outputs: (records[COMPACT_DTYPE] or None, significant[SIG_DTYPE] sorted by SNP)."""
        snp_end = self.n_snps if snp_end is None else snp_end
        n = snp_end - snp_begin
        rec = np.zeros(n, COMPACT_DTYPE) if records else None
        sig = np.zeros(sig_capacity, SIG_DTYPE) if p_threshold > 0 else None
        n_sig = C.c_uint64()
        rc = self.L.gwasdev_marginal_scan_compact(self.h, snp_begin, snp_end, _ptr(rec), p_threshold, _ptr(sig), sig_capacity if sig is not None else 0,
                                                  C.byref(n_sig), 0)
        if rc == 4:   # GWASDEV_EOVERFLOW: grow and retry once
            return self.marginal_scan_compact(snp_begin, snp_end, records=records, p_threshold=p_threshold, sig_capacity=int(n_sig.value))
        _check(rc, "gwasdev_marginal_scan_compact")
        return rec, (sig[: n_sig.value].copy() if sig is not None else None)

    def marginal_scan_compact_into(self, snp_begin, snp_end, records=None, p_threshold=0.0, sig=None, sig_capacity=0, on_device=True) -> int:
        """Raw-pointer call of gwasdev_marginal_scan_compact; returns the number of significant SNPs."""
        n_sig = C.c_uint64()
        _check(self.L.gwasdev_marginal_scan_compact(self.h, snp_begin, snp_end, _ptr(records), p_threshold, _ptr(sig), sig_capacity, C.byref(n_sig),
                                                    1 if on_device else 0), "gwasdev_marginal_scan_compact")
        return int(n_sig.value)

    def marginal_accumulate(self, acc, snp_begin: int = 0, snp_end: int | None = None, on_device: bool = False):
        """acc[8 per SNP] += this sample block's case/control genotype counts (streaming in sample blocks)."""
        snp_end = self.n_snps if snp_end is None else snp_end
        _check(self.L.gwasdev_marginal_accumulate(self.h, snp_begin, snp_end, _ptr(acc), 1 if on_device else 0),
               "gwasdev_marginal_accumulate")

    def last_scan_ms(self) -> float:
        return float(self.L.gwasdev_last_scan_ms(self.h))

    def counts(self, mode: int, snp_begin: int = 0, snp_end: int | None = None) -> np.ndarray:
        snp_end = self.n_snps if snp_end is None else snp_end
        out = np.zeros((snp_end - snp_begin, 4 if mode == 0 else 8), np.uint32)
        _check(self.L.gwasdev_counts(self.h, snp_begin, snp_end, mode, _ptr(out)), "gwasdev_counts")
        return out

    # -- linkage disequilibrium
    def _sample_blocks(self, sample_mask):
        """None, P uint16 blocks (bit c&15 of block c>>4), or a bool per sample."""
        if sample_mask is None:
            return None
        m = np.asarray(sample_mask)
        if m.dtype == bool:
            assert m.shape == (self.n_samples,), m.shape
            bits = np.zeros(self.P * 16, np.uint8)
            bits[: self.n_samples] = m
            return np.packbits(bits, bitorder="little").view(np.uint16).copy()
        m = np.ascontiguousarray(m, np.uint16)
        assert m.shape == (self.P,), m.shape
        return m

    def ld_window(self, window: int, r2_threshold: float = 0.2, snp_begin: int = 0, snp_end: int | None = None, sample_mask=None,
                  band: bool = False, capacity: int = 1 << 20, pairs: bool = True):
        """Genotypic r^2 of every pair snp_begin <= i < j < snp_end with j - i <= window (gwasdev_ld_window). Returns (pairs
        [LD_PAIR_DTYPE] with r2 >= r2_threshold sorted by (i, j), or None; band (n, window) float32 of r2 or None; LdStats).
        The list grows to the size needed when `capacity` is too small."""
        snp_end = self.n_snps if snp_end is None else snp_end
        mask = self._sample_blocks(sample_mask)
        out = np.zeros(capacity, LD_PAIR_DTYPE) if pairs else None
        b = np.zeros((max(snp_end - snp_begin, 0), window), np.float32) if band else None
        st, got = LdStats(), C.c_uint64()
        rc = self.L.gwasdev_ld_window(self.h, snp_begin, snp_end, window, _ptr(mask), r2_threshold, _ptr(out), capacity if pairs else 0,
                                      C.byref(got), _ptr(b), C.byref(st), 0)
        if rc == 4 and pairs:   # GWASDEV_EOVERFLOW: re-run with the size needed
            return self.ld_window(window, r2_threshold, snp_begin, snp_end, sample_mask, band, int(got.value), pairs)
        _check(rc, "gwasdev_ld_window")
        return (out[: got.value].copy() if pairs else None), b, st

    def ld_pairs(self, pi, pj, sample_mask=None) -> np.ndarray:
        """Genotypic r^2 of given pairs at any distance (i != j, either order): LD_PAIR_DTYPE records with i < j."""
        pi, pj = self._pairs(pi, pj)
        out = np.zeros(len(pi), LD_PAIR_DTYPE)
        _check(self.L.gwasdev_ld_pairs(self.h, len(pi), _ptr(pi), _ptr(pj), _ptr(self._sample_blocks(sample_mask)), _ptr(out)),
               "gwasdev_ld_pairs")
        return out

    def ld_prune(self, window: int, r2_threshold: float, snp_begin: int = 0, snp_end: int | None = None, sample_mask=None) -> np.ndarray:
        """Greedy LD pruning (see ld_prune): ld_window at r2_threshold, then the host rule. Returns a bool keep mask over the range."""
        snp_end = self.n_snps if snp_end is None else snp_end
        pairs, _, _ = self.ld_window(window, r2_threshold, snp_begin, snp_end, sample_mask)
        return ld_prune(pairs, window, r2_threshold, snp_begin, snp_end)

    # -- pairs
    def _pairs(self, pi, pj):
        pi = np.ascontiguousarray(pi, np.uint32).ravel()
        pj = np.ascontiguousarray(pj, np.uint32).ravel()
        assert len(pi) == len(pj)
        return pi, pj

    def pair_tables(self, pi, pj, mode: int = 3) -> np.ndarray:
        pi, pj = self._pairs(pi, pj)
        out = np.zeros((len(pi), 32), np.uint32)
        _check(self.L.gwasdev_pair_tables(self.h, len(pi), _ptr(pi), _ptr(pj), mode, _ptr(out)), "gwasdev_pair_tables")
        return out

    def ksa(self, pi, pj) -> np.ndarray:
        pi, pj = self._pairs(pi, pj)
        out = np.zeros(len(pi))
        _check(self.L.gwasdev_ksa(self.h, len(pi), _ptr(pi), _ptr(pj), _ptr(out)), "gwasdev_ksa")
        return out

    def ksa_screen_f32(self, pi, pj) -> np.ndarray:
        pi, pj = self._pairs(pi, pj)
        out = np.zeros(len(pi), np.float32)
        _check(self.L.gwasdev_ksa_screen_f32(self.h, len(pi), _ptr(pi), _ptr(pj), _ptr(out)), "gwasdev_ksa_screen_f32")
        return out

    def ksa_screen_mma_f32(self, pi, pj) -> np.ndarray:
        """[n, 2]: fp32 statistic of the tensor-core epilogue and its upper-bound pre-filter value."""
        pi, pj = self._pairs(pi, pj)
        out = np.zeros((len(pi), 2), np.float32)
        _check(self.L.gwasdev_ksa_screen_mma_f32(self.h, len(pi), _ptr(pi), _ptr(pj), _ptr(out)), "gwasdev_ksa_screen_mma_f32")
        return out

    def set_pair_engine(self, engine: int):
        """0 auto, 1 AND+POPC tiles, 2 tensor cores (tcgen05)."""
        _check(self.L.gwasdev_set_pair_engine(self.h, engine), "gwasdev_set_pair_engine")

    def mma_tile_counts(self, I: int, J: int) -> np.ndarray:
        """Raw corner counts of tile pair (A-block I of 64 SNPs, B-block J of 128 SNPs): [64, 128, 2 classes, 4 cells]."""
        out = np.zeros((64, 128, 2, 4), np.uint32)
        _check(self.L.gwasdev_mma_tile_counts(self.h, I, J, _ptr(out)), "gwasdev_mma_tile_counts")
        return out

    def gtest(self, pi, pj):
        pi, pj = self._pairs(pi, pj)
        s, z = np.zeros(len(pi)), np.zeros(len(pi))
        _check(self.L.gwasdev_gtest(self.h, len(pi), _ptr(pi), _ptr(pj), _ptr(s), _ptr(z)), "gwasdev_gtest")
        return s, z

    def epi_pairs(self, pi, pj, mode: int = 1):
        """EpistasisPerformance's pair body: tables by overload `mode`, pairwise.c likelihood-ratio test, pchisq(ll, 4)."""
        pi, pj = self._pairs(pi, pj)
        ll, p = np.zeros(len(pi)), np.zeros(len(pi))
        _check(self.L.gwasdev_epi_pairs(self.h, len(pi), _ptr(pi), _ptr(pj), mode, _ptr(ll), _ptr(p)), "gwasdev_epi_pairs")
        return ll, p

    def pairwise_topk(self, top_k: int, threshold: float = 30.0, shard: int = 0, n_shards: int = 1, hits=None, on_device: bool = False):
        """The top_k pairs with the largest statistic above `threshold`, sorted by (i, j): (hits, PairStats)."""
        st = PairStats()
        n = C.c_uint64()
        own = hits is None
        if own:
            assert not on_device
            hits = np.zeros(top_k, HIT_DTYPE)
        _check(self.L.gwasdev_pairwise_topk(self.h, threshold, top_k, shard, n_shards, _ptr(hits), C.byref(n), C.byref(st),
                                            1 if on_device else 0), "gwasdev_pairwise_topk")
        return (hits[: n.value].copy() if own else int(n.value)), st

    def replicate(self, device: int) -> "GenoStore":
        """Copy of this store (table, options, selection) on another device of the same process."""
        other = GenoStore.__new__(GenoStore)
        other.L = self.L
        other.h = C.c_void_p()
        _check(self.L.gwasdev_replicate(self.h, device, C.byref(other.h)), "gwasdev_replicate")
        other.n_snps, other.n_samples, other.device, other.P = self.n_snps, self.n_samples, device, self.P
        other.n_case, other.n_ctrl = self.n_case, self.n_ctrl
        return other

    def pairwise_scan(self, threshold: float = 30.0, shard: int = 0, n_shards: int = 1, capacity: int = 1 << 20,
                      hits=None, on_device: bool = False):
        """computeBoost's pre-screen. Returns (hits[HIT_DTYPE] sorted by (i, j), PairStats).
        With on_device=True, `hits` must be a device buffer of capacity*16 bytes (torch tensor or address)."""
        st = PairStats()
        n = C.c_uint64()
        own = hits is None
        if own:
            assert not on_device
            hits = np.zeros(capacity, HIT_DTYPE)
        rc = self.L.gwasdev_pairwise_scan(self.h, threshold, shard, n_shards, _ptr(hits), capacity, C.byref(n),
                                          C.byref(st), 1 if on_device else 0)
        if rc == 4 and own:   # GWASDEV_EOVERFLOW: grow and retry once
            return self.pairwise_scan(threshold, shard, n_shards, int(n.value), None, False)
        _check(rc, "gwasdev_pairwise_scan")
        return (hits[: n.value].copy() if own else int(n.value)), st
