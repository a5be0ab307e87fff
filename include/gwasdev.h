/*
 * gwasdev.h -- C-ABI of the B200-native association hot path (libgwasdev.so).
 *
 * Drop-in boundary for libgwaspp's case/control association path: everything the reference's
 * GenoTable virtuals and test-class functions do for that path, as plain C entry points with plain
 * pointers and sizes. No C++ types, exceptions or torch types cross this boundary. All functions
 * return 0 on success and a non-zero status otherwise; gwasdev_last_error() gives the message
 * (the reference's convention on this path is assert/abort; the C++ adapter in
 * libgwaspp_b200/host asserts on non-zero to mimic it).
 *
 * Citations are relative to the reference tree's src/libgwaspp/ unless stated otherwise.
 * There is no CPU fallback: every compute entry point fails with GWASDEV_ENODEVICE without a GPU.
 */
#ifndef GWASDEV_H
#define GWASDEV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GWASDEV_API __attribute__((visibility("default")))
#else
#define GWASDEV_API
#endif

#define GWASDEV_OK 0
#define GWASDEV_EINVAL 1     /* bad argument / call order */
#define GWASDEV_ENODEVICE 2  /* no CUDA device, or a CUDA runtime error */
#define GWASDEV_ENOMEM 3
#define GWASDEV_EOVERFLOW 4  /* caller's hit buffer too small; *n_hits holds the needed size */

typedef struct gwasdev_store gwasdev_store;   /* device-resident genotype store, opaque */

/* genetics/genotype/common_genotype.h:101-106 (marginal_information), byte-compatible: 192 bytes.
 * frequency_table order is {aa, ab, bb, xx} (common_genotype.h:67-75). */
typedef struct {
    uint32_t margins[4], cases[4], controls[4];
    double dMarginalEntropy, dMarginalEntropy_Y;
    double dPbc[8];   /* P(genotype | class): cases[4] then controls[4] */
    double dPca[8];   /* P(class | genotype): cases[4] then controls[4] */
} gwasdev_marginal_information;

/* Per-SNP association statistics written by the marginal scan (64 bytes).
 * maf_ref_* is MinorAlleleFrequency() of algorithms/maf_func.h:46-54 (which returns max(f, 1-f));
 * maf_pooled is the true minor-allele frequency over called genotypes of cases+controls.
 * The chi-square tests have no counterpart in the reference; they are specified in DESIGN.md. */
typedef struct {
    double maf_ref_case, maf_ref_ctrl, maf_pooled, df_genotypic;
    double chi2_allelic, p_allelic, chi2_genotypic, p_genotypic;
} gwasdev_snp_stats;

/* Compact per-SNP result for host consumers (32 bytes instead of the 96 of counts + gwasdev_snp_stats): the eight genotype
 * counts as 16-bit integers (both classes below 65 536 samples) and the four test results in fp32 (north star: fp32
 * p-values, 1e-5 relative on significant hits). p-values below the fp32 range flush towards 0; such SNPs are in the
 * significant list of gwasdev_marginal_scan_compact with all their statistics in fp64. */
typedef struct {
    uint16_t cases[4], controls[4];   /* {aa, ab, bb, xx} per class */
    float chi2_allelic, p_allelic, chi2_genotypic, p_genotypic;
} gwasdev_snp_compact;

/* One SNP whose allelic or genotypic p-value is below the caller's threshold (48 bytes). */
typedef struct {
    uint32_t snp, df_genotypic;
    double maf_pooled, chi2_allelic, p_allelic, chi2_genotypic, p_genotypic;
} gwasdev_sig_snp;

/* One screened SNP pair: SNPInteractionPair of algorithms/epistasis_func.h:59-60. */
typedef struct {
    uint32_t i, j;   /* i < j, table row indices */
    double stat;     /* KSA screening statistic (epistasis_func.cpp:424-470) */
} gwasdev_hit;

typedef struct {
    uint64_t pairs_tested;   /* pairs (i<j) this call covered */
    uint64_t candidates;     /* pairs kept by the fp32 screen (threshold - margin) before exact re-scoring */
    uint64_t hits;           /* pairs whose fp64 statistic exceeds the threshold */
    uint64_t word_cells;     /* algorithmic 32-bit AND+POPC word-cells = pairs * 4 * (ceil(nca/32)+ceil(nco/32)) */
    double screen_ms;        /* device time of the tiled screen kernel (CUDA events) */
    double total_ms;         /* device time of the whole call incl. re-scoring */
    uint32_t tiles, tiles_nine_cell;
    uint32_t engine;         /* engine used for the tiles without missing calls: 1 AND+POPC, 2 tensor cores */
    uint32_t reserved;
} gwasdev_pair_stats;

/* ---- lifecycle ------------------------------------------------------------------------------ */
GWASDEV_API const char *gwasdev_last_error(void);
GWASDEV_API int gwasdev_device_count(void);
/* Replaces `new CompressedGenotypeTable5(markers, individs)` (genetics/genetic_data.cpp:60-79,
 * genotype/compressed_genotype_table5.cpp:34-153): allocates the raw store in HBM on `device`. */
GWASDEV_API int gwasdev_create(uint64_t n_snps, uint32_t n_samples, int device, gwasdev_store **out);
GWASDEV_API void gwasdev_destroy(gwasdev_store *s);
/* Run this store's kernels on a caller-owned CUDA stream (cudaStream_t as void*); default is stream 0. */
GWASDEV_API int gwasdev_set_stream(gwasdev_store *s, void *cuda_stream);
/* Kernels launched by this library in this process so far (bench.py's gpu_launches). */
GWASDEV_API uint64_t gwasdev_launch_count(void);
GWASDEV_API int gwasdev_synchronize(gwasdev_store *s);

/* Explicit knobs of a store. The library reads no environment variables: everything that changes which kernel runs is
 * set here, per store, and defaults (0) are the measured best. Used by the tests to force the alternative code paths
 * on small fixtures and by the timing scripts under tools/. */
#define GWASDEV_OPT_SELECT_KERNEL 0  /* K0: 0 auto (register form up to 32 768 samples), 1 table-driven form */
#define GWASDEV_OPT_LANES_PER_ROW 1  /* K1 / K1': 0 auto, or 8 / 16 / 32 lanes cooperating on one row */
#define GWASDEV_OPT_INGEST_CHUNK 2   /* file loaders: bytes of text per device chunk (0: 32 MiB mapped / 4 MiB .gz) */
#define GWASDEV_OPT_SCAN_PIECES 3    /* host-output scans: pieces whose D2H copies overlap the next piece (0 auto, 1..8) */
#define GWASDEV_OPT_MASKED_SCAN 4    /* 0 auto (first scan after a selection counts through the masks); 1 always compact first */
#define GWASDEV_OPT_TRACE 5          /* 1: phase timings of the pairwise scan / compaction / G-test on stderr */
#define GWASDEV_OPT_FOUR_PLANE 6     /* 0 auto; 1: tiles with missing calls stay on the 9-cell AND+POPC kernel */
#define GWASDEV_OPT_ROW_TOTALS 7     /* K1': 0 auto (row totals cached per table when the classes partition the cohort); 1 never */
#define GWASDEV_OPT_CAND_CAPACITY 8  /* pairwise screen: candidate buffer entries (0 auto); small values exercise the overflow paths */
#define GWASDEV_OPT_CLASSIC_PLANES 9 /* two-plane tensor-core screen: 0 auto (every SNP puts its two rarest genotype classes on the tensor cores);
                                        1: always the two homozygote planes, as the reference's shortcut counts them */
#define GWASDEV_OPT_PERM_OPERAND_BYTES 10 /* permutation test: device bytes the SNP-plane operand may keep resident (0 auto: a quarter
                                             of the device memory); a larger table is expanded and multiplied one SNP chunk at a time (at least
                                             64 SNPs, the kernel's tile), as is a table whose operand finds the device too full */
#define GWASDEV_OPT_COUNT 16
GWASDEV_API int gwasdev_set_option(gwasdev_store *s, int option, long long value);

/* ---- geometry ------------------------------------------------------------------------------- */
/* 16-bit blocks per bit-plane for n samples: pad4(n/16 + 1) (compressed_genotype_table5.cpp:55-64). */
GWASDEV_API uint32_t gwasdev_plane_blocks(uint32_t n);

/* ---- loading -------------------------------------------------------------------------------- */
/* Host-side row packer with the reference's text semantics: GenoTable::addGenotypeRow(const char*, ...)
 * (compressed_genotype_table5.cpp:277-365) incl. the first-seen label state machine
 * (common_genotype.h:257-304). row receives [hdr][plane1: P][plane2: P] 16-bit blocks, P =
 * gwasdev_plane_blocks(n_samples). Returns GWASDEV_EINVAL where the reference would abort. */
GWASDEV_API int gwasdev_pack_row_text(const char *txt, size_t len, uint32_t n_samples, uint16_t *row);
/* The same for one sample block of a row that is loaded in several blocks (streaming, see
 * gwasdev_marginal_accumulate): *label_state carries the row's header word from block to block (0 before the
 * first block), so that genotype labels stay first-seen over the whole row as in the reference. */
GWASDEV_API int gwasdev_pack_row_text_block(const char *txt, size_t len, uint32_t n_samples, uint16_t *row,
                                uint16_t *label_state);
/* Upload / download n_rows rows in that layout (row stride 2P+1 blocks, host memory). */
GWASDEV_API int gwasdev_put_rows(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, const uint16_t *rows);
GWASDEV_API int gwasdev_get_rows(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, uint16_t *rows);
/* GenoTable::operator()(r, c) + decodeGenotype (compressed_genotype_table5.cpp:400-432,1225-1231). */
GWASDEV_API int gwasdev_call_at(gwasdev_store *s, uint64_t row, uint32_t col, char out[3]);

/* ---- file / text ingestion on the device (SURVEY.md 8f1) ---------------------------------------------
 * Transposed-PLINK text straight into the store: replaces TpedGenotypeFile::parseNextGenotypeRecord
 * (genetics/individual/tped_genotype_file.cpp:110-185: trim, four marker fields, alleles 1234 -> ACGT, one allele
 * every other character) + GenoTable::addGenotypeRow (compressed_genotype_table5.cpp:277-365) for every line of
 * `text`. Lines end in '\n'; blank lines are skipped; the k-th non-blank line becomes row first_row + k. Only whole
 * lines are consumed: *bytes_used (may be NULL) is the offset after the last '\n', the caller keeps the rest for
 * its next call. *rows_done (may be NULL) = rows written. The host does not look at the text beyond finding that
 * last newline: line index, label resolution and bit-packing run on the device. GWASDEV_EINVAL where the reference
 * aborts (third spelling of one genotype kind) and for lines without four marker fields or more lines than rows. */
GWASDEV_API int gwasdev_put_tped_text(gwasdev_store *s, uint64_t first_row, const char *text, size_t len, uint64_t *rows_done,
                          size_t *bytes_used);
/* Table dimensions of a TPED file (plain or .gz): non-blank lines, and the genotype columns of the first line counted
 * the way the reference sizes its row buffer (tped_genotype_file.cpp:132-136). */
GWASDEV_API int gwasdev_tped_dims(const char *path, uint64_t *n_rows, uint32_t *n_samples);
/* Whole TPED file (plain or .gz, read through zlib) into rows first_row.., double-buffered through pinned memory so
 * that reading chunk k+1 overlaps the device work on chunk k. A .gz needs no rewind: dims and load each open it once
 * (the reference's two-pass reader seeks, which its gzstream cannot: individual_genotype_file.cpp:94). */
GWASDEV_API int gwasdev_load_tped(gwasdev_store *s, const char *path, uint64_t first_row, uint64_t *rows_done);
/* gwasdev_tped_dims + gwasdev_create + gwasdev_load_tped in ONE pass over a plain file: the sample count comes from the
 * first genotype line, the row capacity from the file size, and the table is trimmed to the rows found (a .gz still
 * takes the counting pass first). What `new CompressedGenotypeTable5` + the two-pass reader do in the reference
 * (genetics/genetic_data.cpp:60-79, individual_genotype_file.cpp:63-106). */
GWASDEV_API int gwasdev_create_from_tped(const char *path, int device, gwasdev_store **out, uint64_t *n_rows, uint32_t *n_samples);
/* PLINK .bed rows (SNP-major, ceil(n_samples/4) bytes per SNP, no magic; 0 = hom A1, 1 = missing, 2 = het,
 * 3 = hom A2) into rows [first_row, first_row + n_rows). alleles (may be NULL = A, C) holds the indices of A1 and A2
 * in "ACGT" per row; labels come out as the text loader would give the same calls spelled A1A1 / A1A2 / A2A2 in
 * sample order. The reference has no .bed reader; this is the input SURVEY.md 8f1 adds. */
GWASDEV_API int gwasdev_put_bed(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, const uint8_t *bed, const uint8_t *alleles);
GWASDEV_API int gwasdev_bed_dims(const char *bed_path, uint32_t n_samples, uint64_t *n_rows);
GWASDEV_API int gwasdev_load_bed(gwasdev_store *s, const char *bed_path, const uint8_t *alleles, uint64_t first_row, uint64_t *rows_done);

/* Synthetic cohort generated directly in HBM: fixed-seed restatement of data/simulate_data.cpp:160-207
 * over one panel of data/maf_spectrum.tab (bin_counts[b] = SNP count at MAF b %). missing_q32/2^32
 * is the per-genotype missing probability. Labels are first-seen, as the text loader would give. */
GWASDEV_API int gwasdev_simulate(gwasdev_store *s, uint64_t seed, const uint32_t bin_counts[51], uint32_t missing_q32);
/* One sample block of that cohort: the store holds samples [first_sample, first_sample + n_samples) of a cohort of
 * n_total_samples; draws and first-seen labels are those of the whole-cohort table. */
GWASDEV_API int gwasdev_simulate_block(gwasdev_store *s, uint64_t seed, const uint32_t bin_counts[51], uint32_t missing_q32,
                           uint32_t first_sample, uint32_t n_total_samples);
/* Host helper: exactly n_case cases (1) among n_samples, the rest controls (0). */
GWASDEV_API int gwasdev_simulate_phenotype(uint64_t seed, uint32_t n_samples, uint32_t n_case, uint8_t *pheno);

/* ---- case / control ------------------------------------------------------------------------- */
/* CaseControlSelectable::selectCaseControl (compressed_genotype_table5.cpp:443-575) with the stream
 * masks of CaseControlSet (genetics/analyzable/case_control_set.cpp:77-150): P blocks each, bit c&15
 * of block c>>4 set for member c. Builds the compacted case/control store (and, lazily, the
 * SNP-tiled pairwise store) on the device; the raw store stays resident, so this can be called
 * again with other masks. */
GWASDEV_API int gwasdev_select_case_control(gwasdev_store *s, const uint16_t *case_mask, const uint16_t *ctrl_mask);
/* Compaction is lazy by default: the call above uploads the masks, and the compacted rows are built (kernel K0) only when
 * something needs that LAYOUT -- the layout probes (gwasdev_get_selected_rows, gwasdev_counts mode 2, gwasdev_pair_tables
 * mode 2), the AND+POPC engine, cohorts beyond the packed accumulator with missing calls, or the second marginal scan of a
 * cohort with samples outside both classes. Marginal scans count through the masks on the raw rows (the reference's
 * mask-on-the-fly overload, :609-657: identical counts), and the tensor-core screen, its fp64 re-score and the G-test read
 * raw rows + masks as well. eager != 0 runs K0 inside gwasdev_select_case_control. */
GWASDEV_API int gwasdev_set_select_mode(gwasdev_store *s, int eager);
/* 1 when the compacted rows of the current selection exist on the device (K0 has run for it), 0 when not, -1 without a selection. */
GWASDEV_API int gwasdev_is_compacted(const gwasdev_store *s);
/* Stream masks for the mask-on-the-fly overloads only -- getCaseControlGenotypeDistribution(r, ccs, ccgd) (:609-657,
 * gwasdev_counts mode 1) and getCaseControlContingencyTable(i, j, ccs, ccct) (:806-895, gwasdev_pair_tables mode 1). As in
 * the reference, they do not touch the pre-selected store: selection, compacted rows, margins and pairwise layouts stay
 * valid. gwasdev_select_case_control sets them too (to its own masks). */
GWASDEV_API int gwasdev_set_stream_masks(gwasdev_store *s, const uint16_t *case_mask, const uint16_t *ctrl_mask);
GWASDEV_API int gwasdev_case_control_counts(gwasdev_store *s, uint32_t *n_case, uint32_t *n_ctrl);
/* Compacted rows in the reference's layout [case p1: Pca][case p2: Pca][ctrl p1: Pco][ctrl p2: Pco]
 * (16-bit blocks, Pca = gwasdev_plane_blocks(n_case)) -- layout-parity probe. */
GWASDEV_API int gwasdev_get_selected_rows(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, uint16_t *rows);

/* ---- marginal scan (K1) --------------------------------------------------------------------- */
/* Per SNP in [snp_begin, snp_end): case/control genotype counts
 * (getCaseControlGenotypeDistribution(rIdx, ccgd, m), compressed_genotype_table5.cpp:703-747),
 * marginal_information (computeMarginalInformation, genotype/common_genotype_func.cpp:173-219 ==
 * computeMargins, algorithms/epistasis_func.cpp:706-721), MinorAlleleFrequency and the chi-square tests.
 * counts: 8 per SNP = cases{aa,ab,bb,xx}, controls{aa,ab,bb,xx}. Any output pointer may be NULL.
 * on_device = 0: outputs are host buffers (copied back inside the call); 1: device buffers. */
GWASDEV_API int gwasdev_marginal_scan(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *counts,
                          gwasdev_marginal_information *mi, gwasdev_snp_stats *stats, int on_device);
/* The same scan with compact outputs, for callers on the far side of PCIe (select_cc_maf needs the two frequency tables
 * per SNP, algorithms/maf_func.cpp:256-267; a chi-square scan needs four numbers): `out` (may be NULL) receives one 32-byte
 * record per SNP; SNPs with min(p_allelic, p_genotypic) < p_threshold are also appended to sig[0..*n_sig) in fp64, sorted
 * by SNP index (sig may be NULL when p_threshold <= 0; more than sig_capacity significant SNPs -> GWASDEV_EOVERFLOW with
 * *n_sig = the number found). Needs both classes below 65 536 samples when out != NULL. Host or device buffers as above. */
GWASDEV_API int gwasdev_marginal_scan_compact(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, gwasdev_snp_compact *out,
                                  double p_threshold, gwasdev_sig_snp *sig, uint64_t sig_capacity, uint64_t *n_sig, int on_device);
/* Streaming in sample blocks (BASELINE configs[4]): genotype counts are additive over disjoint sample blocks, which the
 * reference cannot exploit (its rows are always whole: compressed_genotype_table5.cpp:703-747 walks one compacted row).
 * A store holding one block of samples (loaded with label state carried over, or gwasdev_simulate_block) adds its
 * case/control counts of SNPs [snp_begin, snp_end) into acc (8 per SNP, device buffer when on_device); after the last
 * block gwasdev_marginal_finalize computes marginal_information (computeMarginalInformation,
 * genotype/common_genotype_func.cpp:173-219) and the statistics from the summed counts -- bit-identical to one scan
 * over the whole cohort. */
GWASDEV_API int gwasdev_marginal_accumulate(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *acc, int on_device);
GWASDEV_API int gwasdev_marginal_finalize(int device, uint64_t n_snps, const uint32_t *counts, gwasdev_marginal_information *mi,
                              gwasdev_snp_stats *stats, int on_device);
/* Device time (ms, CUDA events) of the scan kernel inside the last gwasdev_marginal_scan call. */
GWASDEV_API double gwasdev_last_scan_ms(gwasdev_store *s);

/* Counts through the other SingleMarkerAnalyzable overloads, for rows [snp_begin, snp_end) (host out):
 * mode 0: getGenotypeDistribution, 4 per SNP {aa,ab,bb,xx} over the raw row (:577-607; xx = N - called,
 *         i.e. what inline_maf_print prints, not the reference's padding-inflated xx -- defect D5);
 * mode 1: mask-on-the-fly getCaseControlGenotypeDistribution(r, ccs, ccgd) (:609-657), 8 per SNP;
 * mode 2: pre-selected getCaseControlGenotypeDistribution(r, ccgd) (:659-701), 8 per SNP. */
GWASDEV_API int gwasdev_counts(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, int mode, uint32_t *out);

/* ---- label-permutation test of the marginal scan (max(T), PLINK --mperm's EMP1 / EMP2) -------------------------------------- */
typedef struct {
    uint64_t n_perm;        /* permutations evaluated by this call */
    uint64_t snps;          /* SNPs covered */
    double gemm_ms;         /* device time of the permutation GEMM kernel(s) (CUDA events) */
    double total_ms;        /* whole call: draws, operands, observed scan, GEMM, reductions */
    uint32_t planes;        /* operand planes per SNP that were multiplied: 2 (no missing calls in the table) or 3 */
    uint32_t built_operand; /* 1 when this call expanded the SNP-plane operand (first call, rows changed, or chunked) */
} gwasdev_perm_stats;

/* Label-permutation test of the current selection over SNPs [snp_begin, snp_end). Permutation first_perm + k makes exactly
 * n_case of the selection's samples (cases + controls-and-not-cases) cases, drawn as gwasdev_permutation_masks describes, or
 * takes case_masks[k] (P blocks each) when case_masks != NULL: any non-empty proper subset of the selection (stratified or
 * family-aware permutations, other traits; the case count may differ between masks). The case genotype counts of every
 * (SNP, permutation) pair come from one int8 tensor-core GEMM over the samples (permutation case bytes x one-hot SNP planes).
 * The observed statistics are those of gwasdev_marginal_scan on the same selection. Outputs (each may be NULL; host or device
 * buffers as on_device), overwritten, not accumulated:
 *   exceed[2*i + {0,1}]      permutations whose chi2_allelic / chi2_genotypic of SNP snp_begin+i is >= the observed one
 *   perm_max[3*k + {0,1,2}]  per permutation: max chi2_allelic, max chi2_genotypic over the df-1 (SNP, permutation) elements,
 *                            the same over the df-2 elements (0 when there are none)
 *   perm_stats               device buffer only: [n_perm][snp_end - snp_begin] x {chi2_allelic, chi2_genotypic}
 * Every statistic is bit-identical to gwasdev_marginal_scan's on the permuted selection. Calls over disjoint first_perm ranges
 * combine by summing exceed and concatenating perm_max. n_perm = 0 is a no-op. */
GWASDEV_API int gwasdev_marginal_permute(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint64_t seed,
                                         uint64_t first_perm, uint64_t n_perm, const uint16_t *case_masks,
                                         uint32_t *exceed, double *perm_max, double *perm_stats,
                                         gwasdev_perm_stats *stats, int on_device);
/* Host arithmetic, no device needed: the case masks (P = gwasdev_plane_blocks(n_samples) blocks each) of permutations
 * first_perm .. first_perm + n_perm - 1 of the selection (case_mask, ctrl_mask). Selected samples (in either mask; a sample in
 * both counts once) are walked in increasing position; with `rank` the position inside the selection, `left` the selected
 * samples not yet visited and `need` the cases still to place, the sample is a case of permutation q iff
 * ((sim_hash(seed, q, rank) >> 32) * left) >> 32 < need (Knuth's selection sampling; exactly |case_mask| cases). */
GWASDEV_API int gwasdev_permutation_masks(uint32_t n_samples, const uint16_t *case_mask, const uint16_t *ctrl_mask,
                                          uint64_t seed, uint64_t first_perm, uint64_t n_perm, uint16_t *out);
/* Host arithmetic: empirical p-values per SNP and test (emp1 / emp2 [2*i + {0 allelic, 1 genotypic}], each may be NULL) from
 * the observed statistics and one or more calls' exceed (summed) and perm_max (concatenated) over n_perm permutations:
 * EMP1 = (exceed + 1) / (n_perm + 1); allelic EMP2 = (1 + #{q : max_a[q] >= chi2_obs}) / (n_perm + 1); genotypic EMP2 compares
 * p-values, minp_q = min(Q1(max_g1[q]), Q2(max_g2[q])) <= Q_df(chi2_obs), with Q_df the chi-square upper tail; df-0 SNPs get 1. */
GWASDEV_API int gwasdev_permutation_pvalues(uint64_t n_snps, uint64_t n_perm, const gwasdev_snp_stats *observed,
                                            const uint32_t *exceed, const double *perm_max, double *emp1, double *emp2);

/* ---- linkage disequilibrium: genotypic r^2 ----------------------------------------------------------------------------------------
 * For a sample set S (every sample of the table, or sample_mask: P 16-bit blocks, bit c&15 of block c>>4 for sample c; NULL = all)
 * and SNPs i, j: x is the allele count under the store's own labels (aa 0, ab 1, bb 2: the {aa, ab, bb} of gwasdev_counts). Over
 * the samples of S called at both SNPs, the exact integer sums n, Sx, Sy, Sxx, Syy, Sxy give, in int64, num = n Sxy - Sx Sy,
 * vx = n Sxx - Sx^2, vy = n Syy - Sy^2, and in fp64 without contraction r2 = (num num) / (vx vy), r = num / sqrt(vx vy): the
 * squared Pearson correlation of allele counts over pairwise-complete samples. Both are NaN when vx = 0 or vy = 0 (a SNP
 * monomorphic over those samples, n < 2). r2 does not depend on the labels; the sign of r does, and labels are first-seen
 * (the first homozygote of a row is aa), so r of two SNPs in perfect LD may be -1. Every entry point below computes r and r2
 * with the same device arithmetic: their values are bit-identical. */
typedef struct {
    uint32_t i, j;      /* i < j, table row indices */
    uint32_t n;         /* samples of S called at both SNPs */
    uint32_t reserved;
    double r, r2;
} gwasdev_ld_pair;      /* 32 bytes */
typedef struct {
    uint64_t pairs_tested;   /* pairs (i, j) of the band this call covered */
    uint64_t pairs_kept;     /* pairs with r2 >= r2_threshold */
    double gemm_ms;          /* device time of the LD GEMM kernel(s) (CUDA events) */
    double total_ms;         /* whole call: operand, GEMM, list sort, copies */
    uint32_t rows_per_snp;   /* operand rows per SNP that were multiplied: 1 (no missing call in S) or 3 */
    uint32_t built_operand;  /* 1 when this call expanded the operand (first call, rows or sample set changed, or chunked) */
} gwasdev_ld_stats;
#define GWASDEV_OPT_LD_OPERAND_BYTES 11 /* LD: device bytes the allele-count operand may keep resident (0 auto: a quarter of the device
                                           memory); a larger table is expanded one chunk of 256-SNP blocks (plus the window's B-SNPs) at a
                                           time, as is a table whose operand finds the device too full */
/* Every pair snp_begin <= i < j < snp_end with j - i <= window (window >= 1; window >= snp_end - snp_begin - 1 is the full LD
 * matrix of the region), from one int8 tensor-core GEMM of the allele-count rows against themselves restricted to the band.
 * Works on a freshly loaded table: no selection is needed.
 *   pairs (may be NULL)  the pairs with r2 >= r2_threshold (fp64 comparison; NaN never qualifies), sorted by (i, j);
 *                        more than `capacity` of them -> GWASDEV_EOVERFLOW with *n_pairs = the number needed
 *   band (may be NULL)   (float)r2 at band[(i - snp_begin) * window + (j - i - 1)], NaN where r2 is undefined or j >= snp_end
 * Host or device buffers as on_device; stats may be NULL. */
GWASDEV_API int gwasdev_ld_window(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t window, const uint16_t *sample_mask,
                                  double r2_threshold, gwasdev_ld_pair *pairs, uint64_t capacity, uint64_t *n_pairs,
                                  float *band, gwasdev_ld_stats *stats, int on_device);
/* Given pairs (pi[k], pj[k]) at any distance, i != j in either order -> out[k] with i < j (host buffers). Counts on the CUDA
 * cores from the raw rows: annotates pair-screen hits and cross-checks the GEMM path. */
GWASDEV_API int gwasdev_ld_pairs(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, const uint16_t *sample_mask,
                                 gwasdev_ld_pair *out);
/* Host arithmetic, no device needed: greedy LD pruning of SNPs [snp_begin, snp_end) from a list of gwasdev_ld_window (same
 * window, threshold at or below r2_threshold; sorted by (i, j), every pair inside the range and the window, else
 * GWASDEV_EINVAL). Walking i upwards, SNP i is kept (keep[i - snp_begin] = 1) unless some kept k with
 * max(snp_begin, i - window) <= k < i has r2(k, i) >= r2_threshold. So no two kept SNPs within the window reach the threshold,
 * and every dropped SNP has a kept SNP before it within the window that does. This is not PLINK's --indep-pairwise: there is
 * no window step, and the earlier SNP always wins, whatever the allele frequencies. */
GWASDEV_API int gwasdev_ld_prune(uint64_t snp_begin, uint64_t snp_end, uint32_t window, double r2_threshold,
                                 const gwasdev_ld_pair *pairs, uint64_t n_pairs, uint8_t *keep);

/* ---- pair tables (K2, per-call virtuals and parity probes) ---------------------------------- */
/* n pairs (pi[k], pj[k]) -> out[k] = case table[16] then control table[16], 4x4 row-major with the xx
 * row/column (common_genotype.h:182-192).
 * mode 0: getContingencyTable (:749-800), un-stratified, in the "case" half;
 * mode 1: mask-on-the-fly getCaseControlContingencyTable(i, j, ccs, ccct) (:806-895);
 * mode 2: pre-selected getCaseControlContingencyTable(i, j, ccct) (:896-987);
 * mode 3: margins overload getCaseControlContingencyTable(i, j, m1, m2, ccct) (:989-1150) -- the hot one.
 * Modes 0-2 reproduce the reference's xx cells including its padding / masked-out inflation. */
GWASDEV_API int gwasdev_pair_tables(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, int mode,
                        uint32_t *out);

/* ---- exhaustive pairwise screen (K2+K3+K5) -------------------------------------------------- */
/* computeBoost's pre-screening loop (algorithms/epistasis_func.cpp:397-486) over every pair i<j whose SNP tile
 * pair belongs to this shard. The pair space is cut into tile pairs (128x128 SNPs for the tensor-core engine,
 * 64x64 for the AND+POPC engine) in a fixed linear order; shards own alternating runs of that order (runs of 64
 * tiles, resp. single tiles), so the n_shards calls with shard = 0..n_shards-1 cover every pair exactly once.
 * Writes the pairs with stat > threshold, sorted by (i, j), into hits[0..*n_hits).
 * hits / on_device as for the marginal scan. Requires gwasdev_select_case_control; computes the margins
 * itself when gwasdev_marginal_scan has not been run over all SNPs. */
GWASDEV_API int gwasdev_pairwise_scan(gwasdev_store *s, double threshold, uint32_t shard, uint32_t n_shards,
                          gwasdev_hit *hits, uint64_t capacity, uint64_t *n_hits,
                          gwasdev_pair_stats *stats, int on_device);
/* The same screen with a bounded result: the top_k pairs with the largest statistic above the threshold (ties at the k-th
 * place go to the smaller (i, j)), sorted by (i, j); hits holds top_k records. computeBoost keeps every pair above its
 * threshold in an unbounded vector (epistasis_func.cpp:388, :482-484); with a low threshold or real data that list has
 * no useful bound, this one does: the kernels raise a device-wide threshold as soon as k better pairs have been seen, so
 * the candidate buffer needs room for a few times k whatever the threshold. Sharded runs return each shard's top_k; the
 * top_k of their union is the global answer (gwasdev_pairwise_scan_multi does that). */
GWASDEV_API int gwasdev_pairwise_topk(gwasdev_store *s, double threshold, uint64_t top_k, uint32_t shard, uint32_t n_shards,
                          gwasdev_hit *hits, uint64_t *n_hits, gwasdev_pair_stats *stats, int on_device);
/* ---- several devices, one host process (the multi-GPU driver a C++ caller reaches) -------------------------------------
 * Copy of a store on another device: headers and raw rows travel device to device (NVLink when peer access is available),
 * options, engine choice and the current selection are re-applied. What a caller does after loading the genotype file once. */
GWASDEV_API int gwasdev_replicate(gwasdev_store *src, int device, gwasdev_store **out);
/* computeBoost's pre-screen (algorithms/epistasis_func.cpp:397-486) over n_stores stores that hold the same table and
 * selection on n_stores different devices: store d runs shard d of n_stores of the tile-pair schedule on its own host thread
 * (as gwasdev_pairwise_scan / gwasdev_pairwise_topk would), the fixed-size hit records are combined with one ncclAllGather
 * (gather = 0; NCCL is loaded at run time, communicators are created once per device list) or with peer copies to
 * stores[0]'s device (gather = 1), and that device merges them: hits[0..*n_hits) in host memory, sorted by (i, j) -- the
 * top_k largest statistics when top_k != 0, every pair above the threshold otherwise (capacity as for gwasdev_pairwise_scan).
 * stats (may be NULL) receives n_stores records, one per shard. Identical to the single-device result. */
GWASDEV_API int gwasdev_pairwise_scan_multi(gwasdev_store *const *stores, uint32_t n_stores, double threshold, uint64_t top_k,
                                gwasdev_hit *hits, uint64_t capacity, uint64_t *n_hits, gwasdev_pair_stats *stats, int gather);
/* computeGTest (as gwasdev_gtest) on n given pairs, the list cut into one contiguous piece per store / device. */
GWASDEV_API int gwasdev_gtest_multi(gwasdev_store *const *stores, uint32_t n_stores, uint64_t n, const uint32_t *pi, const uint32_t *pj,
                        double *stat, double *z);
/* Engine for the tile pairs without missing calls. 0 (default): tensor cores (tcgen05 kind::i8 GEMM over signed
 * one-hot bytes, pairwise_mma.cu) when n_case < 16384 and n_ctrl < 131072, else AND+POPC tiles; 1: AND+POPC
 * tiles; 2: tensor cores or GWASDEV_EINVAL. Tile pairs with missing calls (the reference's other branch,
 * compressed_genotype_table5.cpp:1000-1067) take the four-plane tensor-core kernel under the same conditions and the
 * 9-cell AND+POPC kernel otherwise. Cohorts with larger classes (below 2^23 samples each) run on the four-plane kernel
 * with one pair of planes per class (no missing calls) or one accumulator per class (missing calls). Results are
 * identical. */
GWASDEV_API int gwasdev_set_pair_engine(gwasdev_store *s, int engine);
/* Host arithmetic only (works without a device): the tile pairs (I <= J, as SNP-block indices) of the screen's schedule that
 * `shard` of `n_shards` owns, in schedule order, and the pairs i < j < n_snps they cover. engine 2: the tensor-core
 * schedule for a table of n_samples individuals (128-SNP blocks; bands of 8 to 16 A-blocks, as many as keep the working set of
 * the 74 concurrent tiles in the L2: 16 at 4 000 samples, 13 at 10 000, 8 from 12 000; shards own alternating runs of 64
 * consecutive tiles); engine 1: the
 * AND+POPC schedule (64-SNP blocks, row-major upper triangle, single tiles round-robin). tiles (may be NULL) receives
 * min(*n_tiles, capacity) (I, J) pairs. */
GWASDEV_API int gwasdev_shard_schedule(uint64_t n_snps, uint64_t n_samples, int engine, uint32_t shard, uint32_t n_shards, uint32_t *tiles, uint64_t capacity,
                           uint64_t *n_tiles, uint64_t *n_pairs);
/* Parity probe of the tensor-core engine: raw corner counts of one tile pair of its schedule (A-block I of 64
 * SNPs, B-block J of 128 SNPs, I/2 <= J): out[(a*128 + b)*8 + {0,1,2,3}] = cases AA_BB, AA_bb, aa_BB, aa_bb
 * (compressed_genotype_table5.cpp:1069-1083), +4: controls (:1118-1132). out holds 64*128*8 values. */
GWASDEV_API int gwasdev_mma_tile_counts(gwasdev_store *s, uint32_t I, uint32_t J, uint32_t *out);
/* Diagnostic twin of gwasdev_ksa_screen_f32 for the tensor-core engine's epilogue: stat[2k] = its fp32 value of
 * the statistic, stat[2k+1] = its cheap upper bound (pairs whose bound is below threshold - margin are dropped
 * without evaluating the logarithms; the bound must never fall below the statistic). */
GWASDEV_API int gwasdev_ksa_screen_mma_f32(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, float *stat);
/* KSA statistic in fp64 for given pairs (the re-scoring kernel on its own; parity probe). */
GWASDEV_API int gwasdev_ksa(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, double *stat);
/* Diagnostic: the screen kernel's fp32 epilogue evaluated on given pairs, to measure its distance from
 * the fp64 statistic (the screen keeps pairs above threshold - margin; see DESIGN.md). */
GWASDEV_API int gwasdev_ksa_screen_f32(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, float *stat);
/* Diagnostic: the G-test's fp64 division on n operand pairs (host buffers) on `device`. q_fast[k] = the branch-free
 * division of the IPF sweeps, q_rn[k] = __ddiv_rn(a[k], b[k]), bad[k] = 1 where the fast sequence leaves its range (the
 * exponent test ptxas applies before its slow path); q_fast has the bits of q_rn wherever bad is 0 and a[k] != 0, and for
 * a[k] = +0 over a finite, normal b[k]. */
GWASDEV_API int gwasdev_fp64_div_probe(int device, uint64_t n, const double *a, const double *b, double *q_fast, double *q_rn,
                                       uint8_t *bad);
/* computeGTest (epistasis_func.cpp:508-704): exact log-linear G statistic by IPF and the allele-joint
 * log-odds z for n pairs (host buffers). The IPF stops when sum |delta mu| <= 1e-3, as the reference's loop does. On some
 * sparse tables (e.g. cells absent in one class) that sum settles on a cycle and never gets there, and the reference
 * loops forever: a fit that has not converged after 1 000 000 sweeps gives stat = NaN. z does not depend on the fit and
 * is always computed. */
GWASDEV_API int gwasdev_gtest(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, double *stat,
                  double *z);
/* pairwise_epi_test of src/test/pairwise.c:50-133 on n dense 3x3x2 tables (cs, ct: 9 ints each) and
 * pchisq(ll, 4, 0, 0) (:44). */
GWASDEV_API int gwasdev_pairwise_epi_test(int device, uint64_t n, const int32_t *cs, const int32_t *ct, double *ll,
                              double *pval);

/* The pair loop of EpistasisPerformance / EpistasisDebug (epistasis_func.cpp:263-347) for n given pairs: the pair's
 * case/control tables by overload `mode` (as gwasdev_pair_tables; the reference uses mode 1), then the likelihood-ratio
 * test of src/test/pairwise.c:50-133 on their 3x3 cores and pchisq(ll, 4, 0, 0), without shipping the tables to the
 * host. (The reference's C++ copy of the test, epistasis_func.cpp:723-892, reads the 4x4 table as if it were 3x3;
 * the C file is its clean form and the parity target, SURVEY.md a19.) */
GWASDEV_API int gwasdev_epi_pairs(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, int mode, double *ll,
                      double *pval);

/* ---- measurement helpers -------------------------------------------------------------------- */
/* Register-only __popc throughput in 32-bit word-cells (AND+POPC) per second on `device`; the
 * integer-pipe roofline denominator of the pairwise screen (SURVEY.md section 8d). */
GWASDEV_API int gwasdev_popc_peak(int device, double *word_cells_per_s, double *sm_clock_mhz);
/* int8 tensor-core throughput of `device` with the screen kernel's own instruction (tcgen05.mma.cta_group::2.kind::i8,
 * M = 256, N = 256, K = 32, operands resident in shared memory, accumulators in TMEM, no TMA traffic, no epilogue), in
 * 1e12 operations per second at 2 operations per multiply-accumulate: the best launch (burst) and the mean over ~50 ms of
 * back-to-back launches (sustained; may be NULL). The tensor-core roofline denominator of the pairwise screen. */
GWASDEV_API int gwasdev_i8_peak(int device, double *tops_burst, double *tops_sustained);
/* Read-only streaming bandwidth (GB/s) of a plain 128-bit-load kernel over `bytes` of HBM on `device`:
 * context for the marginal scan's roofline next to the driver-measured copy bandwidth. */
GWASDEV_API int gwasdev_hbm_read_peak(int device, uint64_t bytes, double *gb_per_s);
/* The same loads past L1 over a buffer of `bytes` (1 to 64 MiB: L2-resident) read `passes` times in one launch: the rate (GB/s) at which
 * the L2 delivers to the SMs, what the tensor-core screens' operand stream runs into (bench.py: roofline.l2_to_sm). */
GWASDEV_API int gwasdev_l2_read_peak(int device, uint64_t bytes, uint32_t passes, double *gb_per_s);

#ifdef __cplusplus
}
#endif
#endif /* GWASDEV_H */
