/* TEST INFRASTRUCTURE -- NOT PRODUCT CODE.
 *
 * CPU restatement (plain C) of libgwaspp's case/control association hot path, used only as the
 * checker in tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg. The product library
 * (libgwaspp_b200/csrc) never includes, links or calls anything declared here.
 *
 * Parity status: PINNED. Every function below is checked in tests/test_oracle_pinning.py against
 * the unmodified reference compiled from /root/reference (oracle/_ref/libgwasref.so, recipe in
 * oracle/ref_build/Makefile), against golden vectors produced by that build (tests/golden/),
 * against scripts/perl/genotype_set_builder.pl expectation files and against the five 3x3x2
 * tables of src/test/pairwise.c:19-37.  EXCEPTION: go_chi2_allelic / go_chi2_genotypic have no
 * counterpart in the reference ("parity unpinned", SURVEY.md section 8c); they are specified in
 * DESIGN.md and cross-checked against scipy.stats only.
 *
 * All file:line citations are relative to /root/reference/src/libgwaspp unless stated otherwise.
 */
#ifndef GWAS_ORACLE_H
#define GWAS_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* genetics/genotype/common_genotype.h:101-106 -- 192 bytes, same field order. */
typedef struct {
    uint32_t margins[4], cases[4], controls[4]; /* each {aa, ab, bb, xx}  (common_genotype.h:67-75) */
    double entropy, entropy_y;                  /* dMarginalEntropy, dMarginalEntropy_Y */
    double pbc[8];                              /* P(genotype | class): cases[4], controls[4] */
    double pca[8];                              /* P(class | genotype): cases[4], controls[4] */
} go_marginal_information;

/* ---- geometry (compressed_genotype_table5.cpp:34-153, :443-471; case_control_set.cpp:34-75) ---- */
int go_plane_blocks(int n);               /* pad4(n/16 + 1) 16-bit blocks for n samples */

/* ---- a4/a6: text row -> [hdr][plane1][plane2], first-seen labels (compressed_genotype_table5.cpp:277-365,
 *      common_genotype.h:257-304). Returns 0, or -1 where the reference would abort on an assert. ---- */
int go_pack_row_text(const char *txt, long len, int n_samples, uint16_t *row /* 2*P+1 */);
/* codes: 0 "AA", 1 "AC", 2 "CC", 3 missing, 4 "CA" */
int go_pack_row_codes(const uint8_t *codes, int n_samples, uint16_t *row);
/* operator()(r,c) + decodeGenotype (compressed_genotype_table5.cpp:400-432,1225-1231): 2 chars + NUL */
void go_call_at(const uint16_t *row, int n_samples, int col, char out[3]);

/* ---- a7: 1-bit stream masks (case_control_set.cpp:77-150); pheno 1 = case, 0 = control ---- */
void go_stream_masks(const uint8_t *pheno, int n_samples, uint16_t *case_mask, uint16_t *ctrl_mask,
                     int *n_case, int *n_ctrl);

/* ---- a8: selectCaseControl (compressed_genotype_table5.cpp:443-575) ----
 * out = [case p1: Pca][case p2: Pca][ctrl p1: Pco][ctrl p2: Pco] 16-bit blocks */
void go_select_row(const uint16_t *row, int n_samples, const uint16_t *case_mask,
                   const uint16_t *ctrl_mask, int n_case, int n_ctrl, uint16_t *out);

/* ---- a9 / a21: genotype counts; out = cases{aa,ab,bb,xx}, controls{aa,ab,bb,xx} ---- */
void go_cc_counts_selected(const uint16_t *sel, int n_case, int n_ctrl, uint32_t out[8]);   /* :659-701 */
void go_cc_counts_masked(const uint16_t *row, int n_samples, const uint16_t *case_mask,
                         const uint16_t *ctrl_mask, int n_case, int n_ctrl, uint32_t out[8]); /* :609-657 */
void go_counts_whole(const uint16_t *row, int n_samples, uint32_t out[4]);                   /* :577-607 */

/* ---- a10: computeMarginalInformation (genotype/common_genotype_func.cpp:173-219), zero-initialised ---- */
void go_marginal_information_fill(const uint32_t ca[4], const uint32_t co[4], uint32_t n_individs,
                                  go_marginal_information *m);
/* ---- a11: MinorAlleleFrequency (algorithms/maf_func.h:46-54): returns max(f, 1-f); *tot = called ---- */
double go_maf_reference(const uint32_t ft[4], double *tot);

/* ---- a14 / a21: pair tables, 4x4 row-major (common_genotype.h:182-192) ---- */
void go_pair_table_margins(const uint16_t *sel_i, const uint16_t *sel_j, int n_case, int n_ctrl,
                           const go_marginal_information *m1, const go_marginal_information *m2,
                           uint32_t ca[16], uint32_t co[16]);                               /* :989-1150 */
void go_pair_table_selected(const uint16_t *sel_i, const uint16_t *sel_j, int n_case, int n_ctrl,
                            uint32_t ca[16], uint32_t co[16]);                              /* :896-987 */
void go_pair_table_masked(const uint16_t *row_i, const uint16_t *row_j, int n_samples,
                          const uint16_t *case_mask, const uint16_t *ctrl_mask,
                          uint32_t ca[16], uint32_t co[16]);                                /* :806-895 */
void go_pair_table_whole(const uint16_t *row_i, const uint16_t *row_j, int n_samples, uint32_t t[16]); /* :749-800 */

/* ---- a17: KSA screening statistic (algorithms/epistasis_func.cpp:424-470) ---- */
double go_ksa(const uint32_t ca[16], const uint32_t co[16], const go_marginal_information *m1,
              const go_marginal_information *m2, int n_individs);
/* ---- a18: exact log-linear G-test by IPF + allele-joint log-odds z (epistasis_func.cpp:508-704) ---- */
void go_gtest(const uint32_t ca[16], const uint32_t co[16], const go_marginal_information *m1,
              const go_marginal_information *m2, uint32_t n_individs, double *stat, double *z);
/* The same with the sweep count and the error scale S = sum |terms added into inter| + |ln tao|. A fit that has not
 * converged after GO_IPF_MAX_SWEEPS sweeps (the reference never returns) gives stat = NaN and GO_IPF_MAX_SWEEPS + 1 sweeps. */
#define GO_IPF_MAX_SWEEPS 1000000u
void go_gtest_ex(const uint32_t ca[16], const uint32_t co[16], const go_marginal_information *m1,
                 const go_marginal_information *m2, uint32_t n_individs, double *stat, double *z, uint32_t *sweeps,
                 double *s_out);
/* ---- a19: pairwise_epi_test (src/test/pairwise.c:50-133) and pchisq upper tail (closed forms) ---- */
double go_pairwise_epi_test(const int cs[9], const int ct[9]);
double go_chisq_upper(double x, int df);

/* ---- not in the reference (parity unpinned): allelic 2x2 and genotypic 2x3 Pearson chi-square ---- */
void go_chi2_allelic(const uint32_t ca[4], const uint32_t co[4], double *chi2, double *p);
void go_chi2_genotypic(const uint32_t ca[4], const uint32_t co[4], double *chi2, double *p, int *df);

/* ---- whole-table drivers over a selected store (rows of 2*(Pca+Pco) blocks) ---- */
void go_compute_margins(const uint16_t *sel, long n_snps, int n_case, int n_ctrl,
                        go_marginal_information *out);                 /* epistasis_func.cpp:706-721 */
/* computeBoost pre-screen (epistasis_func.cpp:397-486) over pairs (i,j), i in [i0,i1), j in (i, n_snps).
 * Writes up to cap hits {i, j, stat > threshold} in (i,j) order; returns the number found.
 * stats_out (may be NULL): [0] pairs visited, [1] NaN statistics, [2] min, [3] max. */
long go_boost_screen(const uint16_t *sel, const go_marginal_information *mar, long n_snps, int n_case,
                     int n_ctrl, long i0, long i1, double threshold, uint32_t *hit_i, uint32_t *hit_j,
                     double *hit_stat, long cap, double *stats_out);

/* ---- synthetic cohort: fixed-seed restatement of data/simulate_data.cpp:160-207 (see DESIGN.md) ---- */
uint64_t go_sim_hash(uint64_t seed, uint64_t a, uint64_t b);
/* codes[n_samples]: 0 major hom "AA", 1 het "AC", 2 minor hom "CC", 3 missing */
void go_sim_row_codes(uint64_t seed, const uint32_t bin_counts[51], long snp, int n_samples,
                      uint32_t missing_q32, uint8_t *codes);
void go_sim_phenotype(uint64_t seed, int n_samples, int n_case, uint8_t *pheno);
/* number of minor alleles the generator places in SNP `snp` (= floor(p * 2N)) */
uint64_t go_sim_minor_alleles(uint64_t seed, const uint32_t bin_counts[51], long snp, int n_samples);

#ifdef __cplusplus
}
#endif
#endif
