/* TEST INFRASTRUCTURE -- NOT PRODUCT CODE.  See gwas_oracle.h for scope, pinning status and the
 * citation convention (paths relative to /root/reference/src/libgwaspp). */
#include "gwas_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define POPC16(x) __builtin_popcount((unsigned)(uint16_t)(x))

/* ------------------------------------------------------------------------------------------------
 * geometry: "always pad the blocks per row by 1" then round up to a 64-bit word (4 blocks)
 * compressed_genotype_table5.cpp:55-64 (rows), :449-463 (case/control streams), case_control_set.cpp:38-52
 * ---------------------------------------------------------------------------------------------- */
int go_plane_blocks(int n) {
    int b = n / 16 + 1;
    if (b % 4) b += 4 - b % 4;
    return b;
}

/* ------------------------------------------------------------------------------------------------
 * a4 + a6: row loader. Alphabet "ACGT" (genotype.h:81); enc = 4*idx(c1)+idx(c2); anything else is
 * unknown (compressed_genotype_table5.cpp:94-118). Codes: first homozygote seen -> 1 (plane1),
 * heterozygote -> 2 (plane2), second homozygote -> 3 (both planes) (common_genotype.h:257-304).
 * The 16-bit header keeps state<<12 | enc1<<8 | enc2<<4 | enc3, including the reference's
 * "head_val &= clear_code" masking, so headers compare bit-for-bit.
 * ---------------------------------------------------------------------------------------------- */
static int allele_index(unsigned char c) {
    switch (c) { case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': return 3; default: return 4; }
}
static int enc_is_hom(int enc) { return enc == 0 || enc == 5 || enc == 10 || enc == 15; } /* :1220-1223 */

typedef struct { uint16_t state, head; int16_t code_of[16]; } label_machine;

static void lm_init(label_machine *lm) { lm->state = 0; lm->head = 0; memset(lm->code_of, 0xFF, sizeof lm->code_of); }

/* returns the 2-bit code for enc, or -1 where HeaderStateMachine's asserts (or the
 * `assert( geno_code < 0x7000 )` at :325) would abort the reference. */
static int lm_code(label_machine *lm, int enc) {
    if (lm->code_of[enc] >= 0) return lm->code_of[enc];
    int hom = enc_is_hom(enc), code, shift;
    uint16_t clear, next;
    switch (lm->state) {
    case 0x0000: clear = 0x0000; if (hom) { next = 0x1000; shift = 8; code = 1; } else { next = 0x2000; shift = 4; code = 2; } break;
    case 0x1000: clear = 0x0F00; if (hom) { next = 0x3000; shift = 0; code = 3; } else { next = 0x4000; shift = 4; code = 2; } break;
    case 0x2000: if (!hom) return -1; clear = 0x00F0; next = 0x4000; shift = 8; code = 1; break;
    case 0x3000: if (hom) return -1;  clear = 0x0F0F; next = 0x7000; shift = 4; code = 2; break;
    case 0x4000: if (!hom) return -1; clear = 0x0FF0; next = 0x7000; shift = 0; code = 3; break;
    default: return -1;
    }
    lm->state = next;
    lm->head = (uint16_t)((lm->head & clear) | next | (enc << shift));
    lm->code_of[enc] = (int16_t)code;
    return code;
}

static void row_set(uint16_t *row, int P, int col, int code) {
    if (code & 1) row[1 + (col >> 4)] |= (uint16_t)(1u << (col & 15));       /* plane1: codes 1,3 */
    if (code & 2) row[1 + P + (col >> 4)] |= (uint16_t)(1u << (col & 15));   /* plane2: codes 2,3 */
}

int go_pack_row_text(const char *txt, long len, int n_samples, uint16_t *row) {
    int P = go_plane_blocks(n_samples);
    memset(row, 0, sizeof(uint16_t) * (size_t)(2 * P + 1));
    label_machine lm; lm_init(&lm);
    /* 2 allele characters + 1 delimiter per sample; the last delimiter is optional (:309-357) */
    long pos = 0;
    for (int col = 0; col < n_samples && pos + 1 < len; ++col, pos += 3) {
        int a = allele_index((unsigned char)txt[pos]), b = allele_index((unsigned char)txt[pos + 1]);
        if (a < 4 && b < 4) {
            int code = lm_code(&lm, 4 * a + b);
            if (code < 0) return -1;
            row_set(row, P, col, code);
        }
    }
    row[0] = lm.head;
    return 0;
}

int go_pack_row_codes(const uint8_t *codes, int n_samples, uint16_t *row) {
    static const int enc_of[5] = {0 /*AA*/, 1 /*AC*/, 5 /*CC*/, -1, 4 /*CA*/};
    int P = go_plane_blocks(n_samples);
    memset(row, 0, sizeof(uint16_t) * (size_t)(2 * P + 1));
    label_machine lm; lm_init(&lm);
    for (int col = 0; col < n_samples; ++col) {
        int enc = enc_of[codes[col]];
        if (enc < 0) continue;
        int code = lm_code(&lm, enc);
        if (code < 0) return -1;
        row_set(row, P, col, code);
    }
    row[0] = lm.head;
    return 0;
}

void go_call_at(const uint16_t *row, int n_samples, int col, char out[3]) {
    static const char letters[] = "ACGT";
    int P = go_plane_blocks(n_samples);
    int b1 = (row[1 + (col >> 4)] >> (col & 15)) & 1, b2 = (row[1 + P + (col >> 4)] >> (col & 15)) & 1;
    int enc;
    if (b1 && b2) enc = row[0] & 0x000F;
    else if (b1) enc = (row[0] & 0x0F00) >> 8;
    else if (b2) enc = (row[0] & 0x00F0) >> 4;
    else { out[0] = '0'; out[1] = '0'; out[2] = 0; return; }   /* err_lookup = "00" (:137-139) */
    out[0] = letters[enc >> 2]; out[1] = letters[enc & 3]; out[2] = 0;
}

/* ------------------------------------------------------------------------------------------------
 * a7: stream masks
 * ---------------------------------------------------------------------------------------------- */
void go_stream_masks(const uint8_t *pheno, int n_samples, uint16_t *case_mask, uint16_t *ctrl_mask,
                     int *n_case, int *n_ctrl) {
    int P = go_plane_blocks(n_samples), nca = 0, nco = 0;
    memset(case_mask, 0, sizeof(uint16_t) * (size_t)P);
    memset(ctrl_mask, 0, sizeof(uint16_t) * (size_t)P);
    for (int s = 0; s < n_samples; ++s) {
        if (pheno[s] == 1) { case_mask[s >> 4] |= (uint16_t)(1u << (s & 15)); ++nca; }
        else if (pheno[s] == 0) { ctrl_mask[s >> 4] |= (uint16_t)(1u << (s & 15)); ++nco; }
    }
    if (n_case) *n_case = nca;
    if (n_ctrl) *n_ctrl = nco;
}

/* ------------------------------------------------------------------------------------------------
 * a8: compaction into dense case / control streams, ascending sample order within a class; a sample
 * flagged in both masks counts as a case (`if( _case & mask ) ... else if( _ctrl & mask )`, :541-561).
 * ---------------------------------------------------------------------------------------------- */
void go_select_row(const uint16_t *row, int n_samples, const uint16_t *case_mask,
                   const uint16_t *ctrl_mask, int n_case, int n_ctrl, uint16_t *out) {
    int P = go_plane_blocks(n_samples), Pca = go_plane_blocks(n_case), Pco = go_plane_blocks(n_ctrl);
    memset(out, 0, sizeof(uint16_t) * (size_t)(2 * (Pca + Pco)));
    uint16_t *ca1 = out, *ca2 = out + Pca, *co1 = out + 2 * Pca, *co2 = out + 2 * Pca + Pco;
    int kca = 0, kco = 0;
    for (int s = 0; s < P * 16; ++s) {
        int blk = s >> 4, bit = s & 15;
        int b1 = (row[1 + blk] >> bit) & 1, b2 = (row[1 + P + blk] >> bit) & 1;
        if ((case_mask[blk] >> bit) & 1) {
            if (b1) ca1[kca >> 4] |= (uint16_t)(1u << (kca & 15));
            if (b2) ca2[kca >> 4] |= (uint16_t)(1u << (kca & 15));
            ++kca;
        } else if ((ctrl_mask[blk] >> bit) & 1) {
            if (b1) co1[kco >> 4] |= (uint16_t)(1u << (kco & 15));
            if (b2) co2[kco >> 4] |= (uint16_t)(1u << (kco & 15));
            ++kco;
        }
    }
}

/* ------------------------------------------------------------------------------------------------
 * a9 / a21: counts. aa = popc(p1) - popc(p1&p2), ab = popc(p2) - popc(p1&p2), bb = popc(p1&p2).
 * ---------------------------------------------------------------------------------------------- */
static void stream_counts(const uint16_t *p1, const uint16_t *p2, const uint16_t *mask, int blocks,
                          uint32_t n_class, uint32_t out[4]) {
    uint32_t s1 = 0, s2 = 0, both = 0;
    for (int b = 0; b < blocks; ++b) {
        uint16_t m = mask ? mask[b] : 0xFFFF, x = p1[b] & m, y = p2[b] & m;
        s1 += POPC16(x); s2 += POPC16(y); both += POPC16(x & y);
    }
    out[0] = s1 - both; out[1] = s2 - both; out[2] = both;
    out[3] = n_class - out[0] - out[1] - out[2];   /* :649-653, :693-697, :737-741 */
}

void go_cc_counts_selected(const uint16_t *sel, int n_case, int n_ctrl, uint32_t out[8]) {
    int Pca = go_plane_blocks(n_case), Pco = go_plane_blocks(n_ctrl);
    stream_counts(sel, sel + Pca, NULL, Pca, (uint32_t)n_case, out);
    stream_counts(sel + 2 * Pca, sel + 2 * Pca + Pco, NULL, Pco, (uint32_t)n_ctrl, out + 4);
}

void go_cc_counts_masked(const uint16_t *row, int n_samples, const uint16_t *case_mask,
                         const uint16_t *ctrl_mask, int n_case, int n_ctrl, uint32_t out[8]) {
    int P = go_plane_blocks(n_samples);
    stream_counts(row + 1, row + 1 + P, case_mask, P, (uint32_t)n_case, out);
    stream_counts(row + 1, row + 1 + P, ctrl_mask, P, (uint32_t)n_ctrl, out + 4);
}

/* whole cohort: xx = popc(~(p1|p2)) over the PADDED words, i.e. padding bits count as missing
 * (:600; SURVEY.md defect D5). The harness prints N - (aa+ab+bb) instead (maf_func.cpp:332). */
void go_counts_whole(const uint16_t *row, int n_samples, uint32_t out[4]) {
    int P = go_plane_blocks(n_samples);
    uint32_t s1 = 0, s2 = 0, both = 0, none = 0;
    for (int b = 0; b < P; ++b) {
        uint16_t x = row[1 + b], y = row[1 + P + b];
        s1 += POPC16(x); s2 += POPC16(y); both += POPC16(x & y); none += POPC16((uint16_t)~(x | y));
    }
    out[0] = s1 - both; out[1] = s2 - both; out[2] = both; out[3] = none;
}

/* ------------------------------------------------------------------------------------------------
 * a10: marginal information. Entries belonging to zero counts are never written by the reference
 * (:202-215); under the zeroing allocator of the oracle build they read as 0.0, which is what the
 * struct holds here after the memset.
 * ---------------------------------------------------------------------------------------------- */
void go_marginal_information_fill(const uint32_t ca[4], const uint32_t co[4], uint32_t n_individs,
                                  go_marginal_information *m) {
    memset(m, 0, sizeof *m);
    memcpy(m->cases, ca, 16);
    memcpy(m->controls, co, 16);
    uint32_t n_ca = ca[0] + ca[1] + ca[2] + ca[3], n_co = co[0] + co[1] + co[2] + co[3];
    for (int g = 0; g < 4; ++g) {
        uint32_t mar = ca[g] + co[g];
        m->margins[g] = mar;
        if (mar > 0) { double t = (double)mar / (double)n_individs; m->entropy += -(t)*log(t); }
        if (ca[g] > 0) {
            double t = (double)ca[g] / n_individs;
            m->entropy_y += -(t)*log(t);
            m->pbc[g] = (double)ca[g] / (double)n_ca;
            m->pca[g] = (double)ca[g] / mar;
        }
        if (co[g] > 0) {
            double t = (double)co[g] / n_individs;
            m->entropy_y += -(t)*log(t);
            m->pbc[4 + g] = (double)co[g] / (double)n_co;
            m->pca[4 + g] = (double)co[g] / (double)mar;
        }
    }
}

double go_maf_reference(const uint32_t ft[4], double *tot_out) {
    double tot = ft[0], maf = 2.0 * tot;
    tot += ft[1]; maf += ft[1];
    tot += ft[2];
    maf /= tot;
    if (maf < 0.5) maf = 1.0 - maf;
    if (tot_out) *tot_out = tot;
    return maf;
}

/* ------------------------------------------------------------------------------------------------
 * a14 / a21: pair tables. One-hot decode of the two planes: bb = p1&p2, aa = p1^bb, ab = p2^bb,
 * xx = ~(p1|p2) (compressed_genotype_table5.h:104-115).
 * ---------------------------------------------------------------------------------------------- */
typedef struct { uint16_t g[4]; } onehot;   /* aa, ab, bb, xx */
static onehot decode(uint16_t p1, uint16_t p2) {
    onehot o; o.g[2] = p1 & p2; o.g[0] = p1 ^ o.g[2]; o.g[1] = p2 ^ o.g[2]; o.g[3] = (uint16_t)~(p1 | p2);
    return o;
}

/* full 4x4 accumulation over `blocks` blocks with optional mask (mask applied to the planes BEFORE
 * the decode, so masked-out samples decode as xx -- :826-857, defect D6). */
static void table_full(const uint16_t *a1, const uint16_t *a2, const uint16_t *b1, const uint16_t *b2,
                       const uint16_t *mask, int blocks, uint32_t t[16]) {
    for (int k = 0; k < blocks; ++k) {
        uint16_t m = mask ? mask[k] : 0xFFFF;
        onehot A = decode(a1[k] & m, a2[k] & m), B = decode(b1[k] & m, b2[k] & m);
        for (int r = 0; r < 4; ++r)
            for (int c = 0; c < 4; ++c) t[4 * r + c] += POPC16(A.g[r] & B.g[c]);
    }
}
static void table_core9(const uint16_t *a1, const uint16_t *a2, const uint16_t *b1, const uint16_t *b2,
                        int blocks, uint32_t t[16]) {
    for (int k = 0; k < blocks; ++k) {
        onehot A = decode(a1[k], a2[k]), B = decode(b1[k], b2[k]);
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) t[4 * r + c] += POPC16(A.g[r] & B.g[c]);
    }
}
static void table_corners(const uint16_t *a1, const uint16_t *a2, const uint16_t *b1, const uint16_t *b2,
                          int blocks, uint32_t t[16]) {
    for (int k = 0; k < blocks; ++k) {
        onehot A = decode(a1[k], a2[k]), B = decode(b1[k], b2[k]);
        t[0] += POPC16(A.g[0] & B.g[0]); t[2] += POPC16(A.g[0] & B.g[2]);
        t[8] += POPC16(A.g[2] & B.g[0]); t[10] += POPC16(A.g[2] & B.g[2]);
    }
}
/* xx row/column from the per-SNP class margins (:1022-1030, :1060-1067) */
static void fill_xx_from_margins(uint32_t t[16], const uint32_t m1[4], const uint32_t m2[4]) {
    t[3] = m1[0] - t[0] - t[2] - t[1];
    t[7] = m1[1] - t[4] - t[6] - t[5];
    t[11] = m1[2] - t[10] - t[8] - t[9];
    t[12] = m2[0] - t[0] - t[8] - t[4];
    t[13] = m2[1] - t[1] - t[9] - t[5];
    t[14] = m2[2] - t[2] - t[10] - t[6];
    t[15] = m2[3] - t[3] - t[7] - t[11];
}
/* no-missing shortcut: cross cells from margins (:1084-1092, :1133-1141); xx cells stay 0 */
static void fill_cross_from_margins(uint32_t t[16], const uint32_t m1[4], const uint32_t m2[4]) {
    t[1] = m1[0] - t[0] - t[2];
    t[9] = m1[2] - t[10] - t[8];
    t[4] = m2[0] - t[0] - t[8];
    t[6] = m2[2] - t[2] - t[10];
    t[5] = m2[1] - t[1] - t[9];
}

void go_pair_table_margins(const uint16_t *si, const uint16_t *sj, int n_case, int n_ctrl,
                           const go_marginal_information *m1, const go_marginal_information *m2,
                           uint32_t ca[16], uint32_t co[16]) {
    int Pca = go_plane_blocks(n_case), Pco = go_plane_blocks(n_ctrl);
    memset(ca, 0, 64); memset(co, 0, 64);
    const uint16_t *ci = si + 2 * Pca, *cj = sj + 2 * Pca;
    if (m1->cases[3] + m1->controls[3] + m2->cases[3] + m2->controls[3]) {   /* :1000 */
        table_core9(si, si + Pca, sj, sj + Pca, Pca, ca);
        fill_xx_from_margins(ca, m1->cases, m2->cases);
        table_core9(ci, ci + Pco, cj, cj + Pco, Pco, co);
        fill_xx_from_margins(co, m1->controls, m2->controls);
    } else {
        table_corners(si, si + Pca, sj, sj + Pca, Pca, ca);
        fill_cross_from_margins(ca, m1->cases, m2->cases);
        table_corners(ci, ci + Pco, cj, cj + Pco, Pco, co);
        fill_cross_from_margins(co, m1->controls, m2->controls);
    }
}

void go_pair_table_selected(const uint16_t *si, const uint16_t *sj, int n_case, int n_ctrl,
                            uint32_t ca[16], uint32_t co[16]) {
    int Pca = go_plane_blocks(n_case), Pco = go_plane_blocks(n_ctrl);
    memset(ca, 0, 64); memset(co, 0, 64);
    table_full(si, si + Pca, sj, sj + Pca, NULL, Pca, ca);
    table_full(si + 2 * Pca, si + 2 * Pca + Pco, sj + 2 * Pca, sj + 2 * Pca + Pco, NULL, Pco, co);
}

void go_pair_table_masked(const uint16_t *ri, const uint16_t *rj, int n_samples,
                          const uint16_t *case_mask, const uint16_t *ctrl_mask,
                          uint32_t ca[16], uint32_t co[16]) {
    int P = go_plane_blocks(n_samples);
    memset(ca, 0, 64); memset(co, 0, 64);
    table_full(ri + 1, ri + 1 + P, rj + 1, rj + 1 + P, case_mask, P, ca);
    table_full(ri + 1, ri + 1 + P, rj + 1, rj + 1 + P, ctrl_mask, P, co);
}

void go_pair_table_whole(const uint16_t *ri, const uint16_t *rj, int n_samples, uint32_t t[16]) {
    int P = go_plane_blocks(n_samples);
    memset(t, 0, 64);
    table_full(ri + 1, ri + 1 + P, rj + 1, rj + 1 + P, NULL, P, t);
}

/* ------------------------------------------------------------------------------------------------
 * a17: KSA screening statistic. For cell (a,b), class k:
 *   Pab = (ca_ab + co_ab) / margins2[b];  p_k = Pab * Pbc_k(m2)[b] * Pca_k(m1)[a];  tau = sum p
 *   I = sum_{c>0} (c/n) ln(c/n)  -  sum_{c>0, p>0} (c/n) ln p ;   stat = 2n (I + ln tau)
 * Same accumulation order as epistasis_func.cpp:424-470 (cases before controls inside a cell,
 * cells row-major). A zero margins2[b] gives 0/0 = NaN, which propagates into stat.
 * ---------------------------------------------------------------------------------------------- */
double go_ksa(const uint32_t ca[16], const uint32_t co[16], const go_marginal_information *m1,
              const go_marginal_information *m2, int n_individs) {
    double tao = 0.0, inter = 0.0;
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) {
            uint32_t nca = ca[4 * a + b], nco = co[4 * a + b];
            double pab = (double)(nca + nco) / (double)m2->margins[b];
            double t2 = pab * m2->pbc[b] * m1->pca[a];
            double t3 = pab * m2->pbc[4 + b] * m1->pca[4 + a];
            tao += t2 + t3;
            if (nca > 0) {
                double t1 = (double)nca / n_individs;
                inter += t1 * log(t1);
                if (t2 > 0) inter += -t1 * log(t2);
            }
            if (nco > 0) {
                double t1 = (double)nco / n_individs;
                inter += t1 * log(t1);
                if (t3 > 0) inter += -t1 * log(t3);
            }
        }
    return (inter + log(tao)) * n_individs * 2.0;
}

/* ------------------------------------------------------------------------------------------------
 * a18: exact homogeneous-association G-test by iterative proportional fitting, then the
 * allele-joint log-odds z.  mu is [class][a][b], started at all ones; one sweep = (1) rescale so
 * that mu_ab. = n_ab. while accumulating mu_a.k and mu_.bk, (2) multiply every cell by
 * (n_a.k / mu_a.k)(n_.bk / mu_.bk) using the per-SNP class margins; stop when sum|delta| <= 1e-3.
 * ---------------------------------------------------------------------------------------------- */
/* The reference loops until convergence; on some sparse tables sum |delta| settles on a cycle (the update multiplies by
 * the row and the column ratio at once) and it never returns. Here, as in gtest_kernel, a fit that has not converged
 * after GO_IPF_MAX_SWEEPS sweeps gives stat = NaN and reports GO_IPF_MAX_SWEEPS + 1 sweeps; z is computed regardless.
 * go_gtest_ex also returns the sweeps run and S = sum of |every term added into inter| + |ln tao|, the scale of the
 * rounding error of the statistic (2n * S * a few ulp). */
void go_gtest_ex(const uint32_t ca[16], const uint32_t co[16], const go_marginal_information *m1,
                 const go_marginal_information *m2, uint32_t n_individs, double *stat, double *z, uint32_t *sweeps_out,
                 double *s_out) {
    double mu[2][9], mu0[2][9], mu_ik[2][3], mu_jk[2][3];
    for (int i = 0; i < 9; ++i) { mu[0][i] = mu[1][i] = 1.0; }
    double err = 18.0;   /* the reference's first error loop never advances its pointers (:551-553) */
    uint32_t sweeps = 0;
    while (err > 0.001 && sweeps <= GO_IPF_MAX_SWEEPS) {
        ++sweeps;
        memcpy(mu0, mu, sizeof mu);
        memset(mu_ik, 0, sizeof mu_ik);
        memset(mu_jk, 0, sizeof mu_jk);
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) {
                int i = 3 * a + b;
                double s = mu[0][i] + mu[1][i];
                uint32_t nab = ca[4 * a + b] + co[4 * a + b];
                if (s > 0) { mu[0][i] = mu[0][i] * nab / s; mu[1][i] = mu[1][i] * nab / s; }
                else { mu[0][i] = 0; mu[1][i] = 0; }
                mu_ik[0][a] += mu[0][i]; mu_ik[1][a] += mu[1][i];
                mu_jk[0][b] += mu[0][i]; mu_jk[1][b] += mu[1][i];
            }
        err = 0.0;
        for (int a = 0; a < 3; ++a) {
            double r1 = mu_ik[0][a] > 0 ? m1->cases[a] / mu_ik[0][a] : 0.0;
            double r2 = mu_ik[1][a] > 0 ? m1->controls[a] / mu_ik[1][a] : 0.0;
            for (int b = 0; b < 3; ++b) {
                int i = 3 * a + b;
                double r3 = mu_jk[0][b] > 0 ? m2->cases[b] / mu_jk[0][b] : 0.0;
                double r4 = mu_jk[1][b] > 0 ? m2->controls[b] / mu_jk[1][b] : 0.0;
                mu[0][i] = mu[0][i] * r1 * r3;
                mu[1][i] = mu[1][i] * r2 * r4;
                err += fabs(mu[0][i] - mu0[0][i]);
                err += fabs(mu[1][i] - mu0[1][i]);
            }
        }
    }
    double tao = 0.0, inter = 0.0, S = 0.0, term;
#define GO_ADD(x) (term = (x), inter += term, S += fabs(term))
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) {
            int i = 3 * a + b;
            double t1, t2;
            uint32_t nca = ca[4 * a + b], nco = co[4 * a + b];
            if (nca > 0) { t1 = (double)nca / n_individs; GO_ADD(t1 * log(t1)); } else t1 = 0.0;
            if (mu[0][i] > 0) { t2 = mu[0][i] / n_individs; GO_ADD(-t1 * log(t2)); tao += t2; }
            if (nco > 0) { t1 = (double)nco / n_individs; GO_ADD(t1 * log(t1)); } else t1 = 0.0;
            if (mu[1][i] > 0) { t2 = mu[1][i] / n_individs; GO_ADD(-t1 * log(t2)); tao += t2; }
        }
#undef GO_ADD
    *stat = sweeps > GO_IPF_MAX_SWEEPS ? NAN : (inter + log(tao)) * n_individs * 2.0;
    if (sweeps_out) *sweeps_out = sweeps;
    if (s_out) *s_out = S + fabs(log(tao));

    /* allele-joint distribution from cells {0,1,2,4,5,6,8,9,10} in 32-bit unsigned arithmetic,
     * products included (:686-700) */
    uint32_t d[8];
    const uint32_t *t = ca;
    for (int k = 0; k < 2; ++k, t = co) {
        d[4 * k + 0] = (t[0] << 2) + (t[1] << 1) + (t[4] << 1) + t[5];
        d[4 * k + 1] = (t[2] << 2) + (t[1] << 1) + (t[6] << 1) + t[5];
        d[4 * k + 2] = (t[8] << 2) + (t[9] << 1) + (t[4] << 1) + t[5];
        d[4 * k + 3] = (t[10] << 2) + (t[9] << 1) + (t[6] << 1) + t[5];
    }
    double or_aff = log((double)(d[0] * d[3]) / (double)(d[1] * d[2]));
    double v_aff = 1 / (double)d[0] + 1 / (double)d[1] + 1 / (double)d[2] + 1 / (double)d[3];
    double or_unf = log((double)(d[4] * d[7]) / (double)(d[5] * d[6]));
    double v_unf = 1 / (double)d[4] + 1 / (double)d[5] + 1 / (double)d[6] + 1 / (double)d[7];
    *z = (or_aff - or_unf) / sqrt(v_aff + v_unf);
}

void go_gtest(const uint32_t ca[16], const uint32_t co[16], const go_marginal_information *m1,
              const go_marginal_information *m2, uint32_t n_individs, double *stat, double *z) {
    go_gtest_ex(ca, co, m1, m2, n_individs, stat, z, NULL, NULL);
}

/* ------------------------------------------------------------------------------------------------
 * a19: stand-alone KSA likelihood ratio from the 3x3x2 table alone (src/test/pairwise.c:50-133):
 * margins re-derived from the table, p(control | A) taken as 1 - p(case | A).
 * ---------------------------------------------------------------------------------------------- */
double go_pairwise_epi_test(const int cs[9], const int ct[9]) {
    int cn[9], cs1[3] = {0, 0, 0}, cs2[3] = {0, 0, 0}, ct1[3] = {0, 0, 0}, ct2[3] = {0, 0, 0};
    int c1[3] = {0, 0, 0}, c2[3] = {0, 0, 0}, ns = 0, nt = 0, n = 0;
    for (int a = 0; a < 3; ++a) {
        for (int b = 0; b < 3; ++b) {
            int i = 3 * a + b;
            cn[i] = cs[i] + ct[i];
            cs1[a] += cs[i]; cs2[b] += cs[i];
            ct1[a] += ct[i]; ct2[b] += ct[i];
            c1[a] += cn[i]; c2[b] += cn[i];
        }
        ns += cs1[a]; nt += ct1[a]; n += c1[a];
    }
    double ll = 0.0, tao = 0.0;
    for (int a = 0; a < 3; ++a) {
        double psa = (double)cs1[a] / c1[a], pta = 1.0 - psa;
        for (int b = 0; b < 3; ++b) {
            int i = 3 * a + b;
            double pab = (double)cn[i] / c2[b];
            double pbs = (double)cs2[b] / ns, pbt = (double)ct2[b] / nt;
            if (cs[i] > 0) ll += cs[i] * log((double)cs[i] / n);
            if (ct[i] > 0) ll += ct[i] * log((double)ct[i] / n);
            double ps = pab * pbs * psa, pt = pab * pbt * pta;
            tao += ps + pt;
            if (ps > 0) ll -= cs[i] * log(ps);
            if (pt > 0) ll -= ct[i] * log(pt);
        }
    }
    ll += n * log(tao);
    return 2.0 * ll;
}

/* pchisq(x, df, lower=0, log=0) of R's standalone Rmath (un-vendored dependency, unpinned version;
 * call sites epistasis_func.cpp:242,294,340 and src/test/pairwise.c:44). Closed forms for the
 * integer degrees of freedom this path can ask for. */
double go_chisq_upper(double x, int df) {
    if (!(x > 0.0)) return x != x ? x : 1.0;
    switch (df) {
    case 1: return erfc(sqrt(0.5 * x));
    case 2: return exp(-0.5 * x);
    case 4: return exp(-0.5 * x) * (1.0 + 0.5 * x);
    default: return NAN;
    }
}

/* ------------------------------------------------------------------------------------------------
 * PARITY UNPINNED (no counterpart in the reference; specification in DESIGN.md / SURVEY.md 8c):
 * allelic 2x2 chi-square on allele counts A_k = 2 aa_k + ab_k, B_k = 2 bb_k + ab_k (df 1) and the
 * genotypic 2x3 Pearson chi-square over non-empty genotype columns (df = columns - 1).
 * Missing genotypes excluded. Degenerate tables give chi2 = 0, p = 1 (df = 0).
 * ---------------------------------------------------------------------------------------------- */
void go_chi2_allelic(const uint32_t ca[4], const uint32_t co[4], double *chi2, double *p) {
    double a_ca = 2.0 * ca[0] + ca[1], b_ca = 2.0 * ca[2] + ca[1];
    double a_co = 2.0 * co[0] + co[1], b_co = 2.0 * co[2] + co[1];
    double r1 = a_ca + b_ca, r2 = a_co + b_co, c1 = a_ca + a_co, c2 = b_ca + b_co, t = r1 + r2;
    if (r1 == 0 || r2 == 0 || c1 == 0 || c2 == 0) { *chi2 = 0.0; *p = 1.0; return; }
    double d = a_ca * b_co - b_ca * a_co;
    *chi2 = t * d * d / (r1 * r2 * c1 * c2);
    *p = go_chisq_upper(*chi2, 1);
}

void go_chi2_genotypic(const uint32_t ca[4], const uint32_t co[4], double *chi2, double *p, int *df_out) {
    double r1 = (double)ca[0] + ca[1] + ca[2], r2 = (double)co[0] + co[1] + co[2], t = r1 + r2;
    int cols = 0;
    double x = 0.0;
    if (r1 > 0 && r2 > 0)
        for (int g = 0; g < 3; ++g) {
            double c = (double)ca[g] + co[g];
            if (c == 0) continue;
            ++cols;
            double e1 = r1 * c / t, e2 = r2 * c / t;
            x += (ca[g] - e1) * (ca[g] - e1) / e1 + (co[g] - e2) * (co[g] - e2) / e2;
        }
    int df = cols > 1 ? cols - 1 : 0;
    if (df_out) *df_out = df;
    if (df == 0) { *chi2 = 0.0; *p = 1.0; return; }
    *chi2 = x;
    *p = go_chisq_upper(x, df);
}

/* ------------------------------------------------------------------------------------------------
 * drivers
 * ---------------------------------------------------------------------------------------------- */
void go_compute_margins(const uint16_t *sel, long n_snps, int n_case, int n_ctrl,
                        go_marginal_information *out) {
    long stride = 2L * (go_plane_blocks(n_case) + go_plane_blocks(n_ctrl));
    for (long i = 0; i < n_snps; ++i) {
        uint32_t c[8];
        go_cc_counts_selected(sel + i * stride, n_case, n_ctrl, c);
        go_marginal_information_fill(c, c + 4, (uint32_t)(n_case + n_ctrl), &out[i]);
    }
}

long go_boost_screen(const uint16_t *sel, const go_marginal_information *mar, long n_snps, int n_case,
                     int n_ctrl, long i0, long i1, double threshold, uint32_t *hit_i, uint32_t *hit_j,
                     double *hit_stat, long cap, double *stats_out) {
    long stride = 2L * (go_plane_blocks(n_case) + go_plane_blocks(n_ctrl));
    long found = 0, visited = 0, nans = 0;
    double mx = -99999999, mn = 999999999;
    for (long i = i0; i < i1 && i < n_snps; ++i)
        for (long j = i + 1; j < n_snps; ++j) {
            uint32_t ca[16], co[16];
            go_pair_table_margins(sel + i * stride, sel + j * stride, n_case, n_ctrl, &mar[i], &mar[j], ca, co);
            double s = go_ksa(ca, co, &mar[i], &mar[j], n_case + n_ctrl);
            ++visited;
            if (s != s) ++nans;
            if (s > mx) mx = s;
            if (s < mn) mn = s;
            if (s > threshold) {
                if (found < cap) { hit_i[found] = (uint32_t)i; hit_j[found] = (uint32_t)j; hit_stat[found] = s; }
                ++found;
            }
        }
    if (stats_out) { stats_out[0] = (double)visited; stats_out[1] = (double)nans; stats_out[2] = mn; stats_out[3] = mx; }
    return found;
}

/* ------------------------------------------------------------------------------------------------
 * synthetic cohort. data/simulate_data.cpp draws, per SNP, a MAF bin with probability proportional
 * to the panel's bin count (:177-188), a frequency p = bin% + U{0..999}/100000 (:191-192), puts
 * s = floor(p * 2N) minor alleles on a uniformly random subset of the 2N allele slots (:193-203) and
 * reads sample i from slots (2i, 2i+1). The reference seeds from time() (:57), so this restatement
 * swaps rand()/random_shuffle for a counter-based hash (splitmix64 finaliser over (seed, a, b)) and
 * sequential selection sampling, which draws the same distribution reproducibly and identically on
 * host and device. Alleles are canonicalised to A (major) / C (minor), het written "AC"
 * (SURVEY.md fact 4). missing_q32 / 2^32 is the per-genotype missing probability (parity tests only).
 * ---------------------------------------------------------------------------------------------- */
uint64_t go_sim_hash(uint64_t seed, uint64_t a, uint64_t b) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ULL * (a + 1) + 0xD1B54A32D192ED03ULL * (b + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

#define GO_SIM_STREAM_BIN   0xFFFFFFFF00000001ULL
#define GO_SIM_STREAM_FREQ  0xFFFFFFFF00000002ULL
#define GO_SIM_STREAM_MISS  0x8000000000000000ULL
#define GO_SIM_STREAM_PHENO 0xFFFFFFFF00000003ULL

uint64_t go_sim_minor_alleles(uint64_t seed, const uint32_t bin_counts[51], long snp, int n_samples) {
    uint64_t total = 0;
    for (int b = 0; b < 51; ++b) total += bin_counts[b];
    uint64_t r = go_sim_hash(seed, (uint64_t)snp, GO_SIM_STREAM_BIN) % total, cum = 0;
    int bin = 50;
    for (int b = 0; b < 51; ++b) { cum += bin_counts[b]; if (r < cum) { bin = b; break; } }
    uint64_t frac = go_sim_hash(seed, (uint64_t)snp, GO_SIM_STREAM_FREQ) % 1000;
    return ((1000ULL * (uint64_t)bin + frac) * 2ULL * (uint64_t)n_samples) / 100000ULL;   /* floor(p * 2N) */
}

void go_sim_row_codes(uint64_t seed, const uint32_t bin_counts[51], long snp, int n_samples,
                      uint32_t missing_q32, uint8_t *codes) {
    uint64_t slots = 2ULL * (uint64_t)n_samples;
    uint64_t want = go_sim_minor_alleles(seed, bin_counts, snp, n_samples);
    uint64_t chosen = 0;
    for (int s = 0; s < n_samples; ++s) {
        int minor = 0;
        for (int h = 0; h < 2; ++h) {
            uint64_t t = 2ULL * (uint64_t)s + (uint64_t)h, left = slots - t;
            uint64_t u = go_sim_hash(seed, (uint64_t)snp, t) >> 32;
            if (((u * left) >> 32) < want - chosen) { ++minor; ++chosen; }
        }
        uint8_t code = (uint8_t)minor;
        if (missing_q32 &&
            (uint32_t)(go_sim_hash(seed, (uint64_t)snp, GO_SIM_STREAM_MISS | (uint64_t)s) >> 32) < missing_q32)
            code = 3;
        codes[s] = code;
    }
}

void go_sim_phenotype(uint64_t seed, int n_samples, int n_case, uint8_t *pheno) {
    uint64_t chosen = 0;
    for (int s = 0; s < n_samples; ++s) {
        uint64_t left = (uint64_t)(n_samples - s);
        uint64_t u = go_sim_hash(seed, GO_SIM_STREAM_PHENO, (uint64_t)s) >> 32;
        if (((u * left) >> 32) < (uint64_t)n_case - chosen) { pheno[s] = 1; ++chosen; } else pheno[s] = 0;
    }
}
