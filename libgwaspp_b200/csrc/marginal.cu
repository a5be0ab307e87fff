// K1: per-SNP marginal scan over the compacted case/control store.
//
// One pass over HBM. A warp owns a contiguous range of SNP rows (ranges are balanced to one row across
// all resident warps). G lanes (8, 16 or 32, chosen on the host so that no lane idles for the cohort's
// row length) cooperate on one row, 32/G rows are in flight per warp, and every lane streams 32-byte
// chunk pairs (128 samples of both bit-planes) four at a time. The three popcount streams the counts
// need -- |p1|, |p2|, |p1&p2| -- are accumulated with carry-save adders (Harley-Seal): three LOP3 pairs
// fold four words into ones/twos state and a single POPC of the fours carry, so the XU pipe (POPC runs
// at 16 lanes/clk/SM and was the limiter of the first version, ncu r1a) sees ~3x fewer instructions.
// Totals are reduced inside the lane group with REDUX and parked in lane (row % 32); after 32 rows every
// lane finishes one SNP in fp64: genotype counts (compressed_genotype_table5.cpp:703-747),
// marginal_information (genotype/common_genotype_func.cpp:173-219), MinorAlleleFrequency
// (algorithms/maf_func.h:46-54) and the allelic / genotypic chi-square tests (DESIGN.md; no reference
// counterpart). Bound: HBM bandwidth; algorithmic bytes = n_samples / 4 per SNP.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace gwasdev {

static_assert(sizeof(gwasdev_snp_compact) == 32 && sizeof(gwasdev_sig_snp) == 48 && sizeof(gwasdev_snp_stats) == 64 &&
              sizeof(gwasdev_marginal_information) == 192, "C-ABI record sizes (include/gwasdev.h)");

struct ChunkPair { uint4 x, y; };   // 4 words of plane 1, 4 words of plane 2 (same 128 samples)

__device__ __forceinline__ ChunkPair ld_pair(const uint4 *p, bool pred) {   // read-once: keep out of L1
    ChunkPair c;
    c.x = make_uint4(0, 0, 0, 0); c.y = make_uint4(0, 0, 0, 0);
    if (pred) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(c.x.x), "=r"(c.x.y), "=r"(c.x.z), "=r"(c.x.w) : "l"(p));
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(c.y.x), "=r"(c.y.y), "=r"(c.y.z), "=r"(c.y.w) : "l"(p + 1));
    }
    return c;
}

// carry-save adder: (hi, lo) = a + b + c per bit position
__device__ __forceinline__ void csa(uint32_t &hi, uint32_t &lo, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t u = a ^ b;
    hi = (a & b) | (u & c);
    lo = u ^ c;
}
// one popcount stream: bit-sliced running count (ones, twos) plus a scalar count of fours
struct HS { uint32_t ones, twos, fours4; };
__device__ __forceinline__ void hs_add4(HS &h, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    uint32_t ta, tb, f;
    csa(ta, h.ones, h.ones, w0, w1);
    csa(tb, h.ones, h.ones, w2, w3);
    csa(f, h.twos, h.twos, ta, tb);
    h.fours4 += __popc(f);
}
__device__ __forceinline__ uint32_t hs_total(const HS &h) { return 4 * h.fours4 + 2 * __popc(h.twos) + __popc(h.ones); }

// |p1| and |p2| go through the carry-save adders (ALU pipe), |p1 & p2| through plain POPC (XU pipe): with
// ~6 LOP3 + 1 POPC per carry-save stream and 4 POPC per plain stream, two-and-one balances the two pipes
// (ALU 2 warp-instr/clk/SM, XU 0.5) better than three-and-none or none-and-three (B200 sweep, DESIGN.md).
__device__ __forceinline__ void accumulate_pair(const ChunkPair &c, HS &h1, HS &h2, HS &hb) {
    hs_add4(h1, c.x.x, c.x.y, c.x.z, c.x.w);
    hs_add4(h2, c.y.x, c.y.y, c.y.z, c.y.w);
    hb.ones += __popc(c.x.x & c.y.x) + __popc(c.x.y & c.y.y);
    hb.twos += __popc(c.x.z & c.y.z) + __popc(c.x.w & c.y.w);
}
__device__ __forceinline__ uint32_t plain_total(const HS &h) { return h.ones + h.twos; }

// chi-square upper tail for df in {1, 2}: pchisq(x, df, lower=0) == gsl_cdf_chisq_Q(x, df)
__device__ __forceinline__ double chisq_upper(double x, int df) {
    if (!(x > 0.0)) return x != x ? x : 1.0;
    return df == 1 ? erfc(sqrt(0.5 * x)) : exp(-0.5 * x);
}

// fp64 arithmetic below uses the _rn intrinsics so that nvcc cannot contract a*b+c into an FMA: the
// reference is compiled for x86-64 without FMA and rounds every product and sum separately.
__device__ __noinline__ void fill_marginal_information(const uint32_t ca[4], const uint32_t co[4],
                                                          uint32_t n_individs, gwasdev_marginal_information &m) {
    const uint32_t n_ca = ca[3] + ca[0] + ca[1] + ca[2], n_co = co[3] + co[0] + co[1] + co[2];
    double h = 0.0, hy = 0.0;
    const double n = (double)n_individs;
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {
        const uint32_t mar = ca[g] + co[g];
        m.margins[g] = mar; m.cases[g] = ca[g]; m.controls[g] = co[g];
        // zero-count classes are left unwritten by the reference and read as 0.0 under its zeroing
        // oracle allocator (SURVEY.md defect D1): write the zeros explicitly.
        double pbc_ca = 0.0, pca_ca = 0.0, pbc_co = 0.0, pca_co = 0.0;
        if (mar > 0) { const double t = __ddiv_rn((double)mar, n); h = __dadd_rn(h, __dmul_rn(-t, log(t))); }
        if (ca[g] > 0) {
            const double t = __ddiv_rn((double)ca[g], n);
            hy = __dadd_rn(hy, __dmul_rn(-t, log(t)));
            pbc_ca = __ddiv_rn((double)ca[g], (double)n_ca);
            pca_ca = __ddiv_rn((double)ca[g], (double)mar);
        }
        if (co[g] > 0) {
            const double t = __ddiv_rn((double)co[g], n);
            hy = __dadd_rn(hy, __dmul_rn(-t, log(t)));
            pbc_co = __ddiv_rn((double)co[g], (double)n_co);
            pca_co = __ddiv_rn((double)co[g], (double)mar);
        }
        m.dPbc[g] = pbc_ca; m.dPbc[4 + g] = pbc_co; m.dPca[g] = pca_ca; m.dPca[4 + g] = pca_co;
    }
    m.dMarginalEntropy = h;
    m.dMarginalEntropy_Y = hy;
}

__device__ __forceinline__ double maf_reference(const uint32_t ft[4]) {   // algorithms/maf_func.h:46-54
    double tot = ft[0], maf = 2.0 * tot;
    tot += ft[1]; maf += ft[1];
    tot += ft[2];
    maf /= tot;
    if (maf < 0.5) maf = 1.0 - maf;
    return maf;
}

// The two chi-square statistics of one SNP. Out of line and shared by fill_stats and the permutation test's epilogue
// (permute_gemm.cuh, compiled in this translation unit), so that both run the same compiled fp64 code: a permuted cohort's
// statistics are bit-identical to a scan of that cohort.
struct Chi2 { double allelic, genotypic; int df; };
__device__ __noinline__ Chi2 chi2_tests(const uint32_t ca[4], const uint32_t co[4]) {
    Chi2 r;
    const double a_ca = 2.0 * ca[0] + ca[1], b_ca = 2.0 * ca[2] + ca[1];
    const double a_co = 2.0 * co[0] + co[1], b_co = 2.0 * co[2] + co[1];
    const double r1 = a_ca + b_ca, r2 = a_co + b_co, c1 = a_ca + a_co, c2 = b_ca + b_co, t = r1 + r2;
    // allelic 2x2, df 1
    if (r1 == 0 || r2 == 0 || c1 == 0 || c2 == 0) r.allelic = 0.0;
    else {
        const double d = a_ca * b_co - b_ca * a_co;
        r.allelic = t * d * d / (r1 * r2 * c1 * c2);
    }
    // genotypic 2x3 Pearson over non-empty genotype columns
    const double g1 = (double)ca[0] + ca[1] + ca[2], g2 = (double)co[0] + co[1] + co[2], gt = g1 + g2;
    int cols = 0;
    double x = 0.0;
    if (g1 > 0 && g2 > 0) {
#pragma unroll 1
        for (int g = 0; g < 3; ++g) {
            const double c = (double)ca[g] + co[g];
            if (c == 0) continue;
            ++cols;
            const double e1 = g1 * c / gt, e2 = g2 * c / gt;
            x += (ca[g] - e1) * (ca[g] - e1) / e1 + (co[g] - e2) * (co[g] - e2) / e2;
        }
    }
    r.df = cols > 1 ? cols - 1 : 0;
    r.genotypic = r.df == 0 ? 0.0 : x;
    return r;
}

__device__ __noinline__ void fill_stats(const uint32_t ca[4], const uint32_t co[4], gwasdev_snp_stats &o) {
    o.maf_ref_case = maf_reference(ca);
    o.maf_ref_ctrl = maf_reference(co);
    const double a_ca = 2.0 * ca[0] + ca[1], b_ca = 2.0 * ca[2] + ca[1];
    const double a_co = 2.0 * co[0] + co[1], b_co = 2.0 * co[2] + co[1];
    const double c1 = a_ca + a_co, c2 = b_ca + b_co, t = (a_ca + b_ca) + (a_co + b_co);
    o.maf_pooled = t > 0 ? fmin(c1, c2) / t : nan("");
    const Chi2 x = chi2_tests(ca, co);
    // chisq_upper(0, df) is 1: the p-value of a degenerate table (statistic 0) as well as of a zero statistic
    o.chi2_allelic = x.allelic;
    o.p_allelic = chisq_upper(x.allelic, 1);
    o.df_genotypic = x.df;
    o.chi2_genotypic = x.genotypic;
    o.p_genotypic = chisq_upper(x.genotypic, x.df);
}

// Where one scan writes. Every pointer may be NULL; outputs are indexed from out_base (the first SNP of the call).
struct ScanOut {
    uint32_t *counts;
    gwasdev_marginal_information *mi;
    gwasdev_snp_stats *stats;
    gwasdev_snp_compact *compact;          // 32-byte records for host consumers
    gwasdev_sig_snp *sig;                  // SNPs with min(p_allelic, p_genotypic) < p_thr, appended through n_sig
    unsigned long long *n_sig;
    uint64_t sig_cap;
    double p_thr;
    uint4 *row_tot;                        // K1': per-SNP totals over all samples, indexed by the absolute SNP (written or read)
    uint64_t out_base;
};

// One SNP's epilogue, kept out of line so that the streaming loop stays small in the instruction cache. Two forms: the
// plain one writes counts / marginal_information / statistics straight into the caller's arrays; the compact one (32-byte
// records, significant-SNP list) needs the statistics in registers first and lives in its own function so that its local
// record does not cost the plain scan a stack frame (0.2296 -> 0.2237 ms at configs[1] when the two were one function).
__device__ __forceinline__ void snp_counts(uint32_t m1c, uint32_t m2c, uint32_t mbc, uint32_t m1t, uint32_t m2t, uint32_t mbt,
                                           uint32_t n_case, uint32_t n_ctrl, uint32_t (&ca)[4], uint32_t (&co)[4]) {
    ca[0] = m1c - mbc; ca[1] = m2c - mbc; ca[2] = mbc; ca[3] = n_case - ca[0] - ca[1] - ca[2];
    co[0] = m1t - mbt; co[1] = m2t - mbt; co[2] = mbt; co[3] = n_ctrl - co[0] - co[1] - co[2];
}

__device__ __noinline__ void finish_snp_plain(uint32_t m1c, uint32_t m2c, uint32_t mbc, uint32_t m1t, uint32_t m2t, uint32_t mbt,
                                              uint32_t n_case, uint32_t n_ctrl, uint64_t o, uint32_t *__restrict__ counts,
                                              gwasdev_marginal_information *__restrict__ mi, gwasdev_snp_stats *__restrict__ stats) {
    uint32_t ca[4], co[4];
    snp_counts(m1c, m2c, mbc, m1t, m2t, mbt, n_case, n_ctrl, ca, co);
    if (counts) {
        uint4 *dst = reinterpret_cast<uint4 *>(counts + 8 * o);
        dst[0] = make_uint4(ca[0], ca[1], ca[2], ca[3]);
        dst[1] = make_uint4(co[0], co[1], co[2], co[3]);
    }
    if (mi) fill_marginal_information(ca, co, n_case + n_ctrl, mi[o]);
    if (stats) fill_stats(ca, co, stats[o]);
}

__device__ __noinline__ void finish_snp_compact(uint32_t m1c, uint32_t m2c, uint32_t mbc, uint32_t m1t, uint32_t m2t, uint32_t mbt,
                                                uint32_t n_case, uint32_t n_ctrl, uint64_t snp, const ScanOut &out) {
    const uint64_t o = snp - out.out_base;
    uint32_t ca[4], co[4];
    snp_counts(m1c, m2c, mbc, m1t, m2t, mbt, n_case, n_ctrl, ca, co);
    gwasdev_snp_stats st;
    fill_stats(ca, co, st);
    if (out.compact) {
        uint4 *dst = reinterpret_cast<uint4 *>(out.compact + o);
        dst[0] = make_uint4(ca[0] | (ca[1] << 16), ca[2] | (ca[3] << 16), co[0] | (co[1] << 16), co[2] | (co[3] << 16));
        dst[1] = make_uint4(__float_as_uint((float)st.chi2_allelic), __float_as_uint((float)st.p_allelic),
                            __float_as_uint((float)st.chi2_genotypic), __float_as_uint((float)st.p_genotypic));
    }
    if (out.sig && (st.p_allelic < out.p_thr || st.p_genotypic < out.p_thr)) {
        const unsigned long long slot = atomicAdd(out.n_sig, 1ull);
        if (slot < out.sig_cap) {
            gwasdev_sig_snp g;
            g.snp = (uint32_t)snp; g.df_genotypic = (uint32_t)st.df_genotypic; g.maf_pooled = st.maf_pooled;
            g.chi2_allelic = st.chi2_allelic; g.p_allelic = st.p_allelic; g.chi2_genotypic = st.chi2_genotypic; g.p_genotypic = st.p_genotypic;
            out.sig[slot] = g;
        }
    }
}

__device__ __forceinline__ void finish_snp(uint32_t m1c, uint32_t m2c, uint32_t mbc, uint32_t m1t, uint32_t m2t, uint32_t mbt,
                                           uint32_t n_case, uint32_t n_ctrl, uint64_t snp, const ScanOut &out) {
    if (out.compact || out.sig) finish_snp_compact(m1c, m2c, mbc, m1t, m2t, mbt, n_case, n_ctrl, snp, out);      // (the compact scan writes no plain outputs)
    else finish_snp_plain(m1c, m2c, mbc, m1t, m2t, mbt, n_case, n_ctrl, snp - out.out_base, out.counts, out.mi, out.stats);
}

// SLOTS = chunk pairs a lane loads back to back (2*SLOTS 128-bit loads in flight per lane)

// one class of one row: lane l of its G-lane group takes chunk pairs l, l+G, ... of Q, SCAN_SLOTS at a
// time with all loads of a round issued before the first is consumed
template <int G, int SLOTS>
__device__ __forceinline__ void scan_class(const uint4 *__restrict__ base, uint32_t Q, uint32_t l, bool row_valid,
                                           uint32_t &s1, uint32_t &s2, uint32_t &sb) {
    HS h1 = {0, 0, 0}, h2 = {0, 0, 0}, hb = {0, 0, 0};
    const uint4 *p = base + 2 * l;
    for (uint32_t q0 = l; q0 < Q; q0 += SLOTS * G, p += 2 * SLOTS * G) {
        ChunkPair c[SLOTS];
#pragma unroll
        for (int u = 0; u < SLOTS; ++u) c[u] = ld_pair(p + 2 * u * G, row_valid && q0 + u * G < Q);
#pragma unroll
        for (int u = 0; u < SLOTS; ++u)
            if (q0 + u * G < Q) accumulate_pair(c[u], h1, h2, hb);     // uniform over the lane group except at the row tail
    }
    s1 = hs_total(h1); s2 = hs_total(h2); sb = plain_total(hb);
}

// The batch loop both scan kernels share: full rounds of 32-row batches dealt round-robin over the warps (neighbouring
// warps stream neighbouring rows), then the rows that do not fill a round split evenly, so that no warp runs a whole
// batch longer than the rest.
template <class Batch>
__device__ __forceinline__ void for_each_batch(uint64_t snp_begin, uint64_t snp_end, Batch batch) {
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t n_snps = snp_end - snp_begin;
    const uint64_t rounds = n_snps / (n_warps * 32);
    for (uint64_t r = 0; r < rounds; ++r) batch(snp_begin + (r * n_warps + warp) * 32, 32u);
    const uint64_t rem_begin = snp_begin + rounds * n_warps * 32, rem = snp_end - rem_begin;
    const uint64_t b0 = rem_begin + warp * rem / n_warps, b1 = rem_begin + (warp + 1) * rem / n_warps;
    for (uint64_t base = b0; base < b1; base += 32) batch(base, (uint32_t)min((uint64_t)32, b1 - base));
}

// grid: persistent, MINB CTAs of 256 threads per SM.
template <int G, int SLOTS, int MINB>
__global__ void __launch_bounds__(256, MINB)
marginal_scan_kernel(const uint4 *__restrict__ sel, uint32_t stride4, uint32_t Qc, uint32_t Qt,
                     uint32_t n_case, uint32_t n_ctrl, uint64_t snp_begin, uint64_t snp_end, const __grid_constant__ ScanOut out) {
    const uint32_t lane = threadIdx.x & 31, g = lane / G, l = lane % G;
    const uint32_t group_mask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (g * G));
    // One batch: up to 32 consecutive rows; in pass `it` the 32/G lane groups work on rows it*(32/G) .. +32/G-1 (so a short
    // batch needs proportionally fewer passes), lane `it` of group g keeps the totals of row it*(32/G) + g, and after the
    // passes every lane finishes one SNP.
    constexpr uint32_t NG = 32 / G;
    const uint32_t my_row = l * NG + g;
    for_each_batch(snp_begin, snp_end, [&](uint64_t base, uint32_t in_batch) {
        const uint32_t passes = (in_batch + NG - 1) / NG;
        uint32_t m1c = 0, m2c = 0, mbc = 0, m1t = 0, m2t = 0, mbt = 0;   // totals of row (base + my_row)
        for (uint32_t it = 0; it < passes; ++it) {
            const uint32_t brow = it * NG + g;
            const bool valid = brow < in_batch;
            const uint4 *row = sel + (base + (valid ? brow : 0)) * (uint64_t)stride4;
            uint32_t s1, s2, sb, t1, t2, tb;
            scan_class<G, SLOTS>(row, Qc, l, valid, s1, s2, sb);
            scan_class<G, SLOTS>(row + 2 * Qc, Qt, l, valid, t1, t2, tb);
            s1 = __reduce_add_sync(group_mask, s1); s2 = __reduce_add_sync(group_mask, s2);
            sb = __reduce_add_sync(group_mask, sb); t1 = __reduce_add_sync(group_mask, t1);
            t2 = __reduce_add_sync(group_mask, t2); tb = __reduce_add_sync(group_mask, tb);
            if (l == it) { m1c = s1; m2c = s2; mbc = sb; m1t = t1; m2t = t2; mbt = tb; }
        }
        if (my_row < in_batch) finish_snp(m1c, m2c, mbc, m1t, m2t, mbt, n_case, n_ctrl, base + my_row, out);
    });
}

// ---- select + scan in one pass (K1') ----------------------------------------------------------------------------
// The same scan on the RAW rows with the class masks applied on the fly: the reference's
// getCaseControlGenotypeDistribution(rIdx, ccs, ccgd) (compressed_genotype_table5.cpp:609-657), which is all that
// select_cc_maf, a permutation or another trait over the resident table needs: no K0, no second copy of the table,
// algorithmic bytes again n_samples / 4 per SNP. A row is [plane 1: Q chunks][plane 2: Q chunks]; the masks (case,
// control-and-not-case: the compaction's classes) sit in shared memory, or, for cohorts whose masks exceed the shared-memory
// budget (SMEM_MASK false), are read from global memory through the read-only path, where every warp of the grid hits the
// same L2 lines.
__device__ __forceinline__ void accumulate_masked(const uint4 &x, const uint4 &y, const uint4 &m, HS &h1, HS &h2, HS &hb) {
    const uint4 xm = make_uint4(x.x & m.x, x.y & m.y, x.z & m.z, x.w & m.w);
    const uint4 ym = make_uint4(y.x & m.x, y.y & m.y, y.z & m.z, y.w & m.w);
    hs_add4(h1, xm.x, xm.y, xm.z, xm.w);
    hs_add4(h2, ym.x, ym.y, ym.z, ym.w);
    hb.ones += __popc(xm.x & y.x) + __popc(xm.y & y.y);     // plain POPC on the XU pipe: the ALU pipe is the busy one
    hb.twos += __popc(xm.z & y.z) + __popc(xm.w & y.w);
}

// MODE 0 (general): six masked popcount streams, any two disjoint classes (samples may belong to neither).
// MODE 1 (partition, first scan of a table): every sample is a case or a control, so the control counts are the row
//         totals minus the case counts and the totals need no mask (three masked + three plain streams); the totals --
//         which depend on the table alone, not on the phenotype -- are written to row_tot on the way.
// MODE 2 (partition, totals cached): three masked streams; the row totals come from row_tot (16 bytes per SNP instead of
//         a second pass over the words). This is what every re-selection over a resident table runs: the ALU work of the
//         compacted scan plus the mask ANDs, without K0 ever having run.
template <int G, int SLOTS, int MINB, int MODE, bool SMEM_MASK = true>
__global__ void __launch_bounds__(256, MINB)
marginal_scan_masked_kernel(const uint4 *__restrict__ raw, uint32_t Q, const uint4 *__restrict__ mask_case,
                            const uint4 *__restrict__ mask_ctrl, uint32_t n_case, uint32_t n_ctrl, uint64_t snp_begin,
                            uint64_t snp_end, const __grid_constant__ ScanOut out) {
    extern __shared__ uint4 sm_mask[];   // [Q] case, then (MODE 0) [Q] control
    if (SMEM_MASK) {
        for (uint32_t q = threadIdx.x; q < (MODE == 0 ? 2 * Q : Q); q += blockDim.x) sm_mask[q] = q < Q ? mask_case[q] : mask_ctrl[q - Q];
        __syncthreads();
    }
    const uint32_t lane = threadIdx.x & 31, g = lane / G, l = lane % G;
    const uint32_t group_mask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (g * G));
    constexpr uint32_t NG = 32 / G;
    const uint32_t my_row = l * NG + g;
    for_each_batch(snp_begin, snp_end, [&](uint64_t base, uint32_t in_batch) {
        const uint32_t passes = (in_batch + NG - 1) / NG;
        uint32_t m1c = 0, m2c = 0, mbc = 0, m1t = 0, m2t = 0, mbt = 0;
        uint4 tot = make_uint4(0, 0, 0, 0);
        if (MODE == 2 && my_row < in_batch) tot = __ldg(out.row_tot + base + my_row);   // in flight during the passes
        for (uint32_t it = 0; it < passes; ++it) {
            const uint32_t brow = it * NG + g;
            const bool valid = brow < in_batch;
            const uint4 *row = raw + (base + (valid ? brow : 0)) * (uint64_t)(2 * Q);
            HS a1 = {0, 0, 0}, a2 = {0, 0, 0}, ab = {0, 0, 0}, b1 = {0, 0, 0}, b2 = {0, 0, 0}, bb = {0, 0, 0};
            for (uint32_t q0 = l; q0 < Q; q0 += SLOTS * G) {
                uint4 x[SLOTS], y[SLOTS];
#pragma unroll
                for (int u = 0; u < SLOTS; ++u) {
                    const uint32_t q = q0 + u * G;
                    x[u] = make_uint4(0, 0, 0, 0); y[u] = x[u];
                    if (valid && q < Q) {
                        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                                     : "=r"(x[u].x), "=r"(x[u].y), "=r"(x[u].z), "=r"(x[u].w) : "l"(row + q));
                        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                                     : "=r"(y[u].x), "=r"(y[u].y), "=r"(y[u].z), "=r"(y[u].w) : "l"(row + Q + q));
                    }
                }
#pragma unroll
                for (int u = 0; u < SLOTS; ++u) {
                    const uint32_t q = q0 + u * G;
                    if (q < Q) {
                        accumulate_masked(x[u], y[u], SMEM_MASK ? sm_mask[q] : __ldg(mask_case + q), a1, a2, ab);
                        if (MODE == 1) { ChunkPair c; c.x = x[u]; c.y = y[u]; accumulate_pair(c, b1, b2, bb); }   // row totals (bits beyond sample N are zero)
                        else if (MODE == 0) accumulate_masked(x[u], y[u], SMEM_MASK ? sm_mask[Q + q] : __ldg(mask_ctrl + q), b1, b2, bb);
                    }
                }
            }
            uint32_t s1 = hs_total(a1), s2 = hs_total(a2), sb = plain_total(ab), t1 = 0, t2 = 0, tb = 0;
            s1 = __reduce_add_sync(group_mask, s1); s2 = __reduce_add_sync(group_mask, s2);
            sb = __reduce_add_sync(group_mask, sb);
            if (MODE != 2) {
                t1 = hs_total(b1); t2 = hs_total(b2); tb = plain_total(bb);
                t1 = __reduce_add_sync(group_mask, t1); t2 = __reduce_add_sync(group_mask, t2); tb = __reduce_add_sync(group_mask, tb);
            }
            if (l == it) { m1c = s1; m2c = s2; mbc = sb; m1t = t1; m2t = t2; mbt = tb; }
        }
        if (my_row < in_batch) {
            if (MODE == 1) {
                if (out.row_tot) out.row_tot[base + my_row] = make_uint4(m1t, m2t, mbt, 0);
                m1t -= m1c; m2t -= m2c; mbt -= mbc;
            } else if (MODE == 2) { m1t = tot.x - m1c; m2t = tot.y - m2c; mbt = tot.z - mbc; }
            finish_snp(m1c, m2c, mbc, m1t, m2t, mbt, n_case, n_ctrl, base + my_row, out);
        }
    });
}

// Streaming in sample blocks: counts are additive over disjoint sample blocks of one cohort.
__global__ void add_counts_kernel(const uint4 *__restrict__ src, uint4 *__restrict__ acc, uint64_t n4) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const uint4 a = acc[i], b = src[i];
    acc[i] = make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
// marginal_information + statistics from finished counts: the scan kernel's own epilogue on given counts
__global__ void finalize_counts_kernel(const uint32_t *__restrict__ counts, uint64_t n, gwasdev_marginal_information *__restrict__ mi,
                                       gwasdev_snp_stats *__restrict__ stats) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t ca[4], co[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) { ca[g] = counts[8 * i + g]; co[g] = counts[8 * i + 4 + g]; }
    const uint32_t n_ind = ca[0] + ca[1] + ca[2] + ca[3] + co[0] + co[1] + co[2] + co[3];
    if (mi) fill_marginal_information(ca, co, n_ind, mi[i]);
    if (stats) fill_stats(ca, co, stats[i]);
}

// Counts on the RAW rows, optionally through the case/control stream masks (mask-on-the-fly overloads
// compressed_genotype_table5.cpp:577-607 and :609-657). One warp per SNP.
__global__ void raw_counts_kernel(const uint32_t *__restrict__ raw, uint32_t Wr, const uint32_t *__restrict__ mca,
                                  const uint32_t *__restrict__ mco, uint32_t n_a, uint32_t n_b, uint64_t snp_begin,
                                  uint64_t snp_end, uint32_t *__restrict__ out, int per_snp) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t snp = snp_begin + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (snp >= snp_end) return;
    const uint32_t *p1 = raw + snp * 2ull * Wr, *p2 = p1 + Wr;
    uint32_t s1 = 0, s2 = 0, sb = 0, t1 = 0, t2 = 0, tb = 0;
    for (uint32_t w = lane; w < Wr; w += 32) {
        const uint32_t x = p1[w], y = p2[w];
        const uint32_t ma = mca ? mca[w] : 0xffffffffu;
        s1 += __popc(x & ma); s2 += __popc(y & ma); sb += __popc(x & y & ma);
        if (mco) { const uint32_t mb = mco[w]; t1 += __popc(x & mb); t2 += __popc(y & mb); tb += __popc(x & y & mb); }
    }
    s1 = __reduce_add_sync(0xffffffffu, s1); s2 = __reduce_add_sync(0xffffffffu, s2); sb = __reduce_add_sync(0xffffffffu, sb);
    t1 = __reduce_add_sync(0xffffffffu, t1); t2 = __reduce_add_sync(0xffffffffu, t2); tb = __reduce_add_sync(0xffffffffu, tb);
    if (lane == 0) {
        uint32_t *o = out + (snp - snp_begin) * per_snp;
        o[0] = s1 - sb; o[1] = s2 - sb; o[2] = sb; o[3] = n_a - s1 - s2 + sb;
        if (per_snp == 8) { o[4] = t1 - tb; o[5] = t2 - tb; o[6] = tb; o[7] = n_b - t1 - t2 + tb; }
    }
}

}  // namespace gwasdev

using namespace gwasdev;

static int lanes_per_row(const gwasdev_store *s, std::initializer_list<uint32_t> class_chunks, int slots) {
    if (s->opt[GWASDEV_OPT_LANES_PER_ROW]) return (int)s->opt[GWASDEV_OPT_LANES_PER_ROW];
    // the width that wastes the fewest lane slots for this cohort; on ties the one that needs the fewest rounds of `slots`
    // chunk pairs per lane (configs[1] on the raw rows: 80 chunk pairs = 16 lanes x 5, one round, measured 0.240 ms against
    // 0.251 ms for 8 lanes x 10, two rounds), then the narrower
    int G = 8;
    double best = 1e30;
    uint32_t best_rounds = 0;
    for (int cand : {8, 16, 32}) {
        double used = 0, have = 0;
        uint32_t rounds = 0;
        for (uint32_t Q : class_chunks) { const uint32_t per = (Q + cand - 1) / cand; used += (double)per * cand; have += Q; rounds += (per + slots - 1) / slots; }
        const double waste = used / have;
        if (waste < best - 1e-9 || (waste < best + 1e-9 && rounds < best_rounds)) { best = waste; G = cand; best_rounds = rounds; }
    }
    return G;
}

// Launch the compacted scan [snp_begin, snp_end) with DEVICE output pointers.
static int scan_compacted(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, const ScanOut &out) {
    int sms = 0;
    GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    const uint32_t Qc = s->Wc / 4, Qt = s->Wt / 4, stride4 = 2 * (Qc + Qt);
    // loads in flight per lane and resident CTAs per SM: 5 chunk pairs, 3 CTAs (B200 sweep, DESIGN.md)
    int slots = 5, minb = 3;
    int G = lanes_per_row(s, {Qc, Qt}, slots);
    const uint64_t n = snp_end - snp_begin;
    const uint4 *sel = reinterpret_cast<const uint4 *>(s->d_sel);
#ifdef GWASDEV_SWEEP
    if (const char *cfg = getenv("GWASDEV_SCAN_CFG")) sscanf(cfg, "%d,%d,%d", &slots, &minb, &G);
#endif
    const unsigned blocks = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sms * minb, (n + 255) / 256));
#define SCAN_LAUNCH(GG, SS, BB)                                                                                          \
    marginal_scan_kernel<GG, SS, BB><<<blocks, 256, 0, s->stream>>>(sel, stride4, Qc, Qt, s->n_case, s->n_ctrl, snp_begin, snp_end, out)
#ifdef GWASDEV_SWEEP
#define SCAN_CFG(GG)                                                                                   \
    do {                                                                                               \
        if (slots == 6 && minb == 3) SCAN_LAUNCH(GG, 6, 3);                                            \
        else if (slots == 5 && minb == 3) SCAN_LAUNCH(GG, 5, 3);                                       \
        else if (slots == 4 && minb == 4) SCAN_LAUNCH(GG, 4, 4);                                       \
        else if (slots == 3 && minb == 4) SCAN_LAUNCH(GG, 3, 4);                                       \
        else if (slots == 8 && minb == 2) SCAN_LAUNCH(GG, 8, 2);                                       \
        else { set_error("GWASDEV_SCAN_CFG=%d,%d is not an instantiated configuration", slots, minb); return GWASDEV_EINVAL; } \
    } while (0)
#else
#define SCAN_CFG(GG) SCAN_LAUNCH(GG, 5, 3)
#endif
    if (G == 8) SCAN_CFG(8);
    else if (G == 16) SCAN_CFG(16);
    else SCAN_CFG(32);
#undef SCAN_CFG
#undef SCAN_LAUNCH
    (void)slots; (void)minb;
    GW_LAUNCHED();
    return GWASDEV_OK;
}

static size_t masked_smem_bytes(const gwasdev_store *s, int mode) { return (mode == 0 ? 2ull : 1ull) * (s->Wr / 4) * sizeof(uint4); }
static bool partitioned(const gwasdev_store *s) { return s->n_case + s->n_ctrl == s->N; }   // nobody outside the two classes
// do the masks of this selection fit in shared memory
static bool masked_fits(const gwasdev_store *s) { return masked_smem_bytes(s, partitioned(s) ? 1 : 0) <= 200 * 1024; }

// The masked scan over the raw rows (no compacted store needed).
static int scan_masked(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, ScanOut out) {
    int sms = 0;
    GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    const uint32_t Q = s->Wr / 4;
    const bool use_tot = partitioned(s) && s->opt[GWASDEV_OPT_ROW_TOTALS] == 0;
    const int mode = !partitioned(s) ? 0 : (use_tot && s->tot_valid ? 2 : 1);
    if (mode == 1 && use_tot) {
        if (!s->d_row_tot) GW_CUDA(cudaMalloc((void **)&s->d_row_tot, s->M * sizeof(uint4)));
        out.row_tot = s->d_row_tot;
    } else out.row_tot = mode == 2 ? s->d_row_tot : nullptr;
    // loads in flight per lane, resident CTAs per SM (B200 sweeps, tools/sweep_mscan.py): modes 0 and 1 are bound by the
    // ALU pipe (occupancy pays more than loads in flight); mode 2 has the compacted scan's instruction mix
    int slots = mode == 2 ? 5 : 2, minb = mode == 2 ? 3 : 4;
    int G = lanes_per_row(s, {Q}, slots);
#ifdef GWASDEV_SWEEP
    if (const char *cfg = getenv("GWASDEV_MSCAN_CFG")) sscanf(cfg, "%d,%d,%d", &slots, &minb, &G);
#endif
    const uint64_t n = snp_end - snp_begin;
    const bool in_smem = masked_smem_bytes(s, mode) <= 200 * 1024;   // else the kernel reads the masks from global memory
    const size_t smem = in_smem ? masked_smem_bytes(s, mode) : 0;
    const unsigned blocks = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sms * minb, (n + 255) / 256));
    const uint4 *raw = reinterpret_cast<const uint4 *>(s->d_raw);
    const uint4 *mca = reinterpret_cast<const uint4 *>(s->d_case_sel_mask), *mco = reinterpret_cast<const uint4 *>(s->d_ctrl_sel_mask);
#define MSCAN1(GG, SS, BB, MM)                                                                                                     \
    do {                                                                                                                           \
        if (!in_smem) marginal_scan_masked_kernel<GG, SS, BB, MM, false><<<blocks, 256, 0, s->stream>>>(raw, Q, mca, mco, s->n_case, s->n_ctrl, snp_begin, snp_end, out); \
        else {                                                                                                                     \
            if (smem > 48 * 1024) GW_CUDA(cudaFuncSetAttribute(marginal_scan_masked_kernel<GG, SS, BB, MM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            marginal_scan_masked_kernel<GG, SS, BB, MM><<<blocks, 256, smem, s->stream>>>(raw, Q, mca, mco, s->n_case, s->n_ctrl, snp_begin, snp_end, out); \
        }                                                                                                                          \
    } while (0)
#define MSCAN(GG, SS, BB)                                                                                                          \
    do { if (mode == 2) MSCAN1(GG, SS, BB, 2); else if (mode == 1) MSCAN1(GG, SS, BB, 1); else MSCAN1(GG, SS, BB, 0); } while (0)
#ifdef GWASDEV_SWEEP
#define MSCAN_G(GG)                                                                                  \
    do {                                                                                             \
        if (slots == 2 && minb == 4) MSCAN(GG, 2, 4);                                                \
        else if (slots == 3 && minb == 4) MSCAN(GG, 3, 4);                                           \
        else if (slots == 4 && minb == 4) MSCAN(GG, 4, 4);                                           \
        else if (slots == 3 && minb == 3) MSCAN(GG, 3, 3);                                           \
        else if (slots == 4 && minb == 3) MSCAN(GG, 4, 3);                                           \
        else if (slots == 5 && minb == 3) MSCAN(GG, 5, 3);                                           \
        else if (slots == 6 && minb == 3) MSCAN(GG, 6, 3);                                           \
        else if (slots == 6 && minb == 2) MSCAN(GG, 6, 2);                                           \
        else if (slots == 8 && minb == 2) MSCAN(GG, 8, 2);                                           \
        else if (slots == 2 && minb == 5) MSCAN(GG, 2, 5);                                           \
        else { set_error("GWASDEV_MSCAN_CFG=%d,%d is not an instantiated configuration", slots, minb); return GWASDEV_EINVAL; } \
    } while (0)
#else
#define MSCAN_G(GG)                                                                                  \
    do { if (mode == 2) MSCAN1(GG, 5, 3, 2); else if (mode == 1) MSCAN1(GG, 2, 4, 1); else MSCAN1(GG, 2, 4, 0); } while (0)
#endif
    if (G == 8) MSCAN_G(8);
    else if (G == 16) MSCAN_G(16);
    else MSCAN_G(32);
#undef MSCAN_G
#undef MSCAN
#undef MSCAN1
    (void)slots; (void)minb;
    GW_LAUNCHED();
    return GWASDEV_OK;
}

// Which kernel a marginal scan runs: the compacted layout when it exists; otherwise through the masks on the raw rows
// (no K0) -- always when the classes partition the cohort (with cached row totals that costs what the compacted scan
// costs), else for the first scan after a selection only: the second builds the compacted layout, which every later
// scan streams with half the popcount work per byte. A selection K0 cannot compact (gwasdev_internal_compact_fits) is
// always scanned through the masks, from global memory when they do not fit in shared memory.
static bool choose_masked(gwasdev_store *s) {
    if (s->sel_built) return false;
    if (!gwasdev_internal_compact_fits(s)) return true;
    if (s->opt[GWASDEV_OPT_MASKED_SCAN] != 0 || !masked_fits(s)) return false;
    return partitioned(s) || s->scans_since_select == 0;
}

// Scan for the other translation units (margins of the pairwise screen, probes): any SNP range, device outputs, the
// kernel the store's state calls for; timed for gwasdev_last_scan_ms.
int gwasdev_internal_scan(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *d_counts,
                          gwasdev_marginal_information *d_mi, gwasdev_snp_stats *d_stats) {
    GW_REQUIRE(s->selected, "call gwasdev_select_case_control first");
    const bool masked = choose_masked(s);
    if (!masked) { const int rc = gwasdev_internal_ensure_compacted(s); if (rc != GWASDEV_OK) return rc; }
    ScanOut out = {};
    out.counts = d_counts; out.mi = d_mi; out.stats = d_stats; out.out_base = snp_begin;
    GW_CUDA(cudaEventRecord(s->ev0, s->stream));
    const int rc = masked ? scan_masked(s, snp_begin, snp_end, out) : scan_compacted(s, snp_begin, snp_end, out);
    if (rc != GWASDEV_OK) return rc;
    if (masked && partitioned(s) && s->opt[GWASDEV_OPT_ROW_TOTALS] == 0 && snp_begin == 0 && snp_end == s->M) s->tot_valid = true;
    GW_CUDA(cudaEventRecord(s->ev1, s->stream));
    return GWASDEV_OK;
}

// the compacted kernel on the compacted rows, whatever the store would choose (layout probe gwasdev_counts mode 2)
static int scan_compacted_forced(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *d_counts) {
    { const int rc = gwasdev_internal_ensure_compacted(s); if (rc != GWASDEV_OK) return rc; }
    ScanOut out = {};
    out.counts = d_counts; out.out_base = snp_begin;
    return scan_compacted(s, snp_begin, snp_end, out);
}

// Shared body of the two public scans: device outputs directly, host outputs through staging buffers in pieces whose
// D2H copies overlap the next piece's scan.
struct HostCopy { void *host; void *dev; size_t bytes_per_snp; };

static int run_scan(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, ScanOut out, int on_device, HostCopy *copies, int n_copies) {
    const uint64_t n = snp_end - snp_begin;
    const bool full = snp_begin == 0 && snp_end == s->M;
    const bool masked = choose_masked(s);
    ++s->scans_since_select;
    if (!masked) { const int rc = gwasdev_internal_ensure_compacted(s); if (rc != GWASDEV_OK) return rc; }
    out.out_base = snp_begin;
    GW_CUDA(cudaEventRecord(s->ev0, s->stream));   // ev0..ev1: the scan kernel(s) of this call (gwasdev_last_scan_ms)
    int pieces = 1;
    if (!on_device) {
        if (!s->copy_stream) {
            GW_CUDA(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
            for (cudaEvent_t &e : s->ev_piece) GW_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        uint64_t out_bytes = 0;
        for (int c = 0; c < n_copies; ++c) out_bytes += n * copies[c].bytes_per_snp;
        pieces = (int)std::max<uint64_t>(1, std::min<uint64_t>(gwasdev_store::MAX_PIECES, out_bytes / (4ull << 20)));   // ~4 MB per piece and at most 8 (tools/r2_kernels.py: 16 MB of
                                                                                                                         // compact records in 4 pieces 0.41 ms against 0.57 ms in one; 48 MB in 8)
        if (s->opt[GWASDEV_OPT_SCAN_PIECES]) pieces = (int)s->opt[GWASDEV_OPT_SCAN_PIECES];
    }
    cudaError_t e = cudaSuccess;
    for (int p = 0; p < pieces && e == cudaSuccess; ++p) {
        const uint64_t b = snp_begin + n * p / pieces, en = snp_begin + n * (p + 1) / pieces, o = b - snp_begin, k = en - b;
        if (k == 0) continue;
        const int rc = masked ? scan_masked(s, b, en, out) : scan_compacted(s, b, en, out);
        if (rc != GWASDEV_OK) return rc;
        if (on_device) continue;
        e = cudaEventRecord(s->ev_piece[p], s->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s->copy_stream, s->ev_piece[p], 0);
        for (int c = 0; c < n_copies && e == cudaSuccess; ++c)
            e = cudaMemcpyAsync((char *)copies[c].host + o * copies[c].bytes_per_snp, (char *)copies[c].dev + o * copies[c].bytes_per_snp,
                                k * copies[c].bytes_per_snp, cudaMemcpyDeviceToHost, s->copy_stream);
    }
    if (e == cudaSuccess) e = cudaEventRecord(s->ev1, s->stream);
    if (!on_device) {
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->copy_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    }
    if (e != cudaSuccess) { set_error("marginal scan: %s", cudaGetErrorString(e)); return GWASDEV_ENODEVICE; }
    if (masked && full && partitioned(s) && s->opt[GWASDEV_OPT_ROW_TOTALS] == 0) s->tot_valid = true;   // every piece wrote its rows' totals
    return GWASDEV_OK;
}

extern "C" {

int gwasdev_marginal_scan(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *counts,
                          gwasdev_marginal_information *mi, gwasdev_snp_stats *stats, int on_device) {
    GW_REQUIRE(s != nullptr, "gwasdev_marginal_scan: NULL store");
    GW_REQUIRE(s->selected, "gwasdev_marginal_scan: call gwasdev_select_case_control first");
    GW_REQUIRE(snp_begin <= snp_end && snp_end <= s->M, "gwasdev_marginal_scan: bad SNP range [%llu, %llu)",
               (unsigned long long)snp_begin, (unsigned long long)snp_end);
    if (snp_begin == snp_end) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    const uint64_t n = snp_end - snp_begin;
    const bool full = snp_begin == 0 && snp_end == s->M;
    ScanOut out = {};
    if (on_device) {
        out.counts = counts; out.mi = mi; out.stats = stats;
        return run_scan(s, snp_begin, snp_end, out, 1, nullptr, 0);
    }
    HostCopy copies[3];
    int nc = 0;
    if (counts) { GW_CUDA(reserve(s->sc_out_counts, n * 8 * sizeof(uint32_t))); out.counts = (uint32_t *)s->sc_out_counts.p; copies[nc++] = {counts, out.counts, 8 * sizeof(uint32_t)}; }
    if (stats) { GW_CUDA(reserve(s->sc_out_stats, n * sizeof(gwasdev_snp_stats))); out.stats = (gwasdev_snp_stats *)s->sc_out_stats.p; copies[nc++] = {stats, out.stats, sizeof(gwasdev_snp_stats)}; }
    if (mi) {
        if (full) {   // keep the full-table margins resident for the pairwise screen
            GW_CUDA(reserve_raw(s->d_mi, s->cap_mi, s->M * sizeof(gwasdev_marginal_information)));
            out.mi = s->d_mi;
        } else { GW_CUDA(reserve(s->sc_out_mi, n * sizeof(gwasdev_marginal_information))); out.mi = (gwasdev_marginal_information *)s->sc_out_mi.p; }
        copies[nc++] = {mi, out.mi, sizeof(gwasdev_marginal_information)};
    }
    const int rc = run_scan(s, snp_begin, snp_end, out, 0, copies, nc);
    if (rc != GWASDEV_OK) return rc;
    if (mi && full) { s->mi_valid = true; s->side_valid = false; s->mma_side_valid = false; }
    return GWASDEV_OK;
}

int gwasdev_marginal_scan_compact(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, gwasdev_snp_compact *out_rec,
                                  double p_threshold, gwasdev_sig_snp *sig, uint64_t sig_capacity, uint64_t *n_sig, int on_device) {
    GW_REQUIRE(s != nullptr, "gwasdev_marginal_scan_compact: NULL store");
    GW_REQUIRE(s->selected, "gwasdev_marginal_scan_compact: call gwasdev_select_case_control first");
    GW_REQUIRE(snp_begin <= snp_end && snp_end <= s->M, "gwasdev_marginal_scan_compact: bad SNP range [%llu, %llu)",
               (unsigned long long)snp_begin, (unsigned long long)snp_end);
    GW_REQUIRE(!out_rec || (s->n_case < 65536 && s->n_ctrl < 65536), "gwasdev_marginal_scan_compact: 16-bit counts need both classes below 65 536 samples");
    const bool want_sig = p_threshold > 0.0;
    GW_REQUIRE(!want_sig || (n_sig && (sig || sig_capacity == 0)), "gwasdev_marginal_scan_compact: a p-value threshold needs sig / n_sig");
    GW_REQUIRE(out_rec || want_sig, "gwasdev_marginal_scan_compact: nothing to compute");
    if (n_sig) *n_sig = 0;
    if (snp_begin == snp_end) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    const uint64_t n = snp_end - snp_begin;
    ScanOut out = {};
    HostCopy copies[1];
    int nc = 0;
    if (out_rec) {
        if (on_device) out.compact = out_rec;
        else { GW_CUDA(reserve(s->sc_out_stats, n * sizeof(gwasdev_snp_compact))); out.compact = (gwasdev_snp_compact *)s->sc_out_stats.p; copies[nc++] = {out_rec, out.compact, sizeof(gwasdev_snp_compact)}; }
    }
    unsigned long long *d_cnt = nullptr;
    if (want_sig) {
        GW_CUDA(reserve(s->sc_cnt, 2 * sizeof(unsigned long long)));
        d_cnt = (unsigned long long *)s->sc_cnt.p;
        GW_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), s->stream));
        out.n_sig = d_cnt; out.sig_cap = sig_capacity; out.p_thr = p_threshold;
        if (on_device) out.sig = sig;
        else { GW_CUDA(reserve(s->sc_out_mi, std::max<uint64_t>(1, sig_capacity) * sizeof(gwasdev_sig_snp))); out.sig = (gwasdev_sig_snp *)s->sc_out_mi.p; }
    }
    const int rc = run_scan(s, snp_begin, snp_end, out, on_device, copies, nc);
    if (rc != GWASDEV_OK) return rc;
    if (want_sig) {
        GW_CUDA(cudaMemcpyAsync(s->h_cnt, d_cnt, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
        GW_CUDA(cudaStreamSynchronize(s->stream));
        const uint64_t found = s->h_cnt[0];
        *n_sig = found;
        if (found > sig_capacity) {
            set_error("gwasdev_marginal_scan_compact: %llu significant SNPs exceed the caller's capacity of %llu", (unsigned long long)found, (unsigned long long)sig_capacity);
            return GWASDEV_EOVERFLOW;
        }
        if (!on_device && found > 0) {
            GW_CUDA(cudaMemcpyAsync(sig, out.sig, found * sizeof(gwasdev_sig_snp), cudaMemcpyDeviceToHost, s->stream));
            GW_CUDA(cudaStreamSynchronize(s->stream));
            std::sort(sig, sig + found, [](const gwasdev_sig_snp &a, const gwasdev_sig_snp &b) { return a.snp < b.snp; });   // appended in completion order
        }
    }
    return GWASDEV_OK;
}

int gwasdev_marginal_accumulate(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *acc, int on_device) {
    GW_REQUIRE(s && acc, "gwasdev_marginal_accumulate: NULL argument");
    GW_REQUIRE(s->selected, "gwasdev_marginal_accumulate: call gwasdev_select_case_control first");
    GW_REQUIRE(snp_begin <= snp_end && snp_end <= s->M, "gwasdev_marginal_accumulate: bad SNP range [%llu, %llu)",
               (unsigned long long)snp_begin, (unsigned long long)snp_end);
    if (snp_begin == snp_end) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    const uint64_t n = snp_end - snp_begin;
    GW_CUDA(reserve(s->sc_out_counts, n * 8 * sizeof(uint32_t)));
    uint32_t *d_counts = (uint32_t *)s->sc_out_counts.p, *d_acc = acc;
    // a block's rows are used once: counted through the masks unless the compacted layout already exists
    int rc = gwasdev_internal_scan(s, snp_begin, snp_end, d_counts, nullptr, nullptr);
    if (rc != GWASDEV_OK) return rc;
    if (!on_device) {
        GW_CUDA(reserve(s->sc_stage, n * 8 * sizeof(uint32_t)));
        d_acc = (uint32_t *)s->sc_stage.p;
        GW_CUDA(cudaMemcpyAsync(d_acc, acc, n * 8 * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    }
    add_counts_kernel<<<(unsigned)((2 * n + 255) / 256), 256, 0, s->stream>>>(reinterpret_cast<const uint4 *>(d_counts),
                                                                              reinterpret_cast<uint4 *>(d_acc), 2 * n);
    GW_LAUNCHED();
    if (!on_device) {
        GW_CUDA(cudaMemcpyAsync(acc, d_acc, n * 8 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
        GW_CUDA(cudaStreamSynchronize(s->stream));
    }
    return GWASDEV_OK;
}
int gwasdev_marginal_finalize(int device, uint64_t n_snps, const uint32_t *counts, gwasdev_marginal_information *mi,
                              gwasdev_snp_stats *stats, int on_device) {
    GW_REQUIRE(counts && (mi || stats), "gwasdev_marginal_finalize: NULL argument");
    if (gwasdev_device_count() <= device || device < 0) { set_error("gwasdev_marginal_finalize: no CUDA device %d", device); return GWASDEV_ENODEVICE; }
    if (n_snps == 0) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(device));
    const uint32_t *d_counts = counts;
    uint32_t *tmp_counts = nullptr;
    gwasdev_marginal_information *d_mi = mi;
    gwasdev_snp_stats *d_stats = stats;
    cudaError_t e = cudaSuccess;
    if (!on_device) {
        e = cudaMalloc(&tmp_counts, n_snps * 8 * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMemcpy(tmp_counts, counts, n_snps * 8 * sizeof(uint32_t), cudaMemcpyHostToDevice);
        d_counts = tmp_counts; d_mi = nullptr; d_stats = nullptr;
        if (e == cudaSuccess && mi) e = cudaMalloc(&d_mi, n_snps * sizeof *mi);
        if (e == cudaSuccess && stats) e = cudaMalloc(&d_stats, n_snps * sizeof *stats);
    }
    if (e == cudaSuccess) {
        finalize_counts_kernel<<<(unsigned)((n_snps + 127) / 128), 128>>>(d_counts, n_snps, d_mi, d_stats);
        ++g_launches;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (!on_device) {
        if (e == cudaSuccess && mi) e = cudaMemcpy(mi, d_mi, n_snps * sizeof *mi, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && stats) e = cudaMemcpy(stats, d_stats, n_snps * sizeof *stats, cudaMemcpyDeviceToHost);
        cudaFree(tmp_counts); if (mi) cudaFree(d_mi); if (stats) cudaFree(d_stats);
    }
    if (e != cudaSuccess) { set_error("gwasdev_marginal_finalize: %s", cudaGetErrorString(e)); return e == cudaErrorMemoryAllocation ? GWASDEV_ENOMEM : GWASDEV_ENODEVICE; }
    return GWASDEV_OK;
}

double gwasdev_last_scan_ms(gwasdev_store *s) {
    if (!s || !s->ev0) return -1.0;
    cudaSetDevice(s->device);
    if (cudaEventSynchronize(s->ev1) != cudaSuccess) { cudaGetLastError(); return -1.0; }
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, s->ev0, s->ev1) != cudaSuccess) { cudaGetLastError(); return -1.0; }
    return ms;
}

int gwasdev_counts(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, int mode, uint32_t *out) {
    GW_REQUIRE(s && out, "gwasdev_counts: NULL argument");
    GW_REQUIRE(mode >= 0 && mode <= 2, "gwasdev_counts: mode %d", mode);
    GW_REQUIRE(snp_begin <= snp_end && snp_end <= s->M, "gwasdev_counts: bad SNP range");
    GW_REQUIRE(mode != 2 || s->selected, "gwasdev_counts: mode 2 needs gwasdev_select_case_control");
    GW_REQUIRE(mode != 1 || s->fly_valid, "gwasdev_counts: mode 1 needs gwasdev_set_stream_masks or gwasdev_select_case_control");
    if (snp_begin == snp_end) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    const uint64_t n = snp_end - snp_begin;
    const int per = mode == 0 ? 4 : 8;
    GW_CUDA(reserve(s->sc_out_counts, n * per * sizeof(uint32_t)));
    uint32_t *d_out = (uint32_t *)s->sc_out_counts.p;
    int rc = GWASDEV_OK;
    cudaError_t e = cudaSuccess;
    if (mode == 2) rc = scan_compacted_forced(s, snp_begin, snp_end, d_out);
    else {
        const unsigned blocks = (unsigned)((n * 32 + 255) / 256);
        raw_counts_kernel<<<blocks, 256, 0, s->stream>>>(s->d_raw, s->Wr, mode == 1 ? s->d_case_mask : nullptr,
                                                         mode == 1 ? s->d_ctrl_mask : nullptr,
                                                         mode == 1 ? s->n_fly_case : s->N, s->n_fly_ctrl, snp_begin, snp_end, d_out, per);   // member counts as given (:649-653)
        ++g_launches;
        e = cudaGetLastError();
    }
    if (rc == GWASDEV_OK && e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, n * per * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream);
    if (rc == GWASDEV_OK && e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    if (rc != GWASDEV_OK) return rc;
    if (e != cudaSuccess) { set_error("gwasdev_counts: %s", cudaGetErrorString(e)); return GWASDEV_ENODEVICE; }
    return GWASDEV_OK;
}

}  // extern "C"

// The permutation test's tensor-core kernel lives in this translation unit so that its epilogue and fill_stats call one
// compiled chi2_tests.
#include "permute_gemm.cuh"
