// K2+K3 on the 5th-generation tensor cores: the four corner cells of every pair's 3x3x2 table as ONE
// signed-byte GEMM per SNP tile pair (tcgen05.mma kind::i8, accumulators in TMEM), fused with the fp32 KSA
// screen. Same results as pair_screen_kernel<false> in pairwise.cu (the AND+POPC engine): the counted
// cells are integers, and the candidates are re-scored in fp64 by rescore_kernel either way.
//
// Reference path replaced: the no-missing shortcut of getCaseControlContingencyTable(i, j, m1, m2, ccct)
// (genotype/compressed_genotype_table5.cpp:1069-1144: AA_BB, AA_bb, aa_BB, aa_bb counted, the other five
// cells from the per-SNP class margins) + computeBoost's KSA statistic and threshold
// (algorithms/epistasis_func.cpp:424-470, :482-484).
//
// Formulation. Row 2s+p of the operand matrix is the one-hot plane p (0: genotype aa, 1: genotype bb) of
// SNP s over the samples, one signed byte per sample: a case sample that has the genotype is +1, a
// control sample that has it is -128, everything else 0. A sample is either case or control for both
// SNPs of a pair, so
//     D[2i+p][2j+q] = sum_samples A*B = n_case(p, q) + 16384 * n_ctrl(p, q)
// exactly in int32 (n_case < 16384, n_ctrl < 131072): one accumulator tile carries both classes.
//
// Kernel. The CTA-pair pipeline of mma_common.cuh (CtaPipe), persistent over tile pairs of (128 A-SNPs = 256 rows,
// 128 per CTA) x (128 B-SNPs = 256 rows, each CTA stages half):
//   loads                 : 2-D SWIZZLE_128B boxes of 128 sample bytes x 128 rows, a CTA's A rows and its half of B;
//                           three stages of two sample blocks, 64 KiB per CTA
//   MMAs                  : tcgen05.mma.cta_group::2.kind::i8, M=256 N=256 K=32, 4 per sample block, into one of
//                           two 256-column TMEM accumulators
//   warps 0-15 epilogue   : each CTA reads its 128 accumulator rows (64 A-SNPs) with tcgen05.ld 32x32b, lane
//                           pairs swap the two planes by shuffle, decode the counts, margins -> 3x3x2 table,
//                           upper bound of the KSA statistic, exact fp32 KSA for the few that pass it,
//                           candidates above threshold - margin
// Tile order keeps a band of A-blocks (8 to 16, see schedule_band) and a sliding window of B-blocks L2-resident.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "mma_common.cuh"

int gwasdev_internal_ensure_side(gwasdev_store *s);   // pairwise.cu: margins, PairSide records, missing-call flags
int gwasdev_internal_set_rows(uint64_t M, const uint32_t *set_a, uint64_t n_a, const uint32_t *set_b, uint64_t n_b, const char *who,
                              std::vector<uint32_t> &map, uint64_t *c1, uint64_t *a1);   // pair_sets.cu

namespace gwasdev {

constexpr int COL_STAGE_BYTES = 32 * 64;                           // column-role records of one epilogue warp's 32 B-SNPs
// A-blocks per L2 band (schedule_band below): with the tile feed the 74 CTA pairs of a B200 work on ~74 consecutive tiles, i.e.
// on the BD A-blocks of the band and a window of ceil(74 / BD) B-blocks; DRAM traffic falls as 1 / BD while that working set
// fits the L2. The largest BD (at most BAND_MAX) whose working set stays below GWASDEV_L2_MB MiB is taken; when none fits
// (rows of 12 000+ samples) the working set is smallest at BD = 8. Measured at configs[3] (2.59 MB blocks) on one box, two
// rounds: 8 -> 2.77-2.78 s, 10 -> 2.75-2.77, 12 -> 2.73-2.74 (19 blocks, 49.2 MB), 13 -> 2.74, 14 -> 2.74-2.75 (51.8 MB),
// 15 -> 2.75-2.76, 16 -> 2.75-2.79 (54.4 MB), 24 -> 3.00 s (72 MB): flat between 12 and 14, the rule picks 13.
#ifndef GWASDEV_L2_MB
#define GWASDEV_L2_MB 48
#endif
constexpr uint32_t BAND_MAX = 16, BAND_FALLBACK = 8, SCHED_PAIRS = 74;
constexpr uint32_t CTRL_SHIFT = 14;                                // (-128)^2 = 2^14

// per-SNP epilogue records, log2 units, class-interleaved so that (case, control) pairs are float2 operands of
// the packed fp32 instructions. Row role (SNP "A" of the pair) / column role (SNP "B"), g = aa, ab, bb:
//   pca[g] = (c_0[g], c_1[g]) / m[g]           w[g] = (c_0[g]/n_0, c_1[g]/n_1) / m[g]  (NaN when m[g] == 0)
//   C_row = sum_kg c_k[g] log2 pca_k[g] + N log2 N          C_col = sum_kg c_k[g] (log2 pbc_k[g] - log2 m[g])
struct __align__(16) MmaRow { float2 pca[3]; float2 cnt[3]; float C; float pad[3]; };
struct __align__(16) MmaCol { float2 w[3];   float2 cnt[3]; float C; float pad[3]; };
static_assert(sizeof(MmaRow) == 64 && sizeof(MmaCol) == 64, "64-byte epilogue records");

// Records of the bound pass (ksa_bound_fast): tau = sum_ab n_ab. W_ab is affine in the four pooled corner counts
// x = (AB, Ab, aB, ab), so only differences against the heterozygote class and two per-SNP dot products are needed:
//   tau = sum_k [ w_k[1] RA_k + pca_k[1] RB_k ] + sum_k [ dA0_k (x1 dB0_k + x2 dB2_k) + dA2_k (x3 dB0_k + x4 dB2_k) ]
//   dA0 = pca[0]-pca[1], dA2 = pca[2]-pca[1], RA_k = pca_k[0] m[0] + pca_k[2] m[2] - pca_k[1] (m[0]+m[2])     (row role)
//   dB0 = w[0]-w[1],     dB2 = w[2]-w[1],     RB_k = w_k[0] m[0] + w_k[1] m[1] + w_k[2] m[2]                  (column role)
// with m[g] the pooled genotype counts. cm[g] = (c_0[g], m[g]): case and pooled counts, the two the bound needs.
struct __align__(16) MmaRowF { float2 dA0, dA2, pca1, RA, cm0, cm2; float C; float pad[3]; };
struct __align__(16) MmaColF { float2 dB0, dB2, w1, RB, cm0, cm1, cm2; float C; float pad; };
static_assert(sizeof(MmaRowF) == 64 && sizeof(MmaColF) == 64, "64-byte bound-pass records");

struct MmaParams {
    uint32_t TB;                // 128-SNP blocks
    uint32_t NKB;               // 128-byte sample blocks per row
    uint32_t n_bands, band;     // bands of the schedule, A-blocks per band
    uint64_t M;
    uint64_t n_tiles;
    uint32_t shard, n_shards;
    const MmaRow *row;
    const MmaCol *col;
    const MmaRowF *rowf;
    const MmaColF *colf;
    const uint8_t *tile_missing;   // per 64-SNP block
    float N;
    float qc, q0;               // upper-bound pre-filter: S <= qc * sum_ab c0^2/cab - q0 (see ksa_upper_bound)
    CandSink sink;
    unsigned long long *tile_counter;   // zero at launch: the CTA pairs draw the shard's tiles from it in schedule order
    uint32_t *dump;             // debug: raw corner counts of tile `dump_tile` only, rows of CTA `dump_rank`
    uint64_t dump_tile;
    uint32_t dump_rank;
    unsigned long long *prof;   // role timers (builds with -DGWASDEV_SWEEP only, GWASDEV_MMA_PROF): per CTA {mma busy, mma waiting for tempty,
                                // mma waiting for full, epilogue busy, epilogue waiting for tfull, producer waiting for empty, tiles} in SM clocks
    // set screens (SETS instantiations only; appended so that the fields above keep their offsets): the shard's tiles as
    // (I2, J), n_tiles of them, and the segment bounds of the gathered sub-table (set_pair_wanted)
    const uint2 *set_tiles;
    uint64_t set_c1, set_a1;
};

// ---- tile order -------------------------------------------------------------------------------------
// Tiles are pairs of 128-SNP blocks (I2 <= J). Band b holds A-blocks [BD b, BD b + BD) for the band height BD of the launch;
// inside a band tiles run column-major over B-blocks J >= BD b, and column c = J - BD b holds the band's A-blocks I2 <= J.
__host__ __device__ inline uint32_t band_height(uint32_t TB, uint32_t b, uint32_t BD) { return min(BD, TB - BD * b); }
__host__ __device__ inline uint32_t column_height(uint32_t na, uint32_t c) { return min(na, c + 1); }
// band height for operand blocks of `block_bytes` (rows of one A-block x bytes per row)
inline uint32_t schedule_band(uint64_t block_bytes) {
#ifdef GWASDEV_BAND_FORCE                    // experiment builds: build.py --variant NAME -DGWASDEV_BAND_FORCE=n
    return GWASDEV_BAND_FORCE;
#endif
    for (uint32_t bd = BAND_MAX; bd >= BAND_FALLBACK; --bd)
        if ((bd + (SCHED_PAIRS + bd - 1) / bd) * block_bytes <= ((uint64_t)GWASDEV_L2_MB << 20)) return bd;
    return BAND_FALLBACK;
}

// Schedule index of the u-th tile of a shard: shards take turns in chunks of SHARD_CHUNK consecutive tiles.
constexpr uint32_t SHARD_CHUNK = 64;
__host__ __device__ inline uint64_t shard_tile(uint64_t u, uint32_t shard, uint32_t n_shards) {
    return ((u / SHARD_CHUNK) * n_shards + shard) * SHARD_CHUNK + u % SHARD_CHUNK;
}
__host__ __device__ inline bool tile_in_shard(uint64_t t, uint32_t shard, uint32_t n_shards) { return (t / SHARD_CHUNK) % n_shards == shard; }
// number of tiles of the shard among the first n tiles of the schedule
__host__ __device__ inline uint64_t shard_tiles_before(uint64_t n, uint32_t shard, uint32_t n_shards) {
    const uint64_t chunk = n / SHARD_CHUNK, rem = n % SHARD_CHUNK;
    uint64_t cnt = (chunk / n_shards) * SHARD_CHUNK + (chunk % n_shards > shard ? SHARD_CHUNK : 0);
    if (chunk % n_shards == shard) cnt += rem;
    return cnt;
}

// Set screens run on a gathered sub-table whose rows are C = A n B, then A \ B, then B \ A (each in table order), with
// c1 = |C| and a1 = |C| + |A \ B|. Pair gi < gj of the sub-table is wanted when gi lies in C, or gi in A \ B and gj in
// B \ A: every unordered pair {i in A, j in B, i != j} exactly once.
__host__ __device__ __forceinline__ bool set_pair_wanted(uint64_t gi, uint64_t gj, uint64_t c1, uint64_t a1) {
    return (gi < c1) | ((gi < a1) & (gj >= a1));
}
// Across segments the sub-table may hold a pair in the other order than the table. The statistic is symmetric in the two SNPs
// except where one of them has an empty genotype class: it is NaN when that is the SNP with the larger table index (0 / 0 in
// ksa_f64) and finite otherwise. So the sub-table's records leave empty classes out (SETS in mma_side_kernel, pair_side_kernel),
// every pair evaluates finite, and the pairs whose statistic is NaN are dropped here from the keys (d_set_keys: table index |
// empty class << 31) of the two SNPs.
__device__ __forceinline__ bool set_pair_live(uint32_t ki, uint32_t kj) {
    const bool rev = (ki & 0x7fffffffu) > (kj & 0x7fffffffu);
    return ((rev ? ki : kj) >> 31) == 0;
}

// Tiles before band b. Every band before the last is full (BD A-blocks, at least BD columns): BD (TB - BD b') - BD (BD - 1) / 2 tiles.
__host__ __device__ inline uint64_t band_offset(uint32_t TB, uint64_t b, uint32_t BD) {
    return b * ((uint64_t)BD * TB) - (uint64_t)(BD * BD) * (b * (b - 1) / 2) - b * (uint64_t)(BD * (BD - 1) / 2);
}

__host__ __device__ inline uint64_t band_tiles(uint32_t TB, uint32_t b, uint32_t BD) {      // tiles in band b (the last one may be short)
    const uint64_t na = band_height(TB, b, BD), cols = TB - BD * b;             // cols >= na
    return na * (na - 1) / 2 + na * (cols - (na - 1));
}
// tiles of the whole schedule
inline uint64_t schedule_tiles(uint32_t TB, uint32_t BD) {
    const uint32_t n_bands = (TB + BD - 1) / BD;
    return band_offset(TB, n_bands - 1, BD) + band_tiles(TB, n_bands - 1, BD);
}

// Position in the schedule: band and index inside the band. Located once with the closed form, then advanced
// with a few integer operations per tile.
struct TileCursor {
    uint32_t b, BD;
    uint64_t r, len;
    __device__ void locate(uint64_t t, uint32_t TB, uint32_t n_bands, uint32_t band) {
        BD = band;
        const double Bc = (double)BD * TB + 0.5 * BD * BD - 0.5 * BD * (BD - 1);
        int64_t k = (int64_t)((Bc - sqrt(fmax(Bc * Bc - 2.0 * BD * BD * (double)t, 0.0))) / (double)(BD * BD));
        k = max((int64_t)0, min(k, (int64_t)n_bands - 1));
        while (k > 0 && band_offset(TB, (uint64_t)k, BD) > t) --k;
        while (k + 1 < (int64_t)n_bands && band_offset(TB, (uint64_t)k + 1, BD) <= t) ++k;
        b = (uint32_t)k; r = t - band_offset(TB, b, BD); len = band_tiles(TB, b, BD);
    }
    __device__ __forceinline__ void advance(uint64_t d, uint32_t TB, uint32_t n_bands) {
        r += d;
        while (r >= len && b + 1 < n_bands) { r -= len; ++b; len = band_tiles(TB, b, BD); }
    }
    __device__ __forceinline__ void decode(uint32_t TB, uint32_t &I2, uint32_t &J) const {
        const uint32_t na = band_height(TB, b, BD), tri = na * (na - 1) / 2;      // columns 0..na-2 hold c+1 tiles each
        uint32_t c, ii;
        if (r < tri) { c = 0; uint32_t q = (uint32_t)r; while (q > c) { q -= c + 1; ++c; } ii = q; }
        else { const uint64_t q = r - tri; c = na - 1 + (uint32_t)(q / na); ii = (uint32_t)(q % na); }
        I2 = BD * b + ii; J = BD * b + c;
    }
};

// The leader producer's side of the tile feed when a kernel computes only some tiles of the schedule (the four-plane kernel:
// those with / without missing calls): draws local indices from the device counter and walks them until a wanted tile turns
// up. The batch drawn at once adapts -- doubled (up to 64) after a batch without a wanted tile, halved after every wanted one --
// so that a cohort whose tiles are all wanted keeps drawing single tiles (tiles in flight stay consecutive) and one with few
// wanted tiles does not pay an atomic per skipped tile.
struct TileDraw {
    unsigned long long *counter;
    uint32_t shard, n_shards, TB, n_bands, band;
    uint64_t last;
    uint64_t u_lo = 0, u_hi = 0, pend = 0, t_cur = 0;
    uint32_t batch = 1, pend_n = 0;
    bool located = false;
    TileCursor cur;
    __device__ __forceinline__ void prefetch() {       // issue the next draw early: its latency hides behind the tile's loads
        if (u_lo == u_hi && pend_n == 0) { pend = atomicAdd(counter, (unsigned long long)batch); pend_n = batch; }
    }
    template <class Wanted> __device__ __forceinline__ bool next(uint32_t &I2, uint32_t &J, Wanted wanted) {
        for (;;) {
            if (u_lo == u_hi) { prefetch(); u_lo = pend; u_hi = pend + pend_n; pend_n = 0; }
            const uint64_t t = shard_tile(u_lo++, shard, n_shards);
            if (t >= last) return false;
            if (!located) { cur.locate(t, TB, n_bands, band); located = true; } else cur.advance(t - t_cur, TB, n_bands);
            t_cur = t;
            cur.decode(TB, I2, J);
            if (wanted(I2, J)) { batch = max(1u, batch >> 1); return true; }
            if (u_lo == u_hi) batch = min(batch << 1, 64u);
        }
    }
};

// ---- fp32 KSA on the four counted corners -----------------------------------------------------------
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// The nine cells of both classes as float2 (x: cases, y: controls) from the four counted corners and the
// per-SNP class counts -- the reference's shortcut (compressed_genotype_table5.cpp:1084-1092, :1133-1141).
struct Cells { float2 n[3][3]; };
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ Cells derive_cells(float2 AB, float2 Ab, float2 aB, float2 ab, const float2 (&ca)[3], const float2 (&cb)[3]) {
    Cells t;
    t.n[0][0] = AB; t.n[0][2] = Ab; t.n[2][0] = aB; t.n[2][2] = ab;
    t.n[0][1] = sub2(sub2(ca[0], AB), Ab);
    t.n[2][1] = sub2(sub2(ca[2], ab), aB);
    t.n[1][0] = sub2(sub2(cb[0], AB), aB);
    t.n[1][2] = sub2(sub2(cb[2], Ab), ab);
    t.n[1][1] = sub2(sub2(cb[1], t.n[0][1]), t.n[2][1]);
    return t;
}

// Cheap rigorous upper bound of the screen statistic. With x = c0/cab, the cell term g2(c0)+g2(c1)-g2(cab) is
// -cab H2(x) (binary entropy, bits), and H2(x) >= H2(x0) + H2'(x0)(x-x0) - qc (x-x0)^2 on [0,1] for the
// cohort's case fraction x0 = n_case/N and the constant qc found on the host. Summed over the table (whose
// cells add up to N samples and n_case cases when no call is missing) the linear part is constant:
//     S <= qc * sum_ab c0^2/cab - q0,      q0 = qc x0 n_case + N H2(x0)
// so stat <= 2 ln2 (N log2 tau + qc Q - q0 - C): nine reciprocals and one logarithm instead of 28 logarithms.
// tau is accumulated on the way and returned for the exact evaluation.
__device__ __forceinline__ float ksa_upper_bound(const Cells &t, const float2 (&pca)[3], const float2 (&w)[3], float Csum,
                                                 float N, float qc, float q0, float &tau_out) {
    float tau = 0.f, Q = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const float2 n = t.n[a][b];
            const float cab = n.x + n.y;
            const float2 wp = __fmul2_rn(w[b], pca[a]);
            tau = fmaf(cab, wp.x + wp.y, tau);
            float r;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(cab + 1.17549435e-38f));
            Q = fmaf(n.x, n.x * r, Q);
        }
    tau_out = tau;
    return 1.3862943611f * (fmaf(N, lg2_approx(tau), fmaf(qc, Q, -q0)) - Csum);
}

// The same bound from the bound-pass records, in log2 units without the 2 ln2 factor and without the constant
// (returns N log2 tau + qc Q; the caller compares against thr2 + q0 + C_row + C_col). Corner counts arrive as
// (case, control); cells are carried as (case, pooled). ~95 instructions, 9 MUFU.RCP + 1 MUFU.LG2.
__device__ __forceinline__ float ksa_bound_fast(float2 AB, float2 Ab, float2 aB, float2 ab, const MmaRowF &A, const float2 (&b)[7],
                                                float N, float qc) {
    // b[] = dB0, dB2, w1, RB, cm0, cm1, cm2 of the column-role record
    AB.y += AB.x; Ab.y += Ab.x; aB.y += aB.x; ab.y += ab.x;                  // (case, pooled)
    const float2 n01 = sub2(sub2(A.cm0, AB), Ab), n21 = sub2(sub2(A.cm2, ab), aB);
    const float2 n10 = sub2(sub2(b[4], AB), aB), n12 = sub2(sub2(b[6], Ab), ab);
    const float2 n11 = sub2(sub2(b[5], n01), n21);
    // tau
    const float2 t0 = __ffma2_rn(A.pca1, b[3], __fmul2_rn(b[2], A.RA));
    const float i1x = fmaf(Ab.y, b[1].x, AB.y * b[0].x), i1y = fmaf(Ab.y, b[1].y, AB.y * b[0].y);
    const float i2x = fmaf(ab.y, b[1].x, aB.y * b[0].x), i2y = fmaf(ab.y, b[1].y, aB.y * b[0].y);
    float tau = t0.x + t0.y;
    tau = fmaf(A.dA0.x, i1x, tau); tau = fmaf(A.dA0.y, i1y, tau);
    tau = fmaf(A.dA2.x, i2x, tau); tau = fmaf(A.dA2.y, i2y, tau);
    // Q = sum c0^2 / cab; an empty cell gives 0 * inf = NaN inside fminf, which returns the other operand, times c0 = 0
    float Q = 0.f;
    const float2 cell[9] = {AB, n01, Ab, n10, n11, n12, aB, n21, ab};
#pragma unroll
    for (int c = 0; c < 9; ++c) {
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(cell[c].y));
        Q = fmaf(cell[c].x, fminf(cell[c].x * r, 1.0f), Q);
    }
    return fmaf(N, lg2_approx(tau), qc * Q);
}

// Exact-formula fp32 value: 2 ln2 (sum g2(n_abk) - sum g2(n_ab.) + N log2 tau - C_row - C_col), equal to
// ksa_screen_f32 of pairwise.cu when neither SNP has a missing call (row/column sums of the table are then the
// per-SNP class counts). g2(n) = n log2 n with g2(0) = 0: n + 2^-126 == n for n >= 1, and 0 * log2(2^-126) = -0.
__device__ __forceinline__ float ksa_screen_cells(const Cells &t, float tau, float Csum, float N) {
    const float2 tiny = make_float2(1.17549435e-38f, 1.17549435e-38f);
    float2 S2 = make_float2(0.f, 0.f);
    float S1 = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const float2 n = t.n[a][b];
            const float cab = n.x + n.y;
            const float2 na = __fadd2_rn(n, tiny);
            S2 = __ffma2_rn(n, make_float2(lg2_approx(na.x), lg2_approx(na.y)), S2);
            S1 = fmaf(-cab, lg2_approx(cab + tiny.x), S1);
        }
    return 1.3862943611f * (fmaf(N, lg2_approx(tau), S2.x + S2.y + S1) - Csum);
}

// D = n_case + 2^14 n_ctrl  ->  (n_case, n_ctrl) as floats, through the 2^23 magic number
__device__ __forceinline__ float2 decode2(uint32_t d) {
    const float2 m = make_float2(__uint_as_float((d & 0x3fffu) | 0x4B000000u), __uint_as_float((d >> CTRL_SHIFT) | 0x4B000000u));
    return __fadd2_rn(m, make_float2(-8388608.0f, -8388608.0f));
}

__device__ __forceinline__ void unpack_record(const uint4 &r0, const uint4 &r1, const uint4 &r2, const uint4 &r3, float2 (&p)[3], float2 (&c)[3], float &C);
__device__ __forceinline__ void load_record_smem(const unsigned char *rec, float2 (&p)[3], float2 (&c)[3], float &C) {
    const uint4 *q = reinterpret_cast<const uint4 *>(rec);
    unpack_record(q[0], q[1], q[2], q[3], p, c, C);
}
__device__ __forceinline__ void load_record(const void *rec, float2 (&p)[3], float2 (&c)[3], float &C) {
    const uint4 *q = reinterpret_cast<const uint4 *>(rec);
    unpack_record(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3), p, c, C);
}
__device__ __forceinline__ void unpack_record(const uint4 &r0, const uint4 &r1, const uint4 &r2, const uint4 &r3, float2 (&p)[3], float2 (&c)[3], float &C) {
    p[0] = make_float2(__uint_as_float(r0.x), __uint_as_float(r0.y)); p[1] = make_float2(__uint_as_float(r0.z), __uint_as_float(r0.w));
    p[2] = make_float2(__uint_as_float(r1.x), __uint_as_float(r1.y)); c[0] = make_float2(__uint_as_float(r1.z), __uint_as_float(r1.w));
    c[1] = make_float2(__uint_as_float(r2.x), __uint_as_float(r2.y)); c[2] = make_float2(__uint_as_float(r2.z), __uint_as_float(r2.w));
    C = __uint_as_float(r3.x);
}

// ---- the kernel -------------------------------------------------------------------------------------
// SETS: set screen on a gathered sub-table -- the leader draws list positions instead of schedule indices and reads (I2, J)
// from p.set_tiles, and a pair counts only when set_pair_wanted and set_pair_live. The whole-table instantiation is unchanged.
using MmaPipe = CtaPipe<MMA_STAGES, KPS, KB_BYTES, EPI_WARPS * COL_STAGE_BYTES>;   // extra: per epilogue warp, 32 column-role records

template <bool SETS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MMA_THREADS, 1)
pair_screen_mma_kernel(const __grid_constant__ CUtensorMap map_ab, const MmaParams p) {
    extern __shared__ unsigned char smem_raw[];
    MmaPipe pipe;
    unsigned char *col_sm = pipe.setup(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = pipe.rank;
    const uint32_t tmem_base = pipe.tmem;

    // The shard's tiles have local indices u = 0, 1, ...; shard_tile(u) is the schedule index. Shards own alternating chunks
    // of SHARD_CHUNK consecutive tiles, so that the tiles a GPU works on at the same time share A- and B-blocks in its L2
    // whatever the number of GPUs. The pair draws its u from p.tile_counter (tile feed).
    const uint64_t last = p.dump ? p.dump_tile + 1 : p.n_tiles;

    if (warp == TMA_WARP) {
        // ===== TMA producer (both CTAs: own 128 A rows, own half of the 256 B rows) =====
        TileCursor cur;
        uint32_t dump_u = 0;
        uint64_t t_cur = 0;
        bool located = false;
        auto next_t = [&]() -> uint64_t {              // schedule index of the next tile of the shard (leader only)
            if (p.dump) return p.dump_tile + dump_u++;
            return shard_tile(atomicAdd(p.tile_counter, 1ull), p.shard, p.n_shards);
        };
        uint64_t t_next = rank == 0 && lane == 0 ? next_t() : 0;   // the leader's producer thread draws one tile ahead
        auto draw = [&](uint32_t &I2, uint32_t &J) -> bool {
            const uint64_t t = t_next;
            if (t >= last) return false;
            if constexpr (SETS) { const uint2 e = p.set_tiles[t]; I2 = e.x; J = e.y; }
            else {
                if (!located) { cur.locate(t, p.TB, p.n_bands, p.band); located = true; }
                else cur.advance(t - t_cur, p.TB, p.n_bands);
                t_cur = t;
                cur.decode(p.TB, I2, J);
            }
            t_next = next_t();                         // in flight while this tile is published and its loads are issued
            return true;
        };
        auto load = [&](uint32_t I2, uint32_t J, unsigned char *dst, uint32_t blk, uint64_t *full) {
            const int a_row = (int)((2 * I2 + rank) * (2 * MMA_A_SNPS)), b_row = (int)(J * MMA_N + rank * MMA_B_SNPS);
            tma_load_2d_pair(dst, &map_ab, (int)(blk * MMA_KB), a_row, full);
            tma_load_2d_pair(dst + A_STAGE_BYTES, &map_ab, (int)(blk * MMA_KB), b_row, full);
        };
        pipe.produce(p.NKB, draw, load, p.prof);
    } else if (warp == MMA_WARP) {
        // ===== MMA issuer (leader CTA only) =====
        pipe.issue(p.NKB, [&](uint32_t d_addr, uint32_t a_addr, uint32_t blk) {
            const uint64_t ad = umma_desc(a_addr), bd = umma_desc(a_addr + A_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < MMA_KB / UMMA_K; ++k)
                tc_mma_i8(d_addr, ad + (uint64_t)(k * UMMA_K >> 4), bd + (uint64_t)(k * UMMA_K >> 4), IDESC_I8, (blk | (uint32_t)k) != 0);
        }, p.prof);
    } else {
        // ===== epilogue (both CTAs: own 64 A-SNPs x the tile's 128 B-SNPs) =====
        const int ew = warp;
        const int q = warp & 3;                       // TMEM lane quadrant this warp may read
        const int g = ew >> 2;                        // column group: 64 accumulator columns = 32 B-SNPs
        const int a_loc = 16 * q + (lane >> 1);       // A-SNP of this lane inside the CTA's 64
        const int pl = lane & 1;                      // plane held by this lane's TMEM row (0: aa, 1: bb)
        GW_PROF(long long prof_tw = 0; const long long prof_e0 = clock64();)
        uint32_t I2, J;
        for (uint64_t tile = 0; pipe.next_warp(lane, (uint32_t)tile, I2, J); ++tile) {
            const uint32_t I = 2 * I2 + rank;         // this CTA's 64-SNP A-block
            const uint64_t gi = (uint64_t)I * MMA_A_SNPS + a_loc;
            // row-role record of this lane's A-SNP. Odd lanes own plane "bb" of A: they see the table with A's
            // genotype labels aa <-> bb exchanged, which the statistic does not depend on, so their record is
            // loaded with the two swapped instead of re-ordering four counts per pair.
            MmaRowF A;
            uint32_t keyA = 0;                        // SETS: this A-SNP's d_set_keys entry, carried in the record's padding
            {
                const uint4 *rq = reinterpret_cast<const uint4 *>(p.rowf + gi);
                const uint4 r0 = __ldg(rq), r1 = __ldg(rq + 1), r2 = __ldg(rq + 2), r3 = __ldg(rq + 3);
                A.dA0 = make_float2(__uint_as_float(r0.x), __uint_as_float(r0.y)); A.dA2 = make_float2(__uint_as_float(r0.z), __uint_as_float(r0.w));
                A.pca1 = make_float2(__uint_as_float(r1.x), __uint_as_float(r1.y)); A.RA = make_float2(__uint_as_float(r1.z), __uint_as_float(r1.w));
                A.cm0 = make_float2(__uint_as_float(r2.x), __uint_as_float(r2.y)); A.cm2 = make_float2(__uint_as_float(r2.z), __uint_as_float(r2.w));
                A.C = __uint_as_float(r3.x);
                if constexpr (SETS) keyA = r3.y;
                if (pl) { float2 x = A.dA0; A.dA0 = A.dA2; A.dA2 = x; x = A.cm0; A.cm0 = A.cm2; A.cm2 = x; }
            }
            const float thr_now = sink_threshold(p.sink);
            const float thrA = thr_now / 1.3862943611f + p.q0 + A.C;   // bound pass, log2 units: N log2 tau + qc Q > thr / (2 ln 2) + q0 + C_row + C_col
            // interior tile: every pair is i < j inside the table and no block has missing calls
            bool interior = (uint64_t)(I + 1) * MMA_A_SNPS <= (uint64_t)J * MMA_B_SNPS && (uint64_t)(J + 1) * MMA_B_SNPS <= p.M &&
                            !p.tile_missing[I] && !p.tile_missing[2 * J] && !p.tile_missing[2 * J + 1];
            if constexpr (SETS) interior = false;     // every pair takes the set rule and set_pair_live
            const bool a_ok = (uint64_t)I * MMA_A_SNPS < p.M && !p.tile_missing[I];
            // missing-call flags of the two 64-SNP halves of the B-block (a half beyond the table counts as flagged)
            const bool b_bad0 = (uint64_t)(2 * J) * TILE >= p.M || p.tile_missing[2 * J];
            const bool b_bad1 = (uint64_t)(2 * J + 1) * TILE >= p.M || p.tile_missing[2 * J + 1];
            const bool b_bad = g < 2 ? b_bad0 : b_bad1;           // this warp's 32 B-SNPs lie in one half
            const bool edge_ok = a_ok && !b_bad;
            // this warp's 32 column-role records: 2 KiB contiguous in global memory -> its private shared-memory slot
            unsigned char *my_col = col_sm + ew * COL_STAGE_BYTES;
            {
                const uint4 *src = reinterpret_cast<const uint4 *>(p.colf + ((uint64_t)J * MMA_B_SNPS + 32 * g));
                uint4 *dst = reinterpret_cast<uint4 *>(my_col);
#pragma unroll
                for (int k = 0; k < 4; ++k) dst[32 * k + lane] = __ldg(src + 32 * k + lane);
                __syncwarp();
            }
            GW_PROF(const long long w2 = clock64();)
            const uint32_t buf = pipe.acc_wait(lane, tile);
            GW_PROF(prof_tw += clock64() - w2;)
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                uint32_t v[32];
                tc_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + buf * ACC_COLS + 64 * g + 32 * h, v);
                tc_wait_ld();
                // columns 4s..4s+3 = B-SNPs b0 = 2s (planes aa, bb) and b1 = 2s+1 of this 16-SNP group. Even lanes
                // (plane aa of A) finish pair (a, b0), odd lanes (plane bb of A) pair (a, b1): each sends the two
                // counts its partner needs and keeps its own two.
                if (p.dump) {
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        const uint32_t keep0 = pl ? v[4 * s + 2] : v[4 * s + 0], keep1 = pl ? v[4 * s + 3] : v[4 * s + 1];
                        const uint32_t send0 = pl ? v[4 * s + 0] : v[4 * s + 2], send1 = pl ? v[4 * s + 1] : v[4 * s + 3];
                        const uint32_t got0 = __shfl_xor_sync(0xffffffffu, send0, 1), got1 = __shfl_xor_sync(0xffffffffu, send1, 1);
                        if (rank != p.dump_rank) continue;
                        const int b_loc = 32 * g + 16 * h + 2 * s + pl;
                        const uint32_t d0 = pl ? got0 : keep0, d1 = pl ? got1 : keep1, d2 = pl ? keep0 : got0, d3 = pl ? keep1 : got1;
                        uint32_t *o = p.dump + ((uint64_t)a_loc * MMA_B_SNPS + b_loc) * 8;
                        o[0] = d0 & 0x3fffu; o[1] = d1 & 0x3fffu; o[2] = d2 & 0x3fffu; o[3] = d3 & 0x3fffu;
                        o[4] = d0 >> CTRL_SHIFT; o[5] = d1 >> CTRL_SHIFT; o[6] = d2 >> CTRL_SHIFT; o[7] = d3 >> CTRL_SHIFT;
                    }
                    continue;
                }
                // pass 1, branch-free so that the eight pairs interleave: upper bound of the statistic
                const uint64_t gj0 = (uint64_t)J * MMA_B_SNPS + 32 * g + 16 * h + pl;
                uint32_t hot = 0;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const uint32_t keep0 = pl ? v[4 * s + 2] : v[4 * s + 0], keep1 = pl ? v[4 * s + 3] : v[4 * s + 1];
                    const uint32_t send0 = pl ? v[4 * s + 0] : v[4 * s + 2], send1 = pl ? v[4 * s + 1] : v[4 * s + 3];
                    const uint32_t got0 = __shfl_xor_sync(0xffffffffu, send0, 1), got1 = __shfl_xor_sync(0xffffffffu, send1, 1);
                    v[4 * s + 0] = keep0; v[4 * s + 1] = keep1; v[4 * s + 2] = got0; v[4 * s + 3] = got1;   // own plane of A first
                    const uint64_t gj = gj0 + 2 * s;
                    float2 b[7]; float Ccol;
                    uint32_t keyB = 0;
                    {
                        const uint4 *cq = reinterpret_cast<const uint4 *>(my_col + (16 * h + 2 * s + pl) * 64);
                        const uint4 r0 = cq[0], r1 = cq[1], r2 = cq[2], r3 = cq[3];
                        b[0] = make_float2(__uint_as_float(r0.x), __uint_as_float(r0.y)); b[1] = make_float2(__uint_as_float(r0.z), __uint_as_float(r0.w));
                        b[2] = make_float2(__uint_as_float(r1.x), __uint_as_float(r1.y)); b[3] = make_float2(__uint_as_float(r1.z), __uint_as_float(r1.w));
                        b[4] = make_float2(__uint_as_float(r2.x), __uint_as_float(r2.y)); b[5] = make_float2(__uint_as_float(r2.z), __uint_as_float(r2.w));
                        b[6] = make_float2(__uint_as_float(r3.x), __uint_as_float(r3.y)); Ccol = __uint_as_float(r3.z);
                        if constexpr (SETS) keyB = r3.w;
                    }
                    const float ub = ksa_bound_fast(decode2(keep0), decode2(keep1), decode2(got0), decode2(got1), A, b, p.N, p.qc);
                    const bool valid = interior | ((gi < gj) & (gj < p.M) & edge_ok &
                                                   (!SETS || (set_pair_wanted(gi, gj, p.set_c1, p.set_a1) & set_pair_live(keyA, keyB))));   // no short-circuit: keeps the pass branch-free
                    hot |= (valid & (ub > thrA + Ccol)) ? (1u << s) : 0u;
                }
                // pass 2, rare: exact fp32 formula for the pairs whose bound passed
                if (__any_sync(0xffffffffu, hot != 0)) {
#pragma unroll 1
                    for (int s = 0; s < 8; ++s) {
                        if (!((hot >> s) & 1u)) continue;
                        uint32_t k0, k1, g0, g1;   // dynamic index into v[]: select instead of local memory
                        k0 = v[0]; k1 = v[1]; g0 = v[2]; g1 = v[3];
#pragma unroll
                        for (int q8 = 1; q8 < 8; ++q8)
                            if (s == q8) { k0 = v[4 * q8]; k1 = v[4 * q8 + 1]; g0 = v[4 * q8 + 2]; g1 = v[4 * q8 + 3]; }
                        const uint64_t gj = gj0 + 2 * s;
                        // the exact-pass operands, rebuilt from the bound-pass records already on chip (no global loads):
                        // pca[g] = dA_g + pca[1], w[g] = dB_g + w[1], control count = pooled - case
                        const MmaColF &B = *reinterpret_cast<const MmaColF *>(my_col + (16 * h + 2 * s + pl) * 64);
                        float2 pca[3], ca[3], w[3], cb[3];
                        pca[1] = A.pca1; pca[0] = __fadd2_rn(A.dA0, A.pca1); pca[2] = __fadd2_rn(A.dA2, A.pca1);
                        ca[0] = make_float2(A.cm0.x, A.cm0.y - A.cm0.x); ca[2] = make_float2(A.cm2.x, A.cm2.y - A.cm2.x); ca[1] = ca[0];
                        w[1] = B.w1; w[0] = __fadd2_rn(B.dB0, B.w1); w[2] = __fadd2_rn(B.dB2, B.w1);
                        cb[0] = make_float2(B.cm0.x, B.cm0.y - B.cm0.x); cb[1] = make_float2(B.cm1.x, B.cm1.y - B.cm1.x);
                        cb[2] = make_float2(B.cm2.x, B.cm2.y - B.cm2.x);
                        const float Crow = A.C, Ccol = B.C;
                        const Cells t = derive_cells(decode2(k0), decode2(k1), decode2(g0), decode2(g1), ca, cb);
                        float tau;
                        (void)ksa_upper_bound(t, pca, w, Crow + Ccol, p.N, p.qc, p.q0, tau);
                        const float stat = ksa_screen_cells(t, tau, Crow + Ccol, p.N);
                        if (stat > thr_now) sink_push(p.sink, (uint32_t)gi, (uint32_t)gj, stat);
                    }
                }
            }
            pipe.acc_release(lane, buf);
        }
        GW_PROF(if (p.prof && lane == 0 && (warp == 0 || warp == 15)) {
            unsigned long long *o = p.prof + blockIdx.x * 8;
            o[warp == 0 ? 3 : 7] = (unsigned long long)(clock64() - prof_e0); if (warp == 0) o[4] = (unsigned long long)prof_tw;
        })
    }
    pipe.teardown();
}

// ---- tensor-core roofline probe ---------------------------------------------------------------------
// The screen kernel's own instruction -- tcgen05.mma.cta_group::2.kind::i8, M = 256, N = 256, K = 32, operands in the
// SWIZZLE_128B K-major layout, accumulators alternating between the two halves of TMEM -- issued back to back on
// operands that stay resident in shared memory: no TMA traffic, no epilogue. What the pair of SMs can do when nothing
// but the MMA pipe and its shared-memory operand reads is in the way; the denominator of roofline.tensor.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
i8_peak_kernel(uint32_t kblocks, uint32_t seed) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (base - smem_u32(smem_raw));
    uint64_t *done = reinterpret_cast<uint64_t *>(sm + KB_BYTES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(done + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    // operands: signed one-hot-like bytes (0, +1, -128) as in the real matrix; the values do not matter for the rate
    for (uint32_t q = tid; q < KB_BYTES / 4; q += blockDim.x) {
        uint32_t h = (q + 1u) * 2654435761u ^ seed ^ (rank * 0x9E3779B9u);
        h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
        uint32_t w = 0;
        for (int b = 0; b < 4; ++b) { const uint32_t r = (h >> (8 * b)) & 7u; w |= (r == 0 ? 0x01u : (r == 1 ? 0x80u : 0u)) << (8 * b); }
        reinterpret_cast<uint32_t *>(sm)[q] = w;
    }
    if (tid == 0) { mbar_init(done, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (warp == 0) tmem_alloc_pair(tmem_slot);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores above -> async-proxy reads of the MMAs
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 1 && lane == 0 && rank == 0) {
        const uint64_t ad = umma_desc(base), bd = umma_desc(base + A_STAGE_BYTES);
        for (uint32_t kb = 0; kb < kblocks; ++kb) {
            const uint32_t d_addr = tmem_base + ((kb >> 4) & 1u) * ACC_COLS;      // 16 sample blocks per accumulator, then the other one
#pragma unroll
            for (int k = 0; k < MMA_KB / UMMA_K; ++k)
                tc_mma_i8(d_addr, ad + (uint64_t)(k * UMMA_K >> 4), bd + (uint64_t)(k * UMMA_K >> 4), IDESC_I8, (kb & 15u) != 0 || k != 0);
        }
        tc_commit_mc(done, 1);            // arrives on the leader's barrier once every MMA above has completed
        mbar_wait_wd(done, 0);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base);
    }
}

// ---- which two genotype classes a SNP puts on the tensor cores ----------------------------------------
// Any two of a SNP's three genotype planes determine the pair tables once the per-SNP class counts are known (the
// reference's own shortcut derives the heterozygote cells from the two homozygote planes, compressed_genotype_table5.cpp:
// 1084-1092). The statistic does not care how a SNP's genotypes are labelled, so every SNP puts its two RAREST classes on
// the tensor cores and derives the commonest one: the operand bytes of a SNP with a 10 % minor allele are then 19 %
// non-zero instead of 82 %, which is what the multipliers and the operand buses toggle on. `derived` (0 aa, 1 ab, 2 bb; 1 =
// the reference's choice) is per SNP; "role" 0 / 2 are the two planes in genotype order, role 1 the derived class, and all
// per-SNP epilogue records are stored by role, so nothing downstream knows.
__device__ __forceinline__ void plane_roles(uint32_t derived, int (&perm)[3]) {
    perm[0] = derived == 0 ? 1 : 0; perm[1] = (int)derived; perm[2] = derived == 2 ? 1 : 2;
}
__global__ void plane_choice_kernel(const gwasdev_marginal_information *__restrict__ mi, uint64_t M, uint64_t Mrec, int classic,
                                    uint8_t *__restrict__ derived) {
    const uint64_t snp = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (snp >= Mrec) return;
    uint32_t d = 1;
    if (!classic && snp < M) {
        const uint32_t a = mi[snp].margins[0], h = mi[snp].margins[1], b = mi[snp].margins[2];
        if (a > h && a >= b) d = 0; else if (b > h && b > a) d = 2;      // ties keep the heterozygote derived
    }
    derived[snp] = (uint8_t)d;
}

// ---- operand matrix: raw rows + class masks -> signed one-hot bytes ------------------------------------

// Operand rows straight from the RAW rows and the selection's class masks (no compaction): a sample's byte is +1
// when it is a case with the genotype, -128 (or +1 in its own plane, LAYOUT 1) when it is a control with it, 0 otherwise --
// wherever the sample sits in the row, because a sample is a case or a control for BOTH SNPs of a pair and the products are
// summed over all samples. One thread per (SNP, 32-sample word of the raw row); a row is 32 * Wr bytes.
//   LAYOUT -1: two planes per SNP (aa, bb), rows 2s + p                     (pair_screen_mma_kernel)
//   LAYOUT  0: four rows per SNP (aa, bb, xx = class member without a call, zero padding), rows 4s + p   (mma4 MODE 0)
//   LAYOUT  1: four rows per SNP (aa cases, bb cases, aa controls, bb controls), every byte +1          (mma4 MODE 1)
__device__ __forceinline__ void store_class_bytes(int8_t *dst, uint32_t xc, uint32_t xt) {     // 32 bytes: +1 for bits of xc, -128 for bits of xt
    uint4 lo, hi;
    lo.x = spread4(xc & 15u) | (spread4(xt & 15u) << 7);                 lo.y = spread4((xc >> 4) & 15u) | (spread4((xt >> 4) & 15u) << 7);
    lo.z = spread4((xc >> 8) & 15u) | (spread4((xt >> 8) & 15u) << 7);   lo.w = spread4((xc >> 12) & 15u) | (spread4((xt >> 12) & 15u) << 7);
    hi.x = spread4((xc >> 16) & 15u) | (spread4((xt >> 16) & 15u) << 7); hi.y = spread4((xc >> 20) & 15u) | (spread4((xt >> 20) & 15u) << 7);
    hi.z = spread4((xc >> 24) & 15u) | (spread4((xt >> 24) & 15u) << 7); hi.w = spread4((xc >> 28) & 15u) | (spread4((xt >> 28) & 15u) << 7);
    reinterpret_cast<uint4 *>(dst)[0] = lo; reinterpret_cast<uint4 *>(dst)[1] = hi;
}

template <int LAYOUT>
__global__ void expand_raw_kernel(const uint32_t *__restrict__ raw, uint32_t Wr, const uint32_t *__restrict__ mca, const uint32_t *__restrict__ mco,
                                  uint32_t kbytes, uint64_t M, const uint8_t *__restrict__ derived, int8_t *__restrict__ mm) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t snp = idx / Wr;
    if (snp >= M) return;
    const uint32_t w = (uint32_t)(idx - snp * Wr);
    const uint32_t p1 = raw[snp * 2ull * Wr + w], p2 = raw[snp * 2ull * Wr + Wr + w], ca = mca[w], co = mco[w];
    const uint32_t bb = p1 & p2, aa = p1 ^ bb;
    constexpr int ROWS = LAYOUT < 0 ? 2 : 4;
    int8_t *row = mm + (ROWS * snp) * (uint64_t)kbytes + 32ull * w;
    if (LAYOUT == 1) {
        store_class_bytes(row, aa & ca, 0u);                     store_class_bytes(row + kbytes, bb & ca, 0u);
        store_class_bytes(row + 2ull * kbytes, aa & co, 0u);     store_class_bytes(row + 3ull * kbytes, bb & co, 0u);
    } else if (LAYOUT == 0) {
        store_class_bytes(row, aa & ca, aa & co);
        store_class_bytes(row + kbytes, bb & ca, bb & co);
        const uint32_t xx = ~(p1 | p2);
        store_class_bytes(row + 2ull * kbytes, xx & ca, xx & co);       // the padding row stays zero (memset)
    } else {
        const uint32_t d = derived[snp], ab = p2 ^ bb;
        const uint32_t g0 = d == 0 ? ab : aa, g2 = d == 2 ? ab : bb;    // roles 0 and 2 (plane_roles)
        store_class_bytes(row, g0 & ca, g0 & co);
        store_class_bytes(row + kbytes, g2 & ca, g2 & co);
    }
}

// =====================================================================================================
// Tiles WITH missing calls on the tensor cores (four planes per SNP).
//
// The four counted corners stay exact when calls are missing; what fails is the margin shortcut for the five cells
// that involve the heterozygote, because "not aa, not bb" is then "ab or missing". With a third one-hot plane per SNP --
// xx, the class members without a call -- the GEMM also yields |aa_A & xx_B|, |bb_A & xx_B|, |xx_A & aa_B|, |xx_A & bb_B|
// and |xx_A & xx_B|, and the nine core cells follow exactly (the reference's other branch,
// compressed_genotype_table5.cpp:1000-1067, counts them with nine AND+POPC streams):
//     AA_Bb = c_A[aa] - AA_BB - AA_bb - AA_xx        aa_Bb likewise          Aa_BB = c_B[aa] - AA_BB - aa_BB - xx_BB
//     Aa_bb likewise        Aa_Bb = c_A[ab] - Aa_BB - Aa_bb - (c_B[xx] - AA_xx - aa_xx - xx_xx)
// with c_X[g] the per-SNP class counts. Operand rows 4s+p: p = 0 aa, 1 bb, 2 xx, 3 zero padding (a power of two keeps
// the pipeline of the two-plane kernel byte for byte: 256 x 256 row tiles, the same TMA boxes, descriptors and barriers;
// a tile is now 64 x 64 SNPs, i.e. one 64-SNP missing-call block against another). The epilogue has no margin shortcut
// and no bound pass: the four lanes that hold the planes of one A-SNP exchange their products so that each owns two of
// the eight pairs of a 32-column load, builds the 3x3x2 table and evaluates ksa_screen_f32 (the epilogue of the
// AND+POPC kernel it replaces). Only tiles with a missing call in either block are computed; the others belong to
// pair_screen_mma_kernel.
// fp32 screen value of a 3x3x2 table whose SNPs may have missing calls: ksa_screen_f32's formula (pair_common.cuh) with the 27
// n log n terms as n * lg2.approx(n + 2^-126) in log2 units (the two-plane kernel's form: 0 * lg2(2^-126) = -0 for an empty cell)
// and the row / column sums taken on the integer table. A column without samples has w = NaN, which reaches tau through
// 0 * NaN exactly as in ksa_screen_f32: such a pair compares false against any threshold.
__device__ __forceinline__ float ksa_screen_table(const uint32_t (&n)[2][3][3], const PairSide &A, const PairSide &B, float N, float lnN) {
    const float tiny = 1.17549435e-38f;
    float S2 = 0.f, tau = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const float c0 = u2f(n[0][a][b]), c1 = u2f(n[1][a][b]), cab = c0 + c1;
            const float W = fmaf(B.w[0][b], A.pca[0][a], B.w[1][b] * A.pca[1][a]);
            tau = fmaf(cab, W, tau);
            S2 = fmaf(c0, lg2_approx(c0 + tiny), S2);
            S2 = fmaf(c1, lg2_approx(c1 + tiny), S2);
            S2 = fmaf(-cab, lg2_approx(cab + tiny), S2);
        }
    float L = 0.f;
    uint32_t total = 0;
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            const uint32_t row = n[k][g][0] + n[k][g][1] + n[k][g][2], col = n[k][0][g] + n[k][1][g] + n[k][2][g];
            L = fmaf(u2f(row), A.lpca[k][g], L);
            L = fmaf(u2f(col), B.lw[k][g], L);
            total += row;
        }
    L = fmaf(u2f(total), lnN, L);
    return 2.0f * fmaf(0.69314718056f, fmaf(N, lg2_approx(tau), S2), -L);
}

constexpr int M4_PLANES = 4;
constexpr int M4_A_SNPS = 2 * MMA_A_SNPS / M4_PLANES;        // 32 A-SNPs per CTA (128 rows)
constexpr int M4_BLK = MMA_N / M4_PLANES;                    // 64 SNPs per schedule block = B-SNPs of a tile
static_assert(M4_BLK == TILE, "the four-plane tiles coincide with the 64-SNP missing-call blocks");

// Shared memory of pair_screen_mma4_kernel<MODE>. The missing-call layouts (modes 0, 2) stage 96 B rows per sample block, and the
// 24 KiB that frees carry the epilogue's product exchange: 1 600 bytes per warp (32 rows of twelve int32, rows skewed by 16 bytes
// per eight lanes so that the quads' reads fall on different banks).
constexpr int M4_XCH_WARP = 1600;
template <int MODE> struct M4Smem {
    static constexpr int CPB = MODE == 1 ? 4 : 3;                                   // accumulator columns per B-SNP
    static constexpr int KBB = A_STAGE_BYTES + MMA_B_SNPS / 4 * CPB * MMA_KB;       // 32 KiB (split classes) or 28 KiB
    static constexpr int XCH = MODE == 1 ? 0 : EPI_WARPS * M4_XCH_WARP;
};
// extra: the exchange rows, then per epilogue warp the PairSide records of its 16 B-SNPs. MODE 2 holds both accumulators per tile.
template <int MODE>
using M4Pipe = CtaPipe<MMA_STAGES, KPS, M4Smem<MODE>::KBB, M4Smem<MODE>::XCH + EPI_WARPS * COL_STAGE_BYTES, MODE == 2 ? 1 : 2>;

struct Mma4Params {
    uint32_t TB, NKB, n_bands, band;
    uint32_t case_kb;              // 128-byte sample blocks of the case range of a row (two-accumulator mode)
    uint64_t M, n_tiles;
    uint32_t shard, n_shards;
    const PairSide *side;
    const uint8_t *tile_missing;   // per 64-SNP block
    float N, lnN;
    CandSink sink;
    unsigned long long *tile_counter;   // zero at launch (tile feed)
    const uint2 *set_tiles;             // set screens (SETS instantiations; appended, as in MmaParams): the shard's tiles, n_tiles of them,
    uint64_t set_c1, set_a1;            // the segment bounds and the sub-table's d_set_keys
    const uint32_t *set_keys;
};

__device__ __forceinline__ uint32_t sel4(uint32_t k, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    const uint32_t lo = (k & 1u) ? b : a, hi = (k & 1u) ? d : c;
    return (k & 2u) ? hi : lo;
}

// SPLIT = false: planes (aa, bb, xx, padding) with the signed case/control bytes, tiles WITH missing calls (above).
// SPLIT = true : planes (aa of the cases, bb of the cases, aa of the controls, bb of the controls), every byte +1, tiles
//                WITHOUT missing calls of cohorts whose class sizes do not fit the packed accumulator of the two-plane
//                kernel (n_case >= 16384 or n_ctrl >= 131072): the two classes land in different products, each a full
//                int32 count, and the five other cells follow from the per-SNP class counts as in the reference's shortcut
//                (compressed_genotype_table5.cpp:1084-1092, :1133-1141). Same pipeline, same 4x MACs.
// MODE 2  : planes (aa, bb, xx, padding), every byte +1, cases and controls accumulated into SEPARATE TMEM accumulators (the
//                K range of a row is class-pure: the MMAs of the case sample blocks go to one, those of the control blocks
//                to the other). Any class sizes with missing calls; the price is the accumulator double buffering (the
//                epilogue of a tile no longer overlaps the MMAs of the next). All tiles of such a cohort take it.
// SETS: set screen as in pair_screen_mma_kernel; the leader walks the list and `wanted` still picks the tiles of this launch.
template <int MODE, bool SETS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MMA_THREADS, 1)
pair_screen_mma4_kernel(const __grid_constant__ CUtensorMap map_ab, const __grid_constant__ CUtensorMap map_b3, const Mma4Params p) {
    constexpr bool SPLIT = MODE == 1, TWOACC = MODE == 2;
    // B side: the padding plane never enters a pair's table, so the missing-call layouts send only three rows per B-SNP to the
    // tensor cores (a 3-D TMA box over the same matrix: sample bytes x 3 of the 4 planes x 32 SNPs = 96 dense rows): N = 192.
    constexpr int CPB = M4Smem<MODE>::CPB;
    constexpr uint32_t IDESC = idesc_i8(M4_BLK * CPB);
    extern __shared__ unsigned char smem_raw[];
    M4Pipe<MODE> pipe;
    unsigned char *xch_sm = pipe.setup(smem_raw);                               // per epilogue warp: product exchange rows (missing-call layouts)
    unsigned char *col_sm = xch_sm + M4Smem<MODE>::XCH;                         // per epilogue warp: PairSide records of its 16 B-SNPs
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = pipe.rank;
    const uint32_t tmem_base = pipe.tmem;

    // the tiles this launch computes: the leader's producer skips the others while it draws (TileDraw), the other roles only see these
    auto wanted = [&](uint32_t I2, uint32_t J) -> bool { return TWOACC || ((p.tile_missing[I2] | p.tile_missing[J]) != 0) != SPLIT; };

    if (warp == TMA_WARP) {
        TileDraw td;
        td.counter = p.tile_counter; td.shard = p.shard; td.n_shards = p.n_shards; td.TB = p.TB; td.n_bands = p.n_bands; td.band = p.band; td.last = p.n_tiles;
        auto draw = [&](uint32_t &I2, uint32_t &J) -> bool {
            if constexpr (SETS) {
                for (;;) {
                    const uint64_t u = atomicAdd(p.tile_counter, 1ull);
                    if (u >= p.n_tiles) return false;
                    const uint2 e = p.set_tiles[u];
                    I2 = e.x; J = e.y;
                    if (wanted(I2, J)) return true;
                }
            } else {
                if (!td.next(I2, J, wanted)) return false;
                td.prefetch();
                return true;
            }
        };
        auto load = [&](uint32_t I2, uint32_t J, unsigned char *dst, uint32_t blk, uint64_t *full) {
            const int a_row = (int)((2 * I2 + rank) * (2 * MMA_A_SNPS)), b_row = (int)(J * MMA_N + rank * MMA_B_SNPS);
            tma_load_2d_pair(dst, &map_ab, (int)(blk * MMA_KB), a_row, full);
            if (SPLIT) tma_load_2d_pair(dst + A_STAGE_BYTES, &map_ab, (int)(blk * MMA_KB), b_row, full);
            else tma_load_3d_pair(dst + A_STAGE_BYTES, &map_b3, (int)(blk * MMA_KB), 0, b_row / M4_PLANES, full);
        };
        pipe.produce(p.NKB, draw, load);
    } else if (warp == MMA_WARP) {
        // TWOACC: the case sample blocks accumulate into the tile's accumulator, the control blocks into the next ACC_COLS columns
        pipe.issue(p.NKB, [&](uint32_t d_addr, uint32_t a_addr, uint32_t blk) {
            const uint64_t ad = umma_desc(a_addr), bd = umma_desc(a_addr + A_STAGE_BYTES);
            const bool ctrl = TWOACC && blk >= p.case_kb;
            const uint32_t d_blk = ctrl ? d_addr + ACC_COLS : d_addr;
            const uint32_t first_blk = ctrl ? p.case_kb : 0u;
#pragma unroll
            for (int k = 0; k < MMA_KB / UMMA_K; ++k)
                tc_mma_i8(d_blk, ad + (uint64_t)(k * UMMA_K >> 4), bd + (uint64_t)(k * UMMA_K >> 4), IDESC, (blk != first_blk) || k != 0);
        });
    } else {
        // ===== epilogue (both CTAs: own 32 A-SNPs x the tile's 64 B-SNPs) =====
        const int ew = warp;
        const int q = warp & 3;                       // TMEM lane quadrant: rows 32q.. = A-SNPs 8q..8q+7 of this CTA
        const int g = ew >> 2;                        // column group: 16 B-SNPs = 16 * CPB accumulator columns
        const int a_loc = 8 * q + (lane >> 2);        // A-SNP of this lane inside the CTA's 32
        const uint32_t pl = (uint32_t)lane & 3u;      // plane held by this lane's TMEM row (0 aa, 1 bb, 2 xx, 3 padding)
        const unsigned qbase = (unsigned)lane & ~3u;
        uint32_t I2, J;
        for (uint64_t tile = 0; pipe.next_warp(lane, (uint32_t)tile, I2, J); ++tile) {
            const uint64_t gi = (uint64_t)I2 * M4_BLK + rank * M4_A_SNPS + a_loc;
            // this warp's 16 column-role records (PairSide, 128 bytes each): 2 KiB contiguous -> its shared-memory slot
            unsigned char *my_col = col_sm + ew * COL_STAGE_BYTES;
            {
                const uint4 *src = reinterpret_cast<const uint4 *>(p.side + ((uint64_t)J * M4_BLK + 16 * g));
                uint4 *dst = reinterpret_cast<uint4 *>(my_col);
#pragma unroll
                for (int k = 0; k < 4; ++k) dst[32 * k + lane] = __ldg(src + 32 * k + lane);
                __syncwarp();
            }
            const PairSide &A = p.side[gi < p.M ? gi : 0];   // read through L1: 8 records per warp, reused for 16 B-SNPs
            const float thr_now = sink_threshold(p.sink);
            const uint32_t buf = pipe.acc_wait(lane, tile);
            // one pair's 3x3x2 table from its products and both SNPs' class counts, then the screen statistic
            auto finish_pair = [&](uint64_t gj, const PairSide &B, const uint32_t (&prod)[CPB][CPB], const uint32_t (&prod_ctl)[3][3]) {
                uint32_t n[2][3][3];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const uint32_t *ca = A.cnt[k], *cb = B.cnt[k];     // aa, ab, bb, xx
                    if (SPLIT) {
                        const uint32_t AB = prod[2 * k][2 * k], Ab = prod[2 * k][2 * k + 1], aB = prod[2 * k + 1][2 * k], ab = prod[2 * k + 1][2 * k + 1];
                        n[k][0][0] = AB; n[k][0][2] = Ab; n[k][2][0] = aB; n[k][2][2] = ab;
                        n[k][0][1] = ca[0] - AB - Ab;
                        n[k][2][1] = ca[2] - aB - ab;
                        n[k][1][0] = cb[0] - AB - aB;
                        n[k][1][2] = cb[2] - Ab - ab;
                        n[k][1][1] = cb[1] - n[k][0][1] - n[k][2][1];
                    } else {
                        uint32_t x[3][3];   // x[P][c]: class-k count of (plane P of A) & (plane c of B); planes aa, bb, xx
#pragma unroll
                        for (int P = 0; P < 3; ++P)
#pragma unroll
                            for (int c = 0; c < 3; ++c)
                                x[P][c] = TWOACC ? (k ? prod_ctl[P][c] : prod[P][c]) : (k ? (prod[P][c] >> CTRL_SHIFT) : (prod[P][c] & 0x3fffu));
                        n[k][0][0] = x[0][0]; n[k][0][2] = x[0][1]; n[k][2][0] = x[1][0]; n[k][2][2] = x[1][1];
                        n[k][0][1] = ca[0] - x[0][0] - x[0][1] - x[0][2];
                        n[k][2][1] = ca[2] - x[1][0] - x[1][1] - x[1][2];
                        n[k][1][0] = cb[0] - x[0][0] - x[1][0] - x[2][0];
                        n[k][1][2] = cb[2] - x[0][1] - x[1][1] - x[2][1];
                        n[k][1][1] = ca[1] - n[k][1][0] - n[k][1][2] - (cb[3] - x[0][2] - x[1][2] - x[2][2]);
                    }
                }
                const float stat = ksa_screen_table(n, A, B, p.N, p.lnN);
                if (stat > thr_now) sink_push(p.sink, (uint32_t)gi, (uint32_t)gj, stat);
            };
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                uint32_t v[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + buf * ACC_COLS + 8 * CPB * (2 * g + h);
                // columns CPB s .. CPB s + CPB - 1 = planes of B-SNP s of this load (s < 8). Lane o of the quad owns the
                // pairs (a, s) for s = o and o + 4 and needs the products of the quad's other planes for them.
                if constexpr (SPLIT) {
                    // through the registers: in rotation r every lane reads from quad lane (o + r) & 3 the four products that lane
                    // holds for the reader's two pairs: D[e][r][c] = product (plane (o + r) & 3 of A, plane c of B-SNP o + 4e).
                    tc_ld32(taddr, v);
                    tc_wait_ld();
                    uint32_t D[2][4][4];
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const uint32_t d = (pl - (uint32_t)r) & 3u;          // the lane that reads from me in this rotation
                        const unsigned src = qbase | ((pl + (uint32_t)r) & 3u);
#pragma unroll
                        for (int e = 0; e < 2; ++e)
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const uint32_t mine = sel4(d, v[16 * e + c], v[16 * e + 4 + c], v[16 * e + 8 + c], v[16 * e + 12 + c]);
                                D[e][r][c] = r == 0 ? mine : __shfl_sync(0xffffffffu, mine, src);
                            }
                    }
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int b_loc = 16 * g + 8 * h + 4 * e + (int)pl;
                        const uint64_t gj = (uint64_t)J * M4_BLK + b_loc;
                        if (!(gi < gj && gj < p.M && (!SETS || (set_pair_wanted(gi, gj, p.set_c1, p.set_a1) && set_pair_live(__ldg(p.set_keys + gi), __ldg(p.set_keys + gj)))))) continue;
                        uint32_t prod[CPB][CPB], none[3][3];                 // plane P of A is what arrived in rotation (P - o) & 3
#pragma unroll
                        for (int P = 0; P < 4; ++P) {
                            const uint32_t r = ((uint32_t)P - pl) & 3u;
#pragma unroll
                            for (int c = 0; c < 4; ++c) prod[P][c] = sel4(r, D[e][0][c], D[e][1][c], D[e][2][c], D[e][3][c]);
                        }
                        finish_pair(gj, *reinterpret_cast<const PairSide *>(my_col + (8 * h + 4 * e + (int)pl) * 128), prod, none);
                    }
                } else {
                    // through shared memory: every lane writes the twelve products it holds for four B-SNPs to its row of the warp's
                    // exchange block (three 16-byte stores) and reads the nine of its pair from the rows of its quad: no selects,
                    // no shuffles, conflict-free both ways (row = 12 words, skewed by 4 words per eight lanes).
                    uint32_t vc[32];
                    if (TWOACC) tc_ld24(taddr + ACC_COLS, vc);
                    tc_ld24(taddr, v);
                    tc_wait_ld();
                    uint32_t *xw = reinterpret_cast<uint32_t *>(xch_sm + ew * M4_XCH_WARP) + 4 * (lane >> 3);
                    uint4 *mine = reinterpret_cast<uint4 *>(xw + 12 * lane);
                    const uint32_t *theirs = xw + 12 * (int)qbase + 3 * (int)pl;
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        uint32_t prod[CPB][CPB], prod_ctl[3][3];
                        __syncwarp();
                        mine[0] = make_uint4(v[12 * e + 0], v[12 * e + 1], v[12 * e + 2], v[12 * e + 3]);
                        mine[1] = make_uint4(v[12 * e + 4], v[12 * e + 5], v[12 * e + 6], v[12 * e + 7]);
                        mine[2] = make_uint4(v[12 * e + 8], v[12 * e + 9], v[12 * e + 10], v[12 * e + 11]);
                        __syncwarp();
#pragma unroll
                        for (int P = 0; P < 3; ++P)
#pragma unroll
                            for (int c = 0; c < 3; ++c) prod[P][c] = theirs[12 * P + c];
                        if (TWOACC) {
                            __syncwarp();
                            mine[0] = make_uint4(vc[12 * e + 0], vc[12 * e + 1], vc[12 * e + 2], vc[12 * e + 3]);
                            mine[1] = make_uint4(vc[12 * e + 4], vc[12 * e + 5], vc[12 * e + 6], vc[12 * e + 7]);
                            mine[2] = make_uint4(vc[12 * e + 8], vc[12 * e + 9], vc[12 * e + 10], vc[12 * e + 11]);
                            __syncwarp();
#pragma unroll
                            for (int P = 0; P < 3; ++P)
#pragma unroll
                                for (int c = 0; c < 3; ++c) prod_ctl[P][c] = theirs[12 * P + c];
                        }
                        const int b_loc = 16 * g + 8 * h + 4 * e + (int)pl;
                        const uint64_t gj = (uint64_t)J * M4_BLK + b_loc;
                        if (gi < gj && gj < p.M && (!SETS || (set_pair_wanted(gi, gj, p.set_c1, p.set_a1) && set_pair_live(__ldg(p.set_keys + gi), __ldg(p.set_keys + gj)))))
                            finish_pair(gj, *reinterpret_cast<const PairSide *>(my_col + (8 * h + 4 * e + (int)pl) * 128), prod, prod_ctl);
                    }
                }
            }
            pipe.acc_release(lane, buf);
        }
    }
    pipe.teardown();
}

// operand rows of the four-plane engine: one thread per (SNP, 32-sample word), 32 bytes of each of aa, bb, xx
// (the padding row 4s+3 stays zero from the memset)
template <int MODE>
__global__ void expand_mma4_kernel(const uint32_t *__restrict__ sel, uint32_t sel_stride, uint32_t Wc, uint32_t Kc, uint32_t Kt,
                                   uint32_t n_case, uint32_t n_ctrl, uint32_t case_bytes, uint32_t kbytes, uint64_t M,
                                   int8_t *__restrict__ mm) {
    const uint32_t K = Kc + Kt;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t snp = idx / K;
    if (snp >= M) return;
    const uint32_t k = (uint32_t)(idx - snp * K);
    const uint32_t *row = sel + snp * (uint64_t)sel_stride;
    uint32_t p1, p2, off, shift, left;
    if (k < Kc) { p1 = row[sel_word(0, 0, k)]; p2 = row[sel_word(0, 1, k)]; off = 32 * k; shift = 0; left = n_case - 32 * k; }
    else { p1 = row[sel_word(2 * Wc, 0, k - Kc)]; p2 = row[sel_word(2 * Wc, 1, k - Kc)]; off = case_bytes + 32 * (k - Kc); shift = 7; left = n_ctrl - 32 * (k - Kc); }
    const uint32_t members = left >= 32 ? 0xffffffffu : ((1u << left) - 1u);     // class members among the word's 32 positions
    const uint32_t bb = p1 & p2, aa = p1 ^ bb, xx = ~(p1 | p2) & members;
    constexpr bool SPLIT = MODE == 1;
    if (MODE != 0) shift = 0;                                // every byte +1: the classes are told apart by the plane / the accumulator
#pragma unroll
    for (int pl = 0; pl < (SPLIT ? 2 : 3); ++pl) {
        const uint32_t x = pl == 0 ? aa : (pl == 1 ? bb : xx);
        const int plane = SPLIT ? (k < Kc ? pl : 2 + pl) : pl;   // split: rows 0,1 hold the cases' aa / bb, rows 2,3 the controls'
        uint4 *dst = reinterpret_cast<uint4 *>(mm + (4 * snp + plane) * (uint64_t)kbytes + off);
        uint4 lo, hi;
        lo.x = spread4(x & 15u) << shift;         lo.y = spread4((x >> 4) & 15u) << shift;
        lo.z = spread4((x >> 8) & 15u) << shift;  lo.w = spread4((x >> 12) & 15u) << shift;
        hi.x = spread4((x >> 16) & 15u) << shift; hi.y = spread4((x >> 20) & 15u) << shift;
        hi.z = spread4((x >> 24) & 15u) << shift; hi.w = spread4((x >> 28) & 15u) << shift;
        dst[0] = lo; dst[1] = hi;
    }
}

// SETS: records of a set screen's sub-table (set_pair_live): an empty class gives w = 0 instead of NaN, and the paddings of the
// bound-pass records carry the SNP's d_set_keys entry (keys)
template <bool SETS>
__global__ void mma_side_kernel(const gwasdev_marginal_information *__restrict__ mi, uint64_t M, uint64_t Mrec, uint32_t n_ind,
                                const uint8_t *__restrict__ derived, MmaRow *__restrict__ row, MmaCol *__restrict__ col, MmaRowF *__restrict__ rowf, MmaColF *__restrict__ colf,
                                const uint32_t *__restrict__ keys) {
    const uint64_t snp = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (snp >= Mrec) return;
    MmaRow r; MmaCol c;
    r.pad[0] = r.pad[1] = r.pad[2] = c.pad[0] = c.pad[1] = c.pad[2] = 0.f;
    const float qnan = __int_as_float(0x7fc00000);
    float rp[2][3], cw[2][3], cn[2][3];
    int perm[3];
    plane_roles(derived[snp], perm);
    if (snp < M) {
        const gwasdev_marginal_information m = mi[snp];
        double Cr = (double)n_ind * log2((double)n_ind), Cc = 0.0;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const uint32_t *cnt = k ? m.controls : m.cases;
#pragma unroll
            for (int role = 0; role < 3; ++role) {         // records are stored by role: planes in genotype order at 0 and 2, the derived class at 1
                const int g = perm[role];
                const double pca = m.dPca[4 * k + g], pbc = m.dPbc[4 * k + g], mar = (double)m.margins[g];
                rp[k][role] = (float)pca;
                cw[k][role] = m.margins[g] > 0 ? (float)(pbc / mar) : (SETS ? 0.f : qnan);
                cn[k][role] = (float)cnt[g];
                if (cnt[g] > 0) { Cr += (double)cnt[g] * log2(pca); Cc += (double)cnt[g] * (log2(pbc) - log2(mar)); }
            }
        }
        r.C = (float)Cr; c.C = (float)Cc;
    } else {
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int g = 0; g < 3; ++g) { rp[k][g] = 0.f; cw[k][g] = qnan; cn[k][g] = 0.f; }
        r.C = c.C = 0.f;
    }
#pragma unroll
    for (int g = 0; g < 3; ++g) {
        r.pca[g] = make_float2(rp[0][g], rp[1][g]); c.w[g] = make_float2(cw[0][g], cw[1][g]);
        r.cnt[g] = c.cnt[g] = make_float2(cn[0][g], cn[1][g]);
    }
    row[snp] = r; col[snp] = c;
    // bound-pass records (fp64 differences and dot products, rounded once)
    MmaRowF rf; MmaColF cf;
    rf.pad[0] = rf.pad[1] = rf.pad[2] = cf.pad = 0.f;
    rf.C = r.C; cf.C = c.C;
    double mp[3], pc[2][3], wc[2][3];
#pragma unroll
    for (int g = 0; g < 3; ++g) {
        mp[g] = (double)cn[0][g] + (double)cn[1][g];
#pragma unroll
        for (int k = 0; k < 2; ++k) { pc[k][g] = (double)rp[k][g]; wc[k][g] = (double)cw[k][g]; }
    }
    float da0[2], da2[2], ra[2], db0[2], db2[2], rb[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        da0[k] = (float)(pc[k][0] - pc[k][1]); da2[k] = (float)(pc[k][2] - pc[k][1]);
        ra[k] = (float)(pc[k][0] * mp[0] + pc[k][2] * mp[2] - pc[k][1] * (mp[0] + mp[2]));
        db0[k] = (float)(wc[k][0] - wc[k][1]); db2[k] = (float)(wc[k][2] - wc[k][1]);
        // a zero pooled count has w = NaN in the reference's sense (0/0) and n_.b = 0: keep the NaN in RB so that
        // tau, and with it the bound, is NaN and the pair is dropped exactly like in the exact formula
        rb[k] = (float)(wc[k][0] * mp[0] + wc[k][1] * mp[1] + wc[k][2] * mp[2]);
    }
    rf.dA0 = make_float2(da0[0], da0[1]); rf.dA2 = make_float2(da2[0], da2[1]);
    rf.pca1 = make_float2(rp[0][1], rp[1][1]); rf.RA = make_float2(ra[0], ra[1]);
    rf.cm0 = make_float2(cn[0][0], (float)mp[0]); rf.cm2 = make_float2(cn[0][2], (float)mp[2]);
    cf.dB0 = make_float2(db0[0], db0[1]); cf.dB2 = make_float2(db2[0], db2[1]);
    cf.w1 = make_float2(cw[0][1], cw[1][1]); cf.RB = make_float2(rb[0], rb[1]);
    cf.cm0 = make_float2(cn[0][0], (float)mp[0]); cf.cm1 = make_float2(cn[0][1], (float)mp[1]); cf.cm2 = make_float2(cn[0][2], (float)mp[2]);
    if constexpr (SETS) {
        const uint32_t key = snp < M ? keys[snp] : 0u;
        rf.pad[0] = cf.pad = __uint_as_float(key);
    }
    rowf[snp] = rf; colf[snp] = cf;
}

// fp32 value of the tensor-core engine's epilogue for given pairs (diagnostic twin of screen_probe_kernel)
__global__ void screen_probe_mma_kernel(const PairSrc src, const uint8_t *__restrict__ derived, const MmaRow *__restrict__ row, const MmaCol *__restrict__ col,
                                        const MmaRowF *__restrict__ rowf, const MmaColF *__restrict__ colf,
                                        const uint32_t *__restrict__ pi, const uint32_t *__restrict__ pj, uint64_t n, float N,
                                        float qc, float q0, float *__restrict__ out) {
    const uint64_t qi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= n) return;
    const uint32_t i = pi[qi], j = pj[qi];
    uint32_t c[2][4];
    {
        uint32_t t0[16], t1[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) { t0[q] = 0; t1[q] = 0; }
        core_counts_src(src, i, j, 0, 1, t0, t1);
        int pa[3], pb[3];
        plane_roles(derived[i], pa); plane_roles(derived[j], pb);
        // the four corners the kernel counts: (role 0 | 2 of A) x (role 0 | 2 of B); AA_BB, AA_bb, aa_BB, aa_bb with the reference's planes
        c[0][0] = t0[4 * pa[0] + pb[0]]; c[0][1] = t0[4 * pa[0] + pb[2]]; c[0][2] = t0[4 * pa[2] + pb[0]]; c[0][3] = t0[4 * pa[2] + pb[2]];
        c[1][0] = t1[4 * pa[0] + pb[0]]; c[1][1] = t1[4 * pa[0] + pb[2]]; c[1][2] = t1[4 * pa[2] + pb[0]]; c[1][3] = t1[4 * pa[2] + pb[2]];
    }
    float2 pca[3], ca[3], w[3], cb[3]; float Crow, Ccol;
    load_record(row + i, pca, ca, Crow);
    load_record(col + j, w, cb, Ccol);
    const Cells t = derive_cells(make_float2((float)c[0][0], (float)c[1][0]), make_float2((float)c[0][1], (float)c[1][1]),
                                 make_float2((float)c[0][2], (float)c[1][2]), make_float2((float)c[0][3], (float)c[1][3]), ca, cb);
    float tau;
    (void)ksa_upper_bound(t, pca, w, Crow + Ccol, N, qc, q0, tau);
    out[2 * qi] = ksa_screen_cells(t, tau, Crow + Ccol, N);
    // the bound exactly as the screen kernel evaluates it
    const MmaRowF A = rowf[i]; const MmaColF B = colf[j];
    const float2 b[7] = {B.dB0, B.dB2, B.w1, B.RB, B.cm0, B.cm1, B.cm2};
    const float ubf = ksa_bound_fast(make_float2((float)c[0][0], (float)c[1][0]), make_float2((float)c[0][1], (float)c[1][1]),
                                     make_float2((float)c[0][2], (float)c[1][2]), make_float2((float)c[0][3], (float)c[1][3]), A, b, N, qc);
    out[2 * qi + 1] = 1.3862943611f * (ubf - q0 - A.C - B.C);
}

}  // namespace gwasdev

using namespace gwasdev;

// ---- host side --------------------------------------------------------------------------------------
bool gwasdev_internal_mma_eligible(const gwasdev_store *s) {
    return s->n_case >= 1 && s->n_ctrl >= 1 && s->n_case < (1u << CTRL_SHIFT) && s->n_ctrl < (1u << (31 - CTRL_SHIFT));
}

// Constants of ksa_upper_bound for a cohort with n_case cases among n samples: the smallest qc (plus a safety
// factor) with H2(x) >= H2(x0) + H2'(x0)(x - x0) - qc (x - x0)^2 on [0, 1], and q0 = qc x0 n_case + n H2(x0).
static void bound_constants(uint32_t n_case, uint32_t n, float *qc_out, float *q0_out) {
    const double x0 = (double)n_case / (double)n;
    auto H = [](double x) { return (x <= 0.0 || x >= 1.0) ? 0.0 : -(x * std::log2(x) + (1.0 - x) * std::log2(1.0 - x)); };
    const double h0 = H(x0), d0 = std::log2((1.0 - x0) / x0);
    double qc = 1.0 / (2.0 * std::log(2.0) * x0 * (1.0 - x0));          // limit x -> x0: -H2''(x0) / 2
    const int G = 1 << 18;
    for (int k = 0; k <= G; ++k) {
        const double x = (double)k / G, dx = x - x0;
        if (std::fabs(dx) < 1e-6) continue;
        qc = std::max(qc, (h0 + d0 * dx - H(x)) / (dx * dx));
    }
    qc *= 1.001;
    *qc_out = (float)qc;
    *q0_out = (float)(qc * x0 * (double)n_case + (double)n * h0);
}

// operand matrix + tensor maps + per-SNP epilogue records + band table; margins must be valid
static int ensure_mma_inputs(gwasdev_store *s) {
    const uint64_t Msnp = (s->M + MMA_B_SNPS - 1) / MMA_B_SNPS * MMA_B_SNPS;
    if (!s->mm_built) {
        GW_CUDA(reserve_raw(s->d_plane_derived, s->cap_plane, Msnp));
        plane_choice_kernel<<<(unsigned)((Msnp + 255) / 256), 256, 0, s->stream>>>(s->d_mi, s->M, Msnp, s->opt[GWASDEV_OPT_CLASSIC_PLANES] != 0, s->d_plane_derived);
        GW_LAUNCHED();
        s->mm_kbytes = 32 * s->Wr;                             // one byte per sample position of the raw row (Wr is a multiple of 4 words: 128-byte blocks)
        s->mm_rows = 2 * Msnp;
        const size_t bytes = (size_t)s->mm_rows * s->mm_kbytes;
        GW_CUDA(reserve_raw(s->d_mm, s->cap_mm, bytes));
        if (Msnp > s->M) GW_CUDA(cudaMemsetAsync(s->d_mm + 2 * s->M * (size_t)s->mm_kbytes, 0, (size_t)(2 * (Msnp - s->M)) * s->mm_kbytes, s->stream));   // rows of the SNPs beyond the table
        const uint64_t work = s->M * s->Wr;
        expand_raw_kernel<-1><<<(unsigned)((work + 255) / 256), 256, 0, s->stream>>>(s->d_raw, s->Wr, s->d_case_sel_mask, s->d_ctrl_sel_mask,
                                                                                   s->mm_kbytes, s->M, s->d_plane_derived, s->d_mm);
        GW_LAUNCHED();
        if (!s->tmap_mm && posix_memalign(&s->tmap_mm, 64, sizeof(CUtensorMap)) != 0) { s->tmap_mm = nullptr; set_error("out of host memory"); return GWASDEV_ENOMEM; }
        int rc;
        if ((rc = encode_operand_map(s->d_mm, s->mm_rows, s->mm_kbytes, 2 * MMA_A_SNPS, (CUtensorMap *)s->tmap_mm)) != GWASDEV_OK) return rc;   // 128-row boxes: a CTA's A rows / its half of B
        // schedule: bands of as many A-blocks as fit 32 MB of operand rows, the last band possibly shorter
        const uint32_t TB = (uint32_t)(Msnp / MMA_BLK);
        s->mm_band = schedule_band((uint64_t)MMA_N * s->mm_kbytes);
        const uint64_t tiles = schedule_tiles(TB, s->mm_band);
        s->mm_tiles = tiles;
        if (s->mma_bound_ncase != s->n_case || s->mma_bound_n != s->n_case + s->n_ctrl) {   // 2.5 ms of host arithmetic: once per class split
            bound_constants(s->n_case, s->n_case + s->n_ctrl, &s->mma_qc, &s->mma_q0);
            s->mma_bound_ncase = s->n_case; s->mma_bound_n = s->n_case + s->n_ctrl;
        }
        s->mm_built = true;
    }
    if (!s->mma_side_valid) {
        MmaRow *row = (MmaRow *)s->d_mma_row; MmaCol *col = (MmaCol *)s->d_mma_col;
        // exact-pass records followed by the bound-pass records
        GW_CUDA(reserve_raw(row, s->cap_mma_row, Msnp * (sizeof(MmaRow) + sizeof(MmaRowF))));
        GW_CUDA(reserve_raw(col, s->cap_mma_col, Msnp * (sizeof(MmaCol) + sizeof(MmaColF))));
        s->d_mma_row = row; s->d_mma_col = col;
        if (s->d_set_keys)
            mma_side_kernel<true><<<(unsigned)((Msnp + 127) / 128), 128, 0, s->stream>>>(s->d_mi, s->M, Msnp, s->n_case + s->n_ctrl, s->d_plane_derived, row, col,
                                                                                       (MmaRowF *)(row + Msnp), (MmaColF *)(col + Msnp), s->d_set_keys);
        else
            mma_side_kernel<false><<<(unsigned)((Msnp + 127) / 128), 128, 0, s->stream>>>(s->d_mi, s->M, Msnp, s->n_case + s->n_ctrl, s->d_plane_derived, row, col,
                                                                                        (MmaRowF *)(row + Msnp), (MmaColF *)(col + Msnp), nullptr);
        GW_LAUNCHED();
        s->mma_side_valid = true;
    }
    return GWASDEV_OK;
}

static uint64_t rect_pairs(uint64_t M, uint64_t i0, uint64_t i1, uint64_t j0, uint64_t j1) {   // pairs i<j, i in [i0,i1), j in [j0,j1), < M
    i1 = std::min(i1, M); j1 = std::min(j1, M);
    if (i1 <= i0 || j1 <= j0) return 0;
    if (i1 <= j0) return (i1 - i0) * (j1 - j0);     // rectangle entirely above the diagonal
    uint64_t n = 0;
    for (uint64_t i = i0; i < i1; ++i) { const uint64_t lo = std::max(j0, i + 1); if (j1 > lo) n += j1 - lo; }
    return n;
}

// Pairs the tensor-core engine covers for this shard: pairs i<j of the tiles t with t % n_shards == shard whose
// two 64-SNP blocks are free of missing calls (flags == nullptr: no block has any).
uint64_t gwasdev_internal_mma_shard_pairs(const gwasdev_store *s, uint32_t shard, uint32_t n_shards, const uint8_t *flags,
                                          uint64_t *tiles_out) {
    const uint64_t M = s->M;
    const uint32_t TB = (uint32_t)((M + MMA_BLK - 1) / MMA_BLK);
    const uint32_t BAND = schedule_band((uint64_t)MMA_N * 32 * s->Wr);          // = s->mm_band once the operands exist
    const uint32_t n_bands = (TB + BAND - 1) / BAND;
    uint64_t pairs = 0, tiles = 0, t = 0;
    for (uint32_t b = 0; b < n_bands; ++b) {
        const uint32_t na = band_height(TB, b, BAND);
        for (uint32_t J = BAND * b; J < TB; ++J) {
            const uint32_t h = column_height(na, J - BAND * b);
            const uint64_t j0 = (uint64_t)J * MMA_BLK, j1 = std::min<uint64_t>(j0 + MMA_BLK, M);
            // tiles t .. t+h-1 are A-blocks I2 = 8b + ii of this column; those of the shard: tile_in_shard(t + ii)
            const uint64_t cnt = shard_tiles_before(t + h, shard, n_shards) - shard_tiles_before(t, shard, n_shards);
            const bool simple = !flags && (uint64_t)(BAND * b + h) * MMA_BLK <= j0;     // full rectangles left of the B-block
            if (cnt == 0) { t += h; continue; }
            if (simple) { tiles += cnt; pairs += cnt * MMA_BLK * (j1 - j0); }
            else {
                for (uint32_t ii = 0; ii < h; ++ii) {
                    if (!tile_in_shard(t + ii, shard, n_shards)) continue;
                    const uint64_t I2 = BAND * b + ii;
                    ++tiles;
                    if (!flags) pairs += rect_pairs(M, I2 * MMA_BLK, (I2 + 1) * MMA_BLK, j0, j0 + MMA_BLK);
                    else
                        for (int sa = 0; sa < 2; ++sa)
                            for (int sb = 0; sb < 2; ++sb) {
                                const uint64_t ia = 2 * I2 + sa, jb = 2ull * J + sb;
                                if (ia * TILE < M && jb * TILE < M && !flags[ia] && !flags[jb])
                                    pairs += rect_pairs(M, ia * TILE, (ia + 1) * TILE, jb * TILE, (jb + 1) * TILE);
                            }
                }
            }
            t += h;
        }
    }
    if (tiles_out) *tiles_out = tiles;
    return pairs;
}

template <bool SETS = false>
static int launch_mma(gwasdev_store *s, MmaParams &p, uint64_t my_tiles) {
#ifdef GWASDEV_SWEEP
    const bool prof = getenv("GWASDEV_MMA_PROF") != nullptr && !p.dump;
#else
    const bool prof = false;
#endif
    unsigned long long *d_prof = nullptr;
    if (prof) {   // 8 timers per CTA; launch_cta_pairs runs at most one CTA per SM
        int sms = 0;
        GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
        GW_CUDA(cudaMalloc(&d_prof, (size_t)sms * 8 * sizeof(unsigned long long)));
        GW_CUDA(cudaMemsetAsync(d_prof, 0, (size_t)sms * 8 * sizeof(unsigned long long), s->stream));
    }
    p.prof = d_prof;
    unsigned pairs = 0;
    { const int rc = launch_cta_pairs(s, pair_screen_mma_kernel<SETS>, MmaPipe::SMEM, my_tiles, p, &pairs, nullptr,
                                         *(const CUtensorMap *)s->tmap_mm);
      if (rc != GWASDEV_OK) return rc; }
    if (prof) {
        std::vector<unsigned long long> h((size_t)2 * pairs * 8);
        GW_CUDA(cudaMemcpyAsync(h.data(), d_prof, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
        GW_CUDA(cudaStreamSynchronize(s->stream));
        cudaFree(d_prof);
        double a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (unsigned c = 0; c < 2 * pairs; ++c) for (int k = 0; k < 8; ++k) a[k] += (double)h[(size_t)c * 8 + k];
        const double nl = pairs, nc = 2.0 * pairs, tiles = a[6] / nl;
        fprintf(stderr, "[gwasdev mma prof] per tile (SM clocks): mma thread %.0f (waits tempty %.0f, full %.0f) | epilogue warp0 %.0f warp15 %.0f "
                        "(waits tfull %.0f) | producer waits empty %.0f | tiles per pair %.0f\n",
                a[0] / nl / tiles, a[1] / nl / tiles, a[2] / nl / tiles, a[3] / nc / tiles, a[7] / nc / tiles, a[4] / nc / tiles, a[5] / nc / tiles, tiles);
    }
    return GWASDEV_OK;
}

static void fill_params(gwasdev_store *s, MmaParams &p, uint32_t shard, uint32_t n_shards) {
    p.TB = (uint32_t)((s->M + MMA_BLK - 1) / MMA_BLK);
    p.NKB = s->mm_kbytes / MMA_KB; p.band = s->mm_band; p.n_bands = (p.TB + p.band - 1) / p.band; p.M = s->M;
    p.shard = shard; p.n_shards = n_shards;
    const uint64_t Msnp = (s->M + MMA_BLK - 1) / MMA_BLK * MMA_BLK;
    p.row = (const MmaRow *)s->d_mma_row; p.col = (const MmaCol *)s->d_mma_col; p.tile_missing = s->d_tile_missing;
    p.rowf = (const MmaRowF *)(p.row + Msnp); p.colf = (const MmaColF *)(p.col + Msnp);
    p.N = (float)(s->n_case + s->n_ctrl);
    p.qc = s->mma_qc; p.q0 = s->mma_q0;
    p.sink = CandSink{};
    p.dump = nullptr; p.dump_tile = 0; p.dump_rank = 0; p.prof = nullptr;
    p.set_tiles = nullptr; p.set_c1 = p.set_a1 = 0;
}

// ---- four-plane engine: host side ---------------------------------------------------------------------
static uint32_t m4_blocks(const gwasdev_store *s) { return (uint32_t)((s->M + M4_BLK - 1) / M4_BLK); }

// bytes per row of the four-plane operand matrix in `mode` (see ensure_mma4_inputs) and the band height that follows from it
static uint32_t m4_kbytes(const gwasdev_store *s, int mode) {
    return mode == 2 ? round_up(s->n_case, MMA_KB) + round_up(s->n_ctrl, MMA_KB) : 32 * s->Wr;
}
static uint32_t m4_band(const gwasdev_store *s, int mode) { return schedule_band((uint64_t)MMA_N * m4_kbytes(s, mode)); }

static int ensure_mma4_inputs(gwasdev_store *s, int mode) {
    if (s->mm4_built && s->mm4_mode == mode) return GWASDEV_OK;
    const uint32_t TB = m4_blocks(s);
    const uint32_t case_bytes = round_up(s->n_case, MMA_KB), ctrl_bytes = round_up(s->n_ctrl, MMA_KB);
    // modes 0 and 1: bytes in raw sample order, straight from the raw rows and the class masks. Mode 2 sends the sample blocks of
    // the case range of K to one accumulator and the control range to the other, so its rows are class-pure: from the compacted rows.
    s->mm4_kbytes = m4_kbytes(s, mode);
    s->mm4_rows = (uint64_t)M4_PLANES * TB * M4_BLK;
    const size_t bytes = (size_t)s->mm4_rows * s->mm4_kbytes;
    GW_CUDA(reserve_raw(s->d_mm4, s->cap_mm4, bytes));
    GW_CUDA(cudaMemsetAsync(s->d_mm4, 0, bytes, s->stream));
    if (mode == 2) {
        { const int rc = gwasdev_internal_ensure_compacted(s); if (rc != GWASDEV_OK) return rc; }
        const uint32_t K = s->Kc + s->Kt;
        const uint64_t work = s->M * K;
        expand_mma4_kernel<2><<<(unsigned)((work + 255) / 256), 256, 0, s->stream>>>(s->d_sel, 2 * (s->Wc + s->Wt), s->Wc, s->Kc, s->Kt, s->n_case, s->n_ctrl,
                                                                                    case_bytes, s->mm4_kbytes, s->M, s->d_mm4);
    } else {
        const uint64_t work = s->M * s->Wr;
        const unsigned blocks = (unsigned)((work + 255) / 256);
        if (mode == 1) expand_raw_kernel<1><<<blocks, 256, 0, s->stream>>>(s->d_raw, s->Wr, s->d_case_sel_mask, s->d_ctrl_sel_mask, s->mm4_kbytes, s->M, nullptr, s->d_mm4);
        else expand_raw_kernel<0><<<blocks, 256, 0, s->stream>>>(s->d_raw, s->Wr, s->d_case_sel_mask, s->d_ctrl_sel_mask, s->mm4_kbytes, s->M, nullptr, s->d_mm4);
    }
    GW_LAUNCHED();
    if (!s->tmap_mm4 && posix_memalign(&s->tmap_mm4, 64, 2 * sizeof(CUtensorMap)) != 0) { s->tmap_mm4 = nullptr; set_error("out of host memory"); return GWASDEV_ENOMEM; }
    { const int rc = encode_operand_map(s->d_mm4, s->mm4_rows, s->mm4_kbytes, 2 * MMA_A_SNPS, (CUtensorMap *)s->tmap_mm4); if (rc != GWASDEV_OK) return rc; }
    {   // the B side of the missing-call layouts: planes 0..2 of 32 SNPs as one dense 96-row box
        encode_tiled_fn encode = nullptr;
        { const int rc = get_encode_tiled(&encode); if (rc != GWASDEV_OK) return rc; }
        cuuint64_t gdim3[3] = {s->mm4_kbytes, (cuuint64_t)M4_PLANES, s->mm4_rows / M4_PLANES};
        cuuint64_t gstride3[2] = {s->mm4_kbytes, (cuuint64_t)M4_PLANES * s->mm4_kbytes};
        cuuint32_t box3[3] = {(cuuint32_t)MMA_KB, 3, (cuuint32_t)(MMA_B_SNPS / 4)};
        cuuint32_t estr3[3] = {1, 1, 1};
        const CUresult r = encode((CUtensorMap *)s->tmap_mm4 + 1, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, s->d_mm4, gdim3, gstride3, box3, estr3, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (three-plane B box) failed (%d)", (int)r); return GWASDEV_ENODEVICE; }
    }
    s->mm4_band = m4_band(s, mode);
    s->mm4_tiles = schedule_tiles(TB, s->mm4_band);
    s->mm4_built = true;
    s->mm4_mode = mode;
    return GWASDEV_OK;
}

// pairs (i < j < M) and tiles of the shard among the tiles with missing calls, in the four-plane schedule
// mode 0: tiles with missing calls; 1: tiles without; 2: all tiles
uint64_t gwasdev_internal_mma4_shard_pairs(gwasdev_store *s, uint32_t shard, uint32_t n_shards, const uint8_t *flags, int mode, uint64_t *tiles_out) {
    const uint32_t TB = m4_blocks(s), BAND = m4_band(s, mode), n_bands = (TB + BAND - 1) / BAND;
    const uint64_t M = s->M;
    uint64_t pairs = 0, tiles = 0, t = 0;
    for (uint32_t b = 0; b < n_bands; ++b) {
        const uint32_t na = band_height(TB, b, BAND);
        for (uint32_t J = BAND * b; J < TB; ++J) {
            const uint32_t h = column_height(na, J - BAND * b);
            for (uint32_t ii = 0; ii < h; ++ii, ++t) {
                const uint32_t I2 = BAND * b + ii;
                if (!tile_in_shard(t, shard, n_shards) || (mode != 2 && ((flags[I2] | flags[J]) != 0) == (mode == 1))) continue;
                ++tiles;
                if (I2 < J && (uint64_t)(J + 1) * M4_BLK <= M) pairs += (uint64_t)M4_BLK * M4_BLK;     // full off-diagonal block
                else pairs += rect_pairs(M, (uint64_t)I2 * M4_BLK, (uint64_t)(I2 + 1) * M4_BLK, (uint64_t)J * M4_BLK, (uint64_t)(J + 1) * M4_BLK);
            }
        }
    }
    if (tiles_out) *tiles_out = tiles;
    return pairs;
}

// ---- set screens: tile lists --------------------------------------------------------------------------
// wanted pairs (set_pair_wanted) of a sub-table of M SNPs inside [i0, i1) x [j0, j1)
static uint64_t set_rect_pairs(uint64_t M, uint64_t c1, uint64_t a1, uint64_t i0, uint64_t i1, uint64_t j0, uint64_t j1) {
    return rect_pairs(M, i0, std::min(i1, c1), j0, j1) + rect_pairs(M, std::max(i0, c1), std::min(i1, a1), std::max(j0, a1), j1);
}

// The set screen's tiles for blocks of `blk` SNPs and bands of `band` A-blocks: the tiles of the whole-table schedule of the
// sub-table that hold a wanted pair, in schedule order, so that the tile feed keeps its L2 banding. Shards take turns in chunks
// of SHARD_CHUNK list positions; the shard's tiles go to `out`. Bands that start at or beyond a1 hold no wanted pair.
static void set_tile_list(uint64_t M, uint64_t c1, uint64_t a1, uint32_t blk, uint32_t band, uint32_t shard, uint32_t n_shards,
                          std::vector<uint2> &out) {
    out.clear();
    const uint32_t TB = (uint32_t)((M + blk - 1) / blk), n_bands = (TB + band - 1) / band;
    uint64_t u = 0;
    for (uint32_t b = 0; b < n_bands && (uint64_t)band * b * blk < a1; ++b) {
        const uint32_t na = band_height(TB, b, band);
        for (uint32_t J = band * b; J < TB; ++J)
            for (uint32_t ii = 0; ii < column_height(na, J - band * b); ++ii) {
                const uint64_t I2 = (uint64_t)band * b + ii;
                if (set_rect_pairs(M, c1, a1, I2 * blk, (I2 + 1) * blk, (uint64_t)J * blk, (uint64_t)(J + 1) * blk) == 0) continue;
                if (tile_in_shard(u++, shard, n_shards)) out.push_back(make_uint2((uint32_t)I2, J));
            }
    }
}

// The shard's tile list of the set screen for the two-plane kernel (mode -1) or the four-plane kernel in `mode` (0, 1, 2;
// see gwasdev_internal_mma4_shard_pairs), and the wanted pairs the kernel computes in it: those of the 64-SNP blocks without
// missing calls (two-plane; flags == nullptr: no block has any), of the tiles with (mode 0) or without (mode 1) missing calls,
// or of every tile (mode 2). *tiles_out = tiles the kernel computes.
uint64_t gwasdev_internal_set_shard_pairs(gwasdev_store *s, uint64_t c1, uint64_t a1, uint32_t shard, uint32_t n_shards, const uint8_t *flags,
                                          int mode, std::vector<uint2> &list, uint64_t *tiles_out) {
    const uint64_t M = s->M;
    uint64_t pairs = 0, tiles = 0;
    if (mode < 0) {
        set_tile_list(M, c1, a1, MMA_BLK, schedule_band((uint64_t)MMA_N * 32 * s->Wr), shard, n_shards, list);
        for (const uint2 &t : list) {
            ++tiles;
            for (int sa = 0; sa < 2; ++sa)
                for (int sb = 0; sb < 2; ++sb) {
                    const uint64_t ia = 2ull * t.x + sa, jb = 2ull * t.y + sb;
                    if (ia * TILE < M && jb * TILE < M && (!flags || (!flags[ia] && !flags[jb])))
                        pairs += set_rect_pairs(M, c1, a1, ia * TILE, (ia + 1) * TILE, jb * TILE, (jb + 1) * TILE);
                }
        }
    } else {
        set_tile_list(M, c1, a1, M4_BLK, m4_band(s, mode), shard, n_shards, list);
        for (const uint2 &t : list) {
            if (mode != 2 && ((flags[t.x] | flags[t.y]) != 0) == (mode == 1)) continue;
            ++tiles;
            pairs += set_rect_pairs(M, c1, a1, (uint64_t)t.x * M4_BLK, (uint64_t)(t.x + 1) * M4_BLK, (uint64_t)t.y * M4_BLK, (uint64_t)(t.y + 1) * M4_BLK);
        }
    }
    if (tiles_out) *tiles_out = tiles;
    return pairs;
}

// Launches the four-plane tensor-core screen over this shard's tiles with missing calls. thr carries the fp32 margin.
// set != nullptr: the set screen over the shard's list instead (shard / n_shards are then part of the list).
int gwasdev_internal_screen_mma4(gwasdev_store *s, const CandSink &sink, uint32_t shard, uint32_t n_shards, int mode, const SetLaunch *set) {
    int rc = ensure_mma4_inputs(s, mode);
    if (rc != GWASDEV_OK) return rc;
    Mma4Params p;
    p.TB = m4_blocks(s); p.NKB = s->mm4_kbytes / MMA_KB; p.band = s->mm4_band; p.n_bands = (p.TB + p.band - 1) / p.band; p.M = s->M; p.n_tiles = s->mm4_tiles;
    p.case_kb = round_up(s->n_case, MMA_KB) / MMA_KB;
    p.shard = shard; p.n_shards = n_shards; p.side = s->d_side; p.tile_missing = s->d_tile_missing;
    const uint32_t n_ind = s->n_case + s->n_ctrl;
    p.N = (float)n_ind; p.lnN = (float)std::log((double)n_ind);
    p.sink = sink;
    p.set_tiles = nullptr; p.set_c1 = p.set_a1 = 0; p.set_keys = s->d_set_keys;
    if (set) { p.n_tiles = set->n_tiles; p.shard = 0; p.n_shards = 1; p.set_tiles = set->tiles; p.set_c1 = set->c1; p.set_a1 = set->a1; }
    const uint64_t my_tiles = shard_tiles_before(p.n_tiles, p.shard, p.n_shards);
    if (my_tiles == 0) return GWASDEV_OK;
    const CUtensorMap *maps = (const CUtensorMap *)s->tmap_mm4;
#define SCREEN4(MODE_, SETS_) launch_cta_pairs(s, pair_screen_mma4_kernel<MODE_, SETS_>, M4Pipe<MODE_>::SMEM, my_tiles, p, nullptr, nullptr, maps[0], maps[1])
    if (set) return mode == 1 ? SCREEN4(1, true) : mode == 2 ? SCREEN4(2, true) : SCREEN4(0, true);
    return mode == 1 ? SCREEN4(1, false) : mode == 2 ? SCREEN4(2, false) : SCREEN4(0, false);
#undef SCREEN4
}

// operands and records of the two kernels ahead of a set screen's timed region
int gwasdev_internal_ensure_mma(gwasdev_store *s) { return ensure_mma_inputs(s); }
int gwasdev_internal_ensure_mma4(gwasdev_store *s, int mode) { return ensure_mma4_inputs(s, mode); }

// Launches the tensor-core screen for this shard's clean tiles. thr already carries the fp32 margin.
// set != nullptr: the set screen over the shard's list instead.
int gwasdev_internal_screen_mma(gwasdev_store *s, const CandSink &sink, uint32_t shard, uint32_t n_shards, const SetLaunch *set) {
    const bool trace = s->opt[GWASDEV_OPT_TRACE] != 0;
    if (trace) cudaEventRecord(s->ev2, s->stream);
    int rc = ensure_mma_inputs(s);
    if (rc != GWASDEV_OK) return rc;
    if (trace) {
        cudaEventRecord(s->ev3, s->stream);
        cudaStreamSynchronize(s->stream);
        float ms = 0.f; cudaEventElapsedTime(&ms, s->ev2, s->ev3);
        fprintf(stderr, "[gwasdev trace] tensor-core operands + per-SNP records %.3f ms\n", ms);
    }
    MmaParams p;
    if (set) {
        fill_params(s, p, 0, 1);
        p.n_tiles = set->n_tiles; p.sink = sink;
        p.set_tiles = set->tiles; p.set_c1 = set->c1; p.set_a1 = set->a1;
        return set->n_tiles == 0 ? GWASDEV_OK : launch_mma<true>(s, p, set->n_tiles);
    }
    fill_params(s, p, shard, n_shards);
    const uint64_t n_tiles = s->mm_tiles;
    p.n_tiles = n_tiles;
    p.sink = sink;
    const uint64_t my_tiles = shard_tiles_before(n_tiles, shard, n_shards);
    if (my_tiles == 0) return GWASDEV_OK;
    return launch_mma(s, p, my_tiles);
}

extern "C" {

// Host arithmetic only (no device): the tile pairs of the screen's schedule that `shard` of `n_shards` owns, in schedule
// order, and the pairs i < j < n_snps they cover. engine 2: tensor-core schedule (128-SNP blocks, bands of 8 to 16 A-blocks
// depending on the row length for n_samples samples, column-major inside a band, shards own alternating runs of 64 consecutive tiles); engine 1: AND+POPC schedule (64-SNP
// blocks, row-major upper triangle, single tiles dealt round-robin).
int gwasdev_shard_schedule(uint64_t n_snps, uint64_t n_samples, int engine, uint32_t shard, uint32_t n_shards, uint32_t *tiles, uint64_t capacity,
                           uint64_t *n_tiles, uint64_t *n_pairs) {
    GW_REQUIRE(n_snps >= 1 && n_samples >= 1 && n_shards >= 1 && shard < n_shards && (engine == 1 || engine == 2), "gwasdev_shard_schedule: bad argument");
    uint64_t cnt = 0, pairs = 0;
    auto take = [&](uint32_t I, uint32_t J, uint32_t blk) {
        if (tiles && cnt < capacity) { tiles[2 * cnt] = I; tiles[2 * cnt + 1] = J; }
        ++cnt;
        pairs += rect_pairs(n_snps, (uint64_t)I * blk, (uint64_t)(I + 1) * blk, (uint64_t)J * blk, (uint64_t)(J + 1) * blk);
    };
    if (engine == 2) {
        const uint32_t BAND = schedule_band((uint64_t)MMA_N * round_up((uint32_t)n_samples, MMA_KB));   // rows are one byte per sample, padded to 128
        const uint32_t TB = (uint32_t)((n_snps + MMA_BLK - 1) / MMA_BLK), n_bands = (TB + BAND - 1) / BAND;
        uint64_t t = 0;
        for (uint32_t b = 0; b < n_bands; ++b) {
            const uint32_t na = band_height(TB, b, BAND);
            for (uint32_t J = BAND * b; J < TB; ++J)
                for (uint32_t ii = 0; ii < column_height(na, J - BAND * b); ++ii, ++t)
                    if (tile_in_shard(t, shard, n_shards)) take(BAND * b + ii, J, MMA_BLK);
        }
    } else {
        const uint32_t T = (uint32_t)((n_snps + TILE - 1) / TILE);
        uint64_t t = 0;
        for (uint32_t I = 0; I < T; ++I)
            for (uint32_t J = I; J < T; ++J, ++t)
                if (t % n_shards == shard) take(I, J, TILE);
    }
    if (n_tiles) *n_tiles = cnt;
    if (n_pairs) *n_pairs = pairs;
    return GWASDEV_OK;
}

int gwasdev_set_schedule(uint64_t n_snps, uint64_t n_samples, uint32_t tile_snps, const uint32_t *set_a, uint64_t n_a, const uint32_t *set_b,
                         uint64_t n_b, uint32_t shard, uint32_t n_shards, uint32_t *tiles, uint64_t capacity, uint64_t *n_tiles, uint64_t *n_pairs) {
    GW_REQUIRE(n_samples >= 1 && n_shards >= 1 && shard < n_shards && (tile_snps == MMA_BLK || tile_snps == M4_BLK),
               "gwasdev_set_schedule: bad argument (tile_snps %u: 128 two-plane, 64 four-plane)", tile_snps);
    std::vector<uint32_t> map;
    uint64_t c1 = 0, a1 = 0;
    int rc = gwasdev_internal_set_rows(n_snps, set_a, n_a, set_b, n_b, "gwasdev_set_schedule", map, &c1, &a1);
    if (rc != GWASDEV_OK) return rc;
    std::vector<uint2> list;
    uint64_t pairs = 0;
    if (map.size() >= 2) {
        // the band of the screen's operand rows: one byte per raw sample position (32 * Wr, gwasdev_create's geometry)
        const uint32_t row_bytes = 32 * round_up(plane_blocks((uint32_t)n_samples) / 2, 4);
        set_tile_list(map.size(), c1, a1, tile_snps, schedule_band((uint64_t)MMA_N * row_bytes), shard, n_shards, list);
        for (const uint2 &t : list)
            pairs += set_rect_pairs(map.size(), c1, a1, (uint64_t)t.x * tile_snps, (uint64_t)(t.x + 1) * tile_snps, (uint64_t)t.y * tile_snps,
                                    (uint64_t)(t.y + 1) * tile_snps);
    }
    for (uint64_t k = 0; tiles && k < std::min<uint64_t>(capacity, list.size()); ++k) { tiles[2 * k] = list[k].x; tiles[2 * k + 1] = list[k].y; }
    if (n_tiles) *n_tiles = list.size();
    if (n_pairs) *n_pairs = pairs;
    return GWASDEV_OK;
}

int gwasdev_set_pair_engine(gwasdev_store *s, int engine) {
    GW_REQUIRE(s != nullptr, "gwasdev_set_pair_engine: NULL store");
    GW_REQUIRE(engine >= 0 && engine <= 2, "gwasdev_set_pair_engine: engine %d (0 auto, 1 popcount, 2 tensor core)", engine);
    s->pair_engine = engine;
    return GWASDEV_OK;
}

// int8 tensor-core throughput of this device with the screen kernel's instruction shape (i8_peak_kernel above):
// *tops_burst = best launch, *tops_sustained = mean over ~50 ms of back-to-back launches (the SM clock drops under the
// tensor cores' power draw), in 1e12 int8 operations per second (2 per multiply-accumulate, as vendors quote it).
int gwasdev_i8_peak(int device, double *tops_burst, double *tops_sustained) {
    GW_REQUIRE(tops_burst != nullptr, "gwasdev_i8_peak: NULL argument");
    if (gwasdev_device_count() <= device || device < 0) { set_error("gwasdev_i8_peak: no CUDA device %d", device); return GWASDEV_ENODEVICE; }
    GW_CUDA(cudaSetDevice(device));
    int sms = 0;
    GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    const size_t smem = 1024 + KB_BYTES + 64;
    GW_CUDA(cudaFuncSetAttribute(i8_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned pairs = (unsigned)std::max(1, sms / 2);
    const uint32_t kblocks = 16384;                                   // 65 536 MMAs per CTA pair: ~5 ms per launch
    const double ops = 2.0 * (double)MMA_M * MMA_N * MMA_KB * (double)kblocks * pairs;
    cudaEvent_t a, b;
    GW_CUDA(cudaEventCreate(&a)); GW_CUDA(cudaEventCreate(&b));
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {                               // warm-up + burst
        GW_CUDA(cudaEventRecord(a));
        i8_peak_kernel<<<2 * pairs, 128, smem>>>(kblocks, 12345u + rep);
        GW_LAUNCHED();
        GW_CUDA(cudaEventRecord(b));
        GW_CUDA(cudaEventSynchronize(b));
        float ms = 0.f;
        GW_CUDA(cudaEventElapsedTime(&ms, a, b));
        if (rep > 0) best = std::max(best, ops / (ms * 1e-3) / 1e12);
    }
    const int reps = 10;
    GW_CUDA(cudaEventRecord(a));
    for (int rep = 0; rep < reps; ++rep) { i8_peak_kernel<<<2 * pairs, 128, smem>>>(kblocks, 777u + rep); GW_LAUNCHED(); }
    GW_CUDA(cudaEventRecord(b));
    GW_CUDA(cudaEventSynchronize(b));
    float ms = 0.f;
    GW_CUDA(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b);
    *tops_burst = best;
    if (tops_sustained) *tops_sustained = ops * reps / (ms * 1e-3) / 1e12;
    return GWASDEV_OK;
}

// Debug / parity probe: the raw corner counts the tensor-core engine accumulates for one tile pair
// (A-block I of 64 SNPs, B-block J of 128 SNPs): out[(a*128 + b)*8 + {0..3}] = case AA_BB, AA_bb, aa_BB, aa_bb,
// +4.. the same for controls.
int gwasdev_mma_tile_counts(gwasdev_store *s, uint32_t I, uint32_t J, uint32_t *out) {
    GW_REQUIRE(s && out, "gwasdev_mma_tile_counts: NULL argument");
    GW_REQUIRE(s->selected, "gwasdev_mma_tile_counts: call gwasdev_select_case_control first");
    GW_REQUIRE(gwasdev_internal_mma_eligible(s), "gwasdev_mma_tile_counts: class sizes outside the tensor-core engine's range");
    GW_CUDA(cudaSetDevice(s->device));
    int rc = gwasdev_internal_ensure_side(s);
    if (rc != GWASDEV_OK) return rc;
    // the probe reports the corners of the two homozygote planes: operands with the reference's planes for this call
    const long long planes_opt = s->opt[GWASDEV_OPT_CLASSIC_PLANES];
    struct Restore { gwasdev_store *s; long long v; ~Restore() { s->opt[GWASDEV_OPT_CLASSIC_PLANES] = v; if (!v) { s->mm_built = false; s->mma_side_valid = false; } } } restore{s, planes_opt};
    if (!planes_opt) { s->opt[GWASDEV_OPT_CLASSIC_PLANES] = 1; s->mm_built = false; s->mma_side_valid = false; }
    if ((rc = ensure_mma_inputs(s)) != GWASDEV_OK) return rc;
    MmaParams p;
    fill_params(s, p, 0, 1);
    GW_REQUIRE(I / 2 < p.TB && J < p.TB && I / 2 <= J, "gwasdev_mma_tile_counts: tile (%u, %u) is not in the schedule", I, J);
    // linear index of (I, J)
    const uint32_t BAND = p.band, I2 = I / 2, b = I2 / BAND, na = band_height(p.TB, b, BAND);
    uint64_t t = band_offset(p.TB, b, BAND);
    for (uint32_t c = 0; c < J - BAND * b; ++c) t += column_height(na, c);
    t += I2 - BAND * b;
    p.n_tiles = s->mm_tiles;
    const size_t bytes = (size_t)MMA_A_SNPS * MMA_B_SNPS * 8 * sizeof(uint32_t);
    GW_CUDA(reserve(s->sc_a, bytes));
    GW_CUDA(cudaMemsetAsync(s->sc_a.p, 0xff, bytes, s->stream));
    p.dump = (uint32_t *)s->sc_a.p; p.dump_tile = t; p.dump_rank = I & 1;
    if ((rc = launch_mma(s, p, 1)) != GWASDEV_OK) return rc;
    GW_CUDA(cudaMemcpyAsync(out, s->sc_a.p, bytes, cudaMemcpyDeviceToHost, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    return GWASDEV_OK;
}

int gwasdev_ksa_screen_mma_f32(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, float *stat) {
    GW_REQUIRE(s && pi && pj && stat, "gwasdev_ksa_screen_mma_f32: NULL argument");
    GW_REQUIRE(s->selected, "gwasdev_ksa_screen_mma_f32: call gwasdev_select_case_control first");
    GW_REQUIRE(gwasdev_internal_mma_eligible(s), "gwasdev_ksa_screen_mma_f32: class sizes outside the tensor-core engine's range");
    for (uint64_t q = 0; q < n; ++q) GW_REQUIRE(pi[q] < s->M && pj[q] < s->M, "gwasdev_ksa_screen_mma_f32: pair outside the table");
    if (n == 0) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    int rc = gwasdev_internal_ensure_side(s);
    if (rc != GWASDEV_OK) return rc;
    if ((rc = ensure_mma_inputs(s)) != GWASDEV_OK) return rc;
    const uint64_t Msnp = (s->M + MMA_BLK - 1) / MMA_BLK * MMA_BLK;
    GW_CUDA(reserve(s->sc_pi, n * 4)); GW_CUDA(reserve(s->sc_pj, n * 4)); GW_CUDA(reserve(s->sc_a, n * 8));
    GW_CUDA(cudaMemcpyAsync(s->sc_pi.p, pi, n * 4, cudaMemcpyHostToDevice, s->stream));
    GW_CUDA(cudaMemcpyAsync(s->sc_pj.p, pj, n * 4, cudaMemcpyHostToDevice, s->stream));
    screen_probe_mma_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s->stream>>>(
        pair_src(s), s->d_plane_derived, (const MmaRow *)s->d_mma_row, (const MmaCol *)s->d_mma_col,
        (const MmaRowF *)((const MmaRow *)s->d_mma_row + Msnp), (const MmaColF *)((const MmaCol *)s->d_mma_col + Msnp),
        (const uint32_t *)s->sc_pi.p, (const uint32_t *)s->sc_pj.p, n, (float)(s->n_case + s->n_ctrl), s->mma_qc, s->mma_q0,
        (float *)s->sc_a.p);
    GW_LAUNCHED();
    GW_CUDA(cudaMemcpyAsync(stat, s->sc_a.p, n * 8, cudaMemcpyDeviceToHost, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    return GWASDEV_OK;
}

}  // extern "C"
