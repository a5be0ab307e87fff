// Device-resident genotype store: creation, row upload/download, synthetic cohort generation,
// case/control compaction (K0) and the SNP-tiled pairwise layout.
//
// Replaces CompressedGenotypeTable5's host table (genetics/genotype/compressed_genotype_table5.cpp:
// initialize :34-153, addGenotypeRow :277-365, operator() :400-432, selectCaseControl :443-575).
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace gwasdev {

static thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

// ---- kernels -------------------------------------------------------------------------------------

// reference row [hdr][plane1: P][plane2: P] (16-bit blocks, odd stride) -> hdr[], raw[M][2][Wr] words
// Bits at or beyond sample N (the reference's row padding) are cleared: every kernel may then take "bit set" as "sample
// has the genotype" without a valid-sample mask.
__global__ void unpack_rows_kernel(const uint16_t *__restrict__ rows, uint32_t P, uint32_t Wr, uint32_t N,
                                   uint16_t *__restrict__ hdr, uint32_t *__restrict__ raw,
                                   uint64_t first_row) {
    const uint64_t r = blockIdx.x;
    const uint16_t *src = rows + r * (2ull * P + 1);
    uint32_t *dst = raw + (first_row + r) * 2ull * Wr;
    if (threadIdx.x == 0) hdr[first_row + r] = src[0];
    for (uint32_t w = threadIdx.x; w < 2 * Wr; w += blockDim.x) {
        const uint32_t plane = w / Wr, k = w % Wr;
        uint32_t v = 0;
        if (2 * k < P) v = src[1 + plane * P + 2 * k];
        if (2 * k + 1 < P) v |= (uint32_t)src[1 + plane * P + 2 * k + 1] << 16;
        if (32 * k + 32 > N) v &= 32 * k >= N ? 0u : (0xffffffffu >> (32 * k + 32 - N));
        dst[w] = v;
    }
}

__global__ void pack_rows_kernel(const uint16_t *__restrict__ hdr, const uint32_t *__restrict__ raw,
                                 uint32_t P, uint32_t Wr, uint16_t *__restrict__ rows, uint64_t first_row) {
    const uint64_t r = blockIdx.x;
    uint16_t *dst = rows + r * (2ull * P + 1);
    const uint32_t *src = raw + (first_row + r) * 2ull * Wr;
    if (threadIdx.x == 0) dst[0] = hdr[first_row + r];
    for (uint32_t b = threadIdx.x; b < 2 * P; b += blockDim.x) {
        const uint32_t plane = b / P, k = b % P;
        dst[1 + b] = (uint16_t)(src[plane * Wr + (k >> 1)] >> ((k & 1) * 16));
    }
}

// K0: case/control compaction (selectCaseControl, compressed_genotype_table5.cpp:520-572) without the
// reference's bit-serial walk. The class mask is fixed for all SNPs, so everything that depends only on
// it is precomputed once on the host: per source word sw the member mask m[sw], the five "move" masks of
// a parallel-suffix bit compress (Hacker's Delight 7-4) and the exclusive rank R[sw] of its first
// member; per output word the first source word that feeds it. One thread then builds one output word
// of both planes with ~15 logic ops per source word instead of 32 single-bit gathers.
struct SelectTables {
    const uint32_t *m;      // [Wr]      member mask per source word
    const uint32_t *mv;     // [Wr][5]   compress move masks
    const uint32_t *rank;   // [Wr + 1]  members before source word sw
    const uint32_t *first;  // [Kout]    first source word contributing to output word o
    const uint32_t *mvl;    // [Wr][5]   move masks of the compress towards the most significant end
    uint32_t n_class, Kout;
};

__device__ __forceinline__ uint32_t compress_bits(uint32_t x, const uint32_t *mv) {
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const uint32_t t = x & mv[i];
        x = (x ^ t) | (t >> (1 << i));
    }
    return x;
}

// One thread per SOURCE word: both planes are compressed once per class and OR-ed into the output row, which is
// assembled in shared memory (a source word's members land in at most two consecutive output words) and then
// written out in the scan layout with full-width stores. SNPS rows per block iteration amortise the two barriers.
template <bool TABLES_IN_SMEM, int SNPS>
__global__ void __launch_bounds__(256)
select_kernel(const uint32_t *__restrict__ raw, uint32_t Wr, SelectTables ca, SelectTables co,
              uint32_t *__restrict__ sel, uint32_t sel_stride, uint32_t Wc, uint32_t Wt, uint64_t M) {
    extern __shared__ uint32_t tab[];   // [SNPS][sel_stride] output rows, then per class: m[Wr], mv[5*Wr], rank[Wr+1]
    const uint32_t per = 7 * Wr + 1;
    uint32_t *rows = tab, *tables = tab + SNPS * sel_stride;
    if (TABLES_IN_SMEM) {
        for (uint32_t q = threadIdx.x; q < 2 * per; q += blockDim.x) tables[q] = q < per ? ca.m[q] : co.m[q - per];
    }
    for (uint32_t q = threadIdx.x; q < SNPS * sel_stride; q += blockDim.x) rows[q] = 0;
    __syncthreads();
    const uint32_t *tm_ca = TABLES_IN_SMEM ? tables : ca.m, *tm_co = TABLES_IN_SMEM ? tables + per : co.m;
    for (uint64_t snp0 = (uint64_t)blockIdx.x * SNPS; snp0 < M; snp0 += (uint64_t)gridDim.x * SNPS) {
        const uint32_t n_here = (uint32_t)min((uint64_t)SNPS, M - snp0);
        for (uint32_t q = threadIdx.x; q < n_here * Wr; q += blockDim.x) {
            const uint32_t r = q / Wr, sw = q - r * Wr;
            const uint32_t *p1 = raw + (snp0 + r) * 2ull * Wr;
            const uint32_t w1 = p1[sw], w2 = p1[Wr + sw];
            uint32_t *row = rows + r * sel_stride;
#pragma unroll
            for (int cls = 0; cls < 2; ++cls) {
                const uint32_t *tm = cls ? tm_co : tm_ca;
                const uint32_t m = tm[sw];
                if (m == 0) continue;
                const uint32_t *mv = tm + Wr + 5 * sw;
                const uint32_t x = compress_bits(w1 & m, mv), y = compress_bits(w2 & m, mv);
                const uint32_t pos = tm[6 * Wr + sw], o = pos >> 5, sh = pos & 31, off = cls ? 2 * Wc : 0;
                if (x) {
                    atomicOr(&row[sel_word(off, 0, o)], x << sh);
                    if (sh && (x >> (32 - sh))) atomicOr(&row[sel_word(off, 0, o + 1)], x >> (32 - sh));
                }
                if (y) {
                    atomicOr(&row[sel_word(off, 1, o)], y << sh);
                    if (sh && (y >> (32 - sh))) atomicOr(&row[sel_word(off, 1, o + 1)], y >> (32 - sh));
                }
            }
        }
        __syncthreads();
        // rows are contiguous in the scan layout: stream them out 16 bytes per thread and clear the buffer
        uint4 *dst = reinterpret_cast<uint4 *>(sel + snp0 * (uint64_t)sel_stride);
        uint4 *src = reinterpret_cast<uint4 *>(rows);
        for (uint32_t q = threadIdx.x; q < n_here * sel_stride / 4; q += blockDim.x) { dst[q] = src[q]; src[q] = make_uint4(0, 0, 0, 0); }
        __syncthreads();
    }
}

// K0, register form (cohorts up to 32 768 samples): thread t owns SOURCE COLUMN t -- the 32-sample word t of every row -- so
// that everything derived from the masks (member mask, the five compress move masks, where the compressed piece lands in
// the output row) is loaded once into registers and the per-row work is two loads, four bit-compresses and the ORs into
// the shared-memory row buffer. The table-driven kernel above spends ~260 instructions per source word on table reads,
// index arithmetic and divisions (ncu r1m); this one ~100.
struct ColumnTables { uint32_t m, mv[5], mul, down, lo, hi; };   // mul = 2^(landing bit); down = 32 - members; lo / hi: word offsets (plane 1) of the piece's two output words

// compress towards the MOST significant end. A stage moves the bits t = x & mv left by k = 2^i: x' = (x ^ t) | (t << k). The
// moved bits land on positions that are empty in x ^ t (a compress never collides) and t is a subset of x, so OR and XOR are
// plain add and subtract: x' = x - t + (t << k) = x + t * (2^k - 1) -- ONE multiply-add on the FMA pipe after ONE LOP3 on the
// ALU pipe, instead of two LOP3 plus a shift (the ALU pipe bounded the r1 form of this kernel: ncu r1q, ALU 68 % busy with
// 44 of its 58 instructions per source word in these stages).
__device__ __forceinline__ uint32_t compress_bits_left(uint32_t x, const uint32_t *mvl) {
#define GW_STAGE(I, MUL) { const uint32_t t = x & mvl[I]; asm("mad.lo.u32 %0, %1, " #MUL ", %0;" : "+r"(x) : "r"(t)); }
    GW_STAGE(0, 1) GW_STAGE(1, 3) GW_STAGE(2, 15) GW_STAGE(3, 255) GW_STAGE(4, 65535)
#undef GW_STAGE
    return x;
}

__device__ __forceinline__ ColumnTables load_column(const SelectTables &t, uint32_t Wr, uint32_t sw, uint32_t class_off, uint32_t W) {
    ColumnTables c;
    c.m = t.m[sw];
#pragma unroll
    for (int i = 0; i < 5; ++i) c.mv[i] = t.mvl[5 * sw + i];
    const uint32_t pos = t.rank[sw], o = pos >> 5;
    c.mul = 1u << (pos & 31);
    c.down = min(32u - (uint32_t)__popc(c.m), 31u);      // an empty column compresses to 0 whatever the shift
    c.lo = sel_word(class_off, 0, min(o, W - 1));
    c.hi = sel_word(class_off, 0, min(o + 1, W - 1));
    return c;
}

// The compressed piece sits in the top bits; one shift brings it down and one 32 x 32 -> 64 bit multiply by 2^(landing bit)
// (IMAD.WIDE, FMA pipe) yields both output words at once.
__device__ __forceinline__ void place_piece(uint32_t *row, const ColumnTables &c, uint32_t w1, uint32_t w2) {
    const uint32_t x = compress_bits_left(w1 & c.m, c.mv) >> c.down, y = compress_bits_left(w2 & c.m, c.mv) >> c.down;
    const unsigned long long px = (unsigned long long)x * c.mul, py = (unsigned long long)y * c.mul;
    atomicOr(&row[c.lo], (uint32_t)px);       // unconditional: a test per OR costs more issue slots than the zero ORs
    atomicOr(&row[c.lo + 4], (uint32_t)py);
    atomicOr(&row[c.hi], (uint32_t)(px >> 32));
    atomicOr(&row[c.hi + 4], (uint32_t)(py >> 32));
}

template <int SNPS>
__global__ void __launch_bounds__(1024)
select_columns_kernel(const uint32_t *__restrict__ raw, uint32_t Wr, SelectTables ca, SelectTables co,
                      uint32_t *__restrict__ sel, uint32_t sel_stride, uint32_t Wc, uint32_t Wt, uint64_t M) {
    extern __shared__ uint32_t rows[];   // [SNPS][sel_stride]
    const uint32_t sw = threadIdx.x;
    const bool live = sw < Wr;
    ColumnTables ta, to;
    if (live) { ta = load_column(ca, Wr, sw, 0, Wc); to = load_column(co, Wr, sw, 2 * Wc, Wt); }
    else { ta = {}; to = {}; }     // a dead lane loads zeros, compresses them to zero and ORs zero into word 0
    for (uint32_t q = threadIdx.x; q < SNPS * sel_stride; q += blockDim.x) rows[q] = 0;
    __syncthreads();
    for (uint64_t snp0 = (uint64_t)blockIdx.x * SNPS; snp0 < M; snp0 += (uint64_t)gridDim.x * SNPS) {
        const uint32_t n_here = (uint32_t)min((uint64_t)SNPS, M - snp0);
        uint32_t w1[SNPS], w2[SNPS];
#pragma unroll
        for (int r = 0; r < SNPS; ++r) {   // all loads of the iteration first
            w1[r] = w2[r] = 0;
            if (live && r < (int)n_here) {
                const uint32_t *p = raw + (snp0 + r) * 2ull * Wr + sw;
                w1[r] = __ldcs(p); w2[r] = __ldcs(p + Wr);
            }
        }
#pragma unroll
        for (int r = 0; r < SNPS; ++r) {
            uint32_t *row = rows + r * sel_stride;
            place_piece(row, ta, w1[r], w2[r]);
            place_piece(row, to, w1[r], w2[r]);
        }
        __syncthreads();
        uint4 *dst = reinterpret_cast<uint4 *>(sel + snp0 * (uint64_t)sel_stride);
        uint4 *src = reinterpret_cast<uint4 *>(rows);
        for (uint32_t q = threadIdx.x; q < n_here * sel_stride / 4; q += blockDim.x) { __stcs(dst + q, src[q]); src[q] = make_uint4(0, 0, 0, 0); }
        __syncthreads();
    }
}

// scan layout -> pairwise layout: one-hot planes aa = p1&~p2, ab = p2&~p1, bb = p1&p2, word-major
// [plane][k][snp] so that 64 consecutive SNPs of one word index are 256 contiguous bytes (one TMA row).
__global__ void build_pairwise_kernel(const uint32_t *__restrict__ sel, uint32_t sel_stride, uint32_t Wc,
                                      uint32_t Wt, uint32_t Kc, uint32_t Kt, uint64_t M, uint64_t Mpad,
                                      uint32_t *__restrict__ pw) {
    const uint64_t snp = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t k = blockIdx.y * blockDim.y + threadIdx.y, K = Kc + Kt;
    if (snp >= Mpad || k >= K) return;
    uint32_t p1 = 0, p2 = 0;
    if (snp < M) {
        const uint32_t *row = sel + snp * (uint64_t)sel_stride;
        if (k < Kc) { p1 = row[sel_word(0, 0, k)]; p2 = row[sel_word(0, 1, k)]; }
        else { p1 = row[sel_word(2 * Wc, 0, k - Kc)]; p2 = row[sel_word(2 * Wc, 1, k - Kc)]; }
    }
    const uint32_t bb = p1 & p2;
    pw[(0ull * K + k) * Mpad + snp] = p1 ^ bb;
    pw[(1ull * K + k) * Mpad + snp] = p2 ^ bb;
    pw[(2ull * K + k) * Mpad + snp] = bb;
}

// compacted rows back in the reference's 16-bit block layout [case p1][case p2][ctrl p1][ctrl p2]
// (layout-parity probe)
__global__ void export_selected_kernel(const uint32_t *__restrict__ sel, uint32_t sel_stride, uint32_t Wc,
                                       uint32_t Wt, uint32_t Pca, uint32_t Pco, uint16_t *__restrict__ out,
                                       uint64_t first_row) {
    const uint64_t r = blockIdx.x;
    const uint32_t *row = sel + (first_row + r) * (uint64_t)sel_stride;
    const uint32_t S = 2 * (Pca + Pco);
    uint16_t *dst = out + r * (uint64_t)S;
    for (uint32_t b = threadIdx.x; b < S; b += blockDim.x) {
        uint32_t off, plane, k, W;
        if (b < Pca) { off = 0; plane = 0; k = b; W = Wc; }
        else if (b < 2 * Pca) { off = 0; plane = 1; k = b - Pca; W = Wc; }
        else if (b < 2 * Pca + Pco) { off = 2 * Wc; plane = 0; k = b - 2 * Pca; W = Wt; }
        else { off = 2 * Wc; plane = 1; k = b - 2 * Pca - Pco; W = Wt; }
        const uint32_t word = (k >> 1) < W ? row[sel_word(off, plane, k >> 1)] : 0u;
        dst[b] = (uint16_t)(word >> ((k & 1) * 16));
    }
}

// Synthetic cohort, one thread per SNP (sequential selection sampling over the 2 * n_total allele slots).
// Distribution restated from data/simulate_data.cpp:160-207; see DESIGN.md "synthetic cohort". The store holds
// samples [s0, s0 + N) of the cohort; draws and first-seen labels are replayed from sample 0, so that sample blocks
// generated one at a time are the columns of the one whole-cohort table (labels included).
__global__ void simulate_kernel(uint64_t seed, const uint32_t *__restrict__ cum_bins, uint32_t N, uint32_t s0, uint32_t n_total,
                                uint32_t missing_q32, uint16_t *__restrict__ hdr,
                                uint32_t *__restrict__ raw, uint32_t Wr, uint64_t M) {
    const uint64_t snp = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (snp >= M) return;
    const uint64_t total = cum_bins[50];
    const uint64_t r = sim_hash(seed, snp, SIM_STREAM_BIN) % total;
    int bin = 50;
    for (int b = 0; b < 51; ++b)
        if (r < cum_bins[b]) { bin = b; break; }
    const uint64_t frac = sim_hash(seed, snp, SIM_STREAM_FREQ) % 1000;
    const uint64_t slots = 2ull * n_total;
    const uint64_t want = ((1000ull * bin + frac) * slots) / 100000ull;   // floor(p * 2N)
    uint64_t chosen = 0;
    Labeler lab;
    lab.reset();
    uint32_t *p1 = raw + snp * 2ull * Wr, *p2 = p1 + Wr;
    uint32_t a = 0, b = 0, w = 0;
    for (uint32_t s = 0; s < s0 + N; ++s) {
        int minor = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint64_t slot = 2ull * s + h, left = slots - slot;
            const uint64_t u = sim_hash(seed, snp, slot) >> 32;
            if (((u * left) >> 32) < want - chosen) { ++minor; ++chosen; }
        }
        bool missing = false;
        if (missing_q32)
            missing = (uint32_t)(sim_hash(seed, snp, SIM_STREAM_MISS | s) >> 32) < missing_q32;
        if (!missing) {
            const int enc = minor == 0 ? 0 : (minor == 1 ? 1 : 5);   // "AA", "AC", "CC"
            const int c = lab.code(enc);
            if (s >= s0) {
                const uint32_t t = (s - s0) & 31;
                a |= (uint32_t)(c & 1) << t;
                b |= (uint32_t)((c >> 1) & 1) << t;
            }
        }
        if (s >= s0 && (((s - s0) & 31) == 31 || s + 1 == s0 + N)) { p1[w] = a; p2[w] = b; ++w; a = 0; b = 0; }
    }
    for (; w < Wr; ++w) { p1[w] = 0; p2[w] = 0; }
    hdr[snp] = lab.head;
}

}  // namespace gwasdev

using namespace gwasdev;

// ---- C-ABI ---------------------------------------------------------------------------------------
extern "C" {

const char *gwasdev_last_error(void) { return g_err; }
uint64_t gwasdev_launch_count(void) { return g_launches; }
uint32_t gwasdev_plane_blocks(uint32_t n) { return plane_blocks(n); }

int gwasdev_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int gwasdev_create(uint64_t n_snps, uint32_t n_samples, int device, gwasdev_store **out) {
    GW_REQUIRE(out != nullptr, "gwasdev_create: out is NULL");
    *out = nullptr;
    GW_REQUIRE(n_snps > 0 && n_samples > 0, "gwasdev_create: empty table (%llu x %u)",
               (unsigned long long)n_snps, n_samples);
    GW_REQUIRE(n_snps < (1ull << 31), "gwasdev_create: more than 2^31 SNPs");
    const int ndev = gwasdev_device_count();
    if (ndev == 0 || device < 0 || device >= ndev) {
        set_error("gwasdev_create: CUDA device %d not available (%d visible); this library has no CPU path",
                  device, ndev);
        return GWASDEV_ENODEVICE;
    }
    GW_CUDA(cudaSetDevice(device));
    gwasdev_store *s = new gwasdev_store();
    s->device = device;
    s->M = n_snps;
    s->N = n_samples;
    s->P = plane_blocks(n_samples);
    s->Wr = round_up(s->P / 2, 4);
    s->Mpad = (n_snps + TILE - 1) / TILE * TILE;
    cudaError_t e = cudaMalloc(&s->d_hdr, n_snps * sizeof(uint16_t));
    if (e == cudaSuccess) e = cudaMalloc(&s->d_raw, n_snps * 2ull * s->Wr * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&s->d_masks, 4ull * s->Wr * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(s->d_masks, 0, 4ull * s->Wr * sizeof(uint32_t));
    s->d_case_mask = s->d_masks; s->d_ctrl_mask = s->d_masks + s->Wr;
    s->d_case_sel_mask = s->d_masks + 2ull * s->Wr; s->d_ctrl_sel_mask = s->d_masks + 3ull * s->Wr;
    if (e == cudaSuccess) e = cudaMemset(s->d_hdr, 0, n_snps * sizeof(uint16_t));
    if (e == cudaSuccess) e = cudaMemset(s->d_raw, 0, n_snps * 2ull * s->Wr * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev2);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev3);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_pw);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&s->h_cnt, 4 * sizeof(unsigned long long));
    if (e != cudaSuccess) {
        set_error("gwasdev_create: %s", cudaGetErrorString(e));
        gwasdev_destroy(s);
        return e == cudaErrorMemoryAllocation ? GWASDEV_ENOMEM : GWASDEV_ENODEVICE;
    }
    *out = s;
    return GWASDEV_OK;
}

static void free_scratch(gwasdev_store::Scratch &sc) { if (sc.p) cudaFree(sc.p); sc.p = nullptr; sc.cap = 0; }

static void invalidate_selection(gwasdev_store *s) {
    s->selected = s->sel_built = s->pw_built = s->mi_valid = s->side_valid = s->mm_built = s->mm4_built = s->mma_side_valid = s->pc_valid = false;
}

}  // extern "C"

void gwasdev_internal_rows_changed(gwasdev_store *s) {
    invalidate_selection(s);
    s->tot_valid = false;
    s->pb_resident = false;   // the permutation test's SNP planes depend on the rows only, not on the selection
    s->pb_missing = -1;
    s->ld_sums_valid = s->ld_resident = false;   // the LD operand depends on the rows and its sample set
}

extern "C" {

void gwasdev_destroy(gwasdev_store *s) {
    if (!s) return;
    cudaSetDevice(s->device);
    gwasdev_internal_free_ingest(s);
    cudaFree(s->d_masks); cudaFree(s->d_row_tot); cudaFree(s->d_case_idx); cudaFree(s->d_ctrl_idx);
    cudaFree(s->d_sel); cudaFree(s->d_pw); cudaFree(s->d_mi); cudaFree(s->d_side); cudaFree(s->d_tile_missing);
    free(s->tmap); free(s->tmap_mm); free(s->tmap_mm4); free(s->tmap_perm); free(s->tmap_ld);
    cudaFree(s->d_pa); cudaFree(s->d_pb); cudaFree(s->d_ld); cudaFree(s->d_ld_mask); cudaFree(s->d_ld_sums);
    cudaFree(s->d_mm); cudaFree(s->d_mm4); cudaFree(s->d_mma_row); cudaFree(s->d_mma_col); cudaFree(s->d_plane_derived); cudaFree(s->d_tile_counter);
    for (gwasdev_store::Scratch *sc : {&s->sc_out_counts, &s->sc_out_stats, &s->sc_out_mi, &s->sc_cnt, &s->sc_cand, &s->sc_keys,
                                      &s->sc_keys2, &s->sc_vals, &s->sc_vals2, &s->sc_sort, &s->sc_hits, &s->sc_pi, &s->sc_pj,
                                      &s->sc_a, &s->sc_b, &s->sc_stage, &s->sc_gather})
        free_scratch(*sc);
    if (s->h_cnt) cudaFreeHost(s->h_cnt);
    cudaFree(s->d_hdr); cudaFree(s->d_raw);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->ev2) cudaEventDestroy(s->ev2);
    if (s->ev3) cudaEventDestroy(s->ev3);
    if (s->ev_pw) cudaEventDestroy(s->ev_pw);
    for (cudaEvent_t e : s->ev_piece) if (e) cudaEventDestroy(e);
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    delete s;
}

int gwasdev_set_stream(gwasdev_store *s, void *cuda_stream) {
    GW_REQUIRE(s != nullptr, "gwasdev_set_stream: NULL store");
    s->stream = (cudaStream_t)cuda_stream;
    return GWASDEV_OK;
}

int gwasdev_set_option(gwasdev_store *s, int option, long long value) {
    GW_REQUIRE(s != nullptr, "gwasdev_set_option: NULL store");
    GW_REQUIRE(option >= 0 && option < GWASDEV_OPT_COUNT, "gwasdev_set_option: unknown option %d", option);
    if (option == GWASDEV_OPT_LANES_PER_ROW)
        GW_REQUIRE(value == 0 || value == 8 || value == 16 || value == 32, "gwasdev_set_option: lanes per row must be 0, 8, 16 or 32");
    if (option == GWASDEV_OPT_SCAN_PIECES) GW_REQUIRE(value >= 0 && value <= gwasdev_store::MAX_PIECES, "gwasdev_set_option: 0..%d pieces", gwasdev_store::MAX_PIECES);
    if (option == GWASDEV_OPT_INGEST_CHUNK) GW_REQUIRE(value == 0 || value >= 64, "gwasdev_set_option: ingest chunks of at least 64 bytes");
    GW_REQUIRE(value >= 0, "gwasdev_set_option: negative value");
    // the tensor-core operand planes and the per-SNP records stored by role follow the plane choice: rebuild them
    if (option == GWASDEV_OPT_CLASSIC_PLANES && value != s->opt[option]) s->mm_built = s->mma_side_valid = false;
    s->opt[option] = value;
    return GWASDEV_OK;
}

int gwasdev_synchronize(gwasdev_store *s) {
    GW_REQUIRE(s != nullptr, "gwasdev_synchronize: NULL store");
    GW_CUDA(cudaSetDevice(s->device));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    return GWASDEV_OK;
}

int gwasdev_pack_row_text(const char *txt, size_t len, uint32_t n_samples, uint16_t *row) {
    return gwasdev_pack_row_text_block(txt, len, n_samples, row, nullptr);
}

int gwasdev_pack_row_text_block(const char *txt, size_t len, uint32_t n_samples, uint16_t *row, uint16_t *label_state) {
    GW_REQUIRE(txt && row, "gwasdev_pack_row_text: NULL argument");
    const uint32_t P = plane_blocks(n_samples);
    memset(row, 0, sizeof(uint16_t) * (2 * (size_t)P + 1));
    static const signed char allele[256] = {
        // index of the allele letter in "ACGT", 4 = unknown (compressed_genotype_table5.cpp:94-100)
#define X4 4, 4, 4, 4
#define X16 X4, X4, X4, X4
        X16, X16, X16, X16,                                        /* 0..63 */
        4, 0, 4, 1, 4, 4, 4, 2, 4, 4, 4, 4, 4, 4, 4, 4,            /* @ A B C D E F G ... */
        4, 4, 4, 4, 3, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4,            /* P Q R S T ... */
        X16, X16, X16, X16, X16, X16, X16, X16, X16, X16
#undef X16
#undef X4
    };
    Labeler lab;
    lab.reset();
    if (label_state && *label_state) {   // continue the row's first-seen labelling after the earlier sample blocks
        const uint16_t h = *label_state, st = h & 0xF000;
        const int e1 = (h >> 8) & 0xF, e2 = (h >> 4) & 0xF, e3 = h & 0xF;
        GW_REQUIRE(st == 0x1000 || st == 0x2000 || st == 0x3000 || st == 0x4000 || st == 0x7000, "gwasdev_pack_row_text_block: bad label state 0x%04x", h);
        lab.head = h;
        if (st == 0x1000 || st == 0x3000 || st == 0x4000 || st == 0x7000) lab.codes |= 1ull << (4 * e1);
        if (st == 0x2000 || st == 0x4000 || st == 0x7000) lab.codes |= 2ull << (4 * e2);
        if (st == 0x3000 || st == 0x7000) lab.codes |= 3ull << (4 * e3);
    }
    size_t pos = 0;
    for (uint32_t col = 0; col < n_samples && pos + 1 < len; ++col, pos += 3) {
        const int a = allele[(unsigned char)txt[pos]], b = allele[(unsigned char)txt[pos + 1]];
        if (a < 4 && b < 4) {
            const int c = lab.code(4 * a + b);
            if (c < 0) {
                set_error("gwasdev_pack_row_text: column %u introduces a third genotype spelling of one kind; "
                          "the reference aborts here (compressed_genotype_table5.cpp:325)", col);
                return GWASDEV_EINVAL;
            }
            if (c & 1) row[1 + (col >> 4)] |= (uint16_t)(1u << (col & 15));
            if (c & 2) row[1 + P + (col >> 4)] |= (uint16_t)(1u << (col & 15));
        }
    }
    row[0] = lab.head;
    if (label_state) *label_state = lab.head;
    return GWASDEV_OK;
}

static const uint64_t STAGE_BYTES = 64ull << 20;

int gwasdev_put_rows(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, const uint16_t *rows) {
    GW_REQUIRE(s && rows, "gwasdev_put_rows: NULL argument");
    GW_REQUIRE(first_row + n_rows <= s->M, "gwasdev_put_rows: rows [%llu, %llu) outside the table of %llu",
               (unsigned long long)first_row, (unsigned long long)(first_row + n_rows), (unsigned long long)s->M);
    if (n_rows == 0) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    const uint64_t row_bytes = (2ull * s->P + 1) * sizeof(uint16_t);
    const uint64_t chunk = std::max<uint64_t>(1, STAGE_BYTES / row_bytes);
    GW_CUDA(reserve(s->sc_stage, std::min(chunk, n_rows) * row_bytes));
    uint16_t *d_stage = (uint16_t *)s->sc_stage.p;
    for (uint64_t r = 0; r < n_rows; r += chunk) {
        const uint64_t n = std::min(chunk, n_rows - r);
        cudaError_t e = cudaMemcpyAsync(d_stage, (const char *)rows + r * row_bytes, n * row_bytes,
                                        cudaMemcpyHostToDevice, s->stream);
        if (e == cudaSuccess) {
            unpack_rows_kernel<<<(unsigned)n, 128, 0, s->stream>>>(d_stage, s->P, s->Wr, s->N, s->d_hdr, s->d_raw, first_row + r);
            ++g_launches;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
        if (e != cudaSuccess) { set_error("gwasdev_put_rows: %s", cudaGetErrorString(e)); return GWASDEV_ENODEVICE; }
    }
    gwasdev_internal_rows_changed(s);
    return GWASDEV_OK;
}

int gwasdev_get_rows(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, uint16_t *rows) {
    GW_REQUIRE(s && rows, "gwasdev_get_rows: NULL argument");
    GW_REQUIRE(first_row + n_rows <= s->M, "gwasdev_get_rows: rows outside the table");
    if (n_rows == 0) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    const uint64_t row_bytes = (2ull * s->P + 1) * sizeof(uint16_t);
    const uint64_t chunk = std::max<uint64_t>(1, STAGE_BYTES / row_bytes);
    GW_CUDA(reserve(s->sc_stage, std::min(chunk, n_rows) * row_bytes));
    uint16_t *d_stage = (uint16_t *)s->sc_stage.p;
    for (uint64_t r = 0; r < n_rows; r += chunk) {
        const uint64_t n = std::min(chunk, n_rows - r);
        pack_rows_kernel<<<(unsigned)n, 128, 0, s->stream>>>(s->d_hdr, s->d_raw, s->P, s->Wr, d_stage, first_row + r);
        ++g_launches;
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync((char *)rows + r * row_bytes, d_stage, n * row_bytes, cudaMemcpyDeviceToHost, s->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
        if (e != cudaSuccess) { set_error("gwasdev_get_rows: %s", cudaGetErrorString(e)); return GWASDEV_ENODEVICE; }
    }
    return GWASDEV_OK;
}

int gwasdev_call_at(gwasdev_store *s, uint64_t row, uint32_t col, char out[3]) {
    GW_REQUIRE(s && out, "gwasdev_call_at: NULL argument");
    GW_REQUIRE(row < s->M && col < s->N, "gwasdev_call_at: (%llu, %u) outside the table", (unsigned long long)row, col);
    GW_CUDA(cudaSetDevice(s->device));
    uint16_t h = 0;
    uint32_t w1 = 0, w2 = 0;
    GW_CUDA(cudaStreamSynchronize(s->stream));
    GW_CUDA(cudaMemcpy(&h, s->d_hdr + row, sizeof h, cudaMemcpyDeviceToHost));
    GW_CUDA(cudaMemcpy(&w1, s->d_raw + row * 2ull * s->Wr + (col >> 5), 4, cudaMemcpyDeviceToHost));
    GW_CUDA(cudaMemcpy(&w2, s->d_raw + row * 2ull * s->Wr + s->Wr + (col >> 5), 4, cudaMemcpyDeviceToHost));
    const int b1 = (w1 >> (col & 31)) & 1, b2 = (w2 >> (col & 31)) & 1;
    int enc;
    if (b1 && b2) enc = h & 0xF;
    else if (b1) enc = (h >> 8) & 0xF;
    else if (b2) enc = (h >> 4) & 0xF;
    else { out[0] = '0'; out[1] = '0'; out[2] = 0; return GWASDEV_OK; }
    out[0] = "ACGT"[enc >> 2]; out[1] = "ACGT"[enc & 3]; out[2] = 0;
    return GWASDEV_OK;
}

int gwasdev_simulate_block(gwasdev_store *s, uint64_t seed, const uint32_t bin_counts[51], uint32_t missing_q32,
                           uint32_t first_sample, uint32_t n_total_samples) {
    GW_REQUIRE(s && bin_counts, "gwasdev_simulate: NULL argument");
    GW_REQUIRE((uint64_t)first_sample + s->N <= n_total_samples, "gwasdev_simulate_block: samples [%u, %llu) outside the cohort of %u",
               first_sample, (unsigned long long)first_sample + s->N, n_total_samples);
    GW_CUDA(cudaSetDevice(s->device));
    uint32_t cum[51];
    uint64_t t = 0;
    for (int b = 0; b < 51; ++b) { t += bin_counts[b]; cum[b] = (uint32_t)t; }
    GW_REQUIRE(t > 0 && t < (1ull << 32), "gwasdev_simulate: bad MAF histogram (total %llu)", (unsigned long long)t);
    uint32_t *d_cum = nullptr;
    GW_CUDA(cudaMalloc(&d_cum, sizeof cum));
    GW_CUDA(cudaMemcpyAsync(d_cum, cum, sizeof cum, cudaMemcpyHostToDevice, s->stream));
    const unsigned threads = 64, blocks = (unsigned)((s->M + threads - 1) / threads);
    simulate_kernel<<<blocks, threads, 0, s->stream>>>(seed, d_cum, s->N, first_sample, n_total_samples, missing_q32, s->d_hdr, s->d_raw,
                                                       s->Wr, s->M);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    cudaFree(d_cum);
    if (e != cudaSuccess) { set_error("gwasdev_simulate: %s", cudaGetErrorString(e)); return GWASDEV_ENODEVICE; }
    gwasdev_internal_rows_changed(s);
    return GWASDEV_OK;
}

int gwasdev_simulate(gwasdev_store *s, uint64_t seed, const uint32_t bin_counts[51], uint32_t missing_q32) {
    GW_REQUIRE(s != nullptr, "gwasdev_simulate: NULL argument");
    return gwasdev_simulate_block(s, seed, bin_counts, missing_q32, 0, s->N);
}

int gwasdev_simulate_phenotype(uint64_t seed, uint32_t n_samples, uint32_t n_case, uint8_t *pheno) {
    GW_REQUIRE(pheno && n_case <= n_samples, "gwasdev_simulate_phenotype: bad argument");
    uint64_t chosen = 0;
    for (uint32_t i = 0; i < n_samples; ++i) {
        const uint64_t left = n_samples - i, u = sim_hash(seed, SIM_STREAM_PHENO, i) >> 32;
        if (((u * left) >> 32) < n_case - chosen) { pheno[i] = 1; ++chosen; } else pheno[i] = 0;
    }
    return GWASDEV_OK;
}

// host-side precomputation of the compress tables for one class
static void build_select_tables(const std::vector<uint32_t> &mask, uint32_t n_class, uint32_t Kout,
                                std::vector<uint32_t> &blob /* m | mv | rank | first */) {
    const uint32_t Wr = (uint32_t)mask.size();
    const uint32_t Kf = std::max(Kout, 1u);
    blob.assign(7ull * Wr + 1 + Kf + 5ull * Wr, 0);
    uint32_t *m = blob.data(), *mv = m + Wr, *rank = m + 6ull * Wr, *first = rank + Wr + 1, *mvl = first + Kf;
    auto rev32 = [](uint32_t v) { uint32_t r = 0; for (int b = 0; b < 32; ++b) r |= ((v >> b) & 1u) << (31 - b); return r; };
    uint32_t r = 0;
    for (uint32_t sw = 0; sw < Wr; ++sw) {
        uint32_t mm = mask[sw];
        m[sw] = mm;
        rank[sw] = r;
        r += (uint32_t)__builtin_popcount(mm);
        for (int left = 0; left < 2; ++left) {   // the left-compress masks are those of the bit-reversed problem, reversed
            uint32_t mq = left ? rev32(mask[sw]) : mm;
            uint32_t mk = ~mq << 1;
            for (int i = 0; i < 5; ++i) {
                uint32_t mp = mk ^ (mk << 1);
                mp ^= mp << 2; mp ^= mp << 4; mp ^= mp << 8; mp ^= mp << 16;
                const uint32_t v = mp & mq;
                if (left) mvl[5 * sw + i] = rev32(v); else mv[5 * sw + i] = v;
                mq = (mq ^ v) | (v >> (1 << i));
                mk &= ~mp;
            }
        }
    }
    rank[Wr] = r;
    (void)n_class;
    uint32_t sw = 0;
    for (uint32_t o = 0; o < Kout; ++o) {
        while (sw < Wr && rank[sw + 1] <= 32 * o) ++sw;   // first source word holding member 32*o
        first[o] = sw;
    }
}

// 16-bit stream-mask blocks -> 32-bit words over the raw sample positions, bits at or beyond sample N dropped
static void mask_words(const uint16_t *blocks, uint32_t P, uint32_t N, uint32_t Wr, uint32_t *out) {
    for (uint32_t w = 0; w < Wr; ++w) {
        uint32_t v = 0;
        if (2 * w < P) v = blocks[2 * w];
        if (2 * w + 1 < P) v |= (uint32_t)blocks[2 * w + 1] << 16;
        if (32 * w + 32 > N) v &= 32 * w >= N ? 0u : (0xffffffffu >> (32 * w + 32 - N));
        out[w] = v;
    }
}
static uint32_t count_bits(const uint32_t *m, uint32_t n) { uint32_t c = 0; for (uint32_t w = 0; w < n; ++w) c += (uint32_t)__builtin_popcount(m[w]); return c; }

int gwasdev_select_case_control(gwasdev_store *s, const uint16_t *case_mask, const uint16_t *ctrl_mask) {
    GW_REQUIRE(s && case_mask && ctrl_mask, "gwasdev_select_case_control: NULL argument");
    GW_CUDA(cudaSetDevice(s->device));
    // member masks as 32-bit words; a sample flagged in both masks is a case for the compaction
    // (compressed_genotype_table5.cpp:541-561) but stays in both masks for the mask-on-the-fly overloads
    const uint32_t Wr = s->Wr;
    std::vector<uint32_t> m(4ull * Wr);
    uint32_t *mca = m.data(), *mco = mca + Wr, *mca_sel = mco + Wr, *mco_sel = mca_sel + Wr;
    mask_words(case_mask, s->P, s->N, Wr, mca);
    mask_words(ctrl_mask, s->P, s->N, Wr, mco);
    for (uint32_t w = 0; w < Wr; ++w) { mca_sel[w] = mca[w]; mco_sel[w] = mco[w] & ~mca[w]; }
    const uint32_t nca = count_bits(mca_sel, Wr), nco = count_bits(mco_sel, Wr);
    GW_REQUIRE(nca + nco > 0, "gwasdev_select_case_control: both masks are empty");
    invalidate_selection(s);
    s->n_case = nca;
    s->n_ctrl = nco;
    s->n_fly_case = nca;
    s->n_fly_ctrl = count_bits(mco, Wr);
    s->Pca = plane_blocks(nca);
    s->Pco = plane_blocks(nco);
    s->Kc = (nca + 31) / 32;
    s->Kt = (nco + 31) / 32;
    s->Wc = round_up(std::max(s->Kc, 1u), 4);
    s->Wt = round_up(std::max(s->Kt, 1u), 4);
    // the four masks in one copy; K0's compress tables are built (host) and uploaded only if K0 ever runs
    GW_CUDA(cudaMemcpyAsync(s->d_masks, m.data(), 4ull * Wr * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));   // m goes out of scope
    s->h_sel_masks.assign(mca_sel, mca_sel + 2ull * Wr);
    s->h_given_masks.assign(case_mask, case_mask + s->P);
    s->h_given_masks.insert(s->h_given_masks.end(), ctrl_mask, ctrl_mask + s->P);
    s->h_fly_masks = s->h_given_masks;
    s->selected = true;
    s->fly_valid = true;
    s->sel_built = false;
    s->scans_since_select = 0;
    // Compaction (K0) is deferred until something needs the compacted layout (layout probes, the AND+POPC engine, a
    // second marginal scan of a cohort with samples outside both classes): scans after a selection count through the
    // masks on the raw rows, the reference's own mask-on-the-fly overload (compressed_genotype_table5.cpp:609-657).
    if (s->eager_select) return gwasdev_internal_ensure_compacted(s);
    return GWASDEV_OK;
}

}  // extern "C"

int gwasdev_internal_replay_settings(const gwasdev_store *src, gwasdev_store *dst) {
    for (int o = 0; o < GWASDEV_OPT_COUNT; ++o) dst->opt[o] = src->opt[o];
    dst->pair_engine = src->pair_engine;
    dst->eager_select = src->eager_select;
    if (src->selected && !src->h_given_masks.empty()) {
        const uint16_t *m = src->h_given_masks.data();
        const int rc = gwasdev_select_case_control(dst, m, m + src->P);
        if (rc != GWASDEV_OK) return rc;
    }
    // the stream masks after the selection, which resets them: gwasdev_set_stream_masks may have replaced them since, and they
    // outlive a row write that drops the selection
    if (src->fly_valid && (!src->selected || src->h_fly_masks != src->h_given_masks)) {
        const uint16_t *m = src->h_fly_masks.data();
        return gwasdev_set_stream_masks(dst, m, m + src->P);
    }
    return GWASDEV_OK;
}

extern "C" {

// Masks of the mask-on-the-fly overloads only (getCaseControlGenotypeDistribution(r, ccs, ..) :609-657,
// getCaseControlContingencyTable(i, j, ccs, ..) :806-895): in the reference these never touch the pre-selected
// m_cases_controls, so the selection, the compacted rows, the margins and the pairwise layouts all stay valid.
int gwasdev_set_stream_masks(gwasdev_store *s, const uint16_t *case_mask, const uint16_t *ctrl_mask) {
    GW_REQUIRE(s && case_mask && ctrl_mask, "gwasdev_set_stream_masks: NULL argument");
    GW_CUDA(cudaSetDevice(s->device));
    const uint32_t Wr = s->Wr;
    std::vector<uint32_t> m(2ull * Wr);
    mask_words(case_mask, s->P, s->N, Wr, m.data());
    mask_words(ctrl_mask, s->P, s->N, Wr, m.data() + Wr);
    s->n_fly_case = count_bits(m.data(), Wr);
    s->n_fly_ctrl = count_bits(m.data() + Wr, Wr);
    GW_CUDA(cudaMemcpyAsync(s->d_masks, m.data(), 2ull * Wr * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    s->h_fly_masks.assign(case_mask, case_mask + s->P);
    s->h_fly_masks.insert(s->h_fly_masks.end(), ctrl_mask, ctrl_mask + s->P);
    s->fly_valid = true;
    return GWASDEV_OK;
}

int gwasdev_set_select_mode(gwasdev_store *s, int eager) {
    GW_REQUIRE(s != nullptr, "gwasdev_set_select_mode: NULL store");
    s->eager_select = eager != 0;
    return GWASDEV_OK;
}

int gwasdev_is_compacted(const gwasdev_store *s) { return (!s || !s->selected) ? -1 : (s->sel_built ? 1 : 0); }

int gwasdev_case_control_counts(gwasdev_store *s, uint32_t *n_case, uint32_t *n_ctrl) {
    GW_REQUIRE(s && s->selected, "gwasdev_case_control_counts: no case/control selection");
    if (n_case) *n_case = s->n_case;
    if (n_ctrl) *n_ctrl = s->n_ctrl;
    return GWASDEV_OK;
}

int gwasdev_get_selected_rows(gwasdev_store *s, uint64_t first_row, uint64_t n_rows, uint16_t *rows) {
    GW_REQUIRE(s && rows, "gwasdev_get_selected_rows: NULL argument");
    GW_REQUIRE(s->selected, "gwasdev_get_selected_rows: call gwasdev_select_case_control first");
    GW_REQUIRE(first_row + n_rows <= s->M, "gwasdev_get_selected_rows: rows outside the table");
    if (n_rows == 0) return GWASDEV_OK;
    GW_CUDA(cudaSetDevice(s->device));
    { const int rc = gwasdev_internal_ensure_compacted(s); if (rc != GWASDEV_OK) return rc; }
    const uint64_t S = 2ull * (s->Pca + s->Pco);
    GW_CUDA(reserve(s->sc_stage, n_rows * S * 2));
    uint16_t *d_out = (uint16_t *)s->sc_stage.p;
    export_selected_kernel<<<(unsigned)n_rows, 128, 0, s->stream>>>(s->d_sel, 2 * (s->Wc + s->Wt), s->Wc, s->Wt, s->Pca, s->Pco, d_out, first_row);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(rows, d_out, n_rows * S * 2, cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) { set_error("gwasdev_get_selected_rows: %s", cudaGetErrorString(e)); return GWASDEV_ENODEVICE; }
    return GWASDEV_OK;
}

}  // extern "C"

// K0 on demand: builds the compacted scan layout from the raw rows with the tables of the last selection.
int gwasdev_internal_ensure_compacted(gwasdev_store *s) {
    GW_REQUIRE(s->selected, "call gwasdev_select_case_control first");
    if (s->sel_built) return GWASDEV_OK;
    GW_REQUIRE(gwasdev_internal_compact_fits(s), "compacted layout: %u selected samples exceed the compaction kernel's row buffer "
               "(about 819 200; scans, screens and permutations need no compacted layout)", s->n_case + s->n_ctrl);
    GW_CUDA(cudaSetDevice(s->device));
    const uint32_t stride = 2 * (s->Wc + s->Wt);
    GW_CUDA(reserve_raw(s->d_sel, s->cap_sel, s->M * (uint64_t)stride * 4));
    {   // compress tables of this selection (host arithmetic over the two masks, 0.05 ms at 10 000 samples)
        std::vector<uint32_t> mca(s->h_sel_masks.begin(), s->h_sel_masks.begin() + s->Wr), mco(s->h_sel_masks.begin() + s->Wr, s->h_sel_masks.end());
        std::vector<uint32_t> bca, bco;
        build_select_tables(mca, s->n_case, s->Kc, bca);
        build_select_tables(mco, s->n_ctrl, s->Kt, bco);
        GW_CUDA(reserve_raw(s->d_case_idx, s->cap_case_idx, bca.size() * 4));
        GW_CUDA(reserve_raw(s->d_ctrl_idx, s->cap_ctrl_idx, bco.size() * 4));
        GW_CUDA(cudaMemcpyAsync(s->d_case_idx, bca.data(), bca.size() * 4, cudaMemcpyHostToDevice, s->stream));
        GW_CUDA(cudaMemcpyAsync(s->d_ctrl_idx, bco.data(), bco.size() * 4, cudaMemcpyHostToDevice, s->stream));
        GW_CUDA(cudaStreamSynchronize(s->stream));   // host vectors go out of scope
    }
    SelectTables ta, to;
    ta.m = s->d_case_idx; ta.mv = ta.m + s->Wr; ta.rank = ta.m + 6ull * s->Wr; ta.first = ta.rank + s->Wr + 1; ta.mvl = ta.first + std::max(s->Kc, 1u); ta.n_class = s->n_case; ta.Kout = s->Kc;
    to.m = s->d_ctrl_idx; to.mv = to.m + s->Wr; to.rank = to.m + 6ull * s->Wr; to.first = to.rank + s->Wr + 1; to.mvl = to.first + std::max(s->Kt, 1u); to.n_class = s->n_ctrl; to.Kout = s->Kt;
    int sms = 0;
    GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    const bool trace = s->opt[GWASDEV_OPT_TRACE] != 0;
    if (trace) cudaEventRecord(s->ev2, s->stream);
    constexpr int SNPS = 4;                                     // rows assembled per block iteration
    const size_t smem_rows = (size_t)SNPS * stride * sizeof(uint32_t);
    const size_t smem_tab = 2 * (7ull * s->Wr + 1) * sizeof(uint32_t);
    if (s->Wr <= 1024 && s->opt[GWASDEV_OPT_SELECT_KERNEL] == 0) {   // register form: one thread per source column
        constexpr int CS = 8;
        const unsigned threads = round_up(s->Wr, 32);
        const size_t smem = (size_t)CS * stride * sizeof(uint32_t);
        GW_CUDA(cudaFuncSetAttribute(select_columns_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        GW_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, select_columns_kernel<CS>, (int)threads, smem));
        const unsigned grid = (unsigned)std::min<uint64_t>((s->M + CS - 1) / CS, (uint64_t)sms * std::max(per_sm, 1));
        select_columns_kernel<CS><<<grid, threads, smem, s->stream>>>(s->d_raw, s->Wr, ta, to, s->d_sel, stride, s->Wc, s->Wt, s->M);
    } else if (smem_rows + smem_tab <= 160 * 1024) {   // tables staged in shared memory (up to ~80 000 samples), else read through L1/L2
        const size_t smem = smem_rows + smem_tab;
        GW_CUDA(cudaFuncSetAttribute(select_kernel<true, SNPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const unsigned per_sm = (unsigned)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / std::max<size_t>(smem, 1)));
        const unsigned grid = (unsigned)std::min<uint64_t>((s->M + SNPS - 1) / SNPS, (uint64_t)sms * per_sm);
        select_kernel<true, SNPS><<<grid, 256, smem, s->stream>>>(s->d_raw, s->Wr, ta, to, s->d_sel, stride, s->Wc, s->Wt, s->M);
    } else {
        GW_CUDA(cudaFuncSetAttribute(select_kernel<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem_rows / SNPS)));
        const unsigned grid = (unsigned)std::min<uint64_t>(s->M, (uint64_t)sms * 4);
        select_kernel<false, 1><<<grid, 256, smem_rows / SNPS, s->stream>>>(s->d_raw, s->Wr, ta, to, s->d_sel, stride, s->Wc, s->Wt, s->M);
    }
    GW_LAUNCHED();
    if (trace) {
        cudaEventRecord(s->ev3, s->stream);
        GW_CUDA(cudaStreamSynchronize(s->stream));
        float ms = 0.f; cudaEventElapsedTime(&ms, s->ev2, s->ev3); fprintf(stderr, "[gwasdev trace] select_kernel %.3f ms\n", ms);
    }
    s->sel_built = true;
    return GWASDEV_OK;
}

// Builds the pairwise layout on first use (called from pairwise.cu).
int gwasdev_internal_build_pairwise(gwasdev_store *s) {
    if (s->pw_built) return GWASDEV_OK;
    GW_REQUIRE(s->selected, "pairwise layout: call gwasdev_select_case_control first");
    { const int rc = gwasdev_internal_ensure_compacted(s); if (rc != GWASDEV_OK) return rc; }
    const uint32_t K = s->Kc + s->Kt;
    GW_CUDA(reserve_raw(s->d_pw, s->cap_pw, 3ull * K * s->Mpad * 4));
    dim3 block(32, 8), grid((unsigned)((s->Mpad + 31) / 32), (K + 7) / 8);
    build_pairwise_kernel<<<grid, block, 0, s->stream>>>(s->d_sel, 2 * (s->Wc + s->Wt), s->Wc, s->Wt, s->Kc, s->Kt, s->M, s->Mpad, s->d_pw);
    GW_LAUNCHED();
    s->pw_built = true;
    return GWASDEV_OK;
}
