// Internal definitions shared by the translation units of libgwasdev.so (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>
#include <vector>

#include "gwasdev.h"

namespace gwasdev {

// ---- error plumbing ------------------------------------------------------------------------------
void set_error(const char *fmt, ...);
extern std::atomic<unsigned long long> g_launches;   // kernels launched by this library (gwasdev_launch_count); stores may be driven from several host threads

#define GW_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            gwasdev::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__,   \
                               __LINE__);                                                          \
            return e_ == cudaErrorMemoryAllocation ? GWASDEV_ENOMEM : GWASDEV_ENODEVICE;           \
        }                                                                                          \
    } while (0)

#define GW_LAUNCHED()                                                                              \
    do {                                                                                           \
        ++gwasdev::g_launches;                                                                     \
        GW_CUDA(cudaGetLastError());                                                               \
    } while (0)

#define GW_REQUIRE(cond, ...)                                                                      \
    do {                                                                                           \
        if (!(cond)) {                                                                             \
            gwasdev::set_error(__VA_ARGS__);                                                       \
            return GWASDEV_EINVAL;                                                                 \
        }                                                                                          \
    } while (0)

// ---- geometry ------------------------------------------------------------------------------------
constexpr int TILE = 64;   // SNPs per side of a pairwise tile

__host__ __device__ inline uint32_t plane_blocks(uint32_t n) {   // pad4(n/16 + 1), 16-bit blocks
    uint32_t b = n / 16 + 1;
    return (b + 3u) & ~3u;
}
__host__ __device__ inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }

// Scan layout of one compacted SNP row (device-private; gwasdev_get_selected_rows converts back to the
// reference's layout): cases then controls; inside a class the two bit-planes are interleaved in
// 16-byte chunks, [p1 words 0-3][p2 words 0-3][p1 words 4-7][p2 words 4-7]..., so that one 32-byte
// load brings 128 samples of both planes. Wc / Wt = words per plane per class (multiples of 4); the
// control block starts at word 2*Wc; row stride = 2*(Wc+Wt) words.
__host__ __device__ inline uint32_t sel_word(uint32_t class_off, uint32_t plane, uint32_t w) {
    return class_off + (w >> 2) * 8 + plane * 4 + (w & 3);
}

// ---- first-seen genotype labelling ---------------------------------------------------------------
// Genotype "encodings" are 4*idx(c1)+idx(c2) over the alphabet ACGT; 0, 5, 10, 15 are homozygous.
// Codes: first homozygote seen in the row -> 1 (plane1), heterozygote -> 2 (plane2), second
// homozygote -> 3 (both). The 16-bit row header keeps state<<12 | enc(code1)<<8 | enc(code2)<<4 |
// enc(code3) with the same bit pattern the reference's header state machine leaves behind
// (genetics/genotype/common_genotype.h:257-304), so stored headers round-trip through decodeGenotype.
struct Labeler {
    uint16_t head;
    uint64_t codes;   // 4 bits per encoding, 0 = not seen yet
    __host__ __device__ void reset() { head = 0; codes = 0; }
    // returns 1..3, or -1 for a sequence the reference rejects (third spelling of a kind)
    __host__ __device__ int code(int enc) {
        int c = (int)((codes >> (4 * enc)) & 0xF);
        if (c) return c;
        const bool hom = (enc == 0 || enc == 5 || enc == 10 || enc == 15);
        const uint16_t state = head & 0xF000;
        uint16_t keep, next;
        int shift;
        if (state == 0x0000)      { keep = 0x0000; if (hom) { next = 0x1000; shift = 8; c = 1; } else { next = 0x2000; shift = 4; c = 2; } }
        else if (state == 0x1000) { keep = 0x0F00; if (hom) { next = 0x3000; shift = 0; c = 3; } else { next = 0x4000; shift = 4; c = 2; } }
        else if (state == 0x2000) { if (!hom) return -1; keep = 0x00F0; next = 0x4000; shift = 8; c = 1; }
        else if (state == 0x3000) { if (hom) return -1;  keep = 0x0F0F; next = 0x7000; shift = 4; c = 2; }
        else if (state == 0x4000) { if (!hom) return -1; keep = 0x0FF0; next = 0x7000; shift = 0; c = 3; }
        else return -1;
        head = (uint16_t)((head & keep) | next | (enc << shift));
        codes |= (uint64_t)c << (4 * enc);
        return c;
    }
};

// ---- counter-based generator for the synthetic cohort (see DESIGN.md, "synthetic cohort") ---------
__host__ __device__ inline uint64_t sim_hash(uint64_t seed, uint64_t a, uint64_t b) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ULL * (a + 1) + 0xD1B54A32D192ED03ULL * (b + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
constexpr uint64_t SIM_STREAM_BIN = 0xFFFFFFFF00000001ULL;
constexpr uint64_t SIM_STREAM_FREQ = 0xFFFFFFFF00000002ULL;
constexpr uint64_t SIM_STREAM_PHENO = 0xFFFFFFFF00000003ULL;
constexpr uint64_t SIM_STREAM_MISS = 0x8000000000000000ULL;

// ---- per-SNP record used by the pairwise screen's fp32 epilogue -----------------------------------
// For SNP x with class counts c_k[g] (k: 0 case, 1 control; g: aa, ab, bb), margins m[g] = c_0[g]+c_1[g]
// and class sizes n_k (incl. missing):
//   pca[k][g]  = c_k[g] / m[g]                       P(class | genotype)      (row role, SNP "A")
//   lpca[k][g] = ln pca[k][g]            (0 when c_k[g] == 0)
//   w[k][g]    = (c_k[g] / n_k) / m[g]               P(genotype | class)/m    (column role, SNP "B"; NaN when m[g]==0)
//   lw[k][g]   = ln(c_k[g] / n_k) - ln m[g]  (0 when c_k[g] == 0)
struct __align__(16) PairSide {
    float pca[2][3];
    float lpca[2][3];
    float w[2][3];
    float lw[2][3];
    uint32_t cnt[2][4];   // c_k[aa, ab, bb, xx]
};
static_assert(sizeof(PairSide) == 128, "PairSide is 128 bytes");

}  // namespace gwasdev

// ---- the store -----------------------------------------------------------------------------------
struct gwasdev_store {
    int device = 0;
    cudaStream_t stream = 0;
    uint64_t M = 0;        // SNPs (rows)
    uint32_t N = 0;        // samples (columns)
    uint32_t P = 0;        // 16-bit blocks per raw plane (reference geometry)
    uint32_t Wr = 0;       // 32-bit words per raw plane on the device (multiple of 4 -> 16-byte rows)
    uint16_t *d_hdr = nullptr;    // [M] row headers
    uint32_t *d_raw = nullptr;    // [M][2][Wr]: plane1 (codes 1,3), plane2 (codes 2,3); sample c = bit c&31 of word c>>5

    // case/control selection
    bool selected = false;        // masks, class sizes and compaction tables of the last selection are on the device
    bool sel_built = false;       // d_sel holds the compacted rows of that selection (K0 has run)
    bool eager_select = false;    // run K0 inside gwasdev_select_case_control (gwasdev_set_select_mode)
    uint32_t scans_since_select = 0;
    uint32_t n_case = 0, n_ctrl = 0;
    uint32_t Pca = 0, Pco = 0;    // reference geometry of the compacted streams (16-bit blocks)
    uint32_t Wc = 0, Wt = 0;      // words per plane per class in the scan layout (multiples of 4)
    uint32_t Kc = 0, Kt = 0;      // tight word counts ceil(n/32) (pairwise layout)
    // class masks over the raw sample positions, [4][Wr] in one allocation (gwasdev_create):
    uint32_t *d_masks = nullptr;
    uint32_t *d_case_mask = nullptr, *d_ctrl_mask = nullptr;           // stream masks of the mask-on-the-fly overloads, as given (a sample may be in both)
    uint32_t *d_case_sel_mask = nullptr, *d_ctrl_sel_mask = nullptr;   // classes of the selection: cases, controls-and-not-cases
    bool fly_valid = false;                                            // on-the-fly masks uploaded (by a selection or gwasdev_set_stream_masks)
    uint32_t n_fly_case = 0, n_fly_ctrl = 0;                           // members of the on-the-fly masks as given (reference: ccs.getCaseCount() / getControlCount())
    std::vector<uint32_t> h_sel_masks;                                 // host copy of the selection masks [2][Wr]: K0's tables are built from it on demand
    std::vector<uint16_t> h_given_masks;                               // the selection's stream masks as given [2][P] (gwasdev_replicate re-applies them)
    std::vector<uint16_t> h_fly_masks;                                 // the on-the-fly masks as given [2][P]: the selection's or gwasdev_set_stream_masks'
    // per-SNP totals over ALL samples (|p1|, |p2|, |p1 & p2|, 0), independent of the phenotype: when the classes partition the
    // cohort the control counts are totals - case counts, so a re-selection's scan needs three masked popcount streams only
    uint4 *d_row_tot = nullptr;
    bool tot_valid = false;
    uint32_t *d_case_idx = nullptr, *d_ctrl_idx = nullptr;     // sample index of the k-th case / control
    uint32_t *d_sel = nullptr;    // scan layout [M][cases: Wc/4 x (p1 chunk, p2 chunk)][controls: Wt/4 x (p1 chunk, p2 chunk)]
    size_t cap_sel = 0, cap_case_idx = 0, cap_ctrl_idx = 0;   // bytes allocated (grow-only)

    // pairwise layout: one-hot planes, word-major so that a 64-SNP tile row is 256 contiguous bytes
    bool pw_built = false;
    uint64_t Mpad = 0;            // M rounded up to a multiple of TILE
    uint32_t *d_pw = nullptr;     // [3 planes aa,ab,bb][K = Kc + Kt][Mpad]
    void *tmap = nullptr;         // host copy of the CUtensorMap over d_pw (128 bytes, 64-byte aligned)

    // margins
    bool mi_valid = false;
    gwasdev_marginal_information *d_mi = nullptr;   // [M]
    gwasdev::PairSide *d_side = nullptr;            // [Mpad]
    uint8_t *d_tile_missing = nullptr;              // [Mpad/TILE] 1 when any SNP of the tile has missing calls
    bool side_valid = false;

    size_t cap_pw = 0, cap_mi = 0, cap_side = 0, cap_tile = 0;

    // tensor-core pair screen (pairwise_mma.cu): signed-byte one-hot rows, K-major
    int pair_engine = 0;          // 0 auto, 1 AND+POPC tiles, 2 tcgen05 tiles (gwasdev_set_pair_engine)
    bool mm_built = false;
    uint64_t mm_rows = 0;         // 2 rows (planes aa, bb) per SNP, SNP count rounded up to 128
    uint32_t mm_kbytes = 0;       // bytes per row of d_mm: 32 * Wr, one byte per sample position of the raw row
    int8_t *d_mm = nullptr;
    void *tmap_mm = nullptr;      // host copies of the two CUtensorMaps (A box, B box)
    void *d_mma_row = nullptr, *d_mma_col = nullptr;   // per-SNP epilogue records (MmaRow / MmaCol)
    uint8_t *d_plane_derived = nullptr;                // per SNP: the genotype class (0 aa, 1 ab, 2 bb) the two-plane operands leave out
    size_t cap_plane = 0;
    unsigned long long *d_tile_counter = nullptr;      // next tile of the running tensor-core screen (its CTA pairs draw their tiles from it)
    uint64_t mm_tiles = 0;        // tile pairs in the tensor-core schedule
    uint32_t mm_band = 0, mm4_band = 0;   // A-blocks per L2 band of the two schedules (pairwise_mma.cu: schedule_band)
    // four-plane operands (aa, bb, xx, padding) for the tiles with missing calls (pair_screen_mma4_kernel)
    bool mm4_built = false;
    int mm4_mode = 0;             // 0: aa/bb/xx planes, packed classes; 1: per-class planes; 2: aa/bb/xx planes, one accumulator per class
    int8_t *d_mm4 = nullptr;
    size_t cap_mm4 = 0;
    uint64_t mm4_rows = 0, mm4_tiles = 0;
    uint32_t mm4_kbytes = 0;      // bytes per row of d_mm4: 32 * Wr (raw sample order; modes 0, 1) or cases | controls padded to 128 each (mode 2)
    void *tmap_mm4 = nullptr;
    float mma_qc = 0.f, mma_q0 = 0.f;   // constants of the upper-bound pre-filter (pairwise_mma.cu)
    uint32_t mma_bound_ncase = 0xffffffffu, mma_bound_n = 0;   // class split they were computed for
    std::vector<uint8_t> h_tile_missing;   // host copy of d_tile_missing (valid with side_valid)
    size_t cap_mm = 0, cap_mma_row = 0, cap_mma_col = 0;
    bool mma_side_valid = false;
    // permutation test (permute.cu): one-hot SNP planes over ALL raw samples, +1 bytes, phenotype-independent -- they survive
    // re-selection and are dropped by gwasdev_internal_rows_changed
    bool pb_resident = false;     // d_pb holds the planes of every SNP of the table
    int pb_missing = -1;          // the table has missing calls (3 planes per SNP) or not (2); -1: not determined yet
    int8_t *d_pb = nullptr;       // [pb_planes * SNPs][32 * Wr]
    int8_t *d_pa = nullptr;       // [permutations][32 * Wr]: +1 where the sample is a case of the permutation
    size_t cap_pb = 0, cap_pa = 0;
    void *tmap_perm = nullptr;    // host copies of the CUtensorMaps over d_pa and d_pb
    // windowed LD (ld.cu): int8 allele-count operand over the sample set S it was built for -- it survives calls with the same S,
    // is rebuilt when S changes and is dropped by gwasdev_internal_rows_changed
    bool ld_sums_valid = false;   // d_ld_sums and ld_missing describe the rows over h_ld_mask
    bool ld_resident = false;     // d_ld holds the operand of every SNP of the table over h_ld_mask
    int ld_missing = 0;           // some sample of S has no call at some SNP: three row types per SNP (x, called, x^2), else one (x)
    std::vector<uint32_t> h_ld_mask;   // S as [Wr] words
    uint32_t *d_ld_mask = nullptr;     // [Wr]
    uint2 *d_ld_sums = nullptr;        // [M] (sum x, sum x^2) over S
    int8_t *d_ld = nullptr;
    size_t cap_ld = 0;
    void *tmap_ld = nullptr;      // host copies of the CUtensorMaps over d_ld (A box, B box)
    bool any_missing = false, any_clean = false;     // over tiles, valid with side_valid
    // gathered sub-table of a set screen (pair_sets.cu): per row, its table index | (1 << 31) when one of its genotype classes aa,
    // ab, bb is empty. Its per-SNP records then leave such a class out of the statistic instead of making it NaN (see set_pair_live)
    uint32_t *d_set_keys = nullptr;
    bool pc_valid = false;                           // cached pair / tile counts of the last pairwise scan's shard
    int pc_engines = 0;
    uint32_t pc_shard = 0, pc_n_shards = 0;
    uint64_t pc_pairs = 0, pc_tiles = 0, pc_nine = 0;

    // grow-only scratch, so that steady-state calls never touch cudaMalloc / cudaFree (both cost
    // milliseconds and cudaFree synchronises the device)
    struct Scratch { void *p = nullptr; size_t cap = 0; };
    Scratch sc_out_counts, sc_out_stats, sc_out_mi;          // host-output staging of the marginal scan
    Scratch sc_cnt, sc_cand, sc_keys, sc_keys2, sc_vals, sc_vals2, sc_sort, sc_hits;   // pairwise scan
    Scratch sc_pi, sc_pj, sc_a, sc_b;                        // pair probes
    Scratch sc_stage;                                        // row upload / download staging
    Scratch sc_gather;                                       // multi-device driver: the shards' hit records after the gather
    unsigned long long *h_cnt = nullptr;                     // pinned host counters
    void *ingest = nullptr;                                  // file / text ingestion state (ingest.cu)

    long long opt[GWASDEV_OPT_COUNT] = {};                   // gwasdev_set_option (explicit knobs; the library reads no environment variables)

    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;   // ev0..ev1: last marginal scan; ev2..ev3: last pair screen
    cudaEvent_t ev_pw = nullptr;                                               // end of the last pairwise scan (its total_ms)
    static constexpr int MAX_PIECES = 8;                     // host-output scans: pieces whose copies overlap the next piece's scan
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_piece[MAX_PIECES] = {};
    double last_scan_ms = 0.0;
};

void gwasdev_internal_free_ingest(gwasdev_store *s);
void gwasdev_internal_rows_changed(gwasdev_store *s);      // raw rows were (re)written: everything derived from them is stale (store.cu)
int gwasdev_internal_ensure_compacted(gwasdev_store *s);   // K0 on demand (store.cu)
// options, pair engine, selection mode and the current selection of src applied to dst, a store over the same samples: what
// gwasdev_replicate and the set screens' gathered sub-tables carry over from the store they copy (store.cu)
int gwasdev_internal_replay_settings(const gwasdev_store *src, gwasdev_store *dst);
// whether K0 can compact the current selection: its largest form stages one compacted row in 200 KiB of shared memory, so
// ceil(n_case / 128) + ceil(n_ctrl / 128) <= 6 400 (about 819 200 selected samples)
inline bool gwasdev_internal_compact_fits(const gwasdev_store *s) { return 2ull * (s->Wc + s->Wt) * sizeof(uint32_t) <= 200 * 1024; }

namespace gwasdev {
// make sure sc holds at least `bytes`; contents are not preserved
inline cudaError_t reserve(gwasdev_store::Scratch &sc, size_t bytes) {
    if (bytes <= sc.cap) return cudaSuccess;
    if (sc.p) cudaFree(sc.p);
    sc.p = nullptr; sc.cap = 0;
    cudaError_t e = cudaMalloc(&sc.p, bytes);
    if (e == cudaSuccess) sc.cap = bytes;
    return e;
}
template <class T> inline cudaError_t reserve_raw(T *&p, size_t &cap, size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc((void **)&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
}
}  // namespace gwasdev
