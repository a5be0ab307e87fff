// Pieces shared by the two pair-screen engines (pairwise.cu: AND+POPC tiles; pairwise_mma.cu: tcgen05 tiles).
#pragma once
#include <cuda.h>
#include <string.h>

#include "common.cuh"

namespace gwasdev {

struct Candidate { uint32_t i, j; float stat; uint32_t pad; };

// Where the screen kernels put the pairs that pass their fp32 test. Threshold mode (hist == nullptr): every pair above
// `thr` (= threshold - margin) is appended; the host re-runs with a larger buffer if it overflowed. Top-k mode: the
// kernels also keep a two-level histogram of the appended statistics over the order-preserving integer image of fp32
// (so it covers any threshold, however low, at under 1 % relative resolution), and whenever the buffer passes a fill mark
// one thread raises a device-wide threshold to the lower edge of the bin above which k candidates have already been seen
// (minus `slack`, twice the fp32 error budget: the final choice is made on the fp64 re-scores) -- a pair below it can no
// longer be among the k best, so the buffer stops growing however low the caller's threshold is.
constexpr int CAND_HIST_COARSE = 256, CAND_HIST_FINE = 65536;     // bins: key >> 24, key >> 16
__host__ __device__ inline uint32_t stat_key(float f) {           // fp32 -> uint32, monotone (total order of non-NaN floats)
#ifdef __CUDA_ARCH__
    const uint32_t b = __float_as_uint(f);
#else
    uint32_t b; memcpy(&b, &f, 4);
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ inline float key_stat(uint32_t k) {
    const uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}
struct CandSink {
    Candidate *cand;
    unsigned long long *n_cand;       // pairs appended so far (may exceed cap)
    unsigned long long cap;
    float thr;                        // static floor
    uint32_t *hist;                   // [CAND_HIST_COARSE + CAND_HIST_FINE] counts per key bin; nullptr: threshold mode
    uint32_t *thr_dyn_key;            // current device-wide threshold as a key (0: not raised yet)
    uint32_t *lost_max_key;           // largest statistic (as a key) among the pairs that found the buffer full
    float slack;
    unsigned long long k_keep;
    unsigned long long raise_from, raise_mask;   // raise when slot + 1 >= raise_from and ((slot + 1) & raise_mask) == 0
};

// One launch of a set screen (pair_sets.cu): the shard's tiles (I2, J) of that kernel's block size in device memory, and the
// segment bounds c1, a1 of the gathered sub-table (set_pair_wanted in pairwise_mma.cu)
struct SetLaunch { const uint2 *tiles; uint64_t n_tiles; uint64_t c1, a1; };
// A set screen on a gathered sub-table: its segment bounds and, on the device, the table row of every sub-table row
struct SetScreen { uint64_t c1, a1; const uint32_t *d_map; };

// threshold the pairs of the next tile are tested against
__device__ __forceinline__ float sink_threshold(const CandSink &s) {
    if (!s.hist) return s.thr;
    uint32_t k;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(k) : "l"(s.thr_dyn_key) : "memory");
    return k ? fmaxf(key_stat(k), s.thr) : s.thr;
}
static __device__ __noinline__ void sink_raise(const uint32_t *hist, uint32_t *thr_dyn_key, float thr, float slack, unsigned long long k_keep) {
    const volatile uint32_t *coarse = hist, *fine = hist + CAND_HIST_COARSE;
    unsigned long long acc = 0;
    for (int c = CAND_HIST_COARSE - 1; c >= 0; --c) {
        const uint32_t n = coarse[c];
        if (acc + n < k_keep) { acc += n; continue; }
        for (int b = 256 * c + 255; b >= 256 * c; --b) {       // the fine bins of this coarse bin (counts may lag the coarse one by in-flight pushes)
            acc += fine[b];
            if (acc >= k_keep) {
                const float t = key_stat((uint32_t)b << 16) - slack;      // lower edge of the bin
                if (t > thr) atomicMax(thr_dyn_key, stat_key(t));
                return;
            }
        }
        return;
    }
}
// append pair (i, j); the caller has checked stat > sink_threshold
__device__ __forceinline__ void sink_push(const CandSink &s, uint32_t i, uint32_t j, float stat) {
    if (s.hist) {
        const uint32_t k = stat_key(stat);
        atomicAdd(s.hist + CAND_HIST_COARSE + (k >> 16), 1u);     // fine first: a reader that sees the coarse count finds at least as much below it
        atomicAdd(s.hist + (k >> 24), 1u);
    }
    const unsigned long long slot = atomicAdd(s.n_cand, 1ull);
    if (slot < s.cap) { Candidate cd; cd.i = i; cd.j = j; cd.stat = stat; cd.pad = 0; s.cand[slot] = cd; }
    else if (s.hist) atomicMax(s.lost_max_key, stat_key(stat));
    if (s.hist && slot + 1 >= s.raise_from && ((slot + 1) & s.raise_mask) == 0) sink_raise(s.hist, s.thr_dyn_key, s.thr, s.slack, s.k_keep);
}

// ---- PTX helpers (mbarrier + TMA) ----------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int x, int y, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}


// Where a per-pair kernel (fp64 re-score, G-test, probes) reads the two SNPs' genotypes: the compacted rows when K0 has run
// for this selection, else the raw rows through the selection's class masks (the operand bytes of the tensor-core screen
// are built the same way, so the pair path never needs the compaction).
struct PairSrc {
    const uint32_t *sel; uint32_t stride, Wc, Wt;              // compacted rows (scan layout) when sel != nullptr ...
    const uint32_t *raw; uint32_t Wr; const uint32_t *mca, *mco;   // ... or raw rows + class masks (cases; controls-and-not-cases)
};
inline PairSrc pair_src(const gwasdev_store *s) {
    PairSrc p;
    p.sel = s->sel_built ? s->d_sel : nullptr; p.stride = 2 * (s->Wc + s->Wt); p.Wc = s->Wc; p.Wt = s->Wt;
    p.raw = s->d_raw; p.Wr = s->Wr; p.mca = s->d_case_sel_mask; p.mco = s->d_ctrl_sel_mask;
    return p;
}
// 3x3 core cells (4x4 row-major, cells 0,1,2,4,5,6,8,9,10) of both classes for pair (i, j); words w = w0, w0 + step, ...
// (one thread: w0 = 0, step = 1; a warp: w0 = lane, step = 32 followed by a warp reduction)
__device__ __forceinline__ void core_counts_src(const PairSrc &p, uint64_t i, uint64_t j, uint32_t w0, uint32_t step, uint32_t ca[16], uint32_t co[16]) {
    auto add9 = [](uint32_t a1, uint32_t a2, uint32_t b1, uint32_t b2, uint32_t m, uint32_t t[16]) {
        const uint32_t abb = a1 & a2 & m, aaa = (a1 & m) ^ abb, aab = (a2 & m) ^ abb, bbb = b1 & b2, baa = b1 ^ bbb, bab = b2 ^ bbb;
        t[0] += __popc(aaa & baa); t[1] += __popc(aaa & bab); t[2] += __popc(aaa & bbb);
        t[4] += __popc(aab & baa); t[5] += __popc(aab & bab); t[6] += __popc(aab & bbb);
        t[8] += __popc(abb & baa); t[9] += __popc(abb & bab); t[10] += __popc(abb & bbb);
    };
    if (p.sel) {
        const uint32_t *ri = p.sel + i * (uint64_t)p.stride, *rj = p.sel + j * (uint64_t)p.stride;
        for (uint32_t w = w0; w < p.Wc; w += step) { const uint32_t x = sel_word(0, 0, w), y = sel_word(0, 1, w); add9(ri[x], ri[y], rj[x], rj[y], 0xffffffffu, ca); }
        for (uint32_t w = w0; w < p.Wt; w += step) { const uint32_t x = sel_word(2 * p.Wc, 0, w), y = sel_word(2 * p.Wc, 1, w); add9(ri[x], ri[y], rj[x], rj[y], 0xffffffffu, co); }
    } else {
        const uint32_t *a1 = p.raw + i * 2ull * p.Wr, *a2 = a1 + p.Wr, *b1 = p.raw + j * 2ull * p.Wr, *b2 = b1 + p.Wr;
        for (uint32_t w = w0; w < p.Wr; w += step) {
            const uint32_t x1 = a1[w], x2 = a2[w], y1 = b1[w], y2 = b2[w];
            add9(x1, x2, y1, y2, p.mca[w], ca);
            add9(x1, x2, y1, y2, p.mco[w], co);
        }
    }
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda at link time)
int get_encode_tiled(encode_tiled_fn *out);

__device__ __forceinline__ float u2f(uint32_t n) { return __uint_as_float(0x4B000000u | n) - 8388608.0f; }   // n < 2^23

// fp32 KSA screen value of a 3x3x2 table with the per-SNP records of both SNPs (see pairwise.cu for the algebra)
__device__ __forceinline__ float g_nlogn(float n) { return n * __logf(fmaxf(n, 1.0f)); }

__device__ __forceinline__ float ksa_screen_f32(const uint32_t (&n)[2][3][3], const PairSide &A, const PairSide &B,
                                                float N, float lnN) {
    float S = 0.f, tau = 0.f, total = 0.f;
    float row[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}}, col[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const float c0 = u2f(n[0][a][b]), c1 = u2f(n[1][a][b]), cab = c0 + c1;
            const float W = fmaf(B.w[0][b], A.pca[0][a], B.w[1][b] * A.pca[1][a]);
            tau = fmaf(cab, W, tau);
            S += g_nlogn(c0) + g_nlogn(c1) - g_nlogn(cab);
            row[0][a] += c0; row[1][a] += c1; col[0][b] += c0; col[1][b] += c1;
            total += cab;
        }
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            S = fmaf(-row[k][g], A.lpca[k][g], S);
            S = fmaf(-col[k][g], B.lw[k][g], S);
        }
    S = fmaf(-total, lnN, S);
    return 2.0f * fmaf(N, logf(tau), S);
}


}  // namespace gwasdev
