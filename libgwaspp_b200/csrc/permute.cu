// Label-permutation test of the marginal scan (max(T): PLINK --mperm's EMP1 and EMP2) on the tensor cores.
//
// Formulation. For permutation q, A[q][c] = 1 when sample position c is a case of q (0 for the other selected samples, the
// samples outside the selection and the padding); for SNP s, the one-hot planes B[3s+p][c] = 1 when sample c has genotype
// p in {aa, bb, xx} (xx: no call), over ALL raw samples. Then (A B^T)[q][3s+p] is the case count of genotype p of SNP s under
// permutation q: one int8 GEMM over the samples (tcgen05.mma kind::i8, every product 0 or 1, plain int32 counts). The
// heterozygote count is n_case(q) - aa - bb - xx, and the control counts are the selection's pooled counts minus the case
// counts (the pooled counts do not depend on the labels; they come from the observed scan the call runs first). A table
// without missing calls sends two planes per SNP (N = 128) instead of three (N = 192).
//
// The B operand depends on the rows only: it stays resident across re-selections while it fits the operand budget
// (GWASDEV_OPT_PERM_OPERAND_BYTES) and is dropped when rows change; above the budget it is expanded one SNP chunk at a time.
// The A operand (a few MB) is rebuilt by every call.
//
// Kernel (perm_gemm_kernel, permute_gemm.cuh, compiled in marginal.cu): the CTA-pair pipeline of mma_common.cuh. Tiles are (256 permutations: 128 TMEM lanes per CTA) x
// (64 SNPs: each CTA stages 32 SNPs of B), taken from a device counter in SNP-major order, so the tiles in flight share a few
// SNP blocks and B is read from DRAM about once per call. One TMEM lane holds one permutation, so a thread owns every plane of
// its (permutation, SNP) elements: the statistics come from the marginal scan's own chi2_tests (bit-identical), the per-permutation
// maxima are register maxima with one atomic per tile, and the exceedance counts are warp ballots with one atomic per SNP.
#include <algorithm>
#include <cmath>
#include <vector>

#include "permute.cuh"

int gwasdev_internal_scan(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t *d_counts,
                          gwasdev_marginal_information *d_mi, gwasdev_snp_stats *d_stats);   // marginal.cu

namespace gwasdev {

__device__ __forceinline__ void store_bits32(int8_t *dst, uint32_t x) {   // 32 bytes: +1 for the set bits of x, 0 elsewhere
    uint4 lo, hi;
    lo.x = spread4(x & 15u);         lo.y = spread4((x >> 4) & 15u);  lo.z = spread4((x >> 8) & 15u);  lo.w = spread4((x >> 12) & 15u);
    hi.x = spread4((x >> 16) & 15u); hi.y = spread4((x >> 20) & 15u); hi.z = spread4((x >> 24) & 15u); hi.w = spread4((x >> 28) & 15u);
    reinterpret_cast<uint4 *>(dst)[0] = lo;
    reinterpret_cast<uint4 *>(dst)[1] = hi;
}

// A operand from the device draws: one thread per permutation row, Knuth's selection sampling over the selected samples in
// increasing raw position (gwasdev_permutation_masks restates it on the host). Rows at or beyond n_perm are zero.
__global__ void perm_draw_kernel(const uint32_t *__restrict__ mca, const uint32_t *__restrict__ mco, uint32_t Wr, uint32_t n_sel,
                                 uint32_t n_case, uint64_t seed, uint64_t first_perm, uint64_t n_perm, uint64_t rows, uint32_t kbytes,
                                 int8_t *__restrict__ pa, uint32_t *__restrict__ ncase) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= rows) return;
    const bool live = k < n_perm;
    ncase[k] = live ? n_case : 0u;
    int8_t *row = pa + k * kbytes;
    uint32_t rank = 0, need = n_case;
    for (uint32_t w = 0; w < Wr; ++w) {
        uint32_t sel = live ? (__ldg(mca + w) | __ldg(mco + w)) : 0u, bits = 0;
        while (sel) {
            const int b = __ffs(sel) - 1;
            sel &= sel - 1;
            const uint64_t u = sim_hash(seed, first_perm + k, rank) >> 32, left = n_sel - rank;
            if (((u * left) >> 32) < need) { bits |= 1u << b; --need; }
            ++rank;
        }
        store_bits32(row + 32 * w, bits);
    }
}

// A operand from caller masks (P 16-bit blocks each, validated on the host): one thread per (row, 32-sample word)
__global__ void perm_masks_kernel(const uint16_t *__restrict__ masks, uint32_t P, uint32_t Wr, uint64_t n_perm, uint64_t rows,
                                  uint32_t kbytes, int8_t *__restrict__ pa) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * Wr) return;
    const uint64_t k = idx / Wr;
    const uint32_t w = (uint32_t)(idx - k * Wr);
    uint32_t bits = 0;
    if (k < n_perm) {
        const uint16_t *m = masks + k * P;
        if (2 * w < P) bits = m[2 * w];
        if (2 * w + 1 < P) bits |= (uint32_t)m[2 * w + 1] << 16;
    }
    store_bits32(pa + k * kbytes + 32 * w, bits);
}

// B operand: planes aa, bb (and xx) of SNPs [snp0, snp0 + n) as rows PL (s - snp0) + p, every sample position +1 when it has
// the genotype. xx is also set at the padding positions beyond sample N: A is zero there.
template <int PL>
__global__ void perm_planes_kernel(const uint32_t *__restrict__ raw, uint32_t Wr, uint64_t snp0, uint64_t n, uint32_t kbytes,
                                   int8_t *__restrict__ pb) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * Wr) return;
    const uint64_t snp = idx / Wr;
    const uint32_t w = (uint32_t)(idx - snp * Wr);
    const uint32_t *r = raw + (snp0 + snp) * 2ull * Wr;
    const uint32_t p1 = __ldg(r + w), p2 = __ldg(r + Wr + w);
    const uint32_t bb = p1 & p2, aa = p1 ^ bb;
    int8_t *dst = pb + PL * snp * kbytes + 32 * w;
    store_bits32(dst, aa);
    store_bits32(dst + kbytes, bb);
    if (PL == 3) store_bits32(dst + 2 * (uint64_t)kbytes, ~(p1 | p2));
}

// 1 into *flag when any of the first N samples of any row has no call
__global__ void any_missing_kernel(const uint32_t *__restrict__ raw, uint32_t Wr, uint32_t N, uint64_t M, int *flag) {
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < M * Wr; idx += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t snp = idx / Wr;
        const uint32_t w = (uint32_t)(idx - snp * Wr);
        const uint32_t valid = 32 * w >= N ? 0u : (32 * w + 32 <= N ? 0xffffffffu : (0xffffffffu >> (32 * w + 32 - N)));
        const uint32_t *r = raw + snp * 2ull * Wr;
        if (~(__ldg(r + w) | __ldg(r + Wr + w)) & valid) { *flag = 1; return; }
    }
}

// chi-square upper tail of the host-side p-value arithmetic (the same function on both sides of every EMP2 comparison)
static double chisq_q(double x, int df) { return x > 0.0 ? (df == 1 ? std::erfc(std::sqrt(0.5 * x)) : std::exp(-0.5 * x)) : 1.0; }

}  // namespace gwasdev

using namespace gwasdev;

// planes of SNPs [snp0, snp0 + n) into d_pb (rows from 0)
static int build_planes(gwasdev_store *s, int PL, uint64_t snp0, uint64_t n) {
    const uint32_t kbytes = 32 * s->Wr;
    GW_CUDA(reserve_raw(s->d_pb, s->cap_pb, (size_t)PL * n * kbytes));
    const uint64_t work = n * s->Wr;
    const unsigned blocks = (unsigned)((work + 255) / 256);
    if (PL == 3) perm_planes_kernel<3><<<blocks, 256, 0, s->stream>>>(s->d_raw, s->Wr, snp0, n, kbytes, s->d_pb);
    else perm_planes_kernel<2><<<blocks, 256, 0, s->stream>>>(s->d_raw, s->Wr, snp0, n, kbytes, s->d_pb);
    GW_LAUNCHED();
    return GWASDEV_OK;
}

// One GEMM launch: the A operand's n_perm permutations (rows of d_pa) x SNPs [i0, i0 + nsnp) of the call, whose B rows start
// at SNP b_snp0 of d_pb (pb_snps SNPs in d_pb).
static int launch_perm(gwasdev_store *s, int PL, PermParams p, uint64_t pa_rows, uint64_t pb_snps, std::vector<cudaEvent_t> &evs) {
    const uint32_t kbytes = 32 * s->Wr;
    CUtensorMap *maps = (CUtensorMap *)s->tmap_perm;
    int rc;
    if ((rc = encode_operand_map(s->d_pa, pa_rows, kbytes, PERM_BLK / 2, &maps[0])) != GWASDEV_OK) return rc;
    if ((rc = encode_operand_map(s->d_pb, (uint64_t)PL * pb_snps, kbytes, PSNP_HALF * PL, &maps[1])) != GWASDEV_OK) return rc;
    p.NKB = kbytes / MMA_KB;
    p.n_tiles = (uint64_t)p.n_pblk * ((p.nsnp + PSNP_BLK - 1) / PSNP_BLK);
    cudaEvent_t e0, e1;
    GW_CUDA(cudaEventCreate(&e0));
    evs.push_back(e0);
    GW_CUDA(cudaEventCreate(&e1));
    evs.push_back(e1);
    { const int rc = gwasdev_internal_perm_gemm(s, PL, p, maps, e0); if (rc != GWASDEV_OK) return rc; }
    GW_CUDA(cudaEventRecord(e1, s->stream));
    return GWASDEV_OK;
}

static int permute_body(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint64_t seed, uint64_t first_perm, uint64_t n_perm,
                        const uint16_t *case_masks, const std::vector<uint32_t> &mask_ncase, uint32_t *exceed, double *perm_max,
                        double *perm_stats, gwasdev_perm_stats *stats, int on_device, std::vector<cudaEvent_t> &evs) {
    const uint64_t n = snp_end - snp_begin;
    const uint32_t kbytes = 32 * s->Wr;
    cudaEvent_t t0, t1;
    GW_CUDA(cudaEventCreate(&t0));
    evs.push_back(t0);
    GW_CUDA(cudaEventCreate(&t1));
    evs.push_back(t1);
    GW_CUDA(cudaEventRecord(t0, s->stream));
    if (!s->tmap_perm && posix_memalign(&s->tmap_perm, 64, 2 * sizeof(CUtensorMap)) != 0) { s->tmap_perm = nullptr; set_error("out of host memory"); return GWASDEV_ENOMEM; }

    // observed statistics and pooled counts of the selection
    GW_CUDA(reserve(s->sc_out_counts, n * 8 * sizeof(uint32_t)));
    GW_CUDA(reserve(s->sc_out_stats, n * sizeof(gwasdev_snp_stats)));
    uint32_t *d_counts = (uint32_t *)s->sc_out_counts.p;
    gwasdev_snp_stats *d_obs = (gwasdev_snp_stats *)s->sc_out_stats.p;
    { const int rc = gwasdev_internal_scan(s, snp_begin, snp_end, d_counts, nullptr, d_obs); if (rc != GWASDEV_OK) return rc; }

    // outputs, accumulated by the kernels from zero
    GW_CUDA(reserve(s->sc_a, n * 2 * sizeof(uint32_t)));
    GW_CUDA(reserve(s->sc_b, n_perm * 3 * sizeof(double)));
    uint32_t *d_exceed = (uint32_t *)s->sc_a.p;
    unsigned long long *d_pmax = (unsigned long long *)s->sc_b.p;
    GW_CUDA(cudaMemsetAsync(d_exceed, 0, n * 2 * sizeof(uint32_t), s->stream));
    GW_CUDA(cudaMemsetAsync(d_pmax, 0, n_perm * 3 * sizeof(double), s->stream));

    // planes per SNP: three when the table has missing calls
    if (s->pb_missing < 0) {
        GW_CUDA(reserve(s->sc_cnt, 2 * sizeof(unsigned long long)));
        int *d_flag = (int *)s->sc_cnt.p;
        GW_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), s->stream));
        int sms = 0;
        GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
        any_missing_kernel<<<(unsigned)sms * 8, 256, 0, s->stream>>>(s->d_raw, s->Wr, s->N, s->M, d_flag);
        GW_LAUNCHED();
        int h = 0;
        GW_CUDA(cudaMemcpyAsync(&h, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
        GW_CUDA(cudaStreamSynchronize(s->stream));
        s->pb_missing = h;
    }
    const int PL = s->pb_missing ? 3 : 2;

    // B operand: resident over the whole table while it fits the budget, else one SNP chunk at a time
    size_t free_b = 0, total_b = 0;
    GW_CUDA(cudaMemGetInfo(&free_b, &total_b));
    uint64_t budget = s->opt[GWASDEV_OPT_PERM_OPERAND_BYTES] ? (uint64_t)s->opt[GWASDEV_OPT_PERM_OPERAND_BYTES] : (uint64_t)total_b / 4;
    const uint64_t snp_bytes = (uint64_t)PL * kbytes;
    bool resident = s->M * snp_bytes <= budget;
    uint64_t chunk = n;
    uint32_t built = 0;
    if (resident && !s->pb_resident) {
        const int rc = build_planes(s, PL, 0, s->M);
        if (rc == GWASDEV_ENOMEM) {              // the device is fuller than the budget assumed: chunks in half of what is free
            cudaGetLastError();
            GW_CUDA(cudaMemGetInfo(&free_b, &total_b));
            budget = free_b / 2;
            resident = false;
        } else if (rc != GWASDEV_OK) return rc;
        else { s->pb_resident = true; built = 1; }
    }
    if (!resident) {   // chunks of whole 64-SNP tiles: at least one, even when the budget is smaller
        s->pb_resident = false;
        chunk = std::max<uint64_t>(PSNP_BLK, budget / snp_bytes / PSNP_BLK * PSNP_BLK);
        built = 1;
    }

    // A operand: permutations in batches of PERM_BATCH
    const uint64_t batch = std::min<uint64_t>(n_perm, PERM_BATCH);
    const uint64_t pa_rows = (batch + PERM_BLK - 1) / PERM_BLK * PERM_BLK;
    GW_CUDA(reserve_raw(s->d_pa, s->cap_pa, (size_t)pa_rows * kbytes));
    GW_CUDA(reserve(s->sc_pi, pa_rows * sizeof(uint32_t)));
    uint32_t *d_ncase = (uint32_t *)s->sc_pi.p;
    if (case_masks) GW_CUDA(reserve(s->sc_pj, batch * s->P * sizeof(uint16_t)));
    const uint64_t n_batches = (n_perm + batch - 1) / batch, n_chunks = (n + chunk - 1) / chunk;
    auto build_a = [&](uint64_t b0, uint64_t nb) -> int {
        if (case_masks) {
            GW_CUDA(cudaMemcpyAsync(s->sc_pj.p, case_masks + b0 * s->P, nb * s->P * sizeof(uint16_t), cudaMemcpyHostToDevice, s->stream));
            std::vector<uint32_t> nc(pa_rows, 0);
            std::copy(mask_ncase.begin() + b0, mask_ncase.begin() + b0 + nb, nc.begin());
            GW_CUDA(cudaMemcpyAsync(d_ncase, nc.data(), pa_rows * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
            GW_CUDA(cudaStreamSynchronize(s->stream));   // nc goes out of scope
            const uint64_t work = pa_rows * s->Wr;
            perm_masks_kernel<<<(unsigned)((work + 255) / 256), 256, 0, s->stream>>>((const uint16_t *)s->sc_pj.p, s->P, s->Wr, nb, pa_rows, kbytes, s->d_pa);
        } else {
            perm_draw_kernel<<<(unsigned)((pa_rows + 127) / 128), 128, 0, s->stream>>>(s->d_case_sel_mask, s->d_ctrl_sel_mask, s->Wr, s->n_case + s->n_ctrl,
                                                                                        s->n_case, seed, first_perm + b0, nb, pa_rows, kbytes, s->d_pa, d_ncase);
        }
        GW_LAUNCHED();
        return GWASDEV_OK;
    };
    for (uint64_t c = 0; c < n_chunks; ++c) {
        const uint64_t c0 = c * chunk, cn = std::min(chunk, n - c0);
        if (!resident) { const int rc = build_planes(s, PL, snp_begin + c0, cn); if (rc != GWASDEV_OK) return rc; }
        for (uint64_t b = 0; b < n_batches; ++b) {
            const uint64_t b0 = b * batch, nb = std::min(batch, n_perm - b0);
            if (c == 0 || n_batches > 1) { const int rc = build_a(b0, nb); if (rc != GWASDEV_OK) return rc; }
            PermParams p = {};
            p.n_pblk = (uint32_t)((nb + PERM_BLK - 1) / PERM_BLK);
            p.b_snp0 = resident ? snp_begin + c0 : 0;
            p.n_perm = nb; p.i0 = c0; p.nsnp = cn; p.n_out = n;
            p.ncase = d_ncase; p.counts = d_counts; p.obs = d_obs; p.exceed = d_exceed; p.pmax = d_pmax + 3 * b0;
            p.pstats = perm_stats ? perm_stats + 2 * b0 * n : nullptr;
            const int rc = launch_perm(s, PL, p, pa_rows, resident ? s->M : cn, evs);
            if (rc != GWASDEV_OK) return rc;
        }
    }

    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (exceed) GW_CUDA(cudaMemcpyAsync(exceed, d_exceed, n * 2 * sizeof(uint32_t), kind, s->stream));
    if (perm_max) GW_CUDA(cudaMemcpyAsync(perm_max, d_pmax, n_perm * 3 * sizeof(double), kind, s->stream));
    GW_CUDA(cudaEventRecord(t1, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    if (stats) {
        float ms = 0.f;
        double gemm = 0.0;
        for (size_t e = 2; e + 1 < evs.size(); e += 2) { GW_CUDA(cudaEventElapsedTime(&ms, evs[e], evs[e + 1])); gemm += ms; }
        GW_CUDA(cudaEventElapsedTime(&ms, t0, t1));
        stats->n_perm = n_perm; stats->snps = n; stats->gemm_ms = gemm; stats->total_ms = ms;
        stats->planes = (uint32_t)PL; stats->built_operand = built;
    }
    return GWASDEV_OK;
}

extern "C" {

int gwasdev_marginal_permute(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint64_t seed, uint64_t first_perm, uint64_t n_perm,
                             const uint16_t *case_masks, uint32_t *exceed, double *perm_max, double *perm_stats, gwasdev_perm_stats *stats,
                             int on_device) {
    GW_REQUIRE(s != nullptr, "gwasdev_marginal_permute: NULL store");
    GW_REQUIRE(s->selected, "gwasdev_marginal_permute: call gwasdev_select_case_control first");
    GW_REQUIRE(snp_begin <= snp_end && snp_end <= s->M, "gwasdev_marginal_permute: bad SNP range [%llu, %llu)",
               (unsigned long long)snp_begin, (unsigned long long)snp_end);
    GW_REQUIRE(!perm_stats || on_device, "gwasdev_marginal_permute: perm_stats must be a device buffer");
    if (stats) *stats = gwasdev_perm_stats{};
    if (n_perm == 0 || snp_begin == snp_end) return GWASDEV_OK;
    const uint32_t n_sel = s->n_case + s->n_ctrl;
    std::vector<uint32_t> mask_ncase;
    if (case_masks) {   // each mask: a non-empty proper subset of the selection
        const std::vector<uint32_t> &m = s->h_sel_masks;   // [cases][controls-and-not-cases], Wr words each
        std::vector<uint16_t> sel16(s->P, 0);
        for (uint32_t b = 0; b < s->P; ++b)
            if (b / 2 < s->Wr) sel16[b] = (uint16_t)((m[b / 2] | m[s->Wr + b / 2]) >> (16 * (b & 1)));
        mask_ncase.resize(n_perm);
        for (uint64_t k = 0; k < n_perm; ++k) {
            uint32_t c = 0;
            for (uint32_t b = 0; b < s->P; ++b) {
                const uint16_t v = case_masks[k * s->P + b];
                GW_REQUIRE((v & ~sel16[b]) == 0, "gwasdev_marginal_permute: case mask %llu has samples outside the selection", (unsigned long long)k);
                c += (uint32_t)__builtin_popcount(v);
            }
            GW_REQUIRE(c >= 1 && c < n_sel, "gwasdev_marginal_permute: case mask %llu leaves a class empty", (unsigned long long)k);
            mask_ncase[k] = c;
        }
    } else GW_REQUIRE(s->n_case >= 1 && s->n_ctrl >= 1, "gwasdev_marginal_permute: the selection has an empty class");
    GW_CUDA(cudaSetDevice(s->device));
    std::vector<cudaEvent_t> evs;
    const int rc = permute_body(s, snp_begin, snp_end, seed, first_perm, n_perm, case_masks, mask_ncase, exceed, perm_max, perm_stats,
                                stats, on_device, evs);
    for (cudaEvent_t e : evs) cudaEventDestroy(e);
    return rc;
}

int gwasdev_permutation_masks(uint32_t n_samples, const uint16_t *case_mask, const uint16_t *ctrl_mask, uint64_t seed, uint64_t first_perm,
                              uint64_t n_perm, uint16_t *out) {
    GW_REQUIRE(case_mask && ctrl_mask && (out || n_perm == 0), "gwasdev_permutation_masks: NULL argument");
    const uint32_t P = plane_blocks(n_samples);
    std::vector<uint32_t> sel;   // selected sample positions, increasing
    uint32_t n_case = 0;
    for (uint32_t c = 0; c < n_samples; ++c) {
        const bool ca = (case_mask[c >> 4] >> (c & 15)) & 1u, co = (ctrl_mask[c >> 4] >> (c & 15)) & 1u;
        if (ca || co) sel.push_back(c);
        n_case += ca;
    }
    const uint32_t n_sel = (uint32_t)sel.size();
    for (uint64_t k = 0; k < n_perm; ++k) {
        uint16_t *o = out + k * P;
        std::fill(o, o + P, (uint16_t)0);
        uint32_t need = n_case;
        for (uint32_t rank = 0; rank < n_sel; ++rank) {
            const uint64_t u = sim_hash(seed, first_perm + k, rank) >> 32, left = n_sel - rank;
            if (((u * left) >> 32) < need) { o[sel[rank] >> 4] |= (uint16_t)(1u << (sel[rank] & 15)); --need; }
        }
    }
    return GWASDEV_OK;
}

int gwasdev_permutation_pvalues(uint64_t n_snps, uint64_t n_perm, const gwasdev_snp_stats *observed, const uint32_t *exceed,
                                const double *perm_max, double *emp1, double *emp2) {
    GW_REQUIRE(observed || !emp2, "gwasdev_permutation_pvalues: EMP2 needs the observed statistics");
    GW_REQUIRE(exceed || !emp1, "gwasdev_permutation_pvalues: EMP1 needs exceed");
    GW_REQUIRE(perm_max || !emp2 || n_perm == 0, "gwasdev_permutation_pvalues: EMP2 needs perm_max");
    const double denom = (double)n_perm + 1.0;
    if (emp1)
        for (uint64_t i = 0; i < 2 * n_snps; ++i) emp1[i] = ((double)exceed[i] + 1.0) / denom;
    if (!emp2) return GWASDEV_OK;
    std::vector<double> max_a(n_perm), minp(n_perm);
    for (uint64_t q = 0; q < n_perm; ++q) {
        max_a[q] = perm_max[3 * q];
        minp[q] = std::min(chisq_q(perm_max[3 * q + 1], 1), chisq_q(perm_max[3 * q + 2], 2));
    }
    std::sort(max_a.begin(), max_a.end());
    std::sort(minp.begin(), minp.end());
    for (uint64_t i = 0; i < n_snps; ++i) {
        const gwasdev_snp_stats &o = observed[i];
        const uint64_t ge = (uint64_t)(max_a.end() - std::lower_bound(max_a.begin(), max_a.end(), o.chi2_allelic));
        emp2[2 * i] = (1.0 + (double)ge) / denom;
        const int df = (int)o.df_genotypic;
        if (df == 0) { emp2[2 * i + 1] = 1.0; continue; }
        const uint64_t le = (uint64_t)(std::upper_bound(minp.begin(), minp.end(), chisq_q(o.chi2_genotypic, df)) - minp.begin());
        emp2[2 * i + 1] = (1.0 + (double)le) / denom;
    }
    return GWASDEV_OK;
}

}  // extern "C"
