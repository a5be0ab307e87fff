// The permutation test's GEMM kernel (see permute.cu for the formulation). Included by marginal.cu only: its epilogue computes
// the statistics with the scan's own out-of-line chi2_tests, so every (SNP, permutation) statistic is bit-identical to a
// scan of the permuted cohort.
#pragma once

#include "permute.cuh"

namespace gwasdev {

template <int PL> struct PermSmem {
    static constexpr int B_BYTES = PSNP_HALF * PL * MMA_KB;      // this CTA's half of B per 128-byte sample block
    static constexpr int KBB = A_STAGE_BYTES + B_BYTES;
    static constexpr int STG = KPS * KBB;
    static constexpr size_t BYTES = 1024 + (size_t)MMA_STAGES * STG + (2 * MMA_STAGES + 4 + 2 * SCHED_SLOTS) * sizeof(uint64_t) +
                                    SCHED_SLOTS * sizeof(uint2) + 16;
    static_assert(KBB % 1024 == 0 && BYTES <= 232448, "stage blocks keep the 1 KiB swizzle alignment; at most 227 KiB per CTA");
};

__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}

// running maximum of a non-negative double: the stored value only grows, so a stale read can only cost an extra atomic
__device__ __forceinline__ void push_max(unsigned long long *dst, double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    if (b > *reinterpret_cast<volatile unsigned long long *>(dst)) atomicMax(dst, b);
}

template <int PL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MMA_THREADS, 1)
perm_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const PermParams p) {
    using S = PermSmem<PL>;
    constexpr uint32_t IDESC = idesc_i8(PSNP_BLK * PL);
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (base - smem_u32(smem_raw));
    uint64_t *full = reinterpret_cast<uint64_t *>(sm + MMA_STAGES * S::STG);
    uint64_t *empty = full + MMA_STAGES;
    uint64_t *tfull = empty + MMA_STAGES;
    uint64_t *tempty = tfull + 2;
    uint64_t *sfull = tempty + 2;                      // tile feed, as in the pair screens
    uint64_t *sempty = sfull + SCHED_SLOTS;
    uint2 *sched = reinterpret_cast<uint2 *>(sempty + SCHED_SLOTS);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(sched + SCHED_SLOTS);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();

    if (tid == 0) {
        for (int s = 0; s < MMA_STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 2 * EPI_WARPS); }
        for (int b = 0; b < SCHED_SLOTS; ++b) { mbar_init(&sfull[b], 1); mbar_init(&sempty[b], SCHED_CONSUMERS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == TMA_WARP) {
        if (lane == 0) {
            uint64_t it = 0;
            uint32_t n_sched = 0;
            for (;;) {
                uint32_t I, J;
                if (rank == 0) {
                    // SNP-major order: consecutive tiles are the permutation blocks of one SNP block
                    const unsigned long long t = atomicAdd(p.tile_counter, 1ull);
                    const bool more = t < p.n_tiles;
                    I = more ? (uint32_t)(t % p.n_pblk) : 0u; J = more ? (uint32_t)(t / p.n_pblk) : 0u;
                    const int slot = (int)(n_sched % SCHED_SLOTS);
                    mbar_wait_wd(&sempty[slot], ((n_sched / SCHED_SLOTS) & 1u) ^ 1u);
                    sched_publish(sched, sfull, slot, more ? I : SCHED_END, J);
                    if (!more) break;
                    ++n_sched;
                } else if (!sched_next(sched, sfull, sempty, n_sched, I, J)) break;
                const int a_row = (int)((2 * I + rank) * (PERM_BLK / 2));
                const int b_row = (int)(PL * (p.b_snp0 + (uint64_t)J * PSNP_BLK + rank * PSNP_HALF));
                for (uint32_t kb = 0; kb < p.NKB; kb += KPS, ++it) {
                    const int st = (int)(it % MMA_STAGES);
                    const uint32_t nk = min((uint32_t)KPS, p.NKB - kb);
                    mbar_wait_wd(&empty[st], (uint32_t)(((it / MMA_STAGES) & 1) ^ 1));
                    unsigned char *dst = sm + st * S::STG;
                    if (rank == 0) mbar_expect_tx(&full[st], nk * 2 * (A_STAGE_BYTES + S::B_BYTES));
                    else mbar_arrive_remote(&full[st], 0);
                    for (uint32_t k2 = 0; k2 < nk; ++k2) {
                        tma_load_2d_pair(dst + k2 * S::KBB, &map_a, (int)((kb + k2) * MMA_KB), a_row, &full[st]);
                        tma_load_2d_pair(dst + k2 * S::KBB + A_STAGE_BYTES, &map_b, (int)((kb + k2) * MMA_KB), b_row, &full[st]);
                    }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0 && rank == 0) {
            uint64_t it = 0, tile_it = 0;
            uint32_t n_sched = 0, I, J;
            while (sched_next(sched, sfull, sempty, n_sched, I, J)) {
                const uint32_t buf = (uint32_t)(tile_it & 1);
                mbar_wait_wd(&tempty[buf], (uint32_t)(((tile_it >> 1) & 1) ^ 1));
                tc_fence_after();
                const uint32_t d_addr = tmem_base + buf * ACC_COLS;
                for (uint32_t kb = 0; kb < p.NKB; kb += KPS, ++it) {
                    const int st = (int)(it % MMA_STAGES);
                    const uint32_t nk = min((uint32_t)KPS, p.NKB - kb);
                    mbar_wait_wd(&full[st], (uint32_t)((it / MMA_STAGES) & 1));
                    tc_fence_after();
                    for (uint32_t k2 = 0; k2 < nk; ++k2) {
                        const uint32_t a_addr = base + st * S::STG + k2 * S::KBB, b_addr = a_addr + A_STAGE_BYTES;
                        const uint64_t ad = umma_desc(a_addr), bd = umma_desc(b_addr);
#pragma unroll
                        for (int k = 0; k < MMA_KB / UMMA_K; ++k)
                            tc_mma_i8(d_addr, ad + (uint64_t)(k * UMMA_K >> 4), bd + (uint64_t)(k * UMMA_K >> 4), IDESC, (kb + k2) != 0 || k != 0);
                    }
                    tc_commit_mc(&empty[st], 3);
                }
                tc_commit_mc(&tfull[buf], 3);
                ++tile_it;
            }
        }
    } else {
        // ===== epilogue (both CTAs): lane quadrant q = 32 permutations of this CTA's 128, column group g = 16 of the 64 SNPs =====
        const int q = warp & 3, g = warp >> 2;
        uint64_t tile_it = 0;
        uint32_t n_sched = 0, I, J;
        while (sched_next_warp(sched, sfull, sempty, lane, n_sched, I, J)) {
            const uint32_t buf = (uint32_t)(tile_it & 1);
            const uint64_t k = (uint64_t)I * PERM_BLK + rank * (PERM_BLK / 2) + 32 * q + lane;   // permutation of this lane
            const bool k_live = k < p.n_perm;
            const uint32_t nca = p.ncase[k];
            if (lane == 0) mbar_wait_wd(&tfull[buf], (uint32_t)((tile_it >> 1) & 1));
            __syncwarp();
            tc_fence_after();
            uint32_t v[2][32];
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + buf * ACC_COLS + PL * 16 * g;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if constexpr (PL == 3) tc_ld24(taddr + 24 * h, v[h]);
                else tc_ld16(taddr + 16 * h, v[h]);
            }
            tc_wait_ld();
            // the accumulator is in registers: hand it back before the fp64 work, so the MMAs run up to two tiles ahead
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(&tempty[buf], 0);
            double max_a = 0.0, max_g1 = 0.0, max_g2 = 0.0;
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const uint64_t loc = (uint64_t)J * PSNP_BLK + 16 * g + 8 * h + s;      // SNP of the chunk (warp-uniform)
                    if (loc >= p.nsnp) continue;
                    const uint64_t i = p.i0 + loc;
                    bool ge_a = false, ge_g = false;
                    if (k_live) {
                        const uint4 *c = reinterpret_cast<const uint4 *>(p.counts + 8 * i);
                        const uint4 c0 = __ldg(c), c1 = __ldg(c + 1);
                        const uint32_t aa = v[h][PL * s], bb = v[h][PL * s + 1], xx = PL == 3 ? v[h][PL * s + 2] : 0u;
                        uint32_t ca[4] = {aa, nca - aa - bb - xx, bb, xx};
                        uint32_t co[4] = {c0.x + c1.x - ca[0], c0.y + c1.y - ca[1], c0.z + c1.z - ca[2], c0.w + c1.w - ca[3]};
                        const Chi2 x = chi2_tests(ca, co);
                        const double xa = x.allelic, xg = x.genotypic;
                        ge_a = xa >= __ldg(&p.obs[i].chi2_allelic);
                        ge_g = xg >= __ldg(&p.obs[i].chi2_genotypic);
                        max_a = fmax(max_a, xa);
                        if (x.df == 1) max_g1 = fmax(max_g1, xg);
                        else if (x.df == 2) max_g2 = fmax(max_g2, xg);
                        if (p.pstats) *reinterpret_cast<double2 *>(p.pstats + 2 * (k * p.n_out + i)) = make_double2(xa, xg);
                    }
                    const uint32_t na = __popc(__ballot_sync(0xffffffffu, ge_a)), ng = __popc(__ballot_sync(0xffffffffu, ge_g));
                    if (lane == 0) {
                        if (na) atomicAdd(p.exceed + 2 * i, na);
                        if (ng) atomicAdd(p.exceed + 2 * i + 1, ng);
                    }
                }
            if (k_live) {
                push_max(p.pmax + 3 * k, max_a);
                push_max(p.pmax + 3 * k + 1, max_g1);
                push_max(p.pmax + 3 * k + 2, max_g2);
            }
            ++tile_it;
        }
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

int gwasdev_internal_perm_gemm(gwasdev_store *s, int PL, const PermParams &p, const CUtensorMap *maps, unsigned pairs) {
#define PERM_GEMM(PL_)                                                                                                    \
    do {                                                                                                                  \
        const size_t smem = PermSmem<PL_>::BYTES;                                                                         \
        GW_CUDA(cudaFuncSetAttribute(perm_gemm_kernel<PL_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));     \
        perm_gemm_kernel<PL_><<<2 * pairs, MMA_THREADS, smem, s->stream>>>(maps[0], maps[1], p);                         \
    } while (0)
    if (PL == 3) PERM_GEMM(3); else PERM_GEMM(2);
#undef PERM_GEMM
    GW_LAUNCHED();
    return GWASDEV_OK;
}

}  // namespace gwasdev
