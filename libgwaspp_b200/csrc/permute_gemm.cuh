// The permutation test's GEMM kernel (see permute.cu for the formulation). Included by marginal.cu only: its epilogue computes
// the statistics with the scan's own out-of-line chi2_tests, so every (SNP, permutation) statistic is bit-identical to a
// scan of the permuted cohort.
#pragma once

#include "permute.cuh"

namespace gwasdev {

template <int PL> struct PermSmem {
    static constexpr int KBB = A_STAGE_BYTES + PSNP_HALF * PL * MMA_KB;   // A rows, then this CTA's half of B, per 128-byte sample block
};
template <int PL> using PermPipe = CtaPipe<MMA_STAGES, KPS, PermSmem<PL>::KBB>;

// running maximum of a non-negative double: the stored value only grows, so a stale read can only cost an extra atomic
__device__ __forceinline__ void push_max(unsigned long long *dst, double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    if (b > *reinterpret_cast<volatile unsigned long long *>(dst)) atomicMax(dst, b);
}

template <int PL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MMA_THREADS, 1)
perm_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const PermParams p) {
    constexpr uint32_t IDESC = idesc_i8(PSNP_BLK * PL);
    extern __shared__ unsigned char smem_raw[];
    PermPipe<PL> pipe;
    pipe.setup(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = pipe.rank;
    const uint32_t tmem_base = pipe.tmem;

    if (warp == TMA_WARP) {
        // SNP-major order: consecutive tiles are the permutation blocks of one SNP block
        auto draw = [&](uint32_t &I, uint32_t &J) -> bool {
            const unsigned long long t = atomicAdd(p.tile_counter, 1ull);
            const bool more = t < p.n_tiles;
            I = more ? (uint32_t)(t % p.n_pblk) : 0u; J = more ? (uint32_t)(t / p.n_pblk) : 0u;
            return more;
        };
        auto load = [&](uint32_t I, uint32_t J, unsigned char *dst, uint32_t blk, uint64_t *full) {
            const int a_row = (int)((2 * I + rank) * (PERM_BLK / 2));
            const int b_row = (int)(PL * (p.b_snp0 + (uint64_t)J * PSNP_BLK + rank * PSNP_HALF));
            tma_load_2d_pair(dst, &map_a, (int)(blk * MMA_KB), a_row, full);
            tma_load_2d_pair(dst + A_STAGE_BYTES, &map_b, (int)(blk * MMA_KB), b_row, full);
        };
        pipe.produce(p.NKB, draw, load);
    } else if (warp == MMA_WARP) {
        pipe.issue(p.NKB, [&](uint32_t d_addr, uint32_t a_addr, uint32_t blk) {
            const uint64_t ad = umma_desc(a_addr), bd = umma_desc(a_addr + A_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < MMA_KB / UMMA_K; ++k)
                tc_mma_i8(d_addr, ad + (uint64_t)(k * UMMA_K >> 4), bd + (uint64_t)(k * UMMA_K >> 4), IDESC, blk != 0 || k != 0);
        });
    } else {
        // ===== epilogue (both CTAs): lane quadrant q = 32 permutations of this CTA's 128, column group g = 16 of the 64 SNPs =====
        const int q = warp & 3, g = warp >> 2;
        uint32_t I, J;
        for (uint32_t tile = 0; pipe.next_warp(lane, tile, I, J); ++tile) {
            const uint64_t k = (uint64_t)I * PERM_BLK + rank * (PERM_BLK / 2) + 32 * q + lane;   // permutation of this lane
            const bool k_live = k < p.n_perm;
            const uint32_t nca = p.ncase[k];
            const uint32_t buf = pipe.acc_wait(lane, tile);
            uint32_t v[2][32];
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + buf * ACC_COLS + PL * 16 * g;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if constexpr (PL == 3) tc_ld24(taddr + 24 * h, v[h]);
                else tc_ld16(taddr + 16 * h, v[h]);
            }
            tc_wait_ld();
            // the accumulator is in registers: hand it back before the fp64 work, so the MMAs run up to two tiles ahead
            pipe.acc_release(lane, buf);
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
        }
    }

    pipe.teardown();
}

int gwasdev_internal_perm_gemm(gwasdev_store *s, int PL, PermParams &p, const CUtensorMap *maps, cudaEvent_t start) {
    if (PL == 3) return launch_cta_pairs(s, perm_gemm_kernel<3>, PermPipe<3>::SMEM, p.n_tiles, p, nullptr, start, maps[0], maps[1]);
    return launch_cta_pairs(s, perm_gemm_kernel<2>, PermPipe<2>::SMEM, p.n_tiles, p, nullptr, start, maps[0], maps[1]);
}

}  // namespace gwasdev
