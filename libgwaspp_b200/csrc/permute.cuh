// Permutation test (permute.cu): tile geometry and launch parameters of its tensor-core kernel, perm_gemm_kernel. The kernel
// itself (permute_gemm.cuh) is compiled in marginal.cu, whose chi2_tests its epilogue calls.
#pragma once

#include "mma_common.cuh"

namespace gwasdev {

constexpr int PERM_BLK = 2 * 2 * MMA_A_SNPS;     // permutations per tile: 128 A rows (TMEM lanes) per CTA
constexpr int PSNP_BLK = 64, PSNP_HALF = 32;     // SNPs per tile / staged by each CTA
constexpr uint64_t PERM_BATCH = 16384;           // permutations per A operand (160 MB at 10 000 samples)

struct PermParams {
    uint32_t NKB;                      // 128-byte sample blocks per row
    uint32_t n_pblk;                   // 256-permutation blocks of the A operand
    uint64_t n_tiles;
    uint64_t b_snp0;                   // B operand row block of the chunk's first SNP
    uint64_t n_perm;                   // live permutations of the A operand
    uint64_t i0, nsnp, n_out;          // call-relative index of the chunk's first SNP, SNPs of the chunk, SNPs of the call
    const uint32_t *ncase;             // [n_pblk * 256] cases per permutation (0 for the padding rows)
    const uint32_t *counts;            // [n_out][8] observed counts (cases aa ab bb xx, controls aa ab bb xx)
    const gwasdev_snp_stats *obs;      // [n_out] observed statistics
    uint32_t *exceed;                  // [n_out][2]
    unsigned long long *pmax;          // [n_perm][3] non-negative doubles as their (order-preserving) bit patterns
    double *pstats;                    // [n_perm][n_out][2] or nullptr
    unsigned long long *tile_counter;  // zero at launch
};

// launches perm_gemm_kernel<PL> on `pairs` CTA pairs over the A / B tensor maps maps[0], maps[1] (marginal.cu)
int gwasdev_internal_perm_gemm(gwasdev_store *s, int PL, const PermParams &p, const CUtensorMap *maps, unsigned pairs);

}  // namespace gwasdev
