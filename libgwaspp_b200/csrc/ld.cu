// Windowed linkage disequilibrium (genotypic r^2, include/gwasdev.h) on the tensor cores.
//
// Formulation. Over a sample set S, SNP s gets int8 rows over the raw sample positions (0 outside S, for missing calls and at
// the padding): x = allele count (aa 0, ab 1, bb 2), and, when some sample of S has no call at some SNP, also c = 1 where called
// and q = x^2. The six sums of a pair are inner products of these rows: one int8 GEMM of the operand against itself (tcgen05.mma
// kind::i8, exact int32 sums), restricted to the band j - i <= window.
//   one row per SNP (no missing call in S): n = |S|, Sx / Sxx are per-SNP sums over S, the GEMM gives Sxy (one MAC per sample
//     and pair);
//   three rows per SNP: A-row type x against B rows (x, c) gives (Sxy, Sx), type c against (x, c, q) gives (Sy, n, Syy), type q
//     against c gives Sxx -- one MMA per A-row type into its own TMEM column range, so one TMEM lane holds one A-SNP with every
//     sum of its pairs and the epilogue needs no exchange between lanes (as in perm_gemm_kernel).
// The operand depends on the rows and S only: it stays resident for the S it was built for within GWASDEV_OPT_LD_OPERAND_BYTES,
// and is otherwise expanded one chunk of 256-SNP A-blocks at a time, together with the B-SNPs of their window.
//
// Kernel (ld_gemm_kernel): the CTA-pair pipeline of mma_common.cuh. A tile is 256 A-SNPs (128 TMEM lanes per CTA) x NB B-SNPs
// (256 for one row per SNP, 32 for three: six accumulator ranges of 32 columns each, double-buffered within the 512 TMEM
// columns). Band tiles (I, J), J from the diagonal block up to the last B-block within the window, are drawn from the device
// tile counter in A-block-major order. The epilogue discards what diagonal and edge tiles compute outside the band (j <= i,
// j - i > window), evaluates ld_stat (the one fp64 function every LD path calls) for every band pair, writes the band and
// appends the pairs at or above the threshold with one atomic per warp; the host sorts the list by (i, j).
#include <algorithm>
#include <cmath>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "mma_common.cuh"

namespace gwasdev {

constexpr int LD_A = 256;        // A-SNPs per tile: 128 per CTA (one operand row group)
constexpr int LD_GRP = 128;      // operand row group: three rows per SNP are stored [x 128][c 128][q 128] per group of 128 SNPs

template <int RT> struct LdCfg {                     // RT: operand rows per SNP (1 or 3)
    static constexpr int NB = RT == 1 ? 256 : 32;    // B-SNPs per tile
    static constexpr int KPS_ = RT == 1 ? 2 : 1;     // 128-byte sample blocks per stage
    static constexpr int STAGES = RT == 1 ? 3 : 4;
    static constexpr int A_BYTES = LD_GRP * RT * MMA_KB;     // per CTA and sample block
    static constexpr int KBB = A_BYTES + NB / 2 * RT * MMA_KB;   // A rows, then this CTA's half of B
    static_assert(6 * NB <= ACC_COLS || RT == 1, "six accumulator ranges per buffer");
};
template <int RT> using LdPipe = CtaPipe<LdCfg<RT>::STAGES, LdCfg<RT>::KPS_, LdCfg<RT>::KBB>;

struct LdParams {
    uint32_t NKB;                  // 128-byte sample blocks per row
    uint32_t nJ;                   // B-blocks per A-block in the schedule
    uint64_t n_tiles;              // A-blocks x nJ
    uint32_t I0;                   // first A-block (operand-relative)
    uint32_t nb_blocks;            // B-blocks of the operand
    uint64_t op0;                  // table row of operand SNP 0
    uint64_t lo, a_end, hi;        // pairs lo <= i < a_end, i < j < hi, j - i <= window
    uint32_t window;
    uint32_t n_all;                // |S| (one row per SNP)
    const uint2 *sums;             // [M] (Sx, Sxx) over S (one row per SNP)
    float *band;                   // or nullptr
    double r2_min;
    gwasdev_ld_pair *list;         // or nullptr (count only)
    unsigned long long cap;
    unsigned long long *n_list;
    unsigned long long *tile_counter;   // zero at launch
};

// The contract's arithmetic, shared by every LD path: exact int64 moments, fp64 without contraction.
__device__ __forceinline__ void ld_stat(uint32_t n, uint32_t sx, uint32_t sy, uint32_t sxx, uint32_t syy, uint32_t sxy, double &r, double &r2) {
    const int64_t num = (int64_t)n * sxy - (int64_t)sx * sy;
    const int64_t vx = (int64_t)n * sxx - (int64_t)sx * sx, vy = (int64_t)n * syy - (int64_t)sy * sy;
    if (vx == 0 || vy == 0) { r = r2 = __longlong_as_double(0x7ff8000000000000ll); return; }
    const double dn = __ll2double_rn(num), v = __dmul_rn(__ll2double_rn(vx), __ll2double_rn(vy));
    r2 = __ddiv_rn(__dmul_rn(dn, dn), v);
    r = __ddiv_rn(dn, __dsqrt_rn(v));
}

// one band pair of the epilogue: band entry, and a list record when r2 >= r2_min (one atomic per warp)
__device__ __forceinline__ void ld_emit(const LdParams &p, bool ok, uint64_t i, uint64_t j, uint32_t n, uint32_t sx, uint32_t sy,
                                        uint32_t sxx, uint32_t syy, uint32_t sxy, int lane) {
    double r = 0.0, r2 = 0.0;
    if (ok) {
        ld_stat(n, sx, sy, sxx, syy, sxy, r, r2);
        if (p.band) p.band[(i - p.lo) * p.window + (j - i - 1)] = (float)r2;
    }
    const bool keep = ok && r2 >= p.r2_min;
    const uint32_t m = __ballot_sync(0xffffffffu, keep);
    if (!m) return;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(p.n_list, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (keep && p.list) {
        const unsigned long long slot = base + __popc(m & ((1u << lane) - 1u));
        if (slot < p.cap) {
            gwasdev_ld_pair rec;
            rec.i = (uint32_t)i; rec.j = (uint32_t)j; rec.n = n; rec.reserved = 0; rec.r = r; rec.r2 = r2;
            p.list[slot] = rec;
        }
    }
}

template <int RT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MMA_THREADS, 1)
ld_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const LdParams p) {
    using S = LdCfg<RT>;
    constexpr int NB = S::NB;
    extern __shared__ unsigned char smem_raw[];
    LdPipe<RT> pipe;
    pipe.setup(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = pipe.rank;
    const uint32_t tmem_base = pipe.tmem;

    if (warp == TMA_WARP) {
        // A-block-major band order; tiles past the operand's last B-block are skipped
        auto draw = [&](uint32_t &I, uint32_t &J) -> bool {
            for (;;) {
                const unsigned long long t = atomicAdd(p.tile_counter, 1ull);
                if (t >= p.n_tiles) { I = J = 0; return false; }
                I = p.I0 + (uint32_t)(t / p.nJ);
                J = I * (LD_A / NB) + (uint32_t)(t % p.nJ);
                if (J < p.nb_blocks) return true;
            }
        };
        auto load = [&](uint32_t I, uint32_t J, unsigned char *d, uint32_t blk, uint64_t *full) {
            const uint32_t ga = 2 * I + rank;                                   // this CTA's A row group
            const uint32_t sb = J * NB + rank * (NB / 2);                      // first B-SNP of this CTA's half
            const int x = (int)(blk * MMA_KB);
            if constexpr (RT == 1) {
                tma_load_2d_pair(d, &map_a, x, (int)(ga * LD_GRP), full);
                tma_load_2d_pair(d + S::A_BYTES, &map_b, x, (int)sb, full);
            } else {
                const uint32_t gb = sb / LD_GRP, rb = sb % LD_GRP;
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    tma_load_2d_pair(d + t * LD_GRP * MMA_KB, &map_a, x, (int)((3 * ga + t) * LD_GRP), full);
                    tma_load_2d_pair(d + S::A_BYTES + t * (NB / 2) * MMA_KB, &map_b, x, (int)((3 * gb + t) * LD_GRP + rb), full);
                }
            }
        };
        pipe.produce(p.NKB, draw, load);
    } else if (warp == MMA_WARP) {
        pipe.issue(p.NKB, [&](uint32_t d_addr, uint32_t a_addr, uint32_t blk) {
            const uint32_t b_addr = a_addr + S::A_BYTES;
#pragma unroll
            for (int k = 0; k < MMA_KB / UMMA_K; ++k) {
                const uint32_t acc = blk != 0 || k != 0;
                const uint64_t ko = (uint64_t)(k * UMMA_K >> 4);
                if constexpr (RT == 1) {
                    tc_mma_i8(d_addr, umma_desc(a_addr) + ko, umma_desc(b_addr) + ko, idesc_i8(NB), acc);
                } else {
                    // per CTA, B holds [x 16][c 16][q 16]: x x (x, c), c x (x, c, q), q x c
                    tc_mma_i8(d_addr, umma_desc(a_addr) + ko, umma_desc(b_addr) + ko, idesc_i8(2 * NB), acc);
                    tc_mma_i8(d_addr + 2 * NB, umma_desc(a_addr + LD_GRP * MMA_KB) + ko, umma_desc(b_addr) + ko, idesc_i8(3 * NB), acc);
                    tc_mma_i8(d_addr + 5 * NB, umma_desc(a_addr + 2 * LD_GRP * MMA_KB) + ko,
                              umma_desc(b_addr + (NB / 2) * MMA_KB) + ko, idesc_i8(NB), acc);
                }
            }
        });
    } else {
        // ===== epilogue (both CTAs): lane quadrant q = 32 A-SNPs of this CTA's 128, column group g = a quarter of the B-SNPs =====
        const int q = warp & 3, g = warp >> 2;
        uint32_t I, J;
        for (uint32_t tile = 0; pipe.next_warp(lane, tile, I, J); ++tile) {
            const uint64_t i = p.op0 + (uint64_t)I * LD_A + rank * LD_GRP + 32 * q + lane;   // A-SNP of this lane
            const bool i_live = i >= p.lo && i < p.a_end;
            const uint64_t iw = i - lane;                                   // the warp's A-SNPs are iw .. iw + 31
            // B-SNPs [j0, j0 + nj) hold no band pair of this warp
            auto outside = [&](uint64_t j0, uint32_t nj) {
                return j0 + nj - 1 <= iw || j0 > iw + 31 + p.window || j0 >= p.hi || iw >= p.a_end || iw + 31 < p.lo;
            };
            const uint32_t buf = pipe.acc_wait(lane, tile);
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + buf * ACC_COLS;
            if constexpr (RT == 1) {
                uint2 si = make_uint2(0, 0);
                if (i_live) si = __ldg(p.sums + i);
                uint32_t v[16];
#pragma unroll 1
                for (int h = 0; h < 4; ++h) {                      // 64 B-SNPs per warp, 16 at a time
                    const int c0 = 64 * g + 16 * h;
                    tc_ld8(taddr + c0, v);
                    tc_ld8(taddr + c0 + 8, v + 8);
                    tc_wait_ld();
                    if (h == 3) pipe.acc_release(lane, buf);       // the accumulator is in registers: hand it back before the fp64 work
                    const uint64_t j0 = p.op0 + (uint64_t)J * NB + c0;
                    if (outside(j0, 16)) continue;
#pragma unroll
                    for (int b = 0; b < 16; ++b) {
                        const uint64_t j = j0 + b;
                        const bool ok = i_live && j > i && j < p.hi && j - i <= p.window;
                        uint2 sj = make_uint2(0, 0);
                        if (j < p.hi) sj = __ldg(p.sums + j);
                        ld_emit(p, ok, i, j, p.n_all, si.x, sj.x, si.y, sj.y, v[b], lane);
                    }
                }
            } else {
                const int h = g >> 1, o = 8 * (g & 1);            // CTA half of the eight B-SNPs, offset inside it
                uint32_t xy[8], xc[8], cx[8], cc[8], cq[8], qc[8];
                tc_ld8(taddr + 32 * h + o, xy);
                tc_ld8(taddr + 32 * h + 16 + o, xc);
                tc_ld8(taddr + 2 * NB + 48 * h + o, cx);
                tc_ld8(taddr + 2 * NB + 48 * h + 16 + o, cc);
                tc_ld8(taddr + 2 * NB + 48 * h + 32 + o, cq);
                tc_ld8(taddr + 5 * NB + 16 * h + o, qc);
                tc_wait_ld();
                pipe.acc_release(lane, buf);
                const uint64_t j0 = p.op0 + (uint64_t)J * NB + 16 * h + o;
                if (outside(j0, 8)) continue;
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const uint64_t j = j0 + b;
                    const bool ok = i_live && j > i && j < p.hi && j - i <= p.window;
                    ld_emit(p, ok, i, j, cc[b], xc[b], cx[b], qc[b], cq[b], xy[b], lane);
                }
            }
        }
    }

    pipe.teardown();
}

// 32 bytes lo_bit + k * hi_bit for the 32 samples of one word
__device__ __forceinline__ void store_count32(int8_t *dst, uint32_t lo, uint32_t hi, uint32_t k) {
    uint32_t b[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) b[t] = spread4((lo >> (4 * t)) & 15u) + k * spread4((hi >> (4 * t)) & 15u);
    reinterpret_cast<uint4 *>(dst)[0] = make_uint4(b[0], b[1], b[2], b[3]);
    reinterpret_cast<uint4 *>(dst)[1] = make_uint4(b[4], b[5], b[6], b[7]);
}

// operand rows of table SNPs [snp0, snp0 + n), zero for the padding SNPs up to n_pad; one thread per (SNP, 32-sample word)
template <int RT>
__global__ void ld_operand_kernel(const uint32_t *__restrict__ raw, const uint32_t *__restrict__ mask, uint32_t Wr, uint64_t snp0,
                                  uint64_t n, uint64_t n_pad, uint32_t kbytes, int8_t *__restrict__ op) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_pad * Wr) return;
    const uint64_t snp = idx / Wr;
    const uint32_t w = (uint32_t)(idx - snp * Wr);
    uint32_t het = 0, hom = 0, called = 0;
    if (snp < n) {
        const uint32_t *r = raw + (snp0 + snp) * 2ull * Wr;
        const uint32_t p1 = __ldg(r + w), p2 = __ldg(r + Wr + w), m = __ldg(mask + w);
        het = p2 & ~p1 & m; hom = p1 & p2 & m; called = (p1 | p2) & m;
    }
    if (RT == 1) {
        store_count32(op + snp * kbytes + 32 * w, het, hom, 2);
    } else {
        int8_t *d = op + ((snp / LD_GRP) * 3 * LD_GRP + snp % LD_GRP) * (uint64_t)kbytes + 32 * w;
        store_count32(d, het, hom, 2);
        store_count32(d + (uint64_t)LD_GRP * kbytes, called, 0, 0);
        store_count32(d + 2ull * LD_GRP * kbytes, het, hom, 4);
    }
}

// per SNP (Sx, Sxx) over S, and *missing = 1 when some sample of S has no call: one warp per SNP
__global__ void ld_sums_kernel(const uint32_t *__restrict__ raw, const uint32_t *__restrict__ mask, uint32_t Wr, uint64_t M,
                               uint2 *__restrict__ sums, int *missing) {
    const uint64_t snp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (snp >= M) return;
    const uint32_t *r = raw + snp * 2ull * Wr;
    uint32_t sx = 0, sxx = 0, miss = 0;
    for (uint32_t w = lane; w < Wr; w += 32) {
        const uint32_t p1 = __ldg(r + w), p2 = __ldg(r + Wr + w), m = __ldg(mask + w);
        const uint32_t het = __popc(p2 & ~p1 & m), hom = __popc(p1 & p2 & m);
        sx += het + 2 * hom; sxx += het + 4 * hom;
        miss |= ~(p1 | p2) & m;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        sx += __shfl_xor_sync(0xffffffffu, sx, o);
        sxx += __shfl_xor_sync(0xffffffffu, sxx, o);
        miss |= __shfl_xor_sync(0xffffffffu, miss, o);
    }
    if (lane == 0) {
        sums[snp] = make_uint2(sx, sxx);
        if (miss) *missing = 1;
    }
}

// gwasdev_ld_pairs: the six sums of given pairs from the raw rows, one warp per pair
__global__ void ld_pairs_kernel(const uint32_t *__restrict__ raw, const uint32_t *__restrict__ mask, uint32_t Wr, uint64_t n,
                                const uint32_t *__restrict__ pi, const uint32_t *__restrict__ pj, gwasdev_ld_pair *__restrict__ out) {
    const uint64_t k = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= n) return;
    const uint32_t i = min(pi[k], pj[k]), j = max(pi[k], pj[k]);
    const uint32_t *a = raw + (uint64_t)i * 2 * Wr, *b = raw + (uint64_t)j * 2 * Wr;
    uint32_t s[6] = {0, 0, 0, 0, 0, 0};   // n, Sx, Sy, Sxx, Syy, Sxy
    for (uint32_t w = lane; w < Wr; w += 32) {
        const uint32_t m = __ldg(mask + w);
        const uint32_t a1 = __ldg(a + w), a2 = __ldg(a + Wr + w), b1 = __ldg(b + w), b2 = __ldg(b + Wr + w);
        const uint32_t ca = (a1 | a2) & m, cb = (b1 | b2) & m, ha = a2 & ~a1, ba = a1 & a2, hb = b2 & ~b1, bb = b1 & b2;
        const uint32_t both = ca & cb;
        const uint32_t nha = __popc(ha & both), nba = __popc(ba & both), nhb = __popc(hb & both), nbb = __popc(bb & both);
        s[0] += __popc(both);
        s[1] += nha + 2 * nba; s[2] += nhb + 2 * nbb;
        s[3] += nha + 4 * nba; s[4] += nhb + 4 * nbb;
        s[5] += __popc(ha & hb & both) + 2 * (__popc(ha & bb & both) + __popc(ba & hb & both)) + 4 * __popc(ba & bb & both);
    }
#pragma unroll
    for (int t = 0; t < 6; ++t)
#pragma unroll
        for (int o = 16; o; o >>= 1) s[t] += __shfl_xor_sync(0xffffffffu, s[t], o);
    if (lane == 0) {
        gwasdev_ld_pair rec;
        rec.i = i; rec.j = j; rec.n = s[0]; rec.reserved = 0;
        ld_stat(s[0], s[1], s[2], s[3], s[4], s[5], rec.r, rec.r2);
        out[k] = rec;
    }
}

__global__ void ld_keys_kernel(const gwasdev_ld_pair *__restrict__ list, uint64_t n, unsigned long long *__restrict__ keys, uint32_t *__restrict__ idx) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    keys[k] = ((unsigned long long)list[k].i << 32) | list[k].j;
    idx[k] = (uint32_t)k;
}

__global__ void ld_gather_kernel(const gwasdev_ld_pair *__restrict__ list, uint64_t n, const uint32_t *__restrict__ idx, gwasdev_ld_pair *__restrict__ out) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = list[idx[k]];
}

}  // namespace gwasdev

using namespace gwasdev;

// S as [Wr] words from P 16-bit blocks (NULL: every sample); bits at or beyond N are refused
static int mask_of(const gwasdev_store *s, const uint16_t *sample_mask, const char *fn, std::vector<uint32_t> &out) {
    out.assign(s->Wr, 0u);
    for (uint32_t c = 0; c < s->P * 16; ++c) {
        const bool in = sample_mask ? ((sample_mask[c >> 4] >> (c & 15)) & 1u) : c < s->N;
        if (!in) continue;
        GW_REQUIRE(c < s->N, "%s: sample_mask has bits at or beyond sample %u", fn, s->N);
        out[c >> 5] |= 1u << (c & 31);
    }
    return GWASDEV_OK;
}

static bool is_device_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice;
}

// per-SNP sums and the missing-call flag of S (cached with S; a new S drops the resident operand)
static int ensure_sums(gwasdev_store *s, const std::vector<uint32_t> &hm) {
    if (s->ld_sums_valid && s->h_ld_mask == hm) return GWASDEV_OK;
    s->ld_sums_valid = s->ld_resident = false;
    if (!s->d_ld_mask) GW_CUDA(cudaMalloc(&s->d_ld_mask, s->Wr * sizeof(uint32_t)));
    if (!s->d_ld_sums) GW_CUDA(cudaMalloc(&s->d_ld_sums, std::max<uint64_t>(1, s->M) * sizeof(uint2)));
    GW_CUDA(cudaMemcpyAsync(s->d_ld_mask, hm.data(), s->Wr * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    GW_CUDA(reserve(s->sc_cnt, 2 * sizeof(unsigned long long)));
    int *d_flag = (int *)s->sc_cnt.p;
    GW_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), s->stream));
    ld_sums_kernel<<<(unsigned)((s->M * 32 + 255) / 256), 256, 0, s->stream>>>(s->d_raw, s->d_ld_mask, s->Wr, s->M, s->d_ld_sums, d_flag);
    GW_LAUNCHED();
    int h = 0;
    GW_CUDA(cudaMemcpyAsync(&h, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    s->ld_missing = h;
    s->h_ld_mask = hm;
    s->ld_sums_valid = true;
    return GWASDEV_OK;
}

static uint64_t ld_pad(uint64_t n) { return (n + LD_A - 1) / LD_A * LD_A; }

// operand of table SNPs [snp0, snp0 + n) into d_ld (SNPs padded to whole 256-SNP blocks)
static int build_operand(gwasdev_store *s, int RT, uint64_t snp0, uint64_t n) {
    const uint32_t kbytes = 32 * s->Wr;
    const uint64_t n_pad = ld_pad(n);
    GW_CUDA(reserve_raw(s->d_ld, s->cap_ld, (size_t)RT * n_pad * kbytes));
    const uint64_t work = n_pad * s->Wr;
    const unsigned blocks = (unsigned)((work + 255) / 256);
    if (RT == 3) ld_operand_kernel<3><<<blocks, 256, 0, s->stream>>>(s->d_raw, s->d_ld_mask, s->Wr, snp0, n, n_pad, kbytes, s->d_ld);
    else ld_operand_kernel<1><<<blocks, 256, 0, s->stream>>>(s->d_raw, s->d_ld_mask, s->Wr, snp0, n, n_pad, kbytes, s->d_ld);
    GW_LAUNCHED();
    return GWASDEV_OK;
}

// one GEMM launch over A-SNPs [a0, a_end) of the operand in d_ld, whose SNP 0 is table row op0 and which holds op_snps SNPs
static int launch_ld(gwasdev_store *s, int RT, LdParams p, uint64_t a0, uint64_t op_snps, std::vector<cudaEvent_t> &evs) {
    const uint32_t kbytes = 32 * s->Wr;
    const int NB = RT == 1 ? LdCfg<1>::NB : LdCfg<3>::NB;
    CUtensorMap *maps = (CUtensorMap *)s->tmap_ld;
    const uint64_t rows = (uint64_t)RT * ld_pad(op_snps);
    int rc;
    if ((rc = encode_operand_map(s->d_ld, rows, kbytes, LD_GRP, &maps[0])) != GWASDEV_OK) return rc;
    if ((rc = encode_operand_map(s->d_ld, rows, kbytes, NB / 2, &maps[1])) != GWASDEV_OK) return rc;
    const uint64_t w_eff = std::min<uint64_t>(p.window, p.hi - p.lo);
    p.NKB = kbytes / MMA_KB;
    p.I0 = (uint32_t)((a0 - p.op0) / LD_A);
    const uint64_t nI = (p.a_end - 1 - p.op0) / LD_A - p.I0 + 1;
    p.nb_blocks = (uint32_t)((std::min(op_snps, p.hi - p.op0) + NB - 1) / NB);   // B-blocks up to the last j
    p.nJ = (uint32_t)std::min<uint64_t>((LD_A - 1 + w_eff) / NB + 1, p.nb_blocks);
    p.n_tiles = nI * p.nJ;
    cudaEvent_t e0, e1;
    GW_CUDA(cudaEventCreate(&e0));
    evs.push_back(e0);
    GW_CUDA(cudaEventCreate(&e1));
    evs.push_back(e1);
    rc = RT == 3 ? launch_cta_pairs(s, ld_gemm_kernel<3>, LdPipe<3>::SMEM, p.n_tiles, p, nullptr, e0, maps[0], maps[1])
                 : launch_cta_pairs(s, ld_gemm_kernel<1>, LdPipe<1>::SMEM, p.n_tiles, p, nullptr, e0, maps[0], maps[1]);
    if (rc != GWASDEV_OK) return rc;
    GW_CUDA(cudaEventRecord(e1, s->stream));
    return GWASDEV_OK;
}

static int ld_window_body(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t window, const std::vector<uint32_t> &hm,
                          double r2_threshold, gwasdev_ld_pair *pairs, uint64_t capacity, uint64_t *n_pairs, float *band,
                          gwasdev_ld_stats *stats, int on_device, std::vector<cudaEvent_t> &evs) {
    const uint64_t n = snp_end - snp_begin;
    const uint32_t kbytes = 32 * s->Wr;
    cudaEvent_t t0, t1;
    GW_CUDA(cudaEventCreate(&t0));
    evs.push_back(t0);
    GW_CUDA(cudaEventCreate(&t1));
    evs.push_back(t1);
    GW_CUDA(cudaEventRecord(t0, s->stream));
    if (!s->tmap_ld && posix_memalign(&s->tmap_ld, 64, 2 * sizeof(CUtensorMap)) != 0) { s->tmap_ld = nullptr; set_error("out of host memory"); return GWASDEV_ENOMEM; }
    { const int rc = ensure_sums(s, hm); if (rc != GWASDEV_OK) return rc; }
    const int RT = s->ld_missing ? 3 : 1;
    uint32_t n_all = 0;
    for (uint32_t w : hm) n_all += (uint32_t)__builtin_popcount(w);

    // outputs: the band starts as NaN everywhere; the list goes to scratch and is sorted at the end
    const uint64_t band_n = n * (uint64_t)window;
    float *d_band = nullptr;
    if (band) {
        if (on_device) d_band = band;
        else { GW_CUDA(reserve(s->sc_b, band_n * sizeof(float))); d_band = (float *)s->sc_b.p; }
        GW_CUDA(cudaMemsetAsync(d_band, 0xff, band_n * sizeof(float), s->stream));
    }
    GW_CUDA(reserve(s->sc_cnt, 2 * sizeof(unsigned long long)));
    unsigned long long *d_nlist = (unsigned long long *)s->sc_cnt.p;
    GW_CUDA(cudaMemsetAsync(d_nlist, 0, sizeof(unsigned long long), s->stream));
    gwasdev_ld_pair *d_list = nullptr;
    if (pairs && capacity) { GW_CUDA(reserve(s->sc_cand, capacity * sizeof(gwasdev_ld_pair))); d_list = (gwasdev_ld_pair *)s->sc_cand.p; }

    // operand: resident over the whole table for S while it fits the budget, else chunks of whole A-blocks plus their window
    size_t free_b = 0, total_b = 0;
    GW_CUDA(cudaMemGetInfo(&free_b, &total_b));
    uint64_t budget = s->opt[GWASDEV_OPT_LD_OPERAND_BYTES] ? (uint64_t)s->opt[GWASDEV_OPT_LD_OPERAND_BYTES] : (uint64_t)total_b / 4;
    const uint64_t snp_bytes = (uint64_t)RT * kbytes;
    bool resident = ld_pad(s->M) * snp_bytes <= budget;
    uint32_t built = 0;
    if (resident && !s->ld_resident) {
        const int rc = build_operand(s, RT, 0, s->M);
        if (rc == GWASDEV_ENOMEM) {             // the device is fuller than the budget assumed: chunks in half of what is free
            cudaGetLastError();
            GW_CUDA(cudaMemGetInfo(&free_b, &total_b));
            budget = free_b / 2;
            resident = false;
        } else if (rc != GWASDEV_OK) return rc;
        else { s->ld_resident = true; built = 1; }
    }
    LdParams p = {};
    p.lo = snp_begin; p.hi = snp_end; p.window = window; p.n_all = n_all; p.sums = s->d_ld_sums; p.band = d_band;
    p.r2_min = r2_threshold; p.list = d_list; p.cap = d_list ? capacity : 0; p.n_list = d_nlist;
    const uint64_t w_eff = std::min<uint64_t>(window, n);
    if (resident) {
        p.op0 = 0; p.a_end = snp_end;
        const int rc = launch_ld(s, RT, p, snp_begin / LD_A * LD_A, s->M, evs);
        if (rc != GWASDEV_OK) return rc;
    } else {   // chunks of whole 256-SNP A-blocks: at least one, even when the budget is smaller
        s->ld_resident = false;
        built = 1;
        const uint64_t fit = budget / snp_bytes;
        const uint64_t chunk = std::max<uint64_t>(LD_A, fit > w_eff + LD_A ? (fit - w_eff) / LD_A * LD_A : LD_A);
        for (uint64_t a0 = snp_begin; a0 < snp_end; a0 += chunk) {
            const uint64_t a_end = std::min(a0 + chunk, snp_end), op_n = std::min(a_end + w_eff, snp_end) - a0;
            { const int rc = build_operand(s, RT, a0, op_n); if (rc != GWASDEV_OK) return rc; }
            p.op0 = a0; p.a_end = a_end;
            const int rc = launch_ld(s, RT, p, a0, op_n, evs);
            if (rc != GWASDEV_OK) return rc;
        }
    }

    unsigned long long found = 0;
    GW_CUDA(cudaMemcpyAsync(&found, d_nlist, sizeof(found), cudaMemcpyDeviceToHost, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (band && !on_device) GW_CUDA(cudaMemcpyAsync(band, d_band, band_n * sizeof(float), kind, s->stream));
    if (n_pairs) *n_pairs = found;
    if (pairs && found > capacity) {
        GW_CUDA(cudaStreamSynchronize(s->stream));
        set_error("gwasdev_ld_window: %llu pairs qualify, capacity %llu", found, (unsigned long long)capacity);
        return GWASDEV_EOVERFLOW;
    }
    if (pairs && found) {   // sort by (i, j)
        GW_CUDA(reserve(s->sc_keys, found * 8));
        GW_CUDA(reserve(s->sc_keys2, found * 8));
        GW_CUDA(reserve(s->sc_vals, found * 4));
        GW_CUDA(reserve(s->sc_vals2, found * 4));
        unsigned long long *kin = (unsigned long long *)s->sc_keys.p, *kout = (unsigned long long *)s->sc_keys2.p;
        uint32_t *vin = (uint32_t *)s->sc_vals.p, *vout = (uint32_t *)s->sc_vals2.p;
        const unsigned g = (unsigned)((found + 255) / 256);
        ld_keys_kernel<<<g, 256, 0, s->stream>>>(d_list, found, kin, vin);
        GW_LAUNCHED();
        size_t tmp = 0;
        GW_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, kin, kout, vin, vout, (int64_t)found, 0, 64, s->stream));
        GW_CUDA(reserve(s->sc_sort, tmp));
        GW_CUDA(cub::DeviceRadixSort::SortPairs(s->sc_sort.p, tmp, kin, kout, vin, vout, (int64_t)found, 0, 64, s->stream));
        gwasdev_ld_pair *d_out = pairs;
        if (!on_device) { GW_CUDA(reserve(s->sc_hits, found * sizeof(gwasdev_ld_pair))); d_out = (gwasdev_ld_pair *)s->sc_hits.p; }
        ld_gather_kernel<<<g, 256, 0, s->stream>>>(d_list, found, vout, d_out);
        GW_LAUNCHED();
        if (!on_device) GW_CUDA(cudaMemcpyAsync(pairs, d_out, found * sizeof(gwasdev_ld_pair), kind, s->stream));
    }
    GW_CUDA(cudaEventRecord(t1, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    if (stats) {
        float ms = 0.f;
        double gemm = 0.0;
        for (size_t e = 2; e + 1 < evs.size(); e += 2) { GW_CUDA(cudaEventElapsedTime(&ms, evs[e], evs[e + 1])); gemm += ms; }
        GW_CUDA(cudaEventElapsedTime(&ms, t0, t1));
        const uint64_t w1 = std::min<uint64_t>(window, n - 1), tested = (n - w1) * w1 + w1 * (w1 - 1) / 2;   // sum over i of min(window, snp_end - 1 - i)
        stats->pairs_tested = tested; stats->pairs_kept = found; stats->gemm_ms = gemm; stats->total_ms = ms;
        stats->rows_per_snp = (uint32_t)RT; stats->built_operand = built;
    }
    return GWASDEV_OK;
}

extern "C" {

int gwasdev_ld_window(gwasdev_store *s, uint64_t snp_begin, uint64_t snp_end, uint32_t window, const uint16_t *sample_mask,
                      double r2_threshold, gwasdev_ld_pair *pairs, uint64_t capacity, uint64_t *n_pairs, float *band,
                      gwasdev_ld_stats *stats, int on_device) {
    GW_REQUIRE(s != nullptr, "gwasdev_ld_window: NULL store");
    GW_REQUIRE(window >= 1, "gwasdev_ld_window: window must be at least 1");
    GW_REQUIRE(snp_begin <= snp_end && snp_end <= s->M, "gwasdev_ld_window: bad SNP range [%llu, %llu)",
               (unsigned long long)snp_begin, (unsigned long long)snp_end);
    GW_REQUIRE(!pairs || n_pairs, "gwasdev_ld_window: pairs needs n_pairs");
    GW_REQUIRE(capacity <= 0xffffffffull, "gwasdev_ld_window: capacity above 2^32 - 1");
    GW_REQUIRE(on_device || (!is_device_ptr(pairs) && !is_device_ptr(band)), "gwasdev_ld_window: device buffers with on_device = 0");
    std::vector<uint32_t> hm;
    { const int rc = mask_of(s, sample_mask, "gwasdev_ld_window", hm); if (rc != GWASDEV_OK) return rc; }
    if (stats) *stats = gwasdev_ld_stats{};
    if (n_pairs) *n_pairs = 0;
    if (snp_end - snp_begin < 2) {   // no pair: the band (one row at most) is all NaN
        if (band && snp_end > snp_begin) {
            if (on_device) GW_CUDA(cudaMemsetAsync(band, 0xff, window * sizeof(float), s->stream));
            else std::fill(band, band + window, std::nanf(""));
        }
        return GWASDEV_OK;
    }
    GW_CUDA(cudaSetDevice(s->device));
    std::vector<cudaEvent_t> evs;
    const int rc = ld_window_body(s, snp_begin, snp_end, window, hm, r2_threshold, pairs, capacity, n_pairs, band, stats, on_device, evs);
    for (cudaEvent_t e : evs) cudaEventDestroy(e);
    return rc;
}

int gwasdev_ld_pairs(gwasdev_store *s, uint64_t n, const uint32_t *pi, const uint32_t *pj, const uint16_t *sample_mask, gwasdev_ld_pair *out) {
    GW_REQUIRE(s != nullptr, "gwasdev_ld_pairs: NULL store");
    if (n == 0) return GWASDEV_OK;
    GW_REQUIRE(pi && pj && out, "gwasdev_ld_pairs: NULL argument");
    GW_REQUIRE(!is_device_ptr(pi) && !is_device_ptr(pj) && !is_device_ptr(out) && !is_device_ptr(sample_mask),
               "gwasdev_ld_pairs: host buffers only");
    for (uint64_t k = 0; k < n; ++k)
        GW_REQUIRE(pi[k] < s->M && pj[k] < s->M && pi[k] != pj[k], "gwasdev_ld_pairs: bad pair %llu (%u, %u)", (unsigned long long)k, pi[k], pj[k]);
    std::vector<uint32_t> hm;
    { const int rc = mask_of(s, sample_mask, "gwasdev_ld_pairs", hm); if (rc != GWASDEV_OK) return rc; }
    GW_CUDA(cudaSetDevice(s->device));
    GW_CUDA(reserve(s->sc_pi, n * sizeof(uint32_t)));
    GW_CUDA(reserve(s->sc_pj, n * sizeof(uint32_t)));
    GW_CUDA(reserve(s->sc_a, s->Wr * sizeof(uint32_t)));
    GW_CUDA(reserve(s->sc_hits, n * sizeof(gwasdev_ld_pair)));
    GW_CUDA(cudaMemcpyAsync(s->sc_pi.p, pi, n * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    GW_CUDA(cudaMemcpyAsync(s->sc_pj.p, pj, n * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    GW_CUDA(cudaMemcpyAsync(s->sc_a.p, hm.data(), s->Wr * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    ld_pairs_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, s->stream>>>(s->d_raw, (const uint32_t *)s->sc_a.p, s->Wr, n, (const uint32_t *)s->sc_pi.p,
                                                                           (const uint32_t *)s->sc_pj.p, (gwasdev_ld_pair *)s->sc_hits.p);
    GW_LAUNCHED();
    GW_CUDA(cudaMemcpyAsync(out, s->sc_hits.p, n * sizeof(gwasdev_ld_pair), cudaMemcpyDeviceToHost, s->stream));
    GW_CUDA(cudaStreamSynchronize(s->stream));
    return GWASDEV_OK;
}

int gwasdev_ld_prune(uint64_t snp_begin, uint64_t snp_end, uint32_t window, double r2_threshold, const gwasdev_ld_pair *pairs,
                     uint64_t n_pairs, uint8_t *keep) {
    GW_REQUIRE(window >= 1, "gwasdev_ld_prune: window must be at least 1");
    GW_REQUIRE(snp_begin <= snp_end, "gwasdev_ld_prune: bad SNP range");
    GW_REQUIRE(keep || snp_begin == snp_end, "gwasdev_ld_prune: NULL keep");
    GW_REQUIRE(pairs || n_pairs == 0, "gwasdev_ld_prune: NULL pairs");
    for (uint64_t k = 0; k < n_pairs; ++k) {
        const gwasdev_ld_pair &q = pairs[k];
        GW_REQUIRE(q.i >= snp_begin && q.i < q.j && q.j < snp_end && q.j - q.i <= window,
                   "gwasdev_ld_prune: pair %llu (%u, %u) outside the range or the window", (unsigned long long)k, q.i, q.j);
        GW_REQUIRE(k == 0 || pairs[k - 1].i < q.i || (pairs[k - 1].i == q.i && pairs[k - 1].j < q.j),
                   "gwasdev_ld_prune: pairs not sorted by (i, j) at %llu", (unsigned long long)k);
    }
    std::fill(keep, keep + (snp_end - snp_begin), (uint8_t)1);
    // SNPs in increasing order: when i is reached, every k < i is final, so a kept i drops the partners it reaches the threshold with
    for (uint64_t k = 0; k < n_pairs; ++k) {
        const gwasdev_ld_pair &q = pairs[k];
        if (keep[q.i - snp_begin] && q.r2 >= r2_threshold) keep[q.j - snp_begin] = 0;
    }
    return GWASDEV_OK;
}

}  // extern "C"
