// tcgen05 building blocks shared by the tensor-core kernels (pairwise_mma.cu: the pair screens; permute.cu: the permutation
// test): CTA-pair geometry, PTX wrappers, the mbarrier helpers, the tile feed and the UMMA descriptors.
#pragma once

#include "pair_common.cuh"

namespace gwasdev {

constexpr int MMA_A_SNPS = 64, MMA_B_SNPS = 128;                   // per CTA: A-SNPs whose rows it owns; B-SNPs of the tile
constexpr int MMA_BLK = 128;                                       // SNPs per schedule block (A-block of the CTA pair = B-block)
constexpr int MMA_M = 4 * MMA_A_SNPS, MMA_N = 2 * MMA_B_SNPS;      // operand rows of one cta_group::2 instruction
constexpr int MMA_KB = 128;                                        // sample bytes per stage (one 128B swizzle row)
constexpr int UMMA_K = 32;                                         // bytes per tcgen05.mma kind::i8
constexpr int MMA_STAGES = 3;
constexpr int KPS = 2;                                             // 128-byte sample blocks per stage (fewer barrier round trips)
constexpr int A_STAGE_BYTES = 2 * MMA_A_SNPS * MMA_KB, B_STAGE_BYTES = MMA_B_SNPS * MMA_KB;   // per CTA and sample block: its A rows, its half of B
constexpr int KB_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;            // 32 KiB per CTA and sample block
constexpr int STAGE_BYTES_MMA = KPS * KB_BYTES;                    // 64 KiB per CTA
constexpr int EPI_WARPS = 16;
constexpr int MMA_THREADS = (2 + EPI_WARPS) * 32;
// The warp scheduler favours the highest warp ids: the two single-thread roles that every stage waits on sit
// above the sixteen epilogue warps (which also makes warp % 4 the TMEM lane quadrant of epilogue warp `warp`).
constexpr int TMA_WARP = EPI_WARPS, MMA_WARP = EPI_WARPS + 1;
constexpr int ACC_COLS = MMA_N;                                    // TMEM columns per accumulator
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;                        // shared::cluster address of the pair's even CTA

// ---- PTX: tcgen05 ------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// arrive on the barrier at the same offset in the CTAs of cta_mask once all earlier MMAs of this thread are done
__device__ __forceinline__ void tc_commit_mc(uint64_t *bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive (no transaction bytes) on the barrier at this offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t *bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
// 2-CTA TMA load: data into this CTA's shared memory, completion bytes on the pair leader's barrier
__device__ __forceinline__ void tma_load_2d_pair(void *dst, const CUtensorMap *map, int x, int y, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar) & PEER_MASK) : "memory");
}
// the same for a 3-D box (sample bytes, planes, SNPs)
__device__ __forceinline__ void tma_load_3d_pair(void *dst, const CUtensorMap *map, int x, int y, int z, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar) & PEER_MASK) : "memory");
}
// 24 accumulator columns (eight B-SNPs of three planes) of this warp's 32 lanes
__device__ __forceinline__ void tc_ld24(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23])
        : "r"(taddr + 16u) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// mbarrier wait with a watchdog: a broken pipeline traps instead of hanging the device
__device__ __forceinline__ void mbar_wait_wd(uint64_t *bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    const long long t0 = clock64();
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.b32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
        if (clock64() - t0 > 8000000000ll) __trap();
    }
}

// ---- tile feed ---------------------------------------------------------------------------------------
// The CTA pairs draw their tiles from one device-wide counter, in schedule order, instead of owning every n-th tile: whatever
// their relative speed, the tiles in flight on the GPU are then ~74 consecutive ones of the schedule (one band of A-blocks and
// a window of ~10 B-blocks, ~50 MB: L2-resident). With fixed ownership the pairs drift apart over the 100 000 tiles each
// processes at configs[3] and the window outgrows the L2 (DRAM reads 6.3 TB per pass against 3.1 TB for eight 1/8 shards).
// One thread of the pair -- the leader's TMA producer -- draws the index, decodes it and publishes (I2, J) in a ring of
// SCHED_SLOTS slots in BOTH CTAs' shared memory; every other role (peer producer, MMA issuer, 2 x 16 epilogue warps) waits on
// its CTA's sfull[slot], reads the slot and arrives on the leader's sempty[slot].
constexpr int SCHED_SLOTS = 4;                 // producer at tile n, epilogue at n - 2: four slots never stall the producer
constexpr uint32_t SCHED_END = 0xffffffffu;
constexpr uint32_t SCHED_CONSUMERS = 2 * EPI_WARPS + 2;   // epilogue warps of both CTAs, the leader's MMA issuer, the peer's producer
__device__ __forceinline__ void mbar_wait_wd_cluster(uint64_t *bar, uint32_t parity) {    // acquires what a remote thread released
    const uint32_t addr = smem_u32(bar);
    const long long t0 = clock64();
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.b32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
        if (clock64() - t0 > 8000000000ll) __trap();
    }
}
// publish (I2, J) in slot `slot` of both CTAs (called by the leader's producer thread)
__device__ __forceinline__ void sched_publish(uint2 *slots, uint64_t *sfull, int slot, uint32_t I2, uint32_t J) {
    asm volatile(
        "{\n\t.reg .b32 rs, rb;\n\t"
        "st.shared.v2.u32 [%0], {%2, %3};\n\t"
        "mapa.shared::cluster.u32 rs, %0, 1;\n\t"
        "st.shared::cluster.v2.u32 [rs], {%2, %3};\n\t"
        "mapa.shared::cluster.u32 rb, %1, 1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [rb];\n\t"
        "mbarrier.arrive.release.cta.shared::cta.b64 _, [%1];\n\t}"
        ::"r"(smem_u32(&slots[slot])), "r"(smem_u32(&sfull[slot])), "r"(I2), "r"(J) : "memory");
}
// single-thread consumer: next tile of the pair, false at the end of the shard
__device__ __forceinline__ bool sched_next(const uint2 *slots, uint64_t *sfull, uint64_t *sempty, uint32_t &n, uint32_t &I2, uint32_t &J) {
    const int slot = (int)(n % SCHED_SLOTS);
    mbar_wait_wd_cluster(&sfull[slot], (n / SCHED_SLOTS) & 1u);
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(I2), "=r"(J) : "r"(smem_u32(&slots[slot])) : "memory");
    if (I2 == SCHED_END) return false;
    mbar_arrive_remote(&sempty[slot], 0);
    ++n;
    return true;
}
// warp-wide consumer (epilogue): lane 0 waits and releases
__device__ __forceinline__ bool sched_next_warp(const uint2 *slots, uint64_t *sfull, uint64_t *sempty, int lane, uint32_t &n, uint32_t &I2, uint32_t &J) {
    const int slot = (int)(n % SCHED_SLOTS);
    if (lane == 0) mbar_wait_wd_cluster(&sfull[slot], (n / SCHED_SLOTS) & 1u);
    __syncwarp();
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(I2), "=r"(J) : "r"(smem_u32(&slots[slot])) : "memory");
    __syncwarp();
    if (I2 == SCHED_END) return false;
    if (lane == 0) mbar_arrive_remote(&sempty[slot], 0);
    ++n;
    return true;
}

// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);          // start address, 16-byte units
    d |= (uint64_t)0 << 16;                                // leading byte offset: unused (one swizzle atom along K)
    d |= (uint64_t)(1024 >> 4) << 32;                      // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                                // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                                // SWIZZLE_128B
    return d;
}
// instruction descriptor kind::i8: D s32, A and B signed 8-bit, both K-major, N >> 3, M >> 4
constexpr uint32_t idesc_i8(int n) { return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(MMA_M >> 4) << 24); }   // M = 256 over the CTA pair
constexpr uint32_t IDESC_I8 = idesc_i8(MMA_N);

// 2-D tensor map over `rows` operand rows of `kbytes` bytes (K-major, SWIZZLE_128B boxes of 128 bytes x box_rows), as the
// permutation test and the LD kernel stage them (permute.cu)
int encode_operand_map(void *ptr, uint64_t rows, uint32_t kbytes, uint32_t box_rows, CUtensorMap *out);

__device__ __forceinline__ uint32_t spread4(uint32_t nibble) { return (nibble * 0x00204081u) & 0x01010101u; }   // bit i -> byte i

}  // namespace gwasdev
