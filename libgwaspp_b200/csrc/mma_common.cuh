// tcgen05 building blocks shared by the tensor-core kernels (pairwise_mma.cu: the pair screens; permute_gemm.cuh: the
// permutation test; ld.cu: windowed LD): CTA-pair geometry, PTX wrappers, the mbarrier helpers, the tile feed, the UMMA
// descriptors, and the CTA-pair pipeline (CtaPipe) with its host launch.
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
// 8 / 16 accumulator columns of this warp's 32 lanes
__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
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
// all 512 TMEM columns of the CTA, by one whole warp in both CTAs of the pair
__device__ __forceinline__ void tmem_alloc_pair(uint32_t *slot) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t tmem) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

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
// single-thread consumer: tile n of the pair (the caller counts), false at the end of the shard
__device__ __forceinline__ bool sched_next(const uint2 *slots, uint64_t *sfull, uint64_t *sempty, uint32_t n, uint32_t &I2, uint32_t &J) {
    const int slot = (int)(n % SCHED_SLOTS);
    mbar_wait_wd_cluster(&sfull[slot], (n / SCHED_SLOTS) & 1u);
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(I2), "=r"(J) : "r"(smem_u32(&slots[slot])) : "memory");
    if (I2 == SCHED_END) return false;
    mbar_arrive_remote(&sempty[slot], 0);
    return true;
}
// warp-wide consumer (epilogue): tile n of the pair (the caller counts), lane 0 waits and releases
__device__ __forceinline__ bool sched_next_warp(const uint2 *slots, uint64_t *sfull, uint64_t *sempty, int lane, uint32_t n, uint32_t &I2, uint32_t &J) {
    const int slot = (int)(n % SCHED_SLOTS);
    if (lane == 0) mbar_wait_wd_cluster(&sfull[slot], (n / SCHED_SLOTS) & 1u);
    __syncwarp();
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(I2), "=r"(J) : "r"(smem_u32(&slots[slot])) : "memory");
    __syncwarp();
    if (I2 == SCHED_END) return false;
    if (lane == 0) mbar_arrive_remote(&sempty[slot], 0);
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
// tensor-core kernels stage them (pairwise.cu)
int encode_operand_map(void *ptr, uint64_t rows, uint32_t kbytes, uint32_t box_rows, CUtensorMap *out);

#ifdef GWASDEV_SWEEP
#define GW_PROF(x) x
#else
#define GW_PROF(x)
#endif

// ---- the CTA-pair pipeline --------------------------------------------------------------------------
// Every tensor-core kernel (the pair screens, the permutation GEMM, the LD GEMM) is a persistent 2-CTA cluster of 18 warps:
//   warp 16 (TMA_WARP)  producer: both CTAs load their rows of each stage; the loads complete on the leader's full[stage]
//   warp 17 (MMA_WARP)  issuer  : (leader only) the MMAs of a stage into the tile's TMEM accumulator; tcgen05.commit multicasts
//                                 empty[stage] and, at the end of the tile, tfull[acc] to both CTAs
//   warps 0-15          epilogue: wait tfull[acc], read TMEM, release tempty[acc] to the leader, then the kernel's own work
// over the tiles that the leader's producer draws and publishes through the tile feed above. CtaPipe holds this protocol; a
// kernel supplies only its draw, its loads of one 128-byte sample block, its MMAs of one sample block and its epilogue.
template <int STAGES> struct PipeBars {
    uint64_t full[STAGES];            // the leader's arrive.expect_tx + the peer producer's arrive; both CTAs' TMA bytes land on it
    uint64_t empty[STAGES];           // one multicast tcgen05.commit
    uint64_t tfull[2];                // one multicast tcgen05.commit
    uint64_t tempty[2];               // every epilogue warp of both CTAs
    uint64_t sfull[SCHED_SLOTS];      // tile feed: slot published / slot read by every consumer of the pair
    uint64_t sempty[SCHED_SLOTS];
    uint2 sched[SCHED_SLOTS];
    uint32_t tmem_slot;
};
// dynamic shared memory of a kernel: 1 KiB alignment slack, the stage ring, the kernel's own region, the barriers
constexpr size_t pipe_smem_bytes(int stages, int stage_bytes, int extra_bytes) {
    return 1024 + (size_t)stages * stage_bytes + extra_bytes + (2 * stages + 4 + 2 * SCHED_SLOTS) * sizeof(uint64_t) +
           SCHED_SLOTS * sizeof(uint2) + 16;
}

// One CTA of the pair. STAGES stages of KPS_ sample blocks of KBB bytes (this CTA's A rows, then its half of B); EXTRA bytes
// of the kernel's own between the ring and the barriers; NACC accumulators of ACC_COLS TMEM columns in flight (1: the epilogue
// of a tile does not overlap the MMAs of the next).
template <int STAGES, int KPS_, int KBB, int EXTRA = 0, int NACC = 2>
struct CtaPipe {
    static constexpr int STG = KPS_ * KBB;
    static constexpr size_t SMEM = pipe_smem_bytes(STAGES, STG, EXTRA);
    static_assert(KBB % 1024 == 0 && SMEM <= 232448, "stage blocks keep the 1 KiB swizzle alignment; at most 227 KiB per CTA");
    unsigned char *sm;                // stage ring (SWIZZLE_128B atoms are 1024-byte aligned)
    uint32_t base;                    // its shared address
    PipeBars<STAGES> *bar;
    uint32_t tmem, rank;              // rank 0: leader of the pair (issues the MMAs, owns full / tempty)

    // barriers, TMEM and the cluster sync of both CTAs; returns the kernel's EXTRA bytes
    __device__ __forceinline__ unsigned char *setup(unsigned char *smem_raw) {
        base = (smem_u32(smem_raw) + 1023u) & ~1023u;
        sm = smem_raw + (base - smem_u32(smem_raw));
        bar = reinterpret_cast<PipeBars<STAGES> *>(sm + STAGES * STG + EXTRA);
        rank = cluster_ctarank();
        if (threadIdx.x == 0) {
            for (int s = 0; s < STAGES; ++s) { mbar_init(&bar->full[s], 2); mbar_init(&bar->empty[s], 1); }
            for (int b = 0; b < 2; ++b) { mbar_init(&bar->tfull[b], 1); mbar_init(&bar->tempty[b], 2 * EPI_WARPS); }
            for (int b = 0; b < SCHED_SLOTS; ++b) { mbar_init(&bar->sfull[b], 1); mbar_init(&bar->sempty[b], SCHED_CONSUMERS); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        if (threadIdx.x / 32 == MMA_WARP) tmem_alloc_pair(&bar->tmem_slot);   // both accumulators
        tc_fence_before();
        cluster_sync_all();                            // barriers initialised and TMEM allocated in both CTAs
        tc_fence_after();
        tmem = bar->tmem_slot;
        return sm + STAGES * STG;
    }
    __device__ __forceinline__ void teardown() {
        tc_fence_before();
        cluster_sync_all();                            // neither CTA leaves while its pair may still touch its SM
        if (threadIdx.x / 32 == MMA_WARP) { tc_fence_after(); tmem_dealloc_pair(tmem); }
    }

    // Producer (lane 0 of TMA_WARP in both CTAs). The leader takes its tiles from draw(I, J) -> false at the end and publishes
    // them; the peer reads them from the feed. load(I, J, dst, blk, full) issues this CTA's loads of sample block blk into dst.
    // prof (role timers, GWASDEV_SWEEP builds): per CTA, [5] = clocks spent waiting for empty.
    template <class Draw, class Load>
    __device__ __forceinline__ void produce(uint32_t NKB, Draw &&draw, Load &&load, unsigned long long *prof = nullptr) {
        if (threadIdx.x % 32 != 0) return;
        uint64_t it = 0;
        GW_PROF(long long prof_pw = 0;)
        for (uint32_t tile = 0;; ++tile) {
            uint32_t I = 0, J = 0;
            if (rank == 0) {
                const bool more = draw(I, J);
                const int slot = (int)(tile % SCHED_SLOTS);
                mbar_wait_wd(&bar->sempty[slot], ((tile / SCHED_SLOTS) & 1u) ^ 1u);
                sched_publish(bar->sched, bar->sfull, slot, more ? I : SCHED_END, J);
                if (!more) break;
            } else if (!sched_next(bar->sched, bar->sfull, bar->sempty, tile, I, J)) break;
            for (uint32_t kb = 0; kb < NKB; kb += KPS_, ++it) {
                const int st = (int)(it % STAGES);
                const uint32_t nk = min((uint32_t)KPS_, NKB - kb);
                GW_PROF(const long long w0 = clock64();)
                mbar_wait_wd(&bar->empty[st], (uint32_t)(((it / STAGES) & 1) ^ 1));
                GW_PROF(prof_pw += clock64() - w0;)
                if (rank == 0) mbar_expect_tx(&bar->full[st], nk * 2 * KBB);
                else mbar_arrive_remote(&bar->full[st], 0);
                for (uint32_t k2 = 0; k2 < nk; ++k2) load(I, J, sm + st * STG + k2 * KBB, kb + k2, &bar->full[st]);
            }
        }
        GW_PROF(if (prof) prof[blockIdx.x * 8 + 5] = (unsigned long long)prof_pw;)
        (void)prof;
    }

    // MMA issuer (lane 0 of MMA_WARP in the leader). mma(d, a, blk) issues the MMAs of sample block blk of the tile, whose
    // stage block starts at shared address a, into the accumulator at TMEM address d (accumulating unless blk is the first).
    // prof: [0] busy, [1] waiting for tempty, [2] waiting for full, [6] tiles.
    template <class Mma>
    __device__ __forceinline__ void issue(uint32_t NKB, Mma &&mma, unsigned long long *prof = nullptr) {
        if (threadIdx.x % 32 != 0 || rank != 0) return;
        uint64_t it = 0;
        uint32_t tile = 0, I, J;
        GW_PROF(long long prof_te = 0; long long prof_fu = 0; const long long prof_t0 = clock64();)
        for (; sched_next(bar->sched, bar->sfull, bar->sempty, tile, I, J); ++tile) {
            const uint32_t buf = tile % NACC;
            GW_PROF(const long long w0 = clock64();)
            mbar_wait_wd(&bar->tempty[buf], ((tile / NACC) & 1u) ^ 1u);
            GW_PROF(prof_te += clock64() - w0;)
            tc_fence_after();
            const uint32_t d_addr = tmem + buf * ACC_COLS;
            for (uint32_t kb = 0; kb < NKB; kb += KPS_, ++it) {
                const int st = (int)(it % STAGES);
                const uint32_t nk = min((uint32_t)KPS_, NKB - kb);
                GW_PROF(const long long w1 = clock64();)
                mbar_wait_wd(&bar->full[st], (uint32_t)((it / STAGES) & 1));
                GW_PROF(prof_fu += clock64() - w1;)
                tc_fence_after();
                for (uint32_t k2 = 0; k2 < nk; ++k2) mma(d_addr, base + st * STG + k2 * KBB, kb + k2);
                tc_commit_mc(&bar->empty[st], 3);      // stage reusable in both CTAs once these MMAs have read it
            }
            tc_commit_mc(&bar->tfull[buf], 3);         // accumulator complete in both CTAs
        }
        GW_PROF(if (prof) {
            unsigned long long *o = prof + blockIdx.x * 8;
            o[0] = (unsigned long long)(clock64() - prof_t0); o[1] = (unsigned long long)prof_te; o[2] = (unsigned long long)prof_fu; o[6] = tile;
        })
        (void)prof;
    }

    // Epilogue warps, counting the pair's tiles n = 0, 1, ...: tile n (false at the end), wait for its accumulator (returns its
    // index; TMEM address tmem + index * ACC_COLS), and hand the accumulator back once its TMEM loads have completed.
    __device__ __forceinline__ bool next_warp(int lane, uint32_t n, uint32_t &I, uint32_t &J) {
        return sched_next_warp(bar->sched, bar->sfull, bar->sempty, lane, n, I, J);
    }
    __device__ __forceinline__ uint32_t acc_wait(int lane, uint64_t n) {
        const uint32_t buf = (uint32_t)(n % NACC);
        if (lane == 0) mbar_wait_wd(&bar->tfull[buf], (uint32_t)((n / NACC) & 1));
        __syncwarp();
        tc_fence_after();
        return buf;
    }
    __device__ __forceinline__ void acc_release(int lane, uint32_t buf) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(&bar->tempty[buf], 0);
    }
};

// Launches a CtaPipe kernel on one CTA pair per TPC, at most one pair per tile, with p.tile_counter zeroed; *pairs_out = the
// pairs. `start` (or nullptr) is recorded right before the kernel, so that an event pair around it times the kernel alone.
template <class Kernel, class Params, class... Maps>
int launch_cta_pairs(gwasdev_store *s, Kernel kernel, size_t smem, uint64_t n_tiles, Params &p, unsigned *pairs_out, cudaEvent_t start,
                     const Maps &...maps) {
    int sms = 0;
    GW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    const unsigned pairs = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sms / 2, n_tiles));
    if (pairs_out) *pairs_out = pairs;
    if (!s->d_tile_counter) GW_CUDA(cudaMalloc(&s->d_tile_counter, sizeof(unsigned long long)));
    GW_CUDA(cudaMemsetAsync(s->d_tile_counter, 0, sizeof(unsigned long long), s->stream));
    p.tile_counter = s->d_tile_counter;
    GW_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (start) GW_CUDA(cudaEventRecord(start, s->stream));
    kernel<<<2 * pairs, MMA_THREADS, smem, s->stream>>>(maps..., p);
    GW_LAUNCHED();
    return GWASDEV_OK;
}

__device__ __forceinline__ uint32_t spread4(uint32_t nibble) { return (nibble * 0x00204081u) & 0x01010101u; }   // bit i -> byte i

}  // namespace gwasdev
