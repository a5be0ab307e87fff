// Pair screens over chosen SNP sets (gwasdev_pairwise_scan_sets): within a set, set-by-all, set-by-set.
//
// The call gathers the rows of A u B into a sub-table on the same device, ordered C = A n B, then A \ B, then B \ A, each
// segment in table order. With c1 = |C| and a1 = |C| + |A \ B|, the wanted pairs gi < gj of the sub-table are those with
// gi < c1, or c1 <= gi < a1 <= gj: every unordered pair {i in A, j in B, i != j} exactly once. The sub-table is an ordinary
// store that takes the parent's options, engine and selection (gwasdev_internal_replay_settings); its margins, per-SNP records,
// missing-call flags and operands come from the whole-table code. The SETS instantiations of the tensor-core screens then run
// over the tiles of its schedule that hold a wanted pair (gwasdev_internal_set_shard_pairs), the candidates are oriented by
// table index before the fp64 re-score and the keys are mapped to table indices before the sort (pair_screen_phase), so that
// every record has the bits of the whole-table screen's and the order and tie rule are the table's. The sub-table is freed
// at the end of the call: its raw rows and operands cost what a table of |A u B| SNPs costs.
#include <algorithm>
#include <vector>

#include "pair_common.cuh"

int gwasdev_internal_pair_scan_sets(gwasdev_store *s, const gwasdev::SetScreen &sets, double threshold, uint64_t top_k, uint32_t shard,
                                    uint32_t n_shards, gwasdev_hit *hits, uint64_t capacity, uint64_t *n_hits, gwasdev_pair_stats *stats,
                                    int on_device);

using namespace gwasdev;

// raw rows rows[k] of the parent -> row k of the sub-table, one thread per 16 bytes of a row (2 Wr words, Wr a multiple of 4),
// and the header words
__global__ void gather_rows_kernel(const uint16_t *__restrict__ hdr, const uint32_t *__restrict__ raw, uint32_t Wr, const uint32_t *__restrict__ rows,
                                   uint64_t n, uint16_t *__restrict__ hdr_out, uint32_t *__restrict__ raw_out) {
    const uint32_t chunks = Wr / 2;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t r = idx / chunks;
    if (r >= n) return;
    const uint32_t c = (uint32_t)(idx - r * chunks);
    const uint64_t src = rows[r];
    reinterpret_cast<uint4 *>(raw_out + r * 2ull * Wr)[c] = reinterpret_cast<const uint4 *>(raw + src * 2ull * Wr)[c];
    if (c == 0) hdr_out[r] = hdr[src];
}

int gwasdev_internal_set_rows(uint64_t M, const uint32_t *set_a, uint64_t n_a, const uint32_t *set_b, uint64_t n_b, const char *who,
                              std::vector<uint32_t> &map, uint64_t *c1, uint64_t *a1) {
    GW_REQUIRE(n_a == 0 || set_a, "%s: set_a is NULL", who);
    if (!set_b) { set_b = set_a; n_b = n_a; }
    GW_REQUIRE(n_b == 0 || set_b, "%s: set_b is NULL", who);
    for (int side = 0; side < 2; ++side) {
        const uint32_t *v = side ? set_b : set_a;
        const uint64_t n = side ? n_b : n_a;
        for (uint64_t k = 0; k < n; ++k) {
            GW_REQUIRE(v[k] < M, "%s: set %c holds SNP %u, the table has %llu", who, side ? 'b' : 'a', v[k], (unsigned long long)M);
            GW_REQUIRE(k == 0 || v[k] > v[k - 1], "%s: set %c is not strictly increasing at position %llu (%u after %u)", who, side ? 'b' : 'a',
                       (unsigned long long)k, v[k], v[k - 1]);
        }
    }
    std::vector<uint32_t> c, amb, bma;
    std::set_intersection(set_a, set_a + n_a, set_b, set_b + n_b, std::back_inserter(c));
    std::set_difference(set_a, set_a + n_a, set_b, set_b + n_b, std::back_inserter(amb));
    std::set_difference(set_b, set_b + n_b, set_a, set_a + n_a, std::back_inserter(bma));
    map = std::move(c);
    *c1 = map.size();
    map.insert(map.end(), amb.begin(), amb.end());
    *a1 = map.size();
    map.insert(map.end(), bma.begin(), bma.end());
    return GWASDEV_OK;
}

extern "C" {

int gwasdev_pairwise_scan_sets(gwasdev_store *s, const uint32_t *set_a, uint64_t n_a, const uint32_t *set_b, uint64_t n_b, double threshold,
                               uint64_t top_k, uint32_t shard, uint32_t n_shards, gwasdev_hit *hits, uint64_t capacity, uint64_t *n_hits,
                               gwasdev_pair_stats *stats, int on_device) {
    GW_REQUIRE(s && n_hits, "gwasdev_pairwise_scan_sets: NULL argument");
    GW_REQUIRE(n_shards >= 1 && shard < n_shards, "gwasdev_pairwise_scan_sets: shard %u of %u", shard, n_shards);
    GW_REQUIRE(s->selected, "gwasdev_pairwise_scan_sets: call gwasdev_select_case_control first");
    GW_REQUIRE(s->pair_engine != 1, "gwasdev_pairwise_scan_sets: set screens run on the tensor-core engines only; this store's pair engine "
               "is 1 (AND+POPC)");
    *n_hits = 0;
    if (stats) memset(stats, 0, sizeof *stats);
    std::vector<uint32_t> map;
    uint64_t c1 = 0, a1 = 0;
    int rc = gwasdev_internal_set_rows(s->M, set_a, n_a, set_b, n_b, "gwasdev_pairwise_scan_sets", map, &c1, &a1);
    if (rc != GWASDEV_OK) return rc;
    if (map.size() < 2) return GWASDEV_OK;                      // no pair: an empty set, or A = B of one SNP
    GW_CUDA(cudaSetDevice(s->device));
    cudaEvent_t ev_start = nullptr;
    GW_CUDA(cudaEventCreate(&ev_start));
    struct Cleanup {
        gwasdev_store *sub = nullptr; cudaEvent_t ev; uint32_t *d_map = nullptr;
        ~Cleanup() { if (d_map) cudaFree(d_map); gwasdev_destroy(sub); cudaEventDestroy(ev); }
    } tidy{nullptr, ev_start};
    GW_CUDA(cudaEventRecord(ev_start, s->stream));
    const uint64_t Ms = map.size();
    if ((rc = gwasdev_create(Ms, s->N, s->device, &tidy.sub)) != GWASDEV_OK) return rc;
    gwasdev_store *sub = tidy.sub;
    sub->stream = s->stream;
    GW_CUDA(cudaMalloc(&tidy.d_map, Ms * sizeof(uint32_t)));
    GW_CUDA(cudaMemcpyAsync(tidy.d_map, map.data(), Ms * sizeof(uint32_t), cudaMemcpyHostToDevice, s->stream));
    const uint64_t work = Ms * (s->Wr / 2);
    gather_rows_kernel<<<(unsigned)((work + 255) / 256), 256, 0, s->stream>>>(s->d_hdr, s->d_raw, s->Wr, tidy.d_map, Ms, sub->d_hdr, sub->d_raw);
    GW_LAUNCHED();
    if ((rc = gwasdev_internal_replay_settings(s, sub)) != GWASDEV_OK) return rc;
    const SetScreen sets = {c1, a1, tidy.d_map};
    rc = gwasdev_internal_pair_scan_sets(sub, sets, threshold, top_k, shard, n_shards, hits, capacity, n_hits, stats, on_device);
    if (stats && (rc == GWASDEV_OK || rc == GWASDEV_EOVERFLOW)) {      // the whole call: gather, selection, operands, screen, re-score, sort
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ev_start, sub->ev_pw) == cudaSuccess) stats->total_ms = ms; else cudaGetLastError();
    }
    return rc;
}

}  // extern "C"
