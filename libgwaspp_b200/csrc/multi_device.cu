// Several B200s driven from ONE host process: the multi-GPU driver the reference's C++ call site can reach.
//
// Reference call site: computeBoost (algorithms/epistasis_func.cpp:349-506) is one C++ function whose pair loop
// (:397-486) visits every pair i < j on one core. Here the caller hands over n stores holding the same table on n
// devices (gwasdev_replicate copies a loaded table to the other devices over NVLink); the tile-pair schedule is cut into
// n shards, one host thread per device runs its shard (screen, fp64 re-score, sort, local top-k), the fixed-size hit
// records are combined with ONE ncclAllGather over NVLink (communicators from ncclCommInitAll, cached per device list)
// and device 0 merges them into the reference's (i, j) emission order. No per-tile traffic between devices.
//
// NCCL is resolved at run time (dlopen of libnccl.so.2: the copy torch has already loaded when the caller is a Python
// process, the system library otherwise), so libgwasdev.so itself has no link-time dependency on it; a box without NCCL
// can still gather through peer copies (gather = 1).
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

int gwasdev_internal_pair_screen(gwasdev_store *s, double threshold, uint64_t top_k, uint32_t shard, uint32_t n_shards, uint64_t *n_hits,
                                 gwasdev_pair_stats *stats);
int gwasdev_internal_pair_emit(gwasdev_store *s, uint64_t found, gwasdev_hit *d_hits);
int gwasdev_internal_merge_hits(gwasdev_store *s, const gwasdev_hit *d_segments, uint32_t n_seg, uint64_t stride, const uint64_t *counts,
                                uint64_t top_k, gwasdev_hit *hits, uint64_t capacity, uint64_t *n_hits);

using namespace gwasdev;

namespace {

struct Nccl {
    void *lib = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    std::map<std::vector<int>, std::vector<ncclComm_t>> comms;   // one communicator set per device list, kept for the process
};
std::mutex g_nccl_mutex;
Nccl g_nccl;

int nccl_load() {
    if (g_nccl.lib) return GWASDEV_OK;
    void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { set_error("gwasdev_pairwise_scan_multi: cannot load libnccl.so.2 (%s); gather = 1 uses peer copies instead", dlerror()); return GWASDEV_ENODEVICE; }
#define SYM(field, name) do { *(void **)(&g_nccl.field) = dlsym(lib, name); if (!g_nccl.field) { set_error("libnccl: symbol %s missing", name); dlclose(lib); return GWASDEV_ENODEVICE; } } while (0)
    SYM(CommInitAll, "ncclCommInitAll"); SYM(CommDestroy, "ncclCommDestroy"); SYM(AllGather, "ncclAllGather");
    SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd"); SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    g_nccl.lib = lib;
    return GWASDEV_OK;
}

#define GW_NCCL(call) do { ncclResult_t r_ = (call); if (r_ != ncclSuccess) { set_error("%s failed: %s", #call, g_nccl.GetErrorString(r_)); return GWASDEV_ENODEVICE; } } while (0)

int nccl_comms(const std::vector<int> &devices, std::vector<ncclComm_t> **out) {
    auto it = g_nccl.comms.find(devices);
    if (it == g_nccl.comms.end()) {
        std::vector<ncclComm_t> c(devices.size());
        GW_NCCL(g_nccl.CommInitAll(c.data(), (int)devices.size(), devices.data()));
        it = g_nccl.comms.emplace(devices, std::move(c)).first;
    }
    *out = &it->second;
    return GWASDEV_OK;
}

}  // namespace

extern "C" {

int gwasdev_replicate(gwasdev_store *src, int device, gwasdev_store **out) {
    GW_REQUIRE(src && out, "gwasdev_replicate: NULL argument");
    *out = nullptr;
    GW_CUDA(cudaSetDevice(src->device));
    GW_CUDA(cudaStreamSynchronize(src->stream));
    gwasdev_store *dst = nullptr;
    int rc = gwasdev_create(src->M, src->N, device, &dst);
    if (rc != GWASDEV_OK) return rc;
    if (device != src->device) {   // direct NVLink path when the driver allows it; cudaMemcpyPeer stages through the host otherwise
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, device, src->device) == cudaSuccess && can) {
            cudaSetDevice(device);
            if (cudaDeviceEnablePeerAccess(src->device, 0) != cudaSuccess) cudaGetLastError();   // already enabled is fine
        }
        cudaGetLastError();
    }
    cudaError_t e = cudaMemcpyPeer(dst->d_hdr, device, src->d_hdr, src->device, src->M * sizeof(uint16_t));
    if (e == cudaSuccess) e = cudaMemcpyPeer(dst->d_raw, device, src->d_raw, src->device, src->M * 2ull * src->Wr * sizeof(uint32_t));
    if (e != cudaSuccess) { set_error("gwasdev_replicate: %s", cudaGetErrorString(e)); gwasdev_destroy(dst); return GWASDEV_ENODEVICE; }
    if ((rc = gwasdev_internal_replay_settings(src, dst)) != GWASDEV_OK) { gwasdev_destroy(dst); return rc; }
    *out = dst;
    return GWASDEV_OK;
}

int gwasdev_pairwise_scan_multi(gwasdev_store *const *stores, uint32_t n_stores, double threshold, uint64_t top_k, gwasdev_hit *hits,
                                uint64_t capacity, uint64_t *n_hits, gwasdev_pair_stats *stats, int gather) {
    GW_REQUIRE(stores && n_hits && n_stores >= 1, "gwasdev_pairwise_scan_multi: NULL argument");
    GW_REQUIRE(gather == 0 || gather == 1, "gwasdev_pairwise_scan_multi: gather %d (0 NCCL all-gather, 1 peer copies)", gather);
    *n_hits = 0;
    std::vector<int> devices(n_stores);
    for (uint32_t d = 0; d < n_stores; ++d) {
        GW_REQUIRE(stores[d] != nullptr, "gwasdev_pairwise_scan_multi: store %u is NULL", d);
        GW_REQUIRE(stores[d]->M == stores[0]->M && stores[d]->N == stores[0]->N && stores[d]->selected &&
                       stores[d]->n_case == stores[0]->n_case && stores[d]->n_ctrl == stores[0]->n_ctrl,
                   "gwasdev_pairwise_scan_multi: store %u does not hold the same table and selection as store 0", d);
        devices[d] = stores[d]->device;
        for (uint32_t q = 0; q < d; ++q) GW_REQUIRE(devices[q] != devices[d], "gwasdev_pairwise_scan_multi: stores %u and %u are on the same device", q, d);
    }
    // ---- one host thread per device: its shard of the tile-pair schedule
    std::vector<uint64_t> found(n_stores, 0);
    std::vector<int> rcs(n_stores, GWASDEV_OK);
    std::vector<std::string> errs(n_stores);
    auto work = [&](uint32_t d) {
        rcs[d] = gwasdev_internal_pair_screen(stores[d], threshold, top_k, d, n_stores, &found[d], stats ? &stats[d] : nullptr);
        if (rcs[d] != GWASDEV_OK) errs[d] = gwasdev_last_error();
    };
    if (n_stores == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (uint32_t d = 0; d < n_stores; ++d) th.emplace_back(work, d);
        for (auto &t : th) t.join();
    }
    for (uint32_t d = 0; d < n_stores; ++d)
        if (rcs[d] != GWASDEV_OK) { set_error("device %d: %s", devices[d], errs[d].c_str()); return rcs[d]; }
    const uint64_t mx = *std::max_element(found.begin(), found.end());
    if (mx == 0) return GWASDEV_OK;
    // ---- fixed-size records: every device unpacks its hits into a send buffer of mx records
    for (uint32_t d = 0; d < n_stores; ++d) {
        gwasdev_store *s = stores[d];
        GW_CUDA(cudaSetDevice(s->device));
        GW_CUDA(reserve(s->sc_hits, mx * sizeof(gwasdev_hit)));
        const int rc = gwasdev_internal_pair_emit(s, found[d], (gwasdev_hit *)s->sc_hits.p);
        if (rc != GWASDEV_OK) return rc;
    }
    gwasdev_store *s0 = stores[0];
    const size_t seg_bytes = mx * sizeof(gwasdev_hit);
    if (n_stores == 1) {
        GW_CUDA(cudaSetDevice(s0->device));
        GW_CUDA(reserve(s0->sc_gather, seg_bytes));
        GW_CUDA(cudaMemcpyAsync(s0->sc_gather.p, s0->sc_hits.p, found[0] * sizeof(gwasdev_hit), cudaMemcpyDeviceToDevice, s0->stream));
    } else if (gather == 0) {
        std::lock_guard<std::mutex> lock(g_nccl_mutex);
        int rc = nccl_load();
        if (rc != GWASDEV_OK) return rc;
        std::vector<ncclComm_t> *comms = nullptr;
        if ((rc = nccl_comms(devices, &comms)) != GWASDEV_OK) return rc;
        for (uint32_t d = 0; d < n_stores; ++d) {
            GW_CUDA(cudaSetDevice(stores[d]->device));
            GW_CUDA(reserve(stores[d]->sc_gather, n_stores * seg_bytes));
        }
        GW_NCCL(g_nccl.GroupStart());
        for (uint32_t d = 0; d < n_stores; ++d)
            GW_NCCL(g_nccl.AllGather(stores[d]->sc_hits.p, stores[d]->sc_gather.p, seg_bytes, ncclUint8, (*comms)[d], stores[d]->stream));
        GW_NCCL(g_nccl.GroupEnd());
        for (uint32_t d = 1; d < n_stores; ++d) {   // the other devices' buffers are free for the next call once their part is done
            GW_CUDA(cudaSetDevice(stores[d]->device));
            GW_CUDA(cudaStreamSynchronize(stores[d]->stream));
        }
    } else {
        GW_CUDA(cudaSetDevice(s0->device));
        GW_CUDA(reserve(s0->sc_gather, n_stores * seg_bytes));
        for (uint32_t d = 0; d < n_stores; ++d) {
            if (found[d] == 0) continue;
            GW_CUDA(cudaSetDevice(stores[d]->device));
            GW_CUDA(cudaStreamSynchronize(stores[d]->stream));
            GW_CUDA(cudaSetDevice(s0->device));
            GW_CUDA(cudaMemcpyPeerAsync((char *)s0->sc_gather.p + d * seg_bytes, s0->device, stores[d]->sc_hits.p, stores[d]->device,
                                        found[d] * sizeof(gwasdev_hit), s0->stream));
        }
    }
    // ---- device 0: union of the shards' lists in (i, j) order (disjoint by construction), top_k of it when asked
    return gwasdev_internal_merge_hits(s0, (const gwasdev_hit *)s0->sc_gather.p, n_stores, mx, found.data(), top_k, hits, capacity, n_hits);
}

// computeGTest (algorithms/epistasis_func.cpp:508-704) on n given pairs, the list cut into one contiguous piece per device.
int gwasdev_gtest_multi(gwasdev_store *const *stores, uint32_t n_stores, uint64_t n, const uint32_t *pi, const uint32_t *pj, double *stat, double *z) {
    GW_REQUIRE(stores && n_stores >= 1 && pi && pj && stat && z, "gwasdev_gtest_multi: NULL argument");
    if (n == 0) return GWASDEV_OK;
    std::vector<int> rcs(n_stores, GWASDEV_OK);
    std::vector<std::string> errs(n_stores);
    auto work = [&](uint32_t d) {
        const uint64_t b = n * d / n_stores, e = n * (d + 1) / n_stores;
        if (e == b) return;
        rcs[d] = gwasdev_gtest(stores[d], e - b, pi + b, pj + b, stat + b, z + b);
        if (rcs[d] != GWASDEV_OK) errs[d] = gwasdev_last_error();
    };
    if (n_stores == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (uint32_t d = 0; d < n_stores; ++d) th.emplace_back(work, d);
        for (auto &t : th) t.join();
    }
    for (uint32_t d = 0; d < n_stores; ++d)
        if (rcs[d] != GWASDEV_OK) { set_error("device %d: %s", stores[d]->device, errs[d].c_str()); return rcs[d]; }
    return GWASDEV_OK;
}

}  // extern "C"
