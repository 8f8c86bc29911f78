// oz_dist.cu — C1 / C2: the two collectives of a training iteration (SURVEY 2.1, 8e), straight over NCCL.
//
//   C1  oz_dist_broadcast_weights   replaces the reference's weight fan-out: temp .h5 -> sftp to the first VM -> scp tree
//                                   (workers.py:203-296).  One ncclBroadcast of the float32 blob into HBM, then the usual
//                                   on-device fold (oz_net_load_weights_dev).
//   C2  oz_dist_gather_examples     replaces the pickled-stdout result gather (workers.py:147-159,180-184): one ncclAllGather
//                                   of the per-rank row counts, one of the padded packed example rows.
//
// Neither sits inside the search loop (games shard by id, nothing is exchanged while they are played).  NCCL is resolved at
// run time with dlopen("libnccl.so.2") - the library a torch process has already loaded (torch's bundled NCCL), or the
// system one - so liboz_b200.so itself has no link-time dependency and still loads on a box without NCCL.
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>

#include <vector>

#include "oz_engine.cuh"

namespace {

struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (h) {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(h, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(h, "ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(h, "ncclCommDestroy");
            api.Broadcast = (decltype(api.Broadcast))dlsym(h, "ncclBroadcast");
            api.AllGather = (decltype(api.AllGather))dlsym(h, "ncclAllGather");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(h, "ncclGetErrorString");
            api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.Broadcast && api.AllGather && api.GetErrorString;
        }
    }
    return &api;
}

#define OZ_NCCL(expr)                                                                                   \
    do {                                                                                                \
        ncclResult_t _r = (expr);                                                                       \
        if (_r != ncclSuccess) {                                                                        \
            oz_set_error("%s failed: %s (%s:%d)", #expr, nccl_api()->GetErrorString(_r), __FILE__, __LINE__); \
            return OZ_ERR_CUDA;                                                                         \
        }                                                                                               \
    } while (0)

int need_api() {
    if (!nccl_api()->ok) {
        const char* why = dlerror();
        oz_set_error("NCCL is not available (dlopen libnccl.so.2: %s)", why ? why : "symbols missing");
        return OZ_ERR_STATE;
    }
    return OZ_OK;
}

}  // namespace

extern "C" int oz_dist_unique_id(uint8_t* id128) {
    OZ_REQUIRE(id128, "null argument");
    int rc = need_api();
    if (rc) return rc;
    ncclUniqueId id;
    OZ_NCCL(nccl_api()->GetUniqueId(&id));
    static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, sizeof(id));
    return OZ_OK;
}

extern "C" int oz_dist_init(oz_engine* e, int32_t rank, int32_t world, const uint8_t* id128) {
    OZ_REQUIRE(e && id128, "null argument");
    OZ_REQUIRE(world >= 1 && rank >= 0 && rank < world, "rank %d / world %d out of range", rank, world);
    if (e->comm) { oz_set_error("oz_dist_init was already called on this engine"); return OZ_ERR_STATE; }
    int rc = need_api();
    if (rc) return rc;
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclComm_t comm = nullptr;
    OZ_NCCL(nccl_api()->CommInitRank(&comm, world, id, rank));
    e->comm = comm;
    e->dist_rank = rank;
    e->dist_world = world;
    return OZ_OK;
}

extern "C" int oz_dist_destroy(oz_engine* e) {
    if (!e || !e->comm) return OZ_OK;
    cudaSetDevice(e->cfg.device);
    cudaStreamSynchronize(e->stream);
    nccl_api()->CommDestroy((ncclComm_t)e->comm);
    e->comm = nullptr;
    return OZ_OK;
}

extern "C" int oz_dist_broadcast_weights(oz_engine* e, const float* blob, int64_t n_floats, int32_t channels, int32_t root) {
    OZ_REQUIRE(e, "null engine");
    if (!e->comm) { oz_set_error("oz_dist_init first"); return OZ_ERR_STATE; }
    OZ_REQUIRE(root >= 0 && root < e->dist_world, "root %d out of range", root);
    OZ_REQUIRE(e->dist_rank != root || blob, "the root rank must pass the weight blob");
    const int32_t plain = channels & ~OZ_NET_FP8;  // the blob does not depend on the precision
    OZ_REQUIRE(n_floats == oz_net_blob_floats(e->cfg.board_size, plain), "weight blob has %lld floats, expected %lld",
               (long long)n_floats, (long long)oz_net_blob_floats(e->cfg.board_size, plain));
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    float* dev = nullptr;
    OZ_CUDA(cudaMalloc((void**)&dev, (size_t)n_floats * 4));
    struct Guard { float* p; ~Guard() { cudaFree(p); } } g{dev};
    if (e->dist_rank == root)
        OZ_CUDA(cudaMemcpyAsync(dev, blob, (size_t)n_floats * 4, cudaMemcpyHostToDevice, e->stream));
    OZ_NCCL(nccl_api()->Broadcast(dev, dev, (size_t)n_floats, ncclFloat32, root, (ncclComm_t)e->comm, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return oz_net_load_weights_dev(e, dev, n_floats, channels);  // folds BN, casts to bf16 (or quantises, OZ_NET_FP8), rebuilds the tables, clears the cache
}

extern "C" int oz_dist_gather_examples(oz_engine* e, const uint64_t* rows, int64_t n_rows, uint64_t* out_rows, int64_t capacity_rows,
                                       int64_t* total_rows) {
    OZ_REQUIRE(e && total_rows && (rows || n_rows == 0) && n_rows >= 0, "bad argument");
    if (!e->comm) { oz_set_error("oz_dist_init first"); return OZ_ERR_STATE; }
    OZ_CUDA(cudaSetDevice(e->cfg.device));
    const int W = e->dist_world;
    // 1. everyone learns everyone's row count
    long long* d_cnt = nullptr;
    OZ_CUDA(cudaMalloc((void**)&d_cnt, sizeof(long long) * (W + 1)));
    struct Guard { void* a; void* b = nullptr; ~Guard() { cudaFree(a); if (b) cudaFree(b); } } g{d_cnt};
    const long long mine = n_rows;
    OZ_CUDA(cudaMemcpyAsync(d_cnt + W, &mine, sizeof(mine), cudaMemcpyHostToDevice, e->stream));
    OZ_NCCL(nccl_api()->AllGather(d_cnt + W, d_cnt, 1, ncclInt64, (ncclComm_t)e->comm, e->stream));
    std::vector<long long> cnt(W);
    OZ_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(long long) * W, cudaMemcpyDeviceToHost, e->stream));
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    long long mx = 0, tot = 0;
    for (int r = 0; r < W; ++r) { mx = cnt[r] > mx ? cnt[r] : mx; tot += cnt[r]; }
    *total_rows = tot;
    if (!out_rows) return OZ_OK;                       // size query
    OZ_REQUIRE(capacity_rows >= tot, "output buffer holds %lld rows, %lld were gathered", (long long)capacity_rows, tot);
    if (mx == 0) return OZ_OK;
    // 2. padded all-gather of the rows (3 x uint64 each), then compaction in rank order on the host
    const size_t slab = (size_t)mx * 3;                // uint64 per rank
    uint64_t* d_rows = nullptr;
    OZ_CUDA(cudaMalloc((void**)&d_rows, sizeof(uint64_t) * slab * (W + 1)));
    g.b = d_rows;
    OZ_CUDA(cudaMemsetAsync(d_rows + slab * W, 0, sizeof(uint64_t) * slab, e->stream));
    if (n_rows)
        OZ_CUDA(cudaMemcpyAsync(d_rows + slab * W, rows, sizeof(uint64_t) * 3 * (size_t)n_rows, cudaMemcpyHostToDevice, e->stream));
    OZ_NCCL(nccl_api()->AllGather(d_rows + slab * W, d_rows, slab, ncclUint64, (ncclComm_t)e->comm, e->stream));
    uint64_t* dst = out_rows;
    for (int r = 0; r < W; ++r) {
        if (cnt[r])
            OZ_CUDA(cudaMemcpyAsync(dst, d_rows + slab * r, sizeof(uint64_t) * 3 * (size_t)cnt[r], cudaMemcpyDeviceToHost, e->stream));
        dst += 3 * cnt[r];
    }
    OZ_CUDA(cudaStreamSynchronize(e->stream));
    return OZ_OK;
}
