// The C ABI's NCCL communicator and the hypothesis-sharded estimate on it.  Host only: compiled by the host compiler.
#include <dlfcn.h>

#include "sfm_host.h"

using namespace sfm;
using namespace sfm_host;

// ---- NCCL behind the C ABI (SURVEY.md 8(b): sfm_nccl_init / sharded estimate without torch) ---------------------
// libnccl is resolved at run time (dlopen): the library a host process already loaded (torch bundles one) is reused,
// otherwise the system's libnccl.so.2.  Only four entry points are needed; their prototypes are restated here so that
// the build does not depend on nccl.h.
struct NcclId { char internal[128]; };  // ncclUniqueId, passed BY VALUE to ncclCommInitRank
static_assert(sizeof(NcclId) == SFM_NCCL_ID_BYTES, "ncclUniqueId is 128 bytes");
namespace {
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;

int nccl_load() {
    if (g_nccl.lib) return 0;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // already in the process (torch)?
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(SFM_ERR_STATE, "libnccl.so.2 not found: %s", dlerror());
    g_nccl.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclGetUniqueId"));
    g_nccl.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(dlsym(h, "ncclCommInitRank"));
    g_nccl.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(h, "ncclAllGather"));
    g_nccl.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
    g_nccl.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy)
        return fail(SFM_ERR_STATE, "libnccl.so.2 lacks a required symbol");
    g_nccl.lib = h;
    return 0;
}
#define NC(call)                                                                                          \
    do {                                                                                                  \
        int e_ = (call);                                                                                  \
        if (e_ != 0)                                                                                      \
            return fail(SFM_ERR_CUDA, "%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(e_) : "?"); \
    } while (0)
}  // namespace

int sfm_nccl_unique_id(void* id_out) {
    if (!id_out) return fail(SFM_ERR_ARG, "null argument");
    if (int r = nccl_load()) return r;
    NC(g_nccl.GetUniqueId(id_out));
    return 0;
}

int sfm_nccl_init(sfm_ctx* c, int rank, int nranks, const void* unique_id) {
    if (int r = use(c)) return r;
    if (!unique_id || nranks < 1 || rank < 0 || rank >= nranks) return fail(SFM_ERR_ARG, "bad communicator arguments");
    if (int r = nccl_load()) return r;
    if (c->nccl_comm) { g_nccl.CommDestroy(c->nccl_comm); c->nccl_comm = nullptr; }
    NcclId id;
    memcpy(&id, unique_id, sizeof id);
    NC(g_nccl.CommInitRank(&c->nccl_comm, nranks, id, rank));
    c->nccl_rank = rank;
    c->nccl_world = nranks;
    return 0;
}

int sfm_nccl_destroy(sfm_ctx* c) {
    if (!c) return 0;
    if (c->nccl_comm && g_nccl.lib) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        g_nccl.CommDestroy(c->nccl_comm);
    }
    c->nccl_comm = nullptr;
    c->nccl_world = 1;
    c->nccl_rank = 0;
    return 0;
}

// One complete hypothesis-sharded estimate on the communicator of sfm_nccl_init, nothing synchronised: this rank's
// hypotheses [rank * hyps_per_rank, (rank + 1) * hyps_per_rank) of the device sampler -> fit -> score -> select, ONE
// ncclAllGather of the SFM_RECORD_BYTES selection records on the context's stream (the path's only collective), merge
// kernel, tail.  Results through sfm_sharded_fetch.
int sfm_two_view_sharded(sfm_ctx* c, uint64_t seed, int64_t hyps_per_rank, double thr, double min_extra, int agg,
                         int mode, double dist_thr) {
    if (int r = use(c)) return r;
    if (!c->nccl_comm) return fail(SFM_ERR_STATE, "sfm_nccl_init first");
    if (c->refine_iters > 0) return fail(SFM_ERR_STATE, "refinement is not supported on hypothesis-sharded runs");
    if (c->batched) return fail(SFM_ERR_STATE, "single-pair call on a batched context");
    if (int r = sample_device(c, seed, 0, (int64_t)c->nccl_rank * hyps_per_rank, hyps_per_rank)) return r;
    if (int r = fit_launch(c, false)) return r;
    if (int r = score_launch(c, thr, min_extra, agg, mode, true, 0, c->n)) return r;
    if (int r = c->gathered.reserve((size_t)c->nccl_world * sizeof(SelectRecord))) return r;
    NC(g_nccl.AllGather(c->record.p, c->gathered.p, sizeof(SelectRecord), /* ncclUint8 */ 1, c->nccl_comm, c->stream));
    return sfm_sharded_tail(c, c->gathered.p, c->nccl_world, c->nccl_rank, hyps_per_rank, mode, thr, dist_thr);
}
