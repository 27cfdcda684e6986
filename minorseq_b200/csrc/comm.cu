// comm.cu -- the path's cross-GPU exchange, native: one ncclAllReduce of the count tensor between
// K1 and K2 (SURVEY.md 8e; BASELINE.json north_star "per-GPU count tensors are combined with a single
// NCCL allreduce over NVLink before calling and phasing"), enqueued on the handle's stream so that
// K1 -> all-reduce -> K2 needs no host synchronisation, plus the all-gather of the compact haplotype
// lists used by ms_phase_groups.
//
// NCCL is bound at run time with dlopen("libnccl.so.2"): inside a PyTorch process this resolves to the
// NCCL build torch already loaded (one NCCL per process), in the stand-alone juliet binary to the
// system library.  One process per GPU; the caller distributes the 128-byte unique id (rank 0 makes it)
// over whatever control channel it has (bench.py: torch.distributed broadcast).
#include <dlfcn.h>
#include <nccl.h>
#include <cstring>
#include "handle.h"

namespace {

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

NcclApi& api() {
    static NcclApi a;
    if (a.lib) return a;
    a.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!a.lib) a.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!a.lib) return a;
    a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(a.lib, "ncclGetUniqueId"));
    a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(a.lib, "ncclCommInitRank"));
    a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(a.lib, "ncclCommDestroy"));
    a.AllReduce = reinterpret_cast<decltype(a.AllReduce)>(dlsym(a.lib, "ncclAllReduce"));
    a.AllGather = reinterpret_cast<decltype(a.AllGather)>(dlsym(a.lib, "ncclAllGather"));
    a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(a.lib, "ncclGetErrorString"));
    a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllReduce && a.AllGather && a.GetErrorString;
    return a;
}

}  // namespace

#define MS_NCCL(h, call)                                                             \
    do {                                                                             \
        ncclResult_t r_ = (call);                                                    \
        if (r_ != ncclSuccess) {                                                     \
            (h)->err = std::string(#call) + ": " + api().GetErrorString(r_);         \
            return MS_ERR_CUDA;                                                      \
        }                                                                            \
    } while (0)

// used by phase.cu
int ms_comm_allgather_bytes(ms_handle* h, const void* d_send, void* d_recv, size_t bytes_per_rank) {
    if (!h->comm) return MS_ERR_ARG;
    MS_NCCL(h, api().AllGather(d_send, d_recv, bytes_per_rank, ncclUint8, static_cast<ncclComm_t>(h->comm), h->stream));
    h->launches++;
    return MS_OK;
}

// used by linkage.cu: in-place int32 sum of the stacked Gram matrix over the ranks, on the handle's stream
int ms_comm_allreduce_i32(ms_handle* h, int32_t* d, size_t count) {
    if (!h->comm) return MS_ERR_ARG;
    MS_STAGE_BEGIN(h, MS_STAGE_LINKAGE_ALLREDUCE);
    MS_NCCL(h, api().AllReduce(d, d, count, ncclInt32, ncclSum, static_cast<ncclComm_t>(h->comm), h->stream));
    MS_STAGE_END(h, MS_STAGE_LINKAGE_ALLREDUCE);
    h->launches++;
    return MS_OK;
}

// used by indel.cu: in-place u32 sum of the indel counts over the ranks, on the handle's stream
int ms_comm_allreduce_u32(ms_handle* h, uint32_t* d, size_t count) {
    if (!h->comm) return MS_ERR_ARG;
    MS_NCCL(h, api().AllReduce(d, d, count, ncclUint32, ncclSum, static_cast<ncclComm_t>(h->comm), h->stream));
    h->launches++;
    return MS_OK;
}

extern "C" void ms_comm_free_internal(ms_handle* h) {
    if (h->comm && api().ok) api().CommDestroy(static_cast<ncclComm_t>(h->comm));
    h->comm = nullptr;
    h->world = 1; h->rank = 0;
}

extern "C" {

int ms_comm_unique_id(char id[128]) {
    if (!id || !api().ok) return MS_ERR_NODEVICE;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId u;
    if (api().GetUniqueId(&u) != ncclSuccess) return MS_ERR_CUDA;
    memcpy(id, &u, 128);
    return MS_OK;
}

int ms_comm_init(ms_handle* h, const char id[128], int rank, int world) {
    if (!h || !id || world < 1 || rank < 0 || rank >= world) return MS_ERR_ARG;
    if (!api().ok) MS_FAIL(h, MS_ERR_NODEVICE, "libnccl.so.2 could not be loaded");
    MS_CUDA(h, cudaSetDevice(h->device));
    ms_comm_free_internal(h);
    h->gcap_hint = 0;   // sizes of the phasing exchange: every rank of the new communicator starts from the same value
    if (world == 1) return MS_OK;
    ncclUniqueId u;
    memcpy(&u, id, 128);
    ncclComm_t c;
    MS_NCCL(h, api().CommInitRank(&c, world, u, rank));
    h->comm = c; h->world = world; h->rank = rank;
    return MS_OK;
}

int ms_comm_size(const ms_handle* h) { return h ? h->world : 0; }

int ms_allreduce_counts(ms_handle* h) {
    MsRange nvtx_range("all-reduce counts");
    if (!h || !h->d_counts) return MS_ERR_ARG;
    if (!h->comm) return MS_OK;  // single rank
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_STAGE_BEGIN(h, MS_STAGE_ALLREDUCE);
    MS_NCCL(h, api().AllReduce(h->d_counts, h->d_counts, static_cast<size_t>(h->L) * 72, ncclUint32, ncclSum,
                               static_cast<ncclComm_t>(h->comm), h->stream));
    MS_STAGE_END(h, MS_STAGE_ALLREDUCE);
    h->launches++;
    return MS_OK;
}

int ms_allreduce_group_counts(ms_handle* h) {
    MsRange nvtx_range("all-reduce group counts");
    if (!h || h->label_groups < 0 || h->label_L != h->L) return MS_ERR_ARG;
    if (!h->comm || h->label_groups == 0) return MS_OK;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_NCCL(h, api().AllReduce(h->b_gcol.p, h->b_gcol.p, static_cast<size_t>(h->label_groups) * h->L * 8, ncclUint32, ncclSum,
                               static_cast<ncclComm_t>(h->comm), h->stream));
    h->launches++;
    return MS_OK;
}

}  // extern "C"
