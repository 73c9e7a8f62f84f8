// Peer mailboxes for the row-sharded coreset loop (SURVEY 8e): every rank owns one device buffer that all ranks of the
// box can write over NVLink (CUDA IPC mapping, one process per GPU).  The persistent coreset kernel uses it for the
// per-pick exchange of (value,row) candidates and of the winning row itself -- no host launch, no NCCL call per pick.
#include <algorithm>
#include <memory>

#include "common.cuh"

struct cmdb_comm {
    int device = 0, rank = 0, world = 1;
    size_t bytes = 0;
    cmdb::Buffer<unsigned char> local;              // this rank's mailbox
    unsigned char *peer[cmdb::kMaxRanks] = {};      // every rank's mailbox as mapped into this process (peer[rank] == local)
    bool imported = false;
    unsigned long long score_epoch = 0;  // round counter of the sharded-scoring exchange (monotone per buffer, same on every rank)
    ~cmdb_comm() {   // peers may still write into the mailbox: synchronise, close the imported mappings, then free it
        cudaSetDevice(device);
        cudaDeviceSynchronize();
        for (int r = 0; r < world; ++r)
            if (r != rank && peer[r]) cudaIpcCloseMemHandle(peer[r]);
    }
};

using namespace cmdb;

extern "C" {

int cmdb_comm_create(int device, int rank, int world, size_t mailbox_bytes, cmdb_comm **out) {
    CMDB_REQUIRE(out, CMDB_ERR_INVALID, "cmdb_comm_create: out is NULL");
    *out = nullptr;
    CMDB_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world, CMDB_ERR_INVALID,
                 "cmdb_comm_create: rank %d / world %d not supported (max %d ranks)", rank, world, kMaxRanks);
    CMDB_REQUIRE(mailbox_bytes >= 64, CMDB_ERR_INVALID, "cmdb_comm_create: mailbox too small");
    CMDB_CUDA(cudaSetDevice(device));
    std::unique_ptr<cmdb_comm> c(new cmdb_comm());
    c->device = device, c->rank = rank, c->world = world, c->bytes = (mailbox_bytes + 255) & ~size_t(255);
    cudaError_t e = c->local.alloc(c->bytes);
    if (e != cudaSuccess || (e = cudaMemset(c->local, 0, c->bytes)) != cudaSuccess) {
        set_error("cmdb_comm_create: %s", cudaGetErrorString(e));
        (void)cudaGetLastError();
        return CMDB_ERR_CUDA;
    }
    c->peer[rank] = c->local;
    *out = c.release();
    return CMDB_OK;
}

int cmdb_comm_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

int cmdb_comm_export(cmdb_comm *c, void *handle_out) {
    CMDB_REQUIRE(c && handle_out, CMDB_ERR_INVALID, "cmdb_comm_export: bad arguments");
    CMDB_CUDA(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    CMDB_CUDA(cudaIpcGetMemHandle(&h, c->local));
    memcpy(handle_out, &h, sizeof(h));
    return CMDB_OK;
}

// handles: [world][cmdb_comm_handle_bytes()] as gathered from every rank's cmdb_comm_export
int cmdb_comm_import(cmdb_comm *c, const void *handles) {
    CMDB_REQUIRE(c && handles, CMDB_ERR_INVALID, "cmdb_comm_import: bad arguments");
    CMDB_REQUIRE(!c->imported, CMDB_ERR_STATE, "cmdb_comm_import: already imported");
    CMDB_CUDA(cudaSetDevice(c->device));
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const unsigned char *)handles + (size_t)r * sizeof(h), sizeof(h));
        void *p = nullptr;
        CMDB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        c->peer[r] = (unsigned char *)p;
    }
    c->imported = true;
    return CMDB_OK;
}

// Clears this rank's mailbox.  Call on every rank, then BARRIER, before each cmdb_coreset_select_sharded: pick epochs
// restart at 1 per call and a peer may begin writing as soon as it enters the kernel.
int cmdb_comm_reset(cmdb_comm *c) {
    CMDB_REQUIRE(c, CMDB_ERR_INVALID, "cmdb_comm_reset: comm is NULL");
    CMDB_CUDA(cudaSetDevice(c->device));
    // flags + key slots only: the replica region behind them is rewritten by every call anyway
    CMDB_CUDA(cudaMemset(c->local, 0, std::min(c->bytes, kCommCoresetBytes)));
    CMDB_CUDA(cudaDeviceSynchronize());
    return CMDB_OK;
}

void cmdb_comm_destroy(cmdb_comm *c) { delete c; }

}  // extern "C"

namespace cmdb {
unsigned long long comm_next_score_epoch(cmdb_comm *c) { return ++c->score_epoch; }

int comm_info(cmdb_comm *c, int *rank, int *world, unsigned char **local, unsigned char **peers, size_t *bytes) {
    CMDB_REQUIRE(c && (c->world == 1 || c->imported), CMDB_ERR_STATE, "comm: call cmdb_comm_import on every rank first");
    *rank = c->rank, *world = c->world, *local = c->local, *bytes = c->bytes;
    for (int r = 0; r < kMaxRanks; ++r) peers[r] = c->peer[r];
    return CMDB_OK;
}
}  // namespace cmdb
