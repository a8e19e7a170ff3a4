// Collectives of the table-wise sharded path behind the C ABI (dlrmb_comm_*): a host that is not
// Python -- DLRM.jl through ccall -- can run BASELINE config 4 without torch.distributed.
//
// New functionality (DLRM.jl is single-process); BASELINE.json north_star / SURVEY.md section 8(b),
// 8(e).  One process per GPU; rank 0 creates an NCCL unique id (dlrmb_comm_unique_id), the host
// program carries its 128 bytes to the other ranks by whatever means it has (a file, a socket, MPI)
// and every rank calls dlrmb_comm_create.  All calls are stream-ordered and must be issued in the
// same order on every rank.
//
//   dlrmb_shard_plan          which rank owns which table (lookup count first, bytes second)
//   dlrmb_shard_plan_mp       the same with per-table pooling factors (weighted by P_k when they differ)
//   dlrmb_comm_a2a_indices    idx_local [ntab][B_local][P] -> idx_owned [t_mine][B_global][P]
//   dlrmb_comm_a2a_indices_mp the `_mp` layout at B_local -> this rank's tables' `_mp` layout at B_global
//   dlrmb_comm_a2a_fwd        pooled [B_global][t_mine][D] (owner) -> T [B_local][1 + ntab][D]
//   dlrmb_comm_a2a_bwd        dT [B_local][1 + ntab][D] -> grads [B_global][t_mine][D] (owner)
//   dlrmb_comm_allreduce_f32  data-parallel dense gradients (sum, in place)
//   dlrmb_comm_allgather      small fixed-size blobs (the IPC handles of dlrmb_xbuf, for the fused
//                             peer-store exchanges of p2p.cu / dlrmb_interaction_bwd_scatter)
//
// NCCL is bound at run time (dlopen of the libnccl.so.2 already in the process, else the system's),
// so libdlrm_b200.so has no link-time dependency on it and single-GPU users never load it.
#include <dlfcn.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace dlrmb {
namespace {

// The slice of the NCCL 2.x API used here (declarations are ABI-stable across 2.x).
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclInt64 = 4, ncclFloat32 = 7 };
enum { ncclSum = 0 };

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

NcclApi& nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);   // the copy the process already uses (torch's)
            if (api.handle) break;
        }
        for (int i = 0; !api.handle && i < 2; ++i) api.handle = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
        if (!api.handle) return;
#define BIND(field, sym) *(void**)(&api.field) = dlsym(api.handle, sym)
        BIND(GetUniqueId, "ncclGetUniqueId");
        BIND(CommInitRank, "ncclCommInitRank");
        BIND(CommDestroy, "ncclCommDestroy");
        BIND(GroupStart, "ncclGroupStart");
        BIND(GroupEnd, "ncclGroupEnd");
        BIND(Send, "ncclSend");
        BIND(Recv, "ncclRecv");
        BIND(AllReduce, "ncclAllReduce");
        BIND(AllGather, "ncclAllGather");
        BIND(GetErrorString, "ncclGetErrorString");
#undef BIND
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.GroupStart && api.GroupEnd && api.Send &&
                 api.Recv && api.AllReduce && api.AllGather && api.GetErrorString;
    });
    return api;
}

#define DLRMB_NCCL(expr)                                                                          \
    do {                                                                                          \
        ncclResult_t _r = (expr);                                                                 \
        if (_r != 0) {                                                                            \
            ::dlrmb::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, nccl().GetErrorString(_r)); \
            return DLRMB_ENCCL;                                                                   \
        }                                                                                         \
    } while (0)

// T[b][slot_of[j]][:] <-> packed[b][j][:] for one peer's block of tables, 16 bytes per thread
template <bool UNPACK>
__global__ void __launch_bounds__(256)
a2a_reorder_kernel(float* __restrict__ T, float* __restrict__ packed, const int32_t* __restrict__ slot_of, int B, int nt,
                   int slots, int C4) {
    const int64_t n = (int64_t)B * nt * C4;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const int c = (int)(i % C4);
        const int64_t r = i / C4;
        const int j = (int)(r % nt);
        const int64_t b = r / nt;
        float4* t = reinterpret_cast<float4*>(T) + ((size_t)b * slots + slot_of[j]) * C4 + c;
        float4* p = reinterpret_cast<float4*>(packed) + (size_t)i;
        if (UNPACK) *t = *p;
        else *p = *t;
    }
}

}  // namespace
}  // namespace dlrmb

struct dlrmb_comm {
    int device = 0, rank = 0, world = 1;
    dlrmb::ncclComm_t comm = nullptr;
    float* stage = nullptr;          // packed exchange buffer
    size_t stage_bytes = 0;
    int32_t* d_slots = nullptr;      // [ntab] interaction slots grouped by owner rank
    int ntab_cached = 0;
    std::vector<int32_t> owner_cached;
    std::vector<std::vector<int>> local;   // local[r] = tables of rank r, ascending
    int sm_count = 148;
};

using namespace dlrmb;

static int comm_prepare(dlrmb_comm* c, const int32_t* owner, int ntab, size_t need_bytes) {
    DLRMB_REQUIRE(c != nullptr && owner != nullptr && ntab > 0, "bad comm arguments");
    bool same = (c->ntab_cached == ntab) && std::equal(owner, owner + ntab, c->owner_cached.begin());
    if (!same) {
        c->local.assign(c->world, {});
        for (int k = 0; k < ntab; ++k) {
            DLRMB_REQUIRE(owner[k] >= 0 && owner[k] < c->world, "owner[%d] = %d outside 0..%d", k, owner[k], c->world - 1);
            c->local[owner[k]].push_back(k);
        }
        std::vector<int32_t> slots;
        for (int r = 0; r < c->world; ++r)
            for (int k : c->local[r]) slots.push_back(1 + k);
        if (c->d_slots) DLRMB_CUDA(cudaFree(c->d_slots));
        c->d_slots = nullptr;
        DLRMB_CUDA(cudaMalloc((void**)&c->d_slots, sizeof(int32_t) * ntab));
        DLRMB_CUDA(cudaMemcpy(c->d_slots, slots.data(), sizeof(int32_t) * ntab, cudaMemcpyHostToDevice));
        c->owner_cached.assign(owner, owner + ntab);
        c->ntab_cached = ntab;
    }
    if (c->stage_bytes < need_bytes) {
        if (c->stage) DLRMB_CUDA(cudaFree(c->stage));
        c->stage = nullptr;
        c->stage_bytes = 0;
        DLRMB_CUDA(cudaMalloc((void**)&c->stage, need_bytes));
        c->stage_bytes = need_bytes;
    }
    return DLRMB_OK;
}

extern "C" {

int32_t dlrmb_shard_plan(int32_t ntab, const int64_t* rows, int32_t world, int32_t* owner) {
    DLRMB_REQUIRE(ntab > 0 && rows && owner && world > 0, "bad shard plan arguments");
    // every table receives B_global * P lookups per step whatever its size, so balance the table COUNT
    // first, then bytes: deal the tables in descending row count, snake order
    std::vector<int> order(ntab);
    for (int k = 0; k < ntab; ++k) order[k] = k;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rows[a] > rows[b]; });
    for (int i = 0; i < ntab; ++i) {
        const int rnd = i / world, pos = i % world;
        owner[order[i]] = (rnd % 2 == 0) ? pos : world - 1 - pos;
    }
    return DLRMB_OK;
}

int32_t dlrmb_shard_plan_mp(int32_t ntab, const int64_t* rows, const int32_t* P, int32_t world, int32_t* owner) {
    DLRMB_REQUIRE(ntab > 0, "ntab must be positive (got %d)", ntab);
    DLRMB_REQUIRE(world > 0, "world must be positive (got %d)", world);
    DLRMB_REQUIRE(rows && owner, "null argument");
    DLRMB_REQUIRE(P != nullptr, "P (per-table pooling factors) is null");
    bool uniform = true;
    for (int k = 0; k < ntab; ++k) {
        DLRMB_REQUIRE(P[k] >= 1, "P[%d] = %d: every pooling factor must be >= 1", k, P[k]);
        uniform = uniform && P[k] == P[0];
    }
    if (uniform) return dlrmb_shard_plan(ntab, rows, world, owner);
    // table k receives B_global * P_k lookups per step: deal the tables longest first (descending P_k, then
    // rows, then id), each to the rank with the fewest lookups so far (ties: fewer rows, then lower rank)
    std::vector<int> order(ntab);
    for (int k = 0; k < ntab; ++k) order[k] = k;
    std::sort(order.begin(), order.end(), [&](int a, int b) {
        if (P[a] != P[b]) return P[a] > P[b];
        if (rows[a] != rows[b]) return rows[a] > rows[b];
        return a < b;
    });
    std::vector<int64_t> load(world, 0), bytes(world, 0);
    for (int k : order) {
        int best = 0;
        for (int r = 1; r < world; ++r)
            if (load[r] < load[best] || (load[r] == load[best] && bytes[r] < bytes[best])) best = r;
        owner[k] = best;
        load[best] += P[k];
        bytes[best] += rows[k];
    }
    return DLRMB_OK;
}

int32_t dlrmb_shard_plan_cw(int32_t ntab, const int64_t* rows, const int32_t* P, int32_t world, int32_t D, int32_t S,
                            int32_t* shards, int32_t* owner) {
    DLRMB_REQUIRE(ntab > 0, "ntab must be positive (got %d)", ntab);
    DLRMB_REQUIRE(world > 0, "world must be positive (got %d)", world);
    DLRMB_REQUIRE(rows && shards && owner, "null argument");
    DLRMB_REQUIRE(P != nullptr, "P (per-table pooling factors) is null");
    DLRMB_REQUIRE(S >= 1 && (S & (S - 1)) == 0, "max_col_shards must be a power of two (got %d)", S);
    DLRMB_REQUIRE(D >= 1, "D must be positive (got %d)", D);
    DLRMB_REQUIRE(S == 1 || (D % S == 0 && (D / S) % 4 == 0),
                  "D / max_col_shards must be a multiple of 4 (D = %d, max_col_shards = %d)", D, S);
    int64_t total = 0;
    for (int k = 0; k < ntab; ++k) {
        DLRMB_REQUIRE(P[k] >= 1, "P[%d] = %d: every pooling factor must be >= 1", k, P[k]);
        total += P[k];
    }
    // halve the hottest table's columns while its share P_k / c_k is above the even share sum(P) / world
    std::vector<int64_t> c(ntab, 1);
    const int64_t cmax = S < world ? S : world;
    for (;;) {
        int k = 0;
        for (int i = 1; i < ntab; ++i) {   // largest P_i / c_i, then more rows, then the lower id
            const int64_t lhs = (int64_t)P[i] * c[k], rhs = (int64_t)P[k] * c[i];
            if (lhs > rhs || (lhs == rhs && rows[i] > rows[k])) k = i;
        }
        if ((int64_t)P[k] * world <= c[k] * total || 2 * c[k] > cmax) break;
        c[k] *= 2;
    }
    int64_t M = 1;
    for (int k = 0; k < ntab; ++k) M = c[k] > M ? c[k] : M;
    for (int k = 0; k < ntab; ++k) {
        shards[k] = (int32_t)c[k];
        for (int j = 0; j < S; ++j) owner[(size_t)k * S + j] = -1;
    }
    if (M == 1) {   // nothing split: the table-wise plan
        std::vector<int32_t> own(ntab);
        int rc = dlrmb_shard_plan_mp(ntab, rows, P, world, own.data());
        if (rc) return rc;
        for (int k = 0; k < ntab; ++k) owner[(size_t)k * S] = own[k];
        return DLRMB_OK;
    }
    // deal the units (k, j) longest first; loads and bytes in units of 1 / M (exact: every c_k divides M)
    std::vector<std::pair<int, int>> units;
    for (int k = 0; k < ntab; ++k)
        for (int j = 0; j < c[k]; ++j) units.emplace_back(k, j);
    std::sort(units.begin(), units.end(), [&](const std::pair<int, int>& a, const std::pair<int, int>& b) {
        const int64_t lhs = (int64_t)P[a.first] * c[b.first], rhs = (int64_t)P[b.first] * c[a.first];
        if (lhs != rhs) return lhs > rhs;
        if (rows[a.first] != rows[b.first]) return rows[a.first] > rows[b.first];
        if (a.first != b.first) return a.first < b.first;
        return a.second < b.second;
    });
    std::vector<int64_t> load(world, 0), bytes(world, 0);
    for (const auto& u : units) {
        const int k = u.first;
        int best = -1;
        for (int r = 0; r < world; ++r) {
            bool holds = false;
            for (int j = 0; j < c[k]; ++j) holds = holds || owner[(size_t)k * S + j] == r;
            if (holds) continue;
            if (best < 0 || load[r] < load[best] || (load[r] == load[best] && bytes[r] < bytes[best])) best = r;
        }
        owner[(size_t)k * S + u.second] = best;
        load[best] += (int64_t)P[k] * (M / c[k]);
        bytes[best] += rows[k] * (M / c[k]);
    }
    return DLRMB_OK;
}

int32_t dlrmb_comm_unique_id(uint8_t* id128) {
    DLRMB_REQUIRE(id128 != nullptr, "id buffer is null");
    if (!nccl().ok) {
        set_error("libnccl.so.2 could not be loaded (%s)", dlerror() ? dlerror() : "symbols missing");
        return DLRMB_ENCCL;
    }
    ncclUniqueId id;
    DLRMB_NCCL(nccl().GetUniqueId(&id));
    memcpy(id128, id.internal, 128);
    return DLRMB_OK;
}

int32_t dlrmb_comm_create(int32_t device, const uint8_t* id128, int32_t rank, int32_t world, dlrmb_comm** out) {
    DLRMB_REQUIRE(out != nullptr && id128 != nullptr, "null argument");
    *out = nullptr;
    DLRMB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "rank %d outside 0..%d", rank, world - 1);
    if (!nccl().ok) {
        set_error("libnccl.so.2 could not be loaded");
        return DLRMB_ENCCL;
    }
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    ncclUniqueId id;
    memcpy(id.internal, id128, 128);
    ncclComm_t comm = nullptr;
    DLRMB_NCCL(nccl().CommInitRank(&comm, world, id, rank));
    dlrmb_comm* c = new dlrmb_comm();
    c->device = device;
    c->rank = rank;
    c->world = world;
    c->comm = comm;
    c->sm_count = device_sm_count(device);
    *out = c;
    return DLRMB_OK;
}

int32_t dlrmb_comm_destroy(dlrmb_comm* c) {
    if (!c) return DLRMB_OK;
    DeviceGuard guard(c->device);
    cudaDeviceSynchronize();
    if (c->comm) nccl().CommDestroy(c->comm);
    cudaFree(c->stage);
    cudaFree(c->d_slots);
    delete c;
    return DLRMB_OK;
}

int32_t dlrmb_comm_info(const dlrmb_comm* c, int32_t* rank, int32_t* world) {
    DLRMB_REQUIRE(c != nullptr, "null comm");
    if (rank) *rank = c->rank;
    if (world) *world = c->world;
    return DLRMB_OK;
}

int32_t dlrmb_comm_a2a_indices(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const void* idx_local,
                               int32_t idx_bytes, int32_t B_local, int32_t P, void* idx_owned, dlrmb_stream stream) {
    DLRMB_REQUIRE(c && idx_local && idx_owned, "null argument");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(B_local > 0 && P > 0, "B_local and P must be positive");
    DeviceGuard guard(c->device);
    int rc = comm_prepare(c, owner, ntab, 0);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t msg = (size_t)B_local * P * idx_bytes;            // one table's indices of one rank's samples
    const char* src = static_cast<const char*>(idx_local);
    char* dst = static_cast<char*>(idx_owned);
    const std::vector<int>& mine = c->local[c->rank];
    DLRMB_NCCL(nccl().GroupStart());
    for (int k = 0; k < ntab; ++k)                                  // table k of my samples -> its owner
        DLRMB_NCCL(nccl().Send(src + (size_t)k * msg, msg, ncclInt8, owner[k], c->comm, s));
    for (int h = 0; h < c->world; ++h)                              // rank h's samples of my table j
        for (size_t j = 0; j < mine.size(); ++j)
            DLRMB_NCCL(nccl().Recv(dst + ((size_t)j * c->world + h) * msg, msg, ncclInt8, h, c->comm, s));
    DLRMB_NCCL(nccl().GroupEnd());
    return DLRMB_OK;
}

int32_t dlrmb_comm_a2a_indices_mp(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const void* idx_local,
                                  int32_t idx_bytes, int32_t B_local, const int32_t* P, void* idx_owned,
                                  dlrmb_stream stream) {
    DLRMB_REQUIRE(c && idx_local && idx_owned, "null argument");
    DLRMB_REQUIRE(P != nullptr, "P (per-table pooling factors) is null");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(B_local > 0, "B_local must be positive");
    for (int k = 0; k < ntab; ++k) DLRMB_REQUIRE(P[k] >= 1, "P[%d] = %d: every pooling factor must be >= 1", k, P[k]);
    DeviceGuard guard(c->device);
    int rc = comm_prepare(c, owner, ntab, 0);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const char* src = static_cast<const char*>(idx_local);
    char* dst = static_cast<char*>(idx_owned);
    const std::vector<int>& mine = c->local[c->rank];
    const size_t Bg = (size_t)B_local * c->world;
    DLRMB_NCCL(nccl().GroupStart());
    size_t off = 0;                                                 // elements: table k's block of my samples
    for (int k = 0; k < ntab; ++k) {
        const size_t n = (size_t)B_local * P[k];
        DLRMB_NCCL(nccl().Send(src + off * idx_bytes, n * idx_bytes, ncclInt8, owner[k], c->comm, s));
        off += n;
    }
    for (int h = 0; h < c->world; ++h) {                            // rank h's samples of my table j: rows
        size_t base = 0;                                            // [h * B_local, (h + 1) * B_local) of its block
        for (int k : mine) {
            const size_t n = (size_t)B_local * P[k];
            DLRMB_NCCL(nccl().Recv(dst + (base + (size_t)h * n) * idx_bytes, n * idx_bytes, ncclInt8, h, c->comm, s));
            base += Bg * P[k];
        }
    }
    DLRMB_NCCL(nccl().GroupEnd());
    return DLRMB_OK;
}

int32_t dlrmb_comm_a2a_fwd(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const float* pooled, int32_t B_local,
                           int32_t D, float* T, dlrmb_stream stream) {
    DLRMB_REQUIRE(c && T, "null argument");
    DLRMB_REQUIRE(B_local > 0 && D > 0 && D % 4 == 0, "B_local must be positive and D a multiple of 4");
    DeviceGuard guard(c->device);
    const size_t recv_floats = (size_t)B_local * ntab * D;
    int rc = comm_prepare(c, owner, ntab, recv_floats * sizeof(float));
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t t_mine = c->local[c->rank].size();
    DLRMB_REQUIRE(t_mine == 0 || pooled != nullptr, "pooled is null");
    DLRMB_NCCL(nccl().GroupStart());
    size_t off = 0;
    for (int h = 0; h < c->world; ++h) {
        if (t_mine)   // my tables, rank h's samples: rows [h * B_local, (h + 1) * B_local) of pooled
            DLRMB_NCCL(nccl().Send(pooled + (size_t)h * B_local * t_mine * D, (size_t)B_local * t_mine * D, ncclFloat32, h, c->comm, s));
        const size_t th = c->local[h].size();
        if (th) DLRMB_NCCL(nccl().Recv(c->stage + off, (size_t)B_local * th * D, ncclFloat32, h, c->comm, s));
        off += (size_t)B_local * th * D;
    }
    DLRMB_NCCL(nccl().GroupEnd());
    off = 0;
    int done = 0;
    for (int h = 0; h < c->world; ++h) {      // packed [B_local][t_h][D] -> T[:, 1 + k, :]
        const int th = (int)c->local[h].size();
        if (!th) continue;
        const int64_t n = (int64_t)B_local * th * (D / 4);
        int64_t blocks = ceil_div64(n, 256 * 4);
        if (blocks > (int64_t)c->sm_count * 8) blocks = (int64_t)c->sm_count * 8;
        a2a_reorder_kernel<true><<<(unsigned)blocks, 256, 0, s>>>(T, c->stage + off, c->d_slots + done, B_local, th, 1 + ntab, D / 4);
        DLRMB_LAUNCH_CHECK();
        off += (size_t)B_local * th * D;
        done += th;
    }
    return DLRMB_OK;
}

int32_t dlrmb_comm_a2a_bwd(dlrmb_comm* c, const int32_t* owner, int32_t ntab, const float* dT, int32_t B_local,
                           int32_t D, float* grads, dlrmb_stream stream) {
    DLRMB_REQUIRE(c && dT, "null argument");
    DLRMB_REQUIRE(B_local > 0 && D > 0 && D % 4 == 0, "B_local must be positive and D a multiple of 4");
    DeviceGuard guard(c->device);
    const size_t send_floats = (size_t)B_local * ntab * D;
    int rc = comm_prepare(c, owner, ntab, send_floats * sizeof(float));
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t t_mine = c->local[c->rank].size();
    DLRMB_REQUIRE(t_mine == 0 || grads != nullptr, "grads is null");
    size_t off = 0;
    int done = 0;
    for (int h = 0; h < c->world; ++h) {      // dT[:, 1 + k, :] of rank h's tables -> packed [B_local][t_h][D]
        const int th = (int)c->local[h].size();
        if (!th) continue;
        const int64_t n = (int64_t)B_local * th * (D / 4);
        int64_t blocks = ceil_div64(n, 256 * 4);
        if (blocks > (int64_t)c->sm_count * 8) blocks = (int64_t)c->sm_count * 8;
        a2a_reorder_kernel<false><<<(unsigned)blocks, 256, 0, s>>>(const_cast<float*>(dT), c->stage + off, c->d_slots + done, B_local,
                                                                 th, 1 + ntab, D / 4);
        DLRMB_LAUNCH_CHECK();
        off += (size_t)B_local * th * D;
        done += th;
    }
    DLRMB_NCCL(nccl().GroupStart());
    off = 0;
    for (int h = 0; h < c->world; ++h) {
        const size_t th = c->local[h].size();
        if (th) DLRMB_NCCL(nccl().Send(c->stage + off, (size_t)B_local * th * D, ncclFloat32, h, c->comm, s));
        off += (size_t)B_local * th * D;
        if (t_mine)
            DLRMB_NCCL(nccl().Recv(grads + (size_t)h * B_local * t_mine * D, (size_t)B_local * t_mine * D, ncclFloat32, h, c->comm, s));
    }
    DLRMB_NCCL(nccl().GroupEnd());
    return DLRMB_OK;
}

int32_t dlrmb_comm_allreduce_f32(dlrmb_comm* c, float* buf, int64_t n, dlrmb_stream stream) {
    DLRMB_REQUIRE(c && buf && n > 0, "bad all-reduce arguments");
    DeviceGuard guard(c->device);
    DLRMB_NCCL(nccl().AllReduce(buf, buf, (size_t)n, ncclFloat32, ncclSum, c->comm, (cudaStream_t)stream));
    return DLRMB_OK;
}

int32_t dlrmb_comm_allgather(dlrmb_comm* c, const void* send, void* recv, int64_t nbytes, dlrmb_stream stream) {
    DLRMB_REQUIRE(c && send && recv && nbytes > 0, "bad all-gather arguments");
    DeviceGuard guard(c->device);
    DLRMB_NCCL(nccl().AllGather(send, recv, (size_t)nbytes, ncclInt8, c->comm, (cudaStream_t)stream));
    return DLRMB_OK;
}

}  // extern "C"
