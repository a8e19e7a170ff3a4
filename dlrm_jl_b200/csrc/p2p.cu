// Fused lookup + exchange for table-wise sharded embeddings: the owner of a table pools its rows
// for the GLOBAL batch and stores every pooled row straight into the interaction input buffer of
// the rank that owns the sample, through NVLink peer mappings (cudaIpc).  This replaces
// "lookup -> staging buffer -> NCCL all-to-all -> unpack" (dlrm_jl_b200/sharded.py) by one kernel:
// the transfer is the kernel's own store stream, posted row by row (whole 128-byte lines), so it
// overlaps the gathers that are still in flight.
//
// New functionality (DLRM.jl is single-process); BASELINE.json north_star / SURVEY.md section 8(e).
#include "common.cuh"
#include "sort_small.cuh"

#include <vector>

struct dlrmb_xbuf {
    int device;
    void* ptr;
    size_t bytes;
};

namespace dlrmb {

constexpr int kMaxPeers = 16;
struct PeerPtrs {
    float* p[kMaxPeers];
};

template <int VEC, typename RowT>
__device__ __forceinline__ typename std::conditional<VEC == 4, float4, float>::type
p2p_ldrow(const float* base, size_t r, size_t D, int c) {
    if constexpr (VEC == 4) return RowIO<RowT>::ldg4(RowIO<RowT>::row(base, r, D), c);
    else return RowIO<RowT>::ldg1(RowIO<RowT>::row(base, r, D), c);
}

int ensure_smem_attr(const void* func, int bytes, unsigned long long* done_mask);

// The lookup's geometry (one flat grid, table k owns CTAs [g.pre[k], g.pre[k+1]) in proportion to
// B_global * P_k * C, lookup_grid_mp of lookup.cu) with a peer-store epilogue: sample b lives on rank
// b / B_local and table k lands at element dstoff[k] of the sample's destination row (slot * D_dest + col0, the
// dest map of dlrmb_tables_set_dest_map; rows are `ostride` floats apart).  P_k == 1 takes the U-chain gather, every other table
// the 4-deep pooling loop in ascending p (the lookup's order, so the pooled rows are bit-identical to
// dlrmb_embedding_fwd).  With SORT_ITEMS > 0 the first g.nlist CTAs sort the tables g.list[]
// (B_global * P_k <= kFusedSortMax) in shared memory, as lookup_sort_mp_kernel does.  Both parameter structs go by value (__grid_constant__: peers.p[h] is read
// with a run-time h straight from the parameter bank), so the launch needs no device copy.
__device__ __forceinline__ float4 p2p_add(float4 a, float4 b) {
    return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}
__device__ __forceinline__ float p2p_add(float a, float b) { return __fadd_rn(a, b); }

template <typename IdxT, int VEC, int U, typename RowT>
__device__ __forceinline__ void lookup_p2p_mp_cta(const TableDesc* __restrict__ desc, const int32_t* __restrict__ dstoff,
                                                  const IdxT* __restrict__ idx, int idx_base, const MpGeom& g,
                                                  uint32_t C, int cshift, uint32_t B_local, const PeerPtrs& peers,
                                                  long long ostride, uint32_t lin) {
    using V = typename std::conditional<VEC == 4, float4, float>::type;
    const int k = mp_find(g.pre, g.ntab, lin);
    const uint32_t cx = lin - g.pre[k], nctas = g.pre[k + 1] - g.pre[k];
    const float* __restrict__ tb = desc[k].base;
    const IdxT* __restrict__ ik = idx + g.off[k];
    const uint32_t P = g.P[k];
    const uint32_t n = g.B * C;
    const uint32_t step = nctas * blockDim.x;
    const size_t D = (size_t)C * VEC;
    const size_t slot_off = (size_t)dstoff[k];

    if (P == 1) {
        for (uint32_t t = cx * blockDim.x + threadIdx.x; t < n; t += step * U) {
            int64_t row[U];
            uint32_t b[U], c[U];
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t tt = t + (uint32_t)u * step;
                ok[u] = tt < n;
                b[u] = cshift >= 0 ? (tt >> cshift) : (tt / C);
                c[u] = tt - b[u] * C;
                row[u] = ok[u] ? (int64_t)__ldg(ik + b[u]) - idx_base : 0;
            }
            V v[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (ok[u]) v[u] = p2p_ldrow<VEC, RowT>(tb, (size_t)row[u], D, c[u]);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (!ok[u]) continue;
                const uint32_t h = b[u] / B_local;
                const uint32_t bl = b[u] - h * B_local;
                reinterpret_cast<V*>(peers.p[h] + (size_t)bl * ostride + slot_off)[c[u]] = v[u];
            }
        }
        return;
    }
    for (uint32_t t = cx * blockDim.x + threadIdx.x; t < n; t += step) {
        const uint32_t b = cshift >= 0 ? (t >> cshift) : (t / C);
        const uint32_t c = t - b * C;
        const IdxT* __restrict__ ip = ik + (size_t)b * P;
        V acc;
        if constexpr (VEC == 4) acc = make_float4(0.f, 0.f, 0.f, 0.f);
        else acc = 0.f;
        uint32_t p = 0;
        for (; p + 4 <= P; p += 4) {
            const int64_t r0 = (int64_t)__ldg(ip + p) - idx_base;
            const int64_t r1 = (int64_t)__ldg(ip + p + 1) - idx_base;
            const int64_t r2 = (int64_t)__ldg(ip + p + 2) - idx_base;
            const int64_t r3 = (int64_t)__ldg(ip + p + 3) - idx_base;
            const V v0 = p2p_ldrow<VEC, RowT>(tb, (size_t)r0, D, c);
            const V v1 = p2p_ldrow<VEC, RowT>(tb, (size_t)r1, D, c);
            const V v2 = p2p_ldrow<VEC, RowT>(tb, (size_t)r2, D, c);
            const V v3 = p2p_ldrow<VEC, RowT>(tb, (size_t)r3, D, c);
            acc = p2p_add(acc, v0);
            acc = p2p_add(acc, v1);
            acc = p2p_add(acc, v2);
            acc = p2p_add(acc, v3);
        }
        for (; p < P; ++p)
            acc = p2p_add(acc, p2p_ldrow<VEC, RowT>(tb, (size_t)((int64_t)__ldg(ip + p) - idx_base), D, c));
        const uint32_t h = b / B_local;
        const uint32_t bl = b - h * B_local;
        reinterpret_cast<V*>(peers.p[h] + (size_t)bl * ostride + slot_off)[c] = acc;
    }
}

template <typename IdxT, int VEC, int U, typename RowT, int SORT_ITEMS>
__global__ void __launch_bounds__(256, (SORT_ITEMS > 0) ? 4 : 1)
lookup_p2p_mp_kernel(const TableDesc* __restrict__ desc, const int32_t* __restrict__ dstoff, const IdxT* __restrict__ idx,
                     int idx_base, const __grid_constant__ MpGeom g, uint32_t C, int cshift, uint32_t B_local,
                     const __grid_constant__ PeerPtrs peers, long long ostride, uint32_t* __restrict__ keys_out,
                     uint32_t* __restrict__ pos_out, int64_t cap, unsigned long long* clk) {
    clock_in(clk, blockIdx.x);
    uint32_t lin = blockIdx.x;
    if constexpr (SORT_ITEMS > 0) {
        extern __shared__ uint32_t sort_smem[];
        if ((int)blockIdx.x < g.nlist) {
            const int k = g.list[blockIdx.x];
            sort_small_body<IdxT, SORT_ITEMS, 256>(idx + g.off[k], idx_base, (int)(g.B * g.P[k]), desc[k].rows,
                                                   keys_out + (size_t)k * cap, pos_out + (size_t)k * cap, sort_smem);
            clock_out(clk, blockIdx.x);
            return;
        }
        lin -= (uint32_t)g.nlist;
    }
    lookup_p2p_mp_cta<IdxT, VEC, U, RowT>(desc, dstoff, idx, idx_base, g, C, cshift, B_local, peers, ostride, lin);
    clock_out(clk, blockIdx.x);
}

// `g` carries ntab, B (= B_global), P and off; gs.nlist > 0 (VEC 4 only) adds the fused sort CTAs of gs.list
template <typename IdxT, int VEC, typename RowT, int SORT_ITEMS>
static int launch_p2p_mp_t(dlrmb_tables* t, const IdxT* idx, int idx_base, const MpGeom& g0, const PeerPtrs& peers,
                           int B_local, int slots, int half, cudaStream_t s) {
    constexpr int U = 4;
    const uint32_t C = t->D / VEC;
    const int64_t n = (int64_t)g0.B * C;
    DLRMB_REQUIRE(n < (1ll << 30), "B * D too large for one lookup launch (%lld chunks)", (long long)n);
    MpGeom g = g0;
    int cshift;
    const int64_t ctas = lookup_grid_mp(t, g, C, &cshift) + (SORT_ITEMS > 0 ? g.nlist : 0);
    size_t smem = 0;
    if constexpr (SORT_ITEMS > 0) {
        smem = SmallSortGeom<SORT_ITEMS, 256>::smem_bytes();
        static unsigned long long done = 0;
        int rc = ensure_smem_attr((const void*)lookup_p2p_mp_kernel<IdxT, VEC, U, RowT, SORT_ITEMS>, (int)smem, &done);
        if (rc) return rc;
    }
    lookup_p2p_mp_kernel<IdxT, VEC, U, RowT, SORT_ITEMS><<<(unsigned)ctas, 256, smem, s>>>(
        t->d_desc, t->d_slotmap, idx, idx_base, g, C, cshift, (uint32_t)B_local, peers, (long long)slots * t->dest_D,
        SORT_ITEMS > 0 ? t->keys[half] : nullptr, SORT_ITEMS > 0 ? t->pos[half] : nullptr, t->cap, clock_slot(CLK_LOOKUP));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <typename IdxT, typename RowT>
static int launch_p2p_mp_i(dlrmb_tables* t, const IdxT* idx, int idx_base, const MpGeom& g, const PeerPtrs& peers,
                           int B_local, int slots, bool vec4, bool with_sort, cudaStream_t s) {
    if (!with_sort)
        return vec4 ? launch_p2p_mp_t<IdxT, 4, RowT, 0>(t, idx, idx_base, g, peers, B_local, slots, 0, s)
                    : launch_p2p_mp_t<IdxT, 1, RowT, 0>(t, idx, idx_base, g, peers, B_local, slots, 0, s);
    // the sort of the coming update, as launch_lookup_sort_mp: tables with L_k <= kFusedSortMax in CTAs of
    // the lookup launch (VEC 4 only), the rest by launch_sort_mp behind it; every table ends in `half`
    const int half = sort_mp_final_half(t, g);
    MpGeom gs = g;
    gs.nlist = 0;
    int64_t fused_max = 0;
    if (vec4)
        for (int k = 0; k < g.ntab; ++k) {
            const int64_t L = (int64_t)g.B * g.P[k];
            if (L <= kFusedSortMax) {
                gs.list[gs.nlist++] = (uint16_t)k;
                if (L > fused_max) fused_max = L;
            }
        }
    int rc;
    if (gs.nlist == 0) {
        rc = vec4 ? launch_p2p_mp_t<IdxT, 4, RowT, 0>(t, idx, idx_base, g, peers, B_local, slots, 0, s)
                  : launch_p2p_mp_t<IdxT, 1, RowT, 0>(t, idx, idx_base, g, peers, B_local, slots, 0, s);
        if (rc) return rc;
        return launch_sort_mp(t, idx, (int)sizeof(IdxT), idx_base, g, 0, half, s);
    }
    rc = fused_max <= 2048 ? launch_p2p_mp_t<IdxT, 4, RowT, 8>(t, idx, idx_base, gs, peers, B_local, slots, half, s)
                           : launch_p2p_mp_t<IdxT, 4, RowT, 16>(t, idx, idx_base, gs, peers, B_local, slots, half, s);
    if (rc) return rc;
    return launch_sort_mp(t, idx, (int)sizeof(IdxT), idx_base, g, kFusedSortMax, half, s);
}

}  // namespace dlrmb

using namespace dlrmb;

extern "C" {

int32_t dlrmb_xbuf_create(int32_t device, int64_t bytes, dlrmb_xbuf** out) {
    DLRMB_REQUIRE(out != nullptr && bytes > 0, "bad xbuf arguments");
    *out = nullptr;
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    void* p = nullptr;
    DLRMB_CUDA(cudaMalloc(&p, (size_t)bytes));
    cudaError_t e = cudaMemset(p, 0, (size_t)bytes);
    if (e != cudaSuccess) {
        cudaFree(p);
        set_error("cudaMemset of a %lld-byte exchange buffer failed: %s", (long long)bytes, cudaGetErrorString(e));
        return DLRMB_ECUDA;
    }
    *out = new dlrmb_xbuf{device, p, (size_t)bytes};
    return DLRMB_OK;
}

int32_t dlrmb_xbuf_destroy(dlrmb_xbuf* x) {
    if (!x) return DLRMB_OK;
    DeviceGuard guard(x->device);
    cudaFree(x->ptr);
    delete x;
    return DLRMB_OK;
}

int32_t dlrmb_xbuf_ptr(dlrmb_xbuf* x, void** dev) {
    DLRMB_REQUIRE(x && dev, "null argument");
    *dev = x->ptr;
    return DLRMB_OK;
}

int32_t dlrmb_xbuf_ipc_handle(dlrmb_xbuf* x, uint8_t* handle64) {
    DLRMB_REQUIRE(x && handle64, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    cudaIpcMemHandle_t h;
    DLRMB_CUDA(cudaIpcGetMemHandle(&h, x->ptr));
    memcpy(handle64, &h, 64);
    return DLRMB_OK;
}

int32_t dlrmb_xbuf_open(int32_t device, const uint8_t* handle64, void** peer_ptr) {
    DLRMB_REQUIRE(handle64 && peer_ptr, "null argument");
    *peer_ptr = nullptr;
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    DLRMB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *peer_ptr = p;
    return DLRMB_OK;
}

int32_t dlrmb_xbuf_close(int32_t device, void* peer_ptr) {
    if (!peer_ptr) return DLRMB_OK;
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    DLRMB_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return DLRMB_OK;
}

static int32_t set_dest_map(dlrmb_tables* t, const int32_t* slots, const int32_t* col0, int32_t D_dest) {
    DLRMB_REQUIRE(t && slots, "null argument");
    DLRMB_REQUIRE(D_dest >= t->D, "D_dest = %d is narrower than the handle's D = %d", D_dest, t->D);
    DeviceGuard guard(t->device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", t->device);
    int max_slot = -1;
    bool vec4 = D_dest % 4 == 0;
    std::vector<int32_t> off(t->ntab);
    for (int k = 0; k < t->ntab; ++k) {
        DLRMB_REQUIRE(slots[k] >= 0, "slot_map[%d] = %d is negative", k, slots[k]);
        const int32_t c0 = col0 ? col0[k] : 0;
        DLRMB_REQUIRE(c0 >= 0 && (int64_t)c0 + t->D <= D_dest, "col0[%d] = %d: columns [%d, %d) leave the destination row of %d",
                      k, c0, c0, c0 + t->D, D_dest);
        DLRMB_REQUIRE(((int64_t)slots[k] + 1) * D_dest < (1ll << 31), "slot_map[%d] = %d: destination offset too large", k,
                      slots[k]);
        if (slots[k] > max_slot) max_slot = slots[k];
        vec4 = vec4 && c0 % 4 == 0;
        off[k] = slots[k] * D_dest + c0;
    }
    if (!t->d_slotmap) DLRMB_CUDA(cudaMalloc((void**)&t->d_slotmap, sizeof(int32_t) * t->ntab));
    DLRMB_CUDA(cudaMemcpy(t->d_slotmap, off.data(), sizeof(int32_t) * t->ntab, cudaMemcpyHostToDevice));
    t->slotmap_max = max_slot;
    t->dest_D = D_dest;
    t->dest_vec4 = vec4;
    return DLRMB_OK;
}

int32_t dlrmb_tables_set_slot_map(dlrmb_tables* t, const int32_t* slots) {
    DLRMB_REQUIRE(t, "null argument");
    return set_dest_map(t, slots, nullptr, t->D);
}

int32_t dlrmb_tables_set_dest_map(dlrmb_tables* t, const int32_t* slots, const int32_t* col0, int32_t D_dest) {
    DLRMB_REQUIRE(t && slots && col0, "null argument");
    return set_dest_map(t, slots, col0, D_dest);
}

// the peer pointers of `world` ranks; vec4: D % 4 == 0, a dest map of 16-byte column offsets and every pointer
// 16-byte aligned
static int peer_ptrs(const dlrmb_tables* t, float* const* peer_T, int world, PeerPtrs* peers, bool* vec4) {
    *vec4 = (t->D % 4 == 0) && t->dest_vec4;
    for (int r = 0; r < kMaxPeers; ++r) {
        peers->p[r] = r < world ? peer_T[r] : nullptr;
        if (r < world) {
            DLRMB_REQUIRE(peer_T[r] != nullptr, "peer_T[%d] is null", r);
            *vec4 = *vec4 && ((reinterpret_cast<uintptr_t>(peer_T[r]) & 15) == 0);
        }
    }
    return DLRMB_OK;
}

static int launch_p2p(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g,
                      const PeerPtrs& peers, int B_local, int slots, bool vec4, bool with_sort, cudaStream_t s) {
    const bool bf = t->elem_bytes == 2;
    if (idx_bytes == 4) {
        const uint32_t* ip = (const uint32_t*)idx;
        return bf ? launch_p2p_mp_i<uint32_t, __nv_bfloat16>(t, ip, idx_base, g, peers, B_local, slots, vec4, with_sort, s)
                  : launch_p2p_mp_i<uint32_t, float>(t, ip, idx_base, g, peers, B_local, slots, vec4, with_sort, s);
    }
    const int64_t* ip = (const int64_t*)idx;
    return bf ? launch_p2p_mp_i<int64_t, __nv_bfloat16>(t, ip, idx_base, g, peers, B_local, slots, vec4, with_sort, s)
              : launch_p2p_mp_i<int64_t, float>(t, ip, idx_base, g, peers, B_local, slots, vec4, with_sort, s);
}

static int32_t embedding_fwd_p2p_impl(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                      int32_t B_global, int32_t P, float* const* peer_T, int32_t world,
                                      int32_t B_local, int32_t slots, bool with_sort, dlrmb_stream stream) {
    DLRMB_REQUIRE(t != nullptr && idx != nullptr && peer_T != nullptr, "null argument");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(idx_base == 0 || idx_base == 1, "idx_base must be 0 or 1 (got %d)", idx_base);
    DLRMB_REQUIRE(P > 0, "P must be positive (got %d)", P);
    DLRMB_REQUIRE(world >= 1 && world <= kMaxPeers, "world must be in 1..%d (got %d)", kMaxPeers, world);
    DLRMB_REQUIRE(B_local > 0 && B_global == B_local * world, "B_global (%d) must equal B_local (%d) * world (%d)",
                  B_global, B_local, world);
    DLRMB_REQUIRE((int64_t)B_global * P <= t->max_lookups, "B*P = %lld exceeds max_lookups = %lld",
                  (long long)B_global * P, (long long)t->max_lookups);
    if (!t->d_slotmap) {
        set_error("dlrmb_embedding_fwd_p2p needs dlrmb_tables_set_slot_map first");
        return DLRMB_ESTATE;
    }
    DLRMB_REQUIRE(slots > t->slotmap_max, "slots = %d does not cover the slot map (largest slot %d)", slots,
                  t->slotmap_max);
    DeviceGuard guard(t->device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", t->device);
    PeerPtrs peers;
    bool vec4;
    int rc = peer_ptrs(t, peer_T, world, &peers, &vec4);
    if (rc) return rc;
    return run_uniform(t, idx, idx_bytes, B_global, P, 0, with_sort,
                       [&](dlrmb_tables* v, const void* gidx, const MpGeom& g, int) {
                           return launch_p2p(v, gidx, idx_bytes, idx_base, g, peers, B_local, slots, vec4, with_sort,
                                             (cudaStream_t)stream);
                       });
}

int32_t dlrmb_embedding_fwd_p2p(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                int32_t B_global, int32_t P, float* const* peer_T, int32_t world,
                                int32_t B_local, int32_t slots, dlrmb_stream stream) {
    return embedding_fwd_p2p_impl(t, idx, idx_bytes, idx_base, B_global, P, peer_T, world, B_local, slots, false, stream);
}

int32_t dlrmb_embedding_fwd_p2p_sort(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                     int32_t B_global, int32_t P, float* const* peer_T, int32_t world,
                                     int32_t B_local, int32_t slots, dlrmb_stream stream) {
    if (t) t->sorted_valid = false;
    return embedding_fwd_p2p_impl(t, idx, idx_bytes, idx_base, B_global, P, peer_T, world, B_local, slots, true, stream);
}

static int32_t embedding_fwd_p2p_mp_impl(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                         int32_t B_global, const int32_t* P, float* const* peer_T, int32_t world,
                                         int32_t B_local, int32_t slots, bool with_sort, dlrmb_stream stream) {
    DLRMB_REQUIRE(t != nullptr && peer_T != nullptr, "null argument");
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B_global, P, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(world >= 1 && world <= kMaxPeers, "world must be in 1..%d (got %d)", kMaxPeers, world);
    DLRMB_REQUIRE(B_local > 0 && (int64_t)B_global == (int64_t)B_local * world,
                  "B_global (%d) must equal B_local (%d) * world (%d)", B_global, B_local, world);
    if (!t->d_slotmap) {
        set_error("dlrmb_embedding_fwd_p2p_mp needs dlrmb_tables_set_slot_map first");
        return DLRMB_ESTATE;
    }
    DLRMB_REQUIRE(slots > t->slotmap_max, "slots = %d does not cover the slot map (largest slot %d)", slots,
                  t->slotmap_max);
    DeviceGuard guard(t->device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", t->device);
    PeerPtrs peers;
    bool vec4;
    rc = peer_ptrs(t, peer_T, world, &peers, &vec4);
    if (rc) return rc;
    rc = launch_p2p(t, idx, idx_bytes, idx_base, g, peers, B_local, slots, vec4, with_sort, (cudaStream_t)stream);
    if (rc) return rc;
    if (with_sort) mark_sorted(t, g, 0);
    return DLRMB_OK;
}

int32_t dlrmb_embedding_fwd_p2p_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                   int32_t B_global, const int32_t* P, float* const* peer_T, int32_t world,
                                   int32_t B_local, int32_t slots, dlrmb_stream stream) {
    return embedding_fwd_p2p_mp_impl(t, idx, idx_bytes, idx_base, B_global, P, peer_T, world, B_local, slots, false,
                                     stream);
}

int32_t dlrmb_embedding_fwd_p2p_sort_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                        int32_t B_global, const int32_t* P, float* const* peer_T, int32_t world,
                                        int32_t B_local, int32_t slots, dlrmb_stream stream) {
    if (t) t->sorted_valid = false;
    return embedding_fwd_p2p_mp_impl(t, idx, idx_bytes, idx_base, B_global, P, peer_T, world, B_local, slots, true,
                                     stream);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Stream-ordered cross-GPU ordering without NCCL: flag barrier over the IPC-mapped buffers
// ---------------------------------------------------------------------------------------------
// Every rank owns a flag array [channels][world] of 32-bit epochs inside a dlrmb_xbuf that its peers
// map.  dlrmb_peer_barrier launches ONE tiny kernel that (1) bumps this rank's epoch of the channel,
// (2) after a system-scope fence stores it into slot [channel][rank] of every rank's array over
// NVLink, (3) waits until all `world` slots of its OWN array have reached the epoch.  Placed on the
// stream behind a kernel that stored into peers' buffers and in front of the kernels that consume
// what the peers stored, it is the ordering point of the fused exchanges: kernel completion makes the
// producer's peer stores visible before the flag store is issued, and nobody passes before every
// rank's flag -- hence every rank's data -- has arrived.  The epoch lives in device memory, so the
// call can be captured into a CUDA graph and replayed.  Each rank must run on its own GPU (the wait
// spins on flags that kernels of other processes set).
namespace dlrmb {

struct PeerFlagPtrs {
    uint32_t* p[kMaxPeers];
};

constexpr int kBarrierChannels = 8;
// state: [0 .. kBarrierChannels) epochs, [kBarrierChannels] = number of timed-out waits

__global__ void __launch_bounds__(32)
peer_barrier_kernel(PeerFlagPtrs peers, int world, int rank, int channel, uint32_t* __restrict__ state,
                    unsigned long long timeout_ns) {
    const int lane = threadIdx.x;
    uint32_t epoch = 0;
    if (lane == 0) {
        epoch = state[channel] + 1u;
        state[channel] = epoch;
    }
    epoch = __shfl_sync(0xffffffffu, epoch, 0);
    if (lane < world) {
        // the stream's earlier kernels (whose peer stores this flag publishes) have completed; the fence
        // orders their effects, as this thread observes them, before the flag store at system scope
        __threadfence_system();
        volatile uint32_t* dst = peers.p[lane] + (size_t)channel * kMaxPeers + rank;
        *dst = epoch;
        const volatile uint32_t* mine = peers.p[rank] + (size_t)channel * kMaxPeers + lane;
        unsigned long long t0 = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        // epochs only grow; compare as a signed distance so a wrap after 2^31 steps stays correct
        while ((int32_t)(*mine - epoch) < 0) {
            __nanosleep(40);
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > timeout_ns) {       // a peer is gone: do not hang the GPU, leave a trace for the host
                atomicAdd(state + kBarrierChannels, 1u);
                break;
            }
        }
    }
    __syncwarp();
    __threadfence_system();
}

// idx_local [ntab][B_local][P] of this rank's samples -> the owners' index buffers
// [t_owner][B_global][P] (rows rank*B_local ...), one 4- or 8-byte store per index over NVLink
struct IdxDest {
    void* base;        // owner's buffer for this table: [B_global][P]
};

template <typename IdxT>
__global__ void __launch_bounds__(256)
indices_scatter_kernel(const IdxT* __restrict__ idx_local, const IdxDest* __restrict__ dests, int ntab, int B_local,
                       int P, int rank) {
    const int k = blockIdx.y;
    const int n = B_local * P;
    const IdxT* src = idx_local + (size_t)k * n;
    IdxT* dst = static_cast<IdxT*>(dests[k].base) + (size_t)rank * n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

// Per-table pooling factors: idx_local is the `_mp` layout at B_local (table k's [B_local][P_k] block at
// element src_off[k]); table k's block lands at dests[k] + rank * B_local * P_k, i.e. rows
// [rank * B_local, (rank + 1) * B_local) of the owner's [B_global][P_k] block.  The geometry goes by value.
struct IdxScatterMpGeom {
    int ntab;
    int B_local;
    uint32_t P[kMpMaxTables];
    int64_t src_off[kMpMaxTables];
};

template <typename IdxT>
__global__ void __launch_bounds__(256)
indices_scatter_mp_kernel(const IdxT* __restrict__ idx_local, const IdxDest* __restrict__ dests,
                          const __grid_constant__ IdxScatterMpGeom g, int rank) {
    const int k = blockIdx.y;
    const int n = g.B_local * (int)g.P[k];
    const IdxT* src = idx_local + g.src_off[k];
    IdxT* dst = static_cast<IdxT*>(dests[k].base) + (size_t)rank * n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

// Column-wise sharding: a split table's block goes to every holder of one of its slices.  Destination i receives
// table dest_table[i]'s block at dests[i] + rank * B_local * P_k, one launch for all destinations.
constexpr int kMaxScatterDests = 1024;
struct IdxScatterListGeom {
    int B_local;
    uint32_t P[kMpMaxTables];
    int64_t src_off[kMpMaxTables];
    uint16_t table[kMaxScatterDests];
};

template <typename IdxT>
__global__ void __launch_bounds__(256)
indices_scatter_list_kernel(const IdxT* __restrict__ idx_local, const IdxDest* __restrict__ dests,
                            const __grid_constant__ IdxScatterListGeom g, int rank) {
    const int k = g.table[blockIdx.y];
    const int n = g.B_local * (int)g.P[k];
    const IdxT* src = idx_local + g.src_off[k];
    IdxT* dst = static_cast<IdxT*>(dests[blockIdx.y].base) + (size_t)rank * n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

}  // namespace dlrmb

extern "C" {

int32_t dlrmb_peer_barrier(int32_t device, uint32_t* const* peer_flags, int32_t world, int32_t rank, int32_t channel,
                           uint32_t* state, dlrmb_stream stream) {
    DLRMB_REQUIRE(peer_flags && state, "null argument");
    DLRMB_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "bad world / rank (%d, %d)", world, rank);
    DLRMB_REQUIRE(channel >= 0 && channel < kBarrierChannels, "channel must be in 0..%d", kBarrierChannels - 1);
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    PeerFlagPtrs peers;
    for (int r = 0; r < kMaxPeers; ++r) {
        peers.p[r] = r < world ? peer_flags[r] : nullptr;
        DLRMB_REQUIRE(r >= world || peer_flags[r] != nullptr, "peer_flags[%d] is null", r);
    }
    peer_barrier_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(peers, world, rank, channel, state, 4000000000ull);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

int64_t dlrmb_peer_barrier_flag_bytes(void) { return (int64_t)kBarrierChannels * kMaxPeers * sizeof(uint32_t); }
int64_t dlrmb_peer_barrier_state_bytes(void) { return (int64_t)(kBarrierChannels + 1) * sizeof(uint32_t); }

int32_t dlrmb_indices_scatter_p2p(int32_t device, const void* idx_local, int32_t idx_bytes, int32_t ntab,
                                  int32_t B_local, int32_t P, const void* const* dests_dev, int32_t rank,
                                  dlrmb_stream stream) {
    DLRMB_REQUIRE(idx_local && dests_dev, "null argument");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(ntab > 0 && ntab <= 65535 && B_local > 0 && P > 0 && rank >= 0, "bad index scatter geometry");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    const int n = B_local * P;
    int bx = (n + 255) / 256;
    if (bx > 64) bx = 64;
    dim3 grid((unsigned)bx, (unsigned)ntab);
    const IdxDest* d = reinterpret_cast<const IdxDest*>(dests_dev);
    if (idx_bytes == 4)
        indices_scatter_kernel<uint32_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)idx_local, d, ntab, B_local, P, rank);
    else
        indices_scatter_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const int64_t*)idx_local, d, ntab, B_local, P, rank);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

int32_t dlrmb_indices_scatter_p2p_mp(int32_t device, const void* idx_local, int32_t idx_bytes, int32_t ntab,
                                     int32_t B_local, const int32_t* P, const void* const* dests_dev, int32_t rank,
                                     dlrmb_stream stream) {
    DLRMB_REQUIRE(idx_local && dests_dev, "null argument");
    DLRMB_REQUIRE(P != nullptr, "P (per-table pooling factors) is null");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(ntab > 0 && ntab <= kMpMaxTables, "ntab must be in 1..%d (got %d)", kMpMaxTables, ntab);
    DLRMB_REQUIRE(B_local > 0 && rank >= 0, "bad index scatter geometry");
    IdxScatterMpGeom g;
    g.ntab = ntab;
    g.B_local = B_local;
    int64_t off = 0;
    int32_t maxP = 0;
    for (int k = 0; k < ntab; ++k) {
        DLRMB_REQUIRE(P[k] >= 1, "P[%d] = %d: every pooling factor must be >= 1", k, P[k]);
        DLRMB_REQUIRE((int64_t)B_local * P[k] < (1ll << 30), "B_local * P[%d] too large", k);
        g.P[k] = (uint32_t)P[k];
        g.src_off[k] = off;
        off += (int64_t)B_local * P[k];
        maxP = P[k] > maxP ? P[k] : maxP;
    }
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    int bx = (int)((B_local * (int64_t)maxP + 255) / 256);
    if (bx > 64) bx = 64;
    dim3 grid((unsigned)bx, (unsigned)ntab);
    const IdxDest* d = reinterpret_cast<const IdxDest*>(dests_dev);
    if (idx_bytes == 4)
        indices_scatter_mp_kernel<uint32_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)idx_local, d, g, rank);
    else
        indices_scatter_mp_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const int64_t*)idx_local, d, g, rank);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

int32_t dlrmb_indices_scatter_p2p_mp_list(int32_t device, const void* idx_local, int32_t idx_bytes, int32_t ntab,
                                          int32_t B_local, const int32_t* P, int32_t ndest, const int32_t* dest_table,
                                          const void* const* dests_dev, int32_t rank, dlrmb_stream stream) {
    DLRMB_REQUIRE(idx_local && dests_dev && dest_table, "null argument");
    DLRMB_REQUIRE(P != nullptr, "P (per-table pooling factors) is null");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(ntab > 0 && ntab <= kMpMaxTables, "ntab must be in 1..%d (got %d)", kMpMaxTables, ntab);
    DLRMB_REQUIRE(ndest > 0 && ndest <= kMaxScatterDests, "ndest must be in 1..%d (got %d)", kMaxScatterDests, ndest);
    DLRMB_REQUIRE(B_local > 0 && rank >= 0, "bad index scatter geometry");
    IdxScatterListGeom g;
    g.B_local = B_local;
    int64_t off = 0;
    int32_t maxP = 0;
    for (int k = 0; k < ntab; ++k) {
        DLRMB_REQUIRE(P[k] >= 1, "P[%d] = %d: every pooling factor must be >= 1", k, P[k]);
        DLRMB_REQUIRE((int64_t)B_local * P[k] < (1ll << 30), "B_local * P[%d] too large", k);
        g.P[k] = (uint32_t)P[k];
        g.src_off[k] = off;
        off += (int64_t)B_local * P[k];
        maxP = P[k] > maxP ? P[k] : maxP;
    }
    for (int i = 0; i < ndest; ++i) {
        DLRMB_REQUIRE(dest_table[i] >= 0 && dest_table[i] < ntab, "dest_table[%d] = %d is not a table (ntab %d)", i,
                      dest_table[i], ntab);
        g.table[i] = (uint16_t)dest_table[i];
    }
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    int bx = (int)((B_local * (int64_t)maxP + 255) / 256);
    if (bx > 64) bx = 64;
    dim3 grid((unsigned)bx, (unsigned)ndest);
    const IdxDest* d = reinterpret_cast<const IdxDest*>(dests_dev);
    if (idx_bytes == 4)
        indices_scatter_list_kernel<uint32_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)idx_local, d, g, rank);
    else
        indices_scatter_list_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const int64_t*)idx_local, d, g, rank);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// One-shot all-reduce of a SMALL float buffer over the IPC-mapped exchange buffers
// ---------------------------------------------------------------------------------------------
// The data-parallel step ends with the all-reduce of the bottom MLP's gradients (0.7 MB): it sits on the
// critical path (bottom MLP backward -> all-reduce -> dense SGD) and is latency-, not bandwidth-bound.
// Every rank owns a buffer [2][world][n] (two halves, alternating by step so that a fast peer's next push
// cannot overwrite what a slow rank is still summing).  push: every rank stores its n floats into slot
// [half][rank] of EVERY rank's buffer over NVLink; flag barrier; sum: every rank adds the `world` slots of
// its own buffer in rank order -- the same order on every rank, so all ranks hold bit-identical sums.
// (world - 1) * n * 4 bytes leave each GPU: right for buffers up to ~1 MB; large buffers stay with NCCL's
// reduce-scatter + all-gather.
namespace dlrmb {

struct PeerFloatPtrs {
    float* p[kMaxPeers];
};

__global__ void __launch_bounds__(256)
allreduce_push_kernel(PeerFloatPtrs peers, int world, int rank, const float4* __restrict__ data, int n4,
                      const uint32_t* __restrict__ state, int channel) {
    const uint32_t half = state[channel] & 1u;           // epoch BEFORE this step's barrier
    const size_t off = ((size_t)half * world + rank) * n4;
    const int peer = blockIdx.y;
    float4* dst = reinterpret_cast<float4*>(peers.p[peer]) + off;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) dst[i] = data[i];
}

__global__ void __launch_bounds__(256)
allreduce_sum_kernel(const float4* __restrict__ mine, int world, float4* __restrict__ data, int n4,
                     const uint32_t* __restrict__ state, int channel) {
    const uint32_t half = (state[channel] - 1u) & 1u;    // the barrier in between has bumped the epoch
    const float4* src = mine + (size_t)half * world * n4;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        float4 acc = src[i];
        for (int r = 1; r < world; ++r) {
            const float4 v = src[(size_t)r * n4 + i];
            acc.x = __fadd_rn(acc.x, v.x); acc.y = __fadd_rn(acc.y, v.y); acc.z = __fadd_rn(acc.z, v.z); acc.w = __fadd_rn(acc.w, v.w);
        }
        data[i] = acc;
    }
}

}  // namespace dlrmb

extern "C" {

int32_t dlrmb_peer_allreduce_f32(int32_t device, float* const* peer_bufs, uint32_t* const* peer_flags, int32_t world,
                                 int32_t rank, int32_t channel, uint32_t* state, float* data, int64_t n,
                                 dlrmb_stream stream) {
    DLRMB_REQUIRE(peer_bufs && peer_flags && state && data, "null argument");
    DLRMB_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "bad world / rank (%d, %d)", world, rank);
    DLRMB_REQUIRE(channel >= 0 && channel < kBarrierChannels, "channel must be in 0..%d", kBarrierChannels - 1);
    DLRMB_REQUIRE(n > 0 && n % 4 == 0 && n < (1ll << 28), "n must be a positive multiple of 4 (got %lld)", (long long)n);
    DLRMB_REQUIRE((reinterpret_cast<uintptr_t>(data) & 15) == 0, "data must be 16-byte aligned");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    PeerFloatPtrs bufs;
    for (int r = 0; r < kMaxPeers; ++r) {
        bufs.p[r] = r < world ? peer_bufs[r] : nullptr;
        DLRMB_REQUIRE(r >= world || peer_bufs[r] != nullptr, "peer_bufs[%d] is null", r);
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int n4 = (int)(n / 4);
    int bx = (n4 + 255) / 256;
    if (bx > 64) bx = 64;
    allreduce_push_kernel<<<dim3((unsigned)bx, (unsigned)world), 256, 0, s>>>(bufs, world, rank, reinterpret_cast<const float4*>(data), n4,
                                                                           state, channel);
    DLRMB_LAUNCH_CHECK();
    int rc = dlrmb_peer_barrier(device, peer_flags, world, rank, channel, state, stream);
    if (rc) return rc;
    int sx = (n4 + 255) / 256;
    if (sx > 592) sx = 592;
    allreduce_sum_kernel<<<(unsigned)sx, 256, 0, s>>>(reinterpret_cast<const float4*>(bufs.p[rank]), world,
                                                     reinterpret_cast<float4*>(data), n4, state, channel);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

}  // extern "C"
