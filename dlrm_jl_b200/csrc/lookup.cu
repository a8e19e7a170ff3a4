// Embedding lookup: gather + sum-pool of rows for every table in one launch.
//
// Replaces maplookup(PreallocationStrategy, tables, sparse) (DLRM.jl src/model/model.jl:161;
// semantics pinned by test/model/model.jl:265-271 and the `concatenated_result` golden).
//
// HBM-bound: per (table, sample) one D*4-byte row read per pooled index and one D*4-byte
// write.  Mapping: one flat grid in which every table owns a range of CTAs, and inside a table
// one thread per 16-byte chunk of an output row (chunk index fastest), so a row is read and
// written by D/4 consecutive lanes as whole 128-byte lines; the index of a row is fetched once
// per lane group through L1.  Every table has its own pooling factor P_k; a uniform batch is
// the case of equal P_k.
// Memory-level parallelism comes from U independent (index -> row) chains per thread when
// P == 1 and from a 4-deep unrolled pooling loop when P > 1.  The pooled sum runs in ascending
// p, so results are bit-identical to the CPU restatement.
#include "common.cuh"
#include "pool_bag.cuh"
#include "sort_small.cuh"

namespace dlrmb {

// P == 1: plain gather.  U independent chains per thread.  `cta` of `nctas` CTAs of 256 threads share
// table k.
template <typename IdxT, int VEC, int U, typename RowT>
__device__ __forceinline__ void lookup_gather_body(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx,
                                                   int idx_base, uint32_t B, uint32_t C, int cshift,
                                                   float* __restrict__ out, int slots, int slot0, int k,
                                                   uint32_t cta, uint32_t nctas) {
    using V = typename Vec<VEC>::type;
    const float* __restrict__ tb = desc[k].base;
    const IdxT* __restrict__ ik = idx + (size_t)k * B;
    const uint32_t n = B * C;
    const uint32_t step = nctas * blockDim.x;
    const size_t D = (size_t)C * VEC;
    float* __restrict__ ob = out + (size_t)(slot0 + k) * D;
    const size_t ostride = (size_t)slots * D;

    for (uint32_t t = cta * blockDim.x + threadIdx.x; t < n; t += step * U) {
        int64_t row[U];
        uint32_t b[U], c[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            uint32_t tt = t + (uint32_t)u * step;
            ok[u] = tt < n;
            b[u] = cshift >= 0 ? (tt >> cshift) : (tt / C);   // C is a power of two for the usual dims
            c[u] = tt - b[u] * C;
            row[u] = ok[u] ? (int64_t)__ldg(ik + b[u]) - idx_base : 0;
        }
        V v[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (ok[u]) v[u] = Vec<VEC>::template ldrow<RowT>(tb, (size_t)row[u], D, c[u]);
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (ok[u]) reinterpret_cast<V*>(ob + (size_t)b[u] * ostride)[c[u]] = v[u];
    }
}

// P > 1: gather + sum-pool, ascending p.
template <typename IdxT, int VEC, typename RowT>
__device__ __forceinline__ void lookup_pool_body(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx,
                                                 int idx_base, uint32_t B, uint32_t P, uint32_t C, int cshift,
                                                 float* __restrict__ out, int slots, int slot0, int k,
                                                 uint32_t cta, uint32_t nctas) {
    using V = typename Vec<VEC>::type;
    const float* __restrict__ tb = desc[k].base;
    const IdxT* __restrict__ ik = idx + (size_t)k * B * P;
    const uint32_t n = B * C;
    const uint32_t step = nctas * blockDim.x;
    const size_t D = (size_t)C * VEC;
    float* __restrict__ ob = out + (size_t)(slot0 + k) * D;
    const size_t ostride = (size_t)slots * D;

    for (uint32_t t = cta * blockDim.x + threadIdx.x; t < n; t += step) {
        const uint32_t b = cshift >= 0 ? (t >> cshift) : (t / C);
        const uint32_t c = t - b * C;
        const IdxT* __restrict__ ip = ik + (size_t)b * P;
        V acc = Vec<VEC>::zero();
        uint32_t p = 0;
        for (; p + 4 <= P; p += 4) {
            int64_t r0 = (int64_t)__ldg(ip + p) - idx_base;
            int64_t r1 = (int64_t)__ldg(ip + p + 1) - idx_base;
            int64_t r2 = (int64_t)__ldg(ip + p + 2) - idx_base;
            int64_t r3 = (int64_t)__ldg(ip + p + 3) - idx_base;
            V v0 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r0, D, c);
            V v1 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r1, D, c);
            V v2 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r2, D, c);
            V v3 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r3, D, c);
            acc = Vec<VEC>::add(acc, v0);
            acc = Vec<VEC>::add(acc, v1);
            acc = Vec<VEC>::add(acc, v2);
            acc = Vec<VEC>::add(acc, v3);
        }
        for (; p < P; ++p) {
            int64_t r = (int64_t)__ldg(ip + p) - idx_base;
            acc = Vec<VEC>::add(acc, Vec<VEC>::template ldrow<RowT>(tb, (size_t)r, D, c));
        }
        reinterpret_cast<V*>(ob + (size_t)b * ostride)[c] = acc;
    }
}

// One flat grid of gather CTAs; table k owns CTAs [g.pre[k], g.pre[k+1]), handed out in proportion to its
// work B * P_k * C (lookup_grid_mp), so a hotness-100 table does not form the tail behind one-hot tables
// holding the same number of CTAs.  The bodies above are pointed at table k (desc + k, its index block, its
// output slot): P_k == 1 takes the U-chain gather, every other table the pooling loop.
template <typename IdxT, int VEC, int U, typename RowT>
__device__ __forceinline__ void lookup_mp_cta(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx,
                                              int idx_base, const MpGeom& g, uint32_t C, int cshift,
                                              float* __restrict__ out, int slots, int slot0, uint32_t lin) {
    const int k = mp_find(g.pre, g.ntab, lin);
    const uint32_t cx = lin - g.pre[k], nx = g.pre[k + 1] - g.pre[k];
    const IdxT* ik = idx + g.off[k];
    if (g.P[k] == 1)
        lookup_gather_body<IdxT, VEC, U, RowT>(desc + k, ik, idx_base, g.B, C, cshift, out, slots, slot0 + k, 0, cx, nx);
    else
        lookup_pool_body<IdxT, VEC, RowT>(desc + k, ik, idx_base, g.B, g.P[k], C, cshift, out, slots, slot0 + k, 0, cx, nx);
}

template <typename IdxT, int VEC, int U, typename RowT>
__global__ void __launch_bounds__(256)
lookup_mp_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx, int idx_base,
                 const __grid_constant__ MpGeom g, uint32_t C, int cshift, float* __restrict__ out, int slots,
                 int slot0, unsigned long long* clk) {
    clock_in(clk, blockIdx.x);
    lookup_mp_cta<IdxT, VEC, U, RowT>(desc, idx, idx_base, g, C, cshift, out, slots, slot0, blockIdx.x);
    clock_out(clk, blockIdx.x);
}

// Training-step form: the lookup and the index sort / dedup of the NEXT sparse update in one launch.
// The sort needs the indices only, and one CTA per table sorts that table's B*P_k keys in shared memory
// (sort_small.cuh) in less time than the gather takes, so the first g.nlist CTAs sort the tables g.list[]
// (L_k <= kFusedSortMax) and the rest gather: the sort costs no launch of its own and no time on the stream.
// (Measured and not kept: the gather CTAs as ONE persistent wave over all tables, every thread walking its CTA's
// share 5 rows at a time with the next round's indices prefetched -- 10.6 vs 12.3 us with L2 flushed before the
// launch, but 10.2 vs 9.6 us back to back and no change in the training step, profiles/r02_lookup_flat.txt.)
template <typename IdxT, int U, typename RowT, int ITEMS>
__global__ void __launch_bounds__(256, 5)
lookup_sort_mp_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx, int idx_base,
                      const __grid_constant__ MpGeom g, uint32_t C, int cshift, float* __restrict__ out, int slots,
                      int slot0, uint32_t* __restrict__ keys_out, uint32_t* __restrict__ pos_out, int64_t cap,
                      unsigned long long* clk) {
    extern __shared__ uint32_t sort_smem[];
    clock_in(clk, blockIdx.x);
    if ((int)blockIdx.x < g.nlist) {
        const int k = g.list[blockIdx.x];
        sort_small_body<IdxT, ITEMS, 256>(idx + g.off[k], idx_base, (int)(g.B * g.P[k]), desc[k].rows,
                                          keys_out + (size_t)k * cap, pos_out + (size_t)k * cap, sort_smem);
        clock_out(clk, blockIdx.x);
        return;
    }
    lookup_mp_cta<IdxT, 4, U, RowT>(desc, idx, idx_base, g, C, cshift, out, slots, slot0, blockIdx.x - g.nlist);
    clock_out(clk, blockIdx.x);
}

// Gather CTAs per table: a launch budget of 32 CTAs per SM split in proportion to B * P_k * C,
// at least one per table and no more than the table has work items for.  Returns the total.
int64_t lookup_grid_mp(const dlrmb_tables* t, MpGeom& g, uint32_t C, int* cshift) {
    constexpr int U = 4;
    int64_t sumP = 0;
    for (int k = 0; k < g.ntab; ++k) sumP += g.P[k];
    const int64_t budget = (int64_t)t->sm_count * 32;
    const int64_t n = (int64_t)g.B * C;
    int64_t total = 0;
    for (int k = 0; k < g.ntab; ++k) {
        const int64_t most = ceil_div64(n, 256 * (g.P[k] == 1 ? U : 1));
        int64_t c = ceil_div64(budget * g.P[k], sumP);
        if (c > most) c = most;
        if (c < 1) c = 1;
        g.pre[k] = (uint32_t)total;
        total += c;
    }
    g.pre[g.ntab] = (uint32_t)total;
    *cshift = -1;
    if ((C & (C - 1)) == 0) {
        int sh = 0;
        while ((1u << sh) < C) ++sh;
        *cshift = sh;
    }
    return total;
}

template <typename IdxT, int VEC, typename RowT>
static int launch_lookup_mp_t(dlrmb_tables* t, const IdxT* idx, int idx_base, const MpGeom& g0, float* out,
                              int slots, int slot0, cudaStream_t s) {
    const uint32_t C = t->D / VEC;
    const int64_t n = (int64_t)g0.B * C;
    DLRMB_REQUIRE(n < (1ll << 30), "B * D too large for one lookup launch (%lld chunks)", (long long)n);
    MpGeom g = g0;
    g.nlist = 0;
    int cshift;
    const int64_t ctas = lookup_grid_mp(t, g, C, &cshift);
    lookup_mp_kernel<IdxT, VEC, 4, RowT><<<(unsigned)ctas, 256, 0, s>>>(t->d_desc, idx, idx_base, g, C, cshift, out, slots,
                                                                       slot0, clock_slot(CLK_LOOKUP));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <typename RowT>
static int launch_lookup_mp_r(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g,
                              float* out, int slots, int slot0, cudaStream_t s) {
    const bool vec4 = (t->D % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    if (idx_bytes == 4) {
        const uint32_t* p = static_cast<const uint32_t*>(idx);
        return vec4 ? launch_lookup_mp_t<uint32_t, 4, RowT>(t, p, idx_base, g, out, slots, slot0, s)
                    : launch_lookup_mp_t<uint32_t, 1, RowT>(t, p, idx_base, g, out, slots, slot0, s);
    }
    const int64_t* p = static_cast<const int64_t*>(idx);
    return vec4 ? launch_lookup_mp_t<int64_t, 4, RowT>(t, p, idx_base, g, out, slots, slot0, s)
                : launch_lookup_mp_t<int64_t, 1, RowT>(t, p, idx_base, g, out, slots, slot0, s);
}

int launch_lookup_mp(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g,
                     float* out, int slots, int slot0, cudaStream_t s) {
    if (t->elem_bytes == 2)
        return launch_lookup_mp_r<__nv_bfloat16>(t, idx, idx_bytes, idx_base, g, out, slots, slot0, s);
    return launch_lookup_mp_r<float>(t, idx, idx_bytes, idx_base, g, out, slots, slot0, s);
}

template <typename IdxT, typename RowT, int ITEMS>
static int launch_lookup_sort_mp_i(dlrmb_tables* t, const IdxT* idx, int idx_base, const MpGeom& g, float* out,
                                   int slots, int slot0, int half, cudaStream_t s) {
    const uint32_t C = t->D / 4;
    int cshift;
    MpGeom gg = g;
    const int64_t ctas = lookup_grid_mp(t, gg, C, &cshift) + g.nlist;
    constexpr size_t smem = SmallSortGeom<ITEMS, 256>::smem_bytes();
    static unsigned long long attr_done = 0;
    int rc = ensure_smem_attr((const void*)lookup_sort_mp_kernel<IdxT, 4, RowT, ITEMS>, (int)smem, &attr_done);
    if (rc) return rc;
    lookup_sort_mp_kernel<IdxT, 4, RowT, ITEMS><<<(unsigned)ctas, 256, smem, s>>>(
        t->d_desc, idx, idx_base, gg, C, cshift, out, slots, slot0, t->keys[half], t->pos[half], t->cap,
        clock_slot(CLK_LOOKUP));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

// lookup + sort for the next update.  Tables with L_k <= kFusedSortMax are sorted by extra CTAs of the
// lookup launch, the others by the stand-alone sort launches that follow (one shared-memory launch for
// L_k <= kSmemSortMax, radix passes above); every table's sorted stream ends in the same ping-pong half.
int launch_lookup_sort_mp(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g,
                          float* out, int slots, int slot0, cudaStream_t s) {
    const int64_t n = (int64_t)g.B * (t->D / 4);
    DLRMB_REQUIRE(n < (1ll << 30), "B * D too large for one lookup launch (%lld chunks)", (long long)n);
    const int half = sort_mp_final_half(t, g);
    const bool vec4 = (t->D % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
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
        rc = launch_lookup_mp(t, idx, idx_bytes, idx_base, g, out, slots, slot0, s);
        if (rc) return rc;
        return launch_sort_mp(t, idx, idx_bytes, idx_base, g, 0, half, s);
    }
    const bool bf = t->elem_bytes == 2;
    const bool small = fused_max <= 2048;
#define DLRMB_LSMP(IdxT, RowT)                                                                                      \
    (small ? launch_lookup_sort_mp_i<IdxT, RowT, 8>(t, static_cast<const IdxT*>(idx), idx_base, gs, out, slots, slot0, half, s) \
           : launch_lookup_sort_mp_i<IdxT, RowT, 16>(t, static_cast<const IdxT*>(idx), idx_base, gs, out, slots, slot0, half, s))
    if (idx_bytes == 4) rc = bf ? DLRMB_LSMP(uint32_t, __nv_bfloat16) : DLRMB_LSMP(uint32_t, float);
    else rc = bf ? DLRMB_LSMP(int64_t, __nv_bfloat16) : DLRMB_LSMP(int64_t, float);
#undef DLRMB_LSMP
    if (rc) return rc;
    return launch_sort_mp(t, idx, idx_bytes, idx_base, g, kFusedSortMax, half, s);
}

// ---- jagged (variable-length) bags ----------------------------------------------------------------
// One flat grid as lookup_mp_kernel: table k owns CTAs [g.pre[k], g.pre[k+1]) (lookup_grid_jagged), a thread
// owns one (bag, 16-byte chunk), reads the bag's two offsets and pools values[o0 .. o1) with pool_bag.  MEAN
// scales the sum by w = fl(1 / n); an empty bag stores +0.0f in both modes.
template <typename IdxT, int VEC, typename RowT, bool MEAN>
__global__ void __launch_bounds__(256)
lookup_jagged_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ values, const IdxT* __restrict__ offsets,
                     int idx_base, const __grid_constant__ MpGeom g, uint32_t B, uint32_t C, int cshift,
                     float* __restrict__ out, int slots, int slot0, unsigned long long* clk) {
    using V = typename Vec<VEC>::type;
    clock_in(clk, blockIdx.x);
    const int k = mp_find(g.pre, g.ntab, blockIdx.x);
    const uint32_t cta = blockIdx.x - g.pre[k], nctas = g.pre[k + 1] - g.pre[k];
    const float* __restrict__ tb = desc[k].base;
    const IdxT* __restrict__ ok = offsets + (size_t)k * B;
    const uint32_t n = B * C;
    const uint32_t step = nctas * blockDim.x;
    const size_t D = (size_t)C * VEC;
    float* __restrict__ ob = out + (size_t)(slot0 + k) * D;
    const size_t ostride = (size_t)slots * D;
    for (uint32_t t = cta * blockDim.x + threadIdx.x; t < n; t += step) {
        const uint32_t b = cshift >= 0 ? (t >> cshift) : (t / C);
        const uint32_t c = t - b * C;
        const int64_t o0 = (int64_t)__ldg(ok + b), o1 = (int64_t)__ldg(ok + b + 1);
        V acc = pool_bag<IdxT, VEC, RowT>(tb, values + o0, (uint32_t)(o1 - o0), idx_base, D, c);
        if (MEAN && o1 > o0) acc = Vec<VEC>::scale(acc, __fdiv_rn(1.0f, (float)(o1 - o0)));
        reinterpret_cast<V*>(ob + (size_t)b * ostride)[c] = acc;
    }
    clock_out(clk, blockIdx.x);
}

// Per-sample weights (the `_weighted` entry points, sum pooling only): lookup_jagged_kernel's grid and thread
// mapping, with row j of a bag scaled by weights[j] before it is added (pool_bag<WEIGHTED>).  The lanes of one bag
// read the same weight, so a weight costs one L1 broadcast per gathered row.
template <typename IdxT, int VEC, typename RowT>
__global__ void __launch_bounds__(256)
lookup_jagged_weighted_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ values,
                              const IdxT* __restrict__ offsets, const float* __restrict__ weights, int idx_base,
                              const __grid_constant__ MpGeom g, uint32_t B, uint32_t C, int cshift,
                              float* __restrict__ out, int slots, int slot0, unsigned long long* clk) {
    using V = typename Vec<VEC>::type;
    clock_in(clk, blockIdx.x);
    const int k = mp_find(g.pre, g.ntab, blockIdx.x);
    const uint32_t cta = blockIdx.x - g.pre[k], nctas = g.pre[k + 1] - g.pre[k];
    const float* __restrict__ tb = desc[k].base;
    const IdxT* __restrict__ ok = offsets + (size_t)k * B;
    const uint32_t n = B * C;
    const uint32_t step = nctas * blockDim.x;
    const size_t D = (size_t)C * VEC;
    float* __restrict__ ob = out + (size_t)(slot0 + k) * D;
    const size_t ostride = (size_t)slots * D;
    for (uint32_t t = cta * blockDim.x + threadIdx.x; t < n; t += step) {
        const uint32_t b = cshift >= 0 ? (t >> cshift) : (t / C);
        const uint32_t c = t - b * C;
        const int64_t o0 = (int64_t)__ldg(ok + b), o1 = (int64_t)__ldg(ok + b + 1);
        reinterpret_cast<V*>(ob + (size_t)b * ostride)[c] =
            pool_bag<IdxT, VEC, RowT, true>(tb, values + o0, (uint32_t)(o1 - o0), idx_base, D, c, weights + o0);
    }
    clock_out(clk, blockIdx.x);
}

// CTAs per table: the lookup_grid_mp budget split in proportion to the table's gathered rows plus its output rows,
// (L_k + B) * C, so a table of long bags is not the tail; at least one per table (its B rows are written even
// when L_k = 0) and no more than it has work items for.
int64_t lookup_grid_jagged(const dlrmb_tables* t, MpGeom& g, uint32_t B, uint32_t C) {
    int64_t sumw = 0;
    for (int k = 0; k < g.ntab; ++k) sumw += (int64_t)g.P[k] + B;
    const int64_t budget = (int64_t)t->sm_count * 32;
    const int64_t most = ceil_div64((int64_t)B * C, 256);
    int64_t total = 0;
    for (int k = 0; k < g.ntab; ++k) {
        int64_t c = ceil_div64(budget * ((int64_t)g.P[k] + B), sumw);
        if (c > most) c = most;
        if (c < 1) c = 1;
        g.pre[k] = (uint32_t)total;
        total += c;
    }
    g.pre[g.ntab] = (uint32_t)total;
    return total;
}

template <typename IdxT, int VEC, typename RowT>
static int launch_lookup_jagged_t(dlrmb_tables* t, const IdxT* values, const IdxT* offsets, const float* weights,
                                  int idx_base, const MpGeom& g0, int B, int pooling, float* out, int slots, int slot0,
                                  cudaStream_t s) {
    const uint32_t C = t->D / VEC;
    const int64_t n = (int64_t)B * C;
    DLRMB_REQUIRE(n < (1ll << 30), "B * D too large for one lookup launch (%lld chunks)", (long long)n);
    MpGeom g = g0;
    const int64_t ctas = lookup_grid_jagged(t, g, (uint32_t)B, C);
    int cshift = -1;
    if ((C & (C - 1)) == 0)
        for (cshift = 0; (1u << cshift) < C; ++cshift) {}
    if (pooling == kJaggedWeighted)
        lookup_jagged_weighted_kernel<IdxT, VEC, RowT><<<(unsigned)ctas, 256, 0, s>>>(
            t->d_desc, values, offsets, weights, idx_base, g, (uint32_t)B, C, cshift, out, slots, slot0,
            clock_slot(CLK_LOOKUP));
    else if (pooling == 1)
        lookup_jagged_kernel<IdxT, VEC, RowT, true><<<(unsigned)ctas, 256, 0, s>>>(
            t->d_desc, values, offsets, idx_base, g, (uint32_t)B, C, cshift, out, slots, slot0, clock_slot(CLK_LOOKUP));
    else
        lookup_jagged_kernel<IdxT, VEC, RowT, false><<<(unsigned)ctas, 256, 0, s>>>(
            t->d_desc, values, offsets, idx_base, g, (uint32_t)B, C, cshift, out, slots, slot0, clock_slot(CLK_LOOKUP));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <typename RowT>
static int launch_lookup_jagged_r(dlrmb_tables* t, const void* values, const void* offsets, const float* w,
                                  int idx_bytes, int idx_base, const MpGeom& g, int B, int pooling, float* out, int slots,
                                  int slot0, cudaStream_t s) {
    const bool vec4 = (t->D % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    if (idx_bytes == 4) {
        const uint32_t* v = static_cast<const uint32_t*>(values);
        const uint32_t* o = static_cast<const uint32_t*>(offsets);
        return vec4 ? launch_lookup_jagged_t<uint32_t, 4, RowT>(t, v, o, w, idx_base, g, B, pooling, out, slots, slot0, s)
                    : launch_lookup_jagged_t<uint32_t, 1, RowT>(t, v, o, w, idx_base, g, B, pooling, out, slots, slot0, s);
    }
    const int64_t* v = static_cast<const int64_t*>(values);
    const int64_t* o = static_cast<const int64_t*>(offsets);
    return vec4 ? launch_lookup_jagged_t<int64_t, 4, RowT>(t, v, o, w, idx_base, g, B, pooling, out, slots, slot0, s)
                : launch_lookup_jagged_t<int64_t, 1, RowT>(t, v, o, w, idx_base, g, B, pooling, out, slots, slot0, s);
}

int launch_lookup_jagged(dlrmb_tables* t, const void* values, const void* offsets, const float* weights, int idx_bytes,
                         int idx_base, const MpGeom& g, int B, int pooling, float* out, int slots, int slot0,
                         cudaStream_t s) {
    if (t->elem_bytes == 2)
        return launch_lookup_jagged_r<__nv_bfloat16>(t, values, offsets, weights, idx_bytes, idx_base, g, B, pooling, out,
                                                     slots, slot0, s);
    return launch_lookup_jagged_r<float>(t, values, offsets, weights, idx_bytes, idx_base, g, B, pooling, out, slots,
                                         slot0, s);
}

// ---- gradient of the pooled rows with respect to the per-sample weights ---------------------------------------
// dw[j] = sum_d dT[b(j)][slot0 + k][d] * table_k[values[j]][d] for every entry j of every bag, in the order the
// header states: a group of G lanes (G = min(32, C rounded up to a power of two), C chunks of VEC floats) owns one
// bag; lane l adds the products of its chunks c = l, l + G, .. in ascending d, acc = fl(acc + fl(g * r)) from
// +0.0f; then the G partials meet in a butterfly, p_l = fl(p_l + p_(l xor s)) for s = G/2 .. 1 (IEEE addition
// commutes, so every lane holds the same bits), and lane 0 stores dw[j].  Four entries are in flight per group;
// the bag's dT row is re-read from L1 for each of them.  A flat grid of ntab * B groups; an empty bag stores
// nothing.
template <int VEC> struct Dot;
template <> struct Dot<4> {
    static __device__ __forceinline__ float acc(float a, float4 g, float4 r) {
        a = __fadd_rn(a, __fmul_rn(g.x, r.x));
        a = __fadd_rn(a, __fmul_rn(g.y, r.y));
        a = __fadd_rn(a, __fmul_rn(g.z, r.z));
        return __fadd_rn(a, __fmul_rn(g.w, r.w));
    }
    static __device__ __forceinline__ float4 ld(const float* p, uint32_t c) {
        return __ldg(reinterpret_cast<const float4*>(p) + c);
    }
};
template <> struct Dot<1> {
    static __device__ __forceinline__ float acc(float a, float g, float r) { return __fadd_rn(a, __fmul_rn(g, r)); }
    static __device__ __forceinline__ float ld(const float* p, uint32_t c) { return __ldg(p + c); }
};

template <typename IdxT, int VEC, typename RowT>
__global__ void __launch_bounds__(256)
weight_grad_jagged_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ values,
                          const IdxT* __restrict__ offsets, int idx_base, uint32_t ntab, uint32_t B, uint32_t C,
                          int glog2, const float* __restrict__ dT, int slots, int slot0, float* __restrict__ dw) {
    using V = typename Vec<VEC>::type;
    const uint32_t G = 1u << glog2;
    const uint32_t lane = threadIdx.x & (G - 1);
    const uint64_t grp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> glog2;
    if (grp >= (uint64_t)ntab * B) return;   // whole groups only: G divides 32
    // the group's lanes, for the shuffles (groups of one warp may walk bags of different lengths)
    const unsigned mask = G == 32 ? 0xffffffffu : (((1u << G) - 1) << ((threadIdx.x & 31) & ~(G - 1)));
    const uint32_t k = (uint32_t)grp / B, b = (uint32_t)grp - k * B;   // ntab * B < 2^32 (the launcher checks)
    const float* __restrict__ tb = desc[k].base;
    const size_t D = (size_t)C * VEC;
    const float* __restrict__ gr = dT + ((size_t)b * slots + slot0 + k) * D;
    const int64_t o0 = (int64_t)__ldg(offsets + (size_t)k * B + b), o1 = (int64_t)__ldg(offsets + (size_t)k * B + b + 1);
    const IdxT* __restrict__ ip = values + o0;
    float* __restrict__ wo = dw + o0;
    const uint32_t n = (uint32_t)(o1 - o0);
    uint32_t p = 0;
    for (; p + 4 <= n; p += 4) {
        const int64_t r0 = (int64_t)__ldg(ip + p) - idx_base;
        const int64_t r1 = (int64_t)__ldg(ip + p + 1) - idx_base;
        const int64_t r2 = (int64_t)__ldg(ip + p + 2) - idx_base;
        const int64_t r3 = (int64_t)__ldg(ip + p + 3) - idx_base;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (uint32_t c = lane; c < C; c += G) {
            const V gv = Dot<VEC>::ld(gr, c);
            const V v0 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r0, D, c);
            const V v1 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r1, D, c);
            const V v2 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r2, D, c);
            const V v3 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r3, D, c);
            a0 = Dot<VEC>::acc(a0, gv, v0);
            a1 = Dot<VEC>::acc(a1, gv, v1);
            a2 = Dot<VEC>::acc(a2, gv, v2);
            a3 = Dot<VEC>::acc(a3, gv, v3);
        }
        for (uint32_t s = G >> 1; s > 0; s >>= 1) {
            a0 = __fadd_rn(a0, __shfl_xor_sync(mask, a0, s, G));
            a1 = __fadd_rn(a1, __shfl_xor_sync(mask, a1, s, G));
            a2 = __fadd_rn(a2, __shfl_xor_sync(mask, a2, s, G));
            a3 = __fadd_rn(a3, __shfl_xor_sync(mask, a3, s, G));
        }
        if (lane == 0) {
            wo[p] = a0;
            wo[p + 1] = a1;
            wo[p + 2] = a2;
            wo[p + 3] = a3;
        }
    }
    for (; p < n; ++p) {
        const int64_t r = (int64_t)__ldg(ip + p) - idx_base;
        float a = 0.f;
        for (uint32_t c = lane; c < C; c += G)
            a = Dot<VEC>::acc(a, Dot<VEC>::ld(gr, c), Vec<VEC>::template ldrow<RowT>(tb, (size_t)r, D, c));
        for (uint32_t s = G >> 1; s > 0; s >>= 1) a = __fadd_rn(a, __shfl_xor_sync(mask, a, s, G));
        if (lane == 0) wo[p] = a;
    }
}

template <typename IdxT, int VEC, typename RowT>
static int launch_weight_grad_jagged_t(dlrmb_tables* t, const IdxT* values, const IdxT* offsets, int idx_base, int B,
                                       const float* dT, int slots, int slot0, float* dw, cudaStream_t s) {
    const uint32_t C = t->D / VEC;
    int glog2 = 0;
    while ((1u << glog2) < C && glog2 < 5) ++glog2;
    const int64_t groups = (int64_t)t->ntab * B;
    DLRMB_REQUIRE(groups <= (int64_t)UINT32_MAX, "batch too large for one weight-gradient launch");
    const int64_t ctas = ceil_div64(groups << glog2, 256);
    weight_grad_jagged_kernel<IdxT, VEC, RowT><<<(unsigned)ctas, 256, 0, s>>>(
        t->d_desc, values, offsets, idx_base, (uint32_t)t->ntab, (uint32_t)B, C, glog2, dT, slots, slot0, dw);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <typename RowT>
static int launch_weight_grad_jagged_r(dlrmb_tables* t, const void* values, const void* offsets, int idx_bytes,
                                       int idx_base, int B, const float* dT, int slots, int slot0, float* dw,
                                       cudaStream_t s) {
    const bool vec4 = t->D % 4 == 0;   // the caller checked dT's alignment
    if (idx_bytes == 4) {
        const uint32_t* v = static_cast<const uint32_t*>(values);
        const uint32_t* o = static_cast<const uint32_t*>(offsets);
        return vec4 ? launch_weight_grad_jagged_t<uint32_t, 4, RowT>(t, v, o, idx_base, B, dT, slots, slot0, dw, s)
                    : launch_weight_grad_jagged_t<uint32_t, 1, RowT>(t, v, o, idx_base, B, dT, slots, slot0, dw, s);
    }
    const int64_t* v = static_cast<const int64_t*>(values);
    const int64_t* o = static_cast<const int64_t*>(offsets);
    return vec4 ? launch_weight_grad_jagged_t<int64_t, 4, RowT>(t, v, o, idx_base, B, dT, slots, slot0, dw, s)
                : launch_weight_grad_jagged_t<int64_t, 1, RowT>(t, v, o, idx_base, B, dT, slots, slot0, dw, s);
}

int launch_weight_grad_jagged(dlrmb_tables* t, const void* values, const void* offsets, int idx_bytes, int idx_base,
                              int B, const float* dT, int slots, int slot0, float* dw, cudaStream_t s) {
    if (t->elem_bytes == 2)
        return launch_weight_grad_jagged_r<__nv_bfloat16>(t, values, offsets, idx_bytes, idx_base, B, dT, slots, slot0,
                                                          dw, s);
    return launch_weight_grad_jagged_r<float>(t, values, offsets, idx_bytes, idx_base, B, dT, slots, slot0, dw, s);
}

// ---- ScaledUniform init (src/model/model.jl:61-65): U(-1/sqrt(rows), 1/sqrt(rows)) ------------
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

template <typename RowT>
__global__ void __launch_bounds__(256)
init_uniform_kernel(float* __restrict__ base, int64_t elems, float scale, uint64_t stream_seed) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    auto* dst = RowIO<RowT>::row(base, 0, 0);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < elems; i += step) {
        uint64_t h = mix64(stream_seed ^ mix64((uint64_t)i));
        float u = (float)(h >> 40) * (1.0f / 16777216.0f);  // [0, 1) on 24 bits
        dst[i] = (RowT)((2.0f * u - 1.0f) * scale);
    }
}

// f32 staging buffer <-> table rows (only used for bf16 storage: upload rounds to nearest even)
template <bool TO_TABLE>
__global__ void __launch_bounds__(256)
convert_rows_kernel(__nv_bfloat16* __restrict__ table, float* __restrict__ buf, int64_t elems) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < elems; i += step) {
        if (TO_TABLE) table[i] = __float2bfloat16_rn(buf[i]);
        else buf[i] = __bfloat162float(table[i]);
    }
}

int launch_convert_rows(dlrmb_tables* t, int k, float* f32_buf, bool to_table, cudaStream_t s) {
    const int64_t elems = t->h_rows[k] * (int64_t)t->D;
    int64_t blocks = ceil_div64(elems, 256 * 4);
    if (blocks > (int64_t)t->sm_count * 16) blocks = (int64_t)t->sm_count * 16;
    auto* table = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(t->slab) + (size_t)t->h_offsets[k] * 2);
    if (to_table) convert_rows_kernel<true><<<(unsigned)blocks, 256, 0, s>>>(table, f32_buf, elems);
    else convert_rows_kernel<false><<<(unsigned)blocks, 256, 0, s>>>(table, f32_buf, elems);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

int launch_init_uniform(dlrmb_tables* t, uint64_t seed, cudaStream_t s) {
    for (int k = 0; k < t->ntab; ++k) {
        int64_t elems = t->h_rows[k] * (int64_t)t->D;
        float scale = 1.0f / sqrtf((float)t->h_rows[k]);
        int64_t blocks = ceil_div64(elems, 256 * 8);
        int64_t cap = (int64_t)t->sm_count * 16;
        if (blocks > cap) blocks = cap;
        uint64_t stream_seed = seed * 0x9E3779B97F4A7C15ull + (uint64_t)(k + 1) * 0xD1B54A32D192ED03ull;
        float* base = reinterpret_cast<float*>(reinterpret_cast<char*>(t->slab) + (size_t)t->h_offsets[k] * t->elem_bytes);
        if (t->elem_bytes == 2)
            init_uniform_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, s>>>(base, elems, scale, stream_seed);
        else
            init_uniform_kernel<float><<<(unsigned)blocks, 256, 0, s>>>(base, elems, scale, stream_seed);
        DLRMB_LAUNCH_CHECK();
    }
    return DLRMB_OK;
}

// ---- optional range check (the reference's hot loops are @inbounds; this is the debug aid) ---
template <typename IdxT>
__global__ void __launch_bounds__(256)
check_indices_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx, int idx_base,
                     int64_t L, unsigned long long* __restrict__ bad /* smallest (table << 40 | pos) */) {
    const int k = blockIdx.y;
    const int64_t rows = desc[k].rows;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += step) {
        int64_t r = (int64_t)idx[(size_t)k * L + i] - idx_base;
        if (r < 0 || r >= rows) {
            unsigned long long code = ((unsigned long long)k << 40) | (unsigned long long)i;
            atomicMin(&bad[0], code);
        }
    }
}

int launch_check_indices(dlrmb_tables* t, const void* d_idx, int idx_bytes, int idx_base, int B,
                         int P, cudaStream_t s, long long* bad_table, long long* bad_pos,
                         long long* bad_val) {
    unsigned long long* d_bad = reinterpret_cast<unsigned long long*>(t->d_uniq);  // scratch reuse
    unsigned long long init[2] = {~0ull, 0ull};
    DLRMB_CUDA(cudaMemcpyAsync(d_bad, init, sizeof(init), cudaMemcpyHostToDevice, s));
    const int64_t L = (int64_t)B * P;
    int64_t bx = ceil_div64(L, 256 * 4);
    if (bx > t->sm_count * 8) bx = t->sm_count * 8;
    dim3 grid((unsigned)bx, (unsigned)t->ntab);
    if (idx_bytes == 4)
        check_indices_kernel<uint32_t><<<grid, 256, 0, s>>>(t->d_desc, (const uint32_t*)d_idx, idx_base, L, d_bad);
    else
        check_indices_kernel<int64_t><<<grid, 256, 0, s>>>(t->d_desc, (const int64_t*)d_idx, idx_base, L, d_bad);
    DLRMB_LAUNCH_CHECK();
    unsigned long long h[2];
    DLRMB_CUDA(cudaMemcpyAsync(h, d_bad, sizeof(h), cudaMemcpyDeviceToHost, s));
    DLRMB_CUDA(cudaStreamSynchronize(s));
    if (h[0] == ~0ull) {
        *bad_table = -1;
        return DLRMB_OK;
    }
    *bad_table = (long long)(h[0] >> 40);
    *bad_pos = (long long)(h[0] & ((1ull << 40) - 1));
    const char* src = (const char*)d_idx + ((size_t)*bad_table * L + (size_t)*bad_pos) * idx_bytes;
    int64_t v64 = 0;
    uint32_t v32 = 0;
    if (idx_bytes == 4) {
        DLRMB_CUDA(cudaMemcpy(&v32, src, 4, cudaMemcpyDeviceToHost));
        v64 = v32;
    } else {
        DLRMB_CUDA(cudaMemcpy(&v64, src, 8, cudaMemcpyDeviceToHost));
    }
    *bad_val = (long long)v64;
    return DLRMB_OK;
}

template <typename IdxT>
__global__ void __launch_bounds__(256)
check_indices_mp_kernel(const TableDesc* __restrict__ desc, const IdxT* __restrict__ idx, int idx_base,
                        const __grid_constant__ MpGeom g, unsigned long long* __restrict__ bad) {
    const int k = blockIdx.y;
    const int64_t rows = desc[k].rows;
    const int64_t L = (int64_t)g.B * g.P[k];
    const IdxT* ik = idx + g.off[k];
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += step) {
        int64_t r = (int64_t)ik[i] - idx_base;
        if (r < 0 || r >= rows) atomicMin(&bad[0], ((unsigned long long)k << 40) | (unsigned long long)i);
    }
}

int launch_check_indices_mp(dlrmb_tables* t, const void* d_idx, int idx_bytes, int idx_base, const MpGeom& g,
                            cudaStream_t s, long long* bad_table, long long* bad_pos, long long* bad_val) {
    unsigned long long* d_bad = reinterpret_cast<unsigned long long*>(t->d_uniq);  // scratch reuse
    unsigned long long init[2] = {~0ull, 0ull};
    DLRMB_CUDA(cudaMemcpyAsync(d_bad, init, sizeof(init), cudaMemcpyHostToDevice, s));
    uint32_t maxP = 0;
    for (int k = 0; k < g.ntab; ++k) maxP = g.P[k] > maxP ? g.P[k] : maxP;
    int64_t bx = ceil_div64((int64_t)g.B * maxP, 256 * 4);
    if (bx > t->sm_count * 8) bx = t->sm_count * 8;
    dim3 grid((unsigned)bx, (unsigned)g.ntab);
    if (idx_bytes == 4)
        check_indices_mp_kernel<uint32_t><<<grid, 256, 0, s>>>(t->d_desc, (const uint32_t*)d_idx, idx_base, g, d_bad);
    else
        check_indices_mp_kernel<int64_t><<<grid, 256, 0, s>>>(t->d_desc, (const int64_t*)d_idx, idx_base, g, d_bad);
    DLRMB_LAUNCH_CHECK();
    unsigned long long h[2];
    DLRMB_CUDA(cudaMemcpyAsync(h, d_bad, sizeof(h), cudaMemcpyDeviceToHost, s));
    DLRMB_CUDA(cudaStreamSynchronize(s));
    if (h[0] == ~0ull) {
        *bad_table = -1;
        return DLRMB_OK;
    }
    *bad_table = (long long)(h[0] >> 40);
    *bad_pos = (long long)(h[0] & ((1ull << 40) - 1));
    const char* src = (const char*)d_idx + ((size_t)g.off[*bad_table] + (size_t)*bad_pos) * idx_bytes;
    int64_t v64 = 0;
    uint32_t v32 = 0;
    if (idx_bytes == 4) {
        DLRMB_CUDA(cudaMemcpy(&v32, src, 4, cudaMemcpyDeviceToHost));
        v64 = v32;
    } else {
        DLRMB_CUDA(cudaMemcpy(&v64, src, 8, cudaMemcpyDeviceToHost));
    }
    *bad_val = (long long)v64;
    return DLRMB_OK;
}

}  // namespace dlrmb
