// Sparse gradient scatter-add fused with the in-place SGD row update.
//
// Replaces the lookup pullback -> SparseEmbeddingUpdate(delta, indices) (DLRM.jl
// src/train/train.jl:144; densified meaning pinned by test/train/backprop.jl:148-158) and
// EmbeddingTables.update!(Flux.Descent(lr), tables, updates, indexers; num_splits, nthreads)
// (call site src/train/train.jl:283-290; Flux Descent = `delta .*= lr; x .-= delta`):
//     table_k[r] -= lr * sum_{(b,p): idx_k[b][p] = r} dT[b][slot0 + k]
//
// Input is the per-table stream sorted by row id (sort.cu).  It is reduced as a three-level,
// fixed-shape tree, so duplicate rows are summed in an order that depends only on the batch
// geometry: no floating-point atomics, bit-reproducible results, one read-modify-write per row.
//
//   level 1  a lane group (one lane per 16-byte chunk of a row) walks a TILE of 4..32 consecutive
//            entries in order, accumulating gradient rows in registers while the row id repeats (a
//            segmented reduction whose segments are the duplicate runs).  A run that lies inside
//            the tile ends in the row's read-modify-write right there.
//   level 2  the lane groups of a CTA cover consecutive tiles (a CHUNK); runs that cross tile
//            boundaries inside the chunk are finished through shared memory by the group that owns
//            the run's first tile.
//   level 3  only runs that cross CHUNK boundaries (hot rows: Zipf heads, tables with a handful of
//            rows) touch global scratch: one "head" and one "carry" partial per chunk, plus a work
//            list of head chunks; every listed run gets a CTA whose lane groups add the carried
//            partials in a fixed strided order and update the row once.  For large batches that is
//            a second launch (update_fixup_kernel).  At DLRM batch sizes, where a launch costs as
//            much as the whole fix-up, level 3 runs inside the same launch (INLINE = true): every CTA
//            counts itself done on its table's counter, and the CTA that finds the count complete --
//            the last one of that table, whichever it is -- lists the table's head chunks and
//            finishes their runs.  Nobody waits for anybody (no spin, no assumption about the order
//            in which CTAs are scheduled), the tables finish independently, and the last CTA re-arms
//            its counter, so an update is one launch and no memset.
//
// HBM traffic per entry: 8 B of (key, position), one D*4-byte gradient row read, and per distinct
// row one D*4-byte read + one D*4-byte write.  The 4 keys / 4 positions of a batch are one 16-byte
// load each, the next batch's are requested before the current batch's rows, and the rows of a
// batch (gradient rows plus the table rows of the runs ending in it) are all in flight together.
#include "common.cuh"

namespace dlrmb {

// Batches of at most this many (table, lookup) entries run the fix-up inside the tiles launch.
constexpr int64_t kUpdateInlineMaxEntries = 1 << 18;

template <int VEC> struct UV;
template <> struct UV<4> {
    using type = float4;
    static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ float4 add(float4 a, float4 b) {
        return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
    }
    // Flux.Descent: delta *= lr; x -= delta  (two roundings, never contracted into an FMA)
    static __device__ __forceinline__ float4 sgd(float4 x, float4 g, float lr) {
        return make_float4(__fsub_rn(x.x, __fmul_rn(lr, g.x)), __fsub_rn(x.y, __fmul_rn(lr, g.y)),
                           __fsub_rn(x.z, __fmul_rn(lr, g.z)), __fsub_rn(x.w, __fmul_rn(lr, g.w)));
    }
    static __device__ __forceinline__ float4 scale(float4 a, float w) {
        return make_float4(__fmul_rn(a.x, w), __fmul_rn(a.y, w), __fmul_rn(a.z, w), __fmul_rn(a.w, w));
    }
};
template <> struct UV<1> {
    using type = float;
    static __device__ __forceinline__ float zero() { return 0.f; }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sgd(float x, float g, float lr) {
        return __fsub_rn(x, __fmul_rn(lr, g));
    }
    static __device__ __forceinline__ float scale(float a, float w) { return __fmul_rn(a, w); }
};

// table-row access in the row's storage type (f32 or bf16); chunk c = floats [c*VEC, c*VEC + VEC)
template <int VEC, typename RowT> struct RowV;
template <typename RowT> struct RowV<4, RowT> {
    static __device__ __forceinline__ float4 load(const float* base, size_t r, size_t D, int c) {
        return RowIO<RowT>::load4(RowIO<RowT>::row(base, r, D), c);
    }
    static __device__ __forceinline__ void store(float* base, size_t r, size_t D, int c, float4 v) {
        RowIO<RowT>::store4(RowIO<RowT>::row(base, r, D), c, v);
    }
};
template <typename RowT> struct RowV<1, RowT> {
    static __device__ __forceinline__ float load(const float* base, size_t r, size_t D, int c) {
        return RowIO<RowT>::load1(RowIO<RowT>::row(base, r, D), c);
    }
    static __device__ __forceinline__ void store(float* base, size_t r, size_t D, int c, float v) {
        RowIO<RowT>::store1(RowIO<RowT>::row(base, r, D), c, v);
    }
};

// per-tile (shared memory) and per-chunk (global) run-boundary flags
enum : uint8_t { FLAG_CARRY_IN = 1, FLAG_CARRY_ENDS = 2, FLAG_HEAD = 4 };

struct UpdateGeom {
    int L, P, tiles, tile, lpr_log2, C, slots, slot0;
    int chunks;          // CTAs (chunks of G tiles) per table
    int G;               // lane groups (= tiles) per CTA of update_tiles_kernel
    int64_t cap, pcap;   // stream stride per table; partial / flag stride per table (in chunks)
};

// Level 3: runs that cross chunk boundaries.  One CTA per listed head chunk: the end of the run is
// found by probing the chunk flags THREADS at a time, lane group `sub` adds the carry partials of
// chunks g+1+sub, g+1+sub+nsub, ... (ascending, four loads in flight), the groups' sums are then
// added in group order on top of the head partial, and the row is updated once.  The order
// depends only on the geometry, so the result is bit-reproducible (the work list's order is not,
// but no arithmetic depends on it).  Scratch written by other CTAs of the same launch is read with
// L1-bypassing loads.
// The run that leaves head chunk g of table k (gm: that table's geometry).
template <int VEC, int NCH, int THREADS, typename RowT>
__device__ __forceinline__ void fixup_one_run(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                                              float lr, const float* partial, const uint8_t* flags, int k, int g,
                                              const UpdateGeom& gm, typename UV<VEC>::type* red, int* s_first) {
    using V = typename UV<VEC>::type;
    const int lpr = 1 << gm.lpr_log2;
    const int tid = threadIdx.x;
    const int sl = tid & (lpr - 1);
    const int sub = tid >> gm.lpr_log2;
    const int nsub = THREADS >> gm.lpr_log2;
    const size_t D = (size_t)gm.C * VEC;
    const int chunk_entries = gm.G * gm.tile;
    {
        const uint8_t* fk = flags + (size_t)k * gm.pcap;
        const float* pk = partial + (size_t)k * gm.pcap * 2 * D;
        // where the run ends: the first later chunk whose carried run stops inside it (the table's
        // last chunk always stops it)
        if (tid == 0) *s_first = 0x7fffffff;
        __syncthreads();
        for (int base = g + 1;; base += THREADS) {
            const int u = base + tid;
            const uint8_t f = (u < gm.chunks) ? __ldcg(fk + u) : (uint8_t)FLAG_CARRY_ENDS;
            if (f & FLAG_CARRY_ENDS) atomicMin(s_first, u);
            __syncthreads();
            if (*s_first != 0x7fffffff) break;
        }
        const int u_last = *s_first;
        V acc[NCH];
#pragma unroll
        for (int m = 0; m < NCH; ++m) acc[m] = UV<VEC>::zero();
        for (int u = g + 1 + sub; u <= u_last; u += 4 * nsub) {
            V v[4][NCH];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int uu = u + q * nsub;
                const V* src = reinterpret_cast<const V*>(pk + (size_t)uu * 2 * D);
#pragma unroll
                for (int m = 0; m < NCH; ++m)
                    if (uu <= u_last && sl + m * lpr < gm.C) v[q][m] = __ldcg(src + sl + m * lpr);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int m = 0; m < NCH; ++m)
                    if (u + q * nsub <= u_last && sl + m * lpr < gm.C) acc[m] = UV<VEC>::add(acc[m], v[q][m]);
        }
#pragma unroll
        for (int m = 0; m < NCH; ++m) red[(sub * NCH + m) * lpr + sl] = acc[m];
        __syncthreads();
        if (sub == 0) {
            const int nact = min(nsub, u_last - g);
            int last = (g + 1) * chunk_entries - 1;          // last entry of the head chunk
            const uint32_t key = keys[(size_t)k * gm.cap + last];
            float* tbase = desc[k].base;
            const V* hp = reinterpret_cast<const V*>(pk + ((size_t)g * 2 + 1) * D);
#pragma unroll
            for (int m = 0; m < NCH; ++m) {
                if (sl + m * lpr < gm.C) {
                    V total = __ldcg(hp + sl + m * lpr);
                    for (int j = 0; j < nact; ++j) total = UV<VEC>::add(total, red[(j * NCH + m) * lpr + sl]);
                    RowV<VEC, RowT>::store(tbase, key, D, sl + m * lpr,
                                           UV<VEC>::sgd(RowV<VEC, RowT>::load(tbase, key, D, sl + m * lpr), total, lr));
                }
            }
        }
        __syncthreads();
    }
}

template <int VEC, int NCH, int THREADS, typename RowT>
__device__ __forceinline__ void fixup_runs(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                                           float lr, const float* partial, const uint8_t* flags,
                                           const uint32_t* head_list, uint32_t n_heads, uint32_t first,
                                           uint32_t stride, const UpdateGeom& gm,
                                           typename UV<VEC>::type* red, int* s_first) {
    for (uint32_t h = first; h < n_heads; h += stride) {
        const int gid = (int)__ldcg(head_list + h);
        const int k = gid / gm.chunks;
        const int g = gid - k * gm.chunks;
        fixup_one_run<VEC, NCH, THREADS, RowT>(desc, keys, lr, partial, flags, k, g, gm, red, s_first);
    }
}

// Level 3 inside the tiles launch: the same arithmetic as fixup_runs, ONE LANE GROUP per listed run (the
// runs of a DLRM-sized batch span a handful of chunks, and a table has up to chunks - 1 of them, so the
// last CTA of a table works on G runs at a time).  The summation order is fixup_runs' -- nsub = 256 /
// lanes-per-row strided partial sums, added in ascending order on top of the head partial -- so both
// paths give the same bits.
template <int VEC, int NCH, typename RowT>
__device__ __forceinline__ void fixup_runs_grouped(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                                                   float lr, const float* partial, const uint8_t* flags,
                                                   const uint32_t* head_list, uint32_t n_heads, int grp, int G,
                                                   int sl, const UpdateGeom& gm) {
    using V = typename UV<VEC>::type;
    const int lpr = 1 << gm.lpr_log2;
    const int nsub = 256 >> gm.lpr_log2;                 // lane groups of update_fixup_kernel
    const size_t D = (size_t)gm.C * VEC;
    const int chunk_entries = gm.G * gm.tile;
    for (uint32_t h = grp; h < n_heads; h += G) {
        const int gid = (int)__ldcg(head_list + h);
        const int k = gid / gm.chunks;
        const int g = gid - k * gm.chunks;
        const uint8_t* fk = flags + (size_t)k * gm.pcap;
        const float* pk = partial + (size_t)k * gm.pcap * 2 * D;
        int u_last = gm.chunks - 1;
        for (int base = g + 1; base < gm.chunks; base += 8) {
            uint8_t f[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) f[q] = (base + q < gm.chunks) ? __ldcg(fk + base + q) : (uint8_t)FLAG_CARRY_ENDS;
            int first = -1;
#pragma unroll
            for (int q = 7; q >= 0; --q)
                if (f[q] & FLAG_CARRY_ENDS) first = q;
            if (first >= 0) {
                u_last = base + first;
                break;
            }
        }
        const int nact = min(nsub, u_last - g);
        const int last = (g + 1) * chunk_entries - 1;    // last entry of the head chunk
        const uint32_t key = keys[(size_t)k * gm.cap + last];
        float* tbase = desc[k].base;
        const V* hp = reinterpret_cast<const V*>(pk + ((size_t)g * 2 + 1) * D);
#pragma unroll
        for (int m = 0; m < NCH; ++m) {
            const int c = sl + m * lpr;
            if (c >= gm.C) continue;
            V total = __ldcg(hp + c);
            const V row = RowV<VEC, RowT>::load(tbase, key, D, c);
            for (int j = 0; j < nact; ++j) {
                V acc = UV<VEC>::zero();
#pragma unroll 4
                for (int u = g + 1 + j; u <= u_last; u += nsub)
                    acc = UV<VEC>::add(acc, __ldcg(reinterpret_cast<const V*>(pk + (size_t)u * 2 * D) + c));
                total = UV<VEC>::add(total, acc);
            }
            RowV<VEC, RowT>::store(tbase, key, D, c, UV<VEC>::sgd(row, total, lr));
        }
    }
}

// Level 3 inside the tiles launch when the table has at most kInlineSmemChunks chunks (every DLRM-sized batch):
// the last CTA of the table has the chunk flags, the list of head chunks and the heads' row ids in shared memory
// (one round of loads), a lane group finds its run's end with ballots over the shared flags, and the head partial,
// the row and the first eight carry partials of the run are requested together -- one more round of loads instead
// of one per partial.  Same summation order as fixup_runs_grouped / fixup_runs, hence the same bits.
constexpr int kInlineSmemChunks = 1024;

template <int VEC, int NCH, typename RowT>
__device__ __forceinline__ void fixup_runs_smem(const TableDesc* __restrict__ desc, float lr, const float* partial,
                                                const uint8_t* s_fl, const uint16_t* s_heads, const uint32_t* s_hkey,
                                                uint32_t n_heads, int k, int grp, int G, int sl, const UpdateGeom& gm) {
    using V = typename UV<VEC>::type;
    const int lpr = 1 << gm.lpr_log2;
    const int nsub = 256 >> gm.lpr_log2;                 // lane groups of update_fixup_kernel
    const size_t D = (size_t)gm.C * VEC;
    const unsigned gshift = (threadIdx.x & 31) & ~(lpr - 1);
    const unsigned gbits = (lpr >= 32) ? 0xffffffffu : ((1u << lpr) - 1u);
    const unsigned gmask = gbits << gshift;
    const float* pk = partial + (size_t)k * gm.pcap * 2 * D;
    float* tbase = desc[k].base;
    for (uint32_t h = grp; h < n_heads; h += G) {
        const int g = s_heads[h];
        const uint32_t key = s_hkey[h];
        int u_last = gm.chunks - 1;
        for (int base = g + 1; base < gm.chunks; base += lpr) {
            const int u = base + sl;
            const bool ends = (u >= gm.chunks) || (s_fl[u] & FLAG_CARRY_ENDS);
            // the ballot also carries the flags of other lane groups of the warp that vote at the same time
            // (the mask names who must take part, not whose bits come back): keep this group's own
            const unsigned b = (__ballot_sync(gmask, ends) >> gshift) & gbits;
            if (b != 0) {
                u_last = min(gm.chunks - 1, base + __ffs((int)b) - 1);
                break;
            }
        }
        const int nact = min(nsub, u_last - g);
        const V* hp = reinterpret_cast<const V*>(pk + ((size_t)g * 2 + 1) * D);
#pragma unroll
        for (int m = 0; m < NCH; ++m) {
            const int c = sl + m * lpr;
            if (c >= gm.C) continue;
            V total = __ldcg(hp + c);
            const V row = RowV<VEC, RowT>::load(tbase, key, D, c);
            for (int jb = 0; jb < nact; jb += 8) {
                V p[8];
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (jb + q < nact) p[q] = __ldcg(reinterpret_cast<const V*>(pk + (size_t)(g + 1 + jb + q) * 2 * D) + c);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (jb + q >= nact) break;
                    V acc = UV<VEC>::add(UV<VEC>::zero(), p[q]);
#pragma unroll 4
                    for (int u = g + 1 + jb + q + nsub; u <= u_last; u += nsub)
                        acc = UV<VEC>::add(acc, __ldcg(reinterpret_cast<const V*>(pk + (size_t)u * 2 * D) + c));
                    total = UV<VEC>::add(total, acc);
                }
            }
            RowV<VEC, RowT>::store(tbase, key, D, c, UV<VEC>::sgd(row, total, lr));
        }
    }
}

// head_count: [0] = listed head chunks (two-launch path), [1 + k] = CTAs of table k that are done
// (INLINE path; zero between launches).
// Chunk `cta` of table k (gm: that table's geometry).  `gid` names the chunk in the two-launch head list,
// `ndone` is the table's chunk count (the INLINE done-counter target), `clk_cta` its stamp slot.
// SCALE (jagged mean pooling or per-sample weights): each gradient row is multiplied by its entry's weight `wts` (f32 bits, the
// stream's layout) before it is accumulated.
template <int VEC, int NCH, int THREADS, typename RowT, bool INLINE, bool SCALE = false>
__device__ __forceinline__ void update_tiles_body(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                                                  const uint32_t* __restrict__ pos, const float* __restrict__ dT, float lr,
                                                  float* __restrict__ partial, uint8_t* __restrict__ flags,
                                                  uint32_t* __restrict__ head_list, uint32_t* __restrict__ head_count,
                                                  const UpdateGeom& gm, int k, int cta, uint32_t gid, uint32_t ndone,
                                                  unsigned long long* clk, unsigned clk_cta,
                                                  const uint32_t* __restrict__ wts = nullptr) {
    using V = typename UV<VEC>::type;
    constexpr int U = 4;
    clock_in(clk, clk_cta);
    __shared__ V s_carry[THREADS * NCH];   // per group: partial of the run carried in from the previous tile
    __shared__ V s_head[THREADS * NCH];    // per group: partial of the run that continues into the next tile
    __shared__ uint8_t s_flag[THREADS];
    __shared__ int s_cta_head;
    __shared__ int s_first;
    __shared__ uint32_t s_nheads;

    const int lpr = 1 << gm.lpr_log2;
    const int G = THREADS >> gm.lpr_log2;
    const int tid = threadIdx.x;
    const int grp = tid >> gm.lpr_log2;
    const int sl = tid & (lpr - 1);
    const int g = cta * G + grp;              // tile index inside table k
    const bool active = g < gm.tiles;
    const size_t D = (size_t)gm.C * VEC;

    const uint32_t* __restrict__ ks = keys + (size_t)k * gm.cap;
    const uint32_t* __restrict__ ps = pos + (size_t)k * gm.cap;
    const uint32_t* __restrict__ ws = SCALE ? wts + (size_t)k * gm.cap : nullptr;
    float* tb = desc[k].base;
    const float* __restrict__ gbase = dT + (size_t)(gm.slot0 + k) * D;
    const size_t gstride = (size_t)gm.slots * D;

    bool chunk_ok[NCH];
#pragma unroll
    for (int m = 0; m < NCH; ++m) chunk_ok[m] = (sl + m * lpr) < gm.C;
    if (tid == 0) s_cta_head = 0;

    uint8_t fl = 0;
    uint32_t last_key = 0;
    V acc[NCH];
#pragma unroll
    for (int m = 0; m < NCH; ++m) acc[m] = UV<VEC>::zero();

    if (active) {
        const int e0 = g * gm.tile;
        const int e1 = min(gm.L, e0 + gm.tile);
        uint4 kq = __ldg(reinterpret_cast<const uint4*>(ks + e0));
        uint4 pq = __ldg(reinterpret_cast<const uint4*>(ps + e0));
        uint4 wq;
        if (SCALE) wq = __ldg(reinterpret_cast<const uint4*>(ws + e0));
        uint32_t kn = (e0 + U < gm.L) ? __ldg(ks + e0 + U) : 0xffffffffu;
        const uint32_t kprev = (e0 > 0) ? __ldg(ks + e0 - 1) : 0xffffffffu;
        const bool cin = e0 > 0 && kprev == kq.x;
        bool cout = false;
        bool first = cin;
        fl = cin ? FLAG_CARRY_IN : 0;

        for (int e = e0; e < e1; e += U) {
            const uint32_t key[U + 1] = {kq.x, kq.y, kq.z, kq.w, kn};
            const uint32_t pp[U] = {pq.x, pq.y, pq.z, pq.w};
            const uint32_t wb[U] = {SCALE ? wq.x : 0u, SCALE ? wq.y : 0u, SCALE ? wq.z : 0u, SCALE ? wq.w : 0u};
            if (e + U < e1) {   // request the next batch's keys / positions now
                kq = __ldg(reinterpret_cast<const uint4*>(ks + e + U));
                pq = __ldg(reinterpret_cast<const uint4*>(ps + e + U));
                if (SCALE) wq = __ldg(reinterpret_cast<const uint4*>(ws + e + U));
                kn = (e + 2 * U < gm.L) ? __ldg(ks + e + 2 * U) : 0xffffffffu;
            }
            bool valid[U], is_end[U];
            V dv[U][NCH], rv[U][NCH];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int ee = e + u;
                valid[u] = ee < e1;
                is_end[u] = valid[u] && ((ee + 1 >= gm.L) || (key[u + 1] != key[u]));
                const uint32_t b = (gm.P == 1) ? pp[u] : pp[u] / (uint32_t)gm.P;
                const V* src = reinterpret_cast<const V*>(gbase + (size_t)b * gstride);
#pragma unroll
                for (int m = 0; m < NCH; ++m)
                    if (valid[u] && chunk_ok[m]) dv[u][m] = __ldg(src + sl + m * lpr);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
#pragma unroll
                for (int m = 0; m < NCH; ++m)
                    if (is_end[u] && chunk_ok[m]) rv[u][m] = RowV<VEC, RowT>::load(tb, key[u], D, sl + m * lpr);
            }
            if (e + U >= e1) {
                cout = (e1 < gm.L) && (e + U == e1) && (key[U] == key[U - 1]);
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (e + u == e1 - 1) last_key = key[u];
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (!valid[u]) continue;
#pragma unroll
                for (int m = 0; m < NCH; ++m)
                    if (chunk_ok[m]) acc[m] = UV<VEC>::add(acc[m], SCALE ? UV<VEC>::scale(dv[u][m], __uint_as_float(wb[u])) : dv[u][m]);
                if (is_end[u]) {
                    if (first) {
                        // run started in an earlier tile: hand the partial sum to its owner
#pragma unroll
                        for (int m = 0; m < NCH; ++m) s_carry[(grp * NCH + m) * lpr + sl] = acc[m];
                        fl |= FLAG_CARRY_ENDS;
                    } else {
#pragma unroll
                        for (int m = 0; m < NCH; ++m)
                            if (chunk_ok[m])
                                RowV<VEC, RowT>::store(tb, key[u], D, sl + m * lpr, UV<VEC>::sgd(rv[u][m], acc[m], lr));
                    }
                    first = false;
#pragma unroll
                    for (int m = 0; m < NCH; ++m) acc[m] = UV<VEC>::zero();
                }
            }
        }
        if (cout) {
            if (first) {   // the whole tile is one run that came in and goes on: pass-through
#pragma unroll
                for (int m = 0; m < NCH; ++m) s_carry[(grp * NCH + m) * lpr + sl] = acc[m];
            } else {
                fl |= FLAG_HEAD;
#pragma unroll
                for (int m = 0; m < NCH; ++m) s_head[(grp * NCH + m) * lpr + sl] = acc[m];
            }
        }
    }
    if (sl == 0) s_flag[grp] = fl;
    __syncthreads();

    // ---- level 2: finish, through shared memory, the runs that cross tiles inside this chunk ----
    const int nact = min(G, gm.tiles - cta * G);     // active groups in this CTA
    float* pcarry = partial + (((size_t)k * gm.pcap + cta) * 2 + 0) * D;
    float* phead = partial + (((size_t)k * gm.pcap + cta) * 2 + 1) * D;
    bool wrote_scratch = false;
    if (active && (fl & FLAG_HEAD)) {
        // this group's last run continues: add the carry partials of the following tiles up to
        // (and including) the first one in which the run ends
        int j = grp + 1;
        bool ended = false;
        V tot[NCH];
#pragma unroll
        for (int m = 0; m < NCH; ++m) tot[m] = s_head[(grp * NCH + m) * lpr + sl];
        for (; j < nact; ++j) {
#pragma unroll
            for (int m = 0; m < NCH; ++m) tot[m] = UV<VEC>::add(tot[m], s_carry[(j * NCH + m) * lpr + sl]);
            if (s_flag[j] & FLAG_CARRY_ENDS) { ended = true; break; }
        }
        if (ended) {
#pragma unroll
            for (int m = 0; m < NCH; ++m)
                if (chunk_ok[m])
                    RowV<VEC, RowT>::store(tb, last_key, D, sl + m * lpr,
                                           UV<VEC>::sgd(RowV<VEC, RowT>::load(tb, last_key, D, sl + m * lpr), tot[m], lr));
        } else {   // the run leaves the chunk: level 3 finishes it
#pragma unroll
            for (int m = 0; m < NCH; ++m)
                if (chunk_ok[m]) reinterpret_cast<V*>(phead)[sl + m * lpr] = tot[m];
            if (sl == 0) {
                s_cta_head = 1;
                // same-launch fix-up from shared memory: the run's row id travels with the chunk's flag
                if (INLINE && gm.chunks <= kInlineSmemChunks) head_list[(size_t)k * gm.pcap + cta] = last_key;
            }
            wrote_scratch = true;
        }
    }
    uint8_t cta_flag = 0;
    if (grp == 0 && (s_flag[0] & FLAG_CARRY_IN)) {
        // the run carried into the chunk: its partial is the carry partials of the leading tiles
        cta_flag = FLAG_CARRY_IN;
        V tot[NCH];
#pragma unroll
        for (int m = 0; m < NCH; ++m) tot[m] = UV<VEC>::zero();
        for (int j = 0; j < nact; ++j) {
#pragma unroll
            for (int m = 0; m < NCH; ++m) tot[m] = UV<VEC>::add(tot[m], s_carry[(j * NCH + m) * lpr + sl]);
            if (s_flag[j] & FLAG_CARRY_ENDS) { cta_flag |= FLAG_CARRY_ENDS; break; }
        }
#pragma unroll
        for (int m = 0; m < NCH; ++m)
            if (chunk_ok[m]) reinterpret_cast<V*>(pcarry)[sl + m * lpr] = tot[m];
        wrote_scratch = true;
    }
    if (INLINE && wrote_scratch) __threadfence();   // partials are visible before this CTA's completion is counted
    __syncthreads();
    if (!INLINE) {
        if (tid == 0) {
            if (s_cta_head) {
                cta_flag |= FLAG_HEAD;
                head_list[atomicAdd(head_count, 1u)] = gid;
            }
            flags[(size_t)k * gm.pcap + cta] = cta_flag;
        }
        clock_out(clk, clk_cta);
        return;
    }

    // ---- level 3 inside this launch: the last CTA of table k to get here finishes the table's
    // chunk-crossing runs (the pattern of the threadfence reduction: publish, fence, count).
    if (tid == 0) {
        if (s_cta_head) cta_flag |= FLAG_HEAD;
        *reinterpret_cast<volatile uint8_t*>(flags + (size_t)k * gm.pcap + cta) = cta_flag;
        __threadfence();
        const uint32_t done = atomicAdd(head_count + 1 + k, 1u) + 1u;
        s_first = (done == ndone) ? 1 : 0;
        if (done == ndone) head_count[1 + k] = 0;   // re-arm for the next launch (every CTA of the table has counted)
        s_nheads = 0;
    }
    __syncthreads();
    if (!s_first) {
        clock_out(clk, clk_cta);
        return;
    }
    __threadfence();
    if (gm.chunks <= kInlineSmemChunks) {
        __shared__ uint8_t s_fl[kInlineSmemChunks];
        __shared__ uint16_t s_heads[kInlineSmemChunks];
        __shared__ uint32_t s_hkey[kInlineSmemChunks];
        const uint8_t* fk = flags + (size_t)k * gm.pcap;
        const uint32_t* hk = head_list + (size_t)k * gm.pcap;
        for (int base = 0; base < gm.chunks; base += THREADS) {
            const int u = base + tid;
            if (u < gm.chunks) {
                const uint8_t f = __ldcg(fk + u);
                const uint32_t key = __ldcg(hk + u);     // meaningful for head chunks only
                s_fl[u] = f;
                if (f & FLAG_HEAD) {
                    const uint32_t slot = atomicAdd(&s_nheads, 1u);
                    s_heads[slot] = (uint16_t)u;
                    s_hkey[slot] = key;
                }
            }
        }
        __syncthreads();
        const uint32_t n_heads = s_nheads;
        if (n_heads != 0) fixup_runs_smem<VEC, NCH, RowT>(desc, lr, partial, s_fl, s_heads, s_hkey, n_heads, k, grp, G, sl, gm);
        __syncthreads();      // thread 0 stamps the exit after every lane group of the CTA has finished its runs
        clock_out(clk, clk_cta);
        return;
    }
    // list the table's head chunks (order irrelevant: distinct runs touch distinct rows)
    uint32_t* my_heads = head_list + (size_t)k * gm.pcap;
    const uint8_t* fk = flags + (size_t)k * gm.pcap;
    for (int base = 0; base < gm.chunks; base += THREADS) {
        const int u = base + tid;
        if (u < gm.chunks && (__ldcg(fk + u) & FLAG_HEAD)) __stcg(my_heads + atomicAdd(&s_nheads, 1u), (uint32_t)(k * gm.chunks + u));
    }
    __syncthreads();
    const uint32_t n_heads = s_nheads;
    if (n_heads != 0) fixup_runs_grouped<VEC, NCH, RowT>(desc, keys, lr, partial, flags, my_heads, n_heads, grp, G, sl, gm);
    __syncthreads();      // thread 0 stamps the exit after every lane group of the CTA has finished its runs
    clock_out(clk, clk_cta);
}

template <int VEC, int NCH, int THREADS, typename RowT, bool INLINE>
__global__ void __launch_bounds__(THREADS, (NCH <= 1) ? 3 : ((NCH <= 2) ? 2 : 1))
update_tiles_kernel(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                    const uint32_t* __restrict__ pos, const float* __restrict__ dT, float lr,
                    float* __restrict__ partial, uint8_t* __restrict__ flags,
                    uint32_t* __restrict__ head_list, uint32_t* __restrict__ head_count, UpdateGeom gm,
                    unsigned long long* clk) {
    const int k = blockIdx.y, cta = blockIdx.x;
    update_tiles_body<VEC, NCH, THREADS, RowT, INLINE>(desc, keys, pos, dT, lr, partial, flags, head_list, head_count, gm,
                                                       k, cta, (uint32_t)(k * gm.chunks + cta), gridDim.x, clk,
                                                       blockIdx.y * gridDim.x + blockIdx.x);
}

template <int VEC, int NCH, typename RowT>
__global__ void __launch_bounds__(256)
update_fixup_kernel(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys, float lr,
                    const float* __restrict__ partial, const uint8_t* __restrict__ flags,
                    const uint32_t* __restrict__ head_list, const uint32_t* __restrict__ head_count,
                    UpdateGeom gm, unsigned long long* clk) {
    using V = typename UV<VEC>::type;
    __shared__ V red[256 * NCH];
    __shared__ int s_first;
    clock_in(clk, blockIdx.x);
    fixup_runs<VEC, NCH, 256, RowT>(desc, keys, lr, partial, flags, head_list, *head_count, blockIdx.x,
                                    gridDim.x, gm, red, &s_first);
    clock_out(clk, blockIdx.x);
}

// ---- per-table pooling factors: one flat grid of sum_k chunks_k CTAs; g.pre maps a CTA to (table, chunk),
// g.P / g.units give each table its P_k and tile count, so every table has its own L_k, tiles and chunks while
// the tile length is the batch's (chosen from the total entry count, as for a uniform batch).  The two-launch
// head list names chunks by their flat CTA id.
__device__ __forceinline__ UpdateGeom update_geom_mp(const UpdateGeom& gm0, const MpGeom& g, int k) {
    UpdateGeom gm = gm0;
    gm.P = (int)g.P[k];
    gm.L = (int)(g.B * g.P[k]);
    gm.tiles = (int)g.units[k];
    gm.chunks = (int)(g.pre[k + 1] - g.pre[k]);
    return gm;
}

template <int VEC, int NCH, int THREADS, typename RowT, bool INLINE>
__global__ void __launch_bounds__(THREADS, (NCH <= 1) ? 3 : ((NCH <= 2) ? 2 : 1))
update_tiles_mp_kernel(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                       const uint32_t* __restrict__ pos, const float* __restrict__ dT, float lr,
                       float* __restrict__ partial, uint8_t* __restrict__ flags,
                       uint32_t* __restrict__ head_list, uint32_t* __restrict__ head_count, UpdateGeom gm0,
                       const __grid_constant__ MpGeom g, unsigned long long* clk) {
    const uint32_t lin = blockIdx.x;
    const int k = mp_find(g.pre, g.ntab, lin);
    const UpdateGeom gm = update_geom_mp(gm0, g, k);
    update_tiles_body<VEC, NCH, THREADS, RowT, INLINE>(desc, keys, pos, dT, lr, partial, flags, head_list, head_count, gm,
                                                       k, (int)(lin - g.pre[k]), lin, (uint32_t)gm.chunks, clk, lin);
}

template <int VEC, int NCH, typename RowT>
__global__ void __launch_bounds__(256)
update_fixup_mp_kernel(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys, float lr,
                       const float* __restrict__ partial, const uint8_t* __restrict__ flags,
                       const uint32_t* __restrict__ head_list, const uint32_t* __restrict__ head_count,
                       UpdateGeom gm0, const __grid_constant__ MpGeom g, unsigned long long* clk) {
    using V = typename UV<VEC>::type;
    __shared__ V red[256 * NCH];
    __shared__ int s_first;
    clock_in(clk, blockIdx.x);
    const uint32_t n_heads = *head_count;
    for (uint32_t h = blockIdx.x; h < n_heads; h += gridDim.x) {
        const uint32_t gid = __ldcg(head_list + h);
        const int k = mp_find(g.pre, g.ntab, gid);
        const UpdateGeom gm = update_geom_mp(gm0, g, k);
        fixup_one_run<VEC, NCH, 256, RowT>(desc, keys, lr, partial, flags, k, (int)(gid - g.pre[k]), gm, red, &s_first);
    }
    clock_out(clk, blockIdx.x);
}

// ---- jagged bags: the `_mp` flat grid over a stream of bag ids (P = 1) with per-table L_k (g.P[k] = L_k, g.B = 1,
// as the jagged sort records them); tables with L_k = 0 own no chunk, and mp_find skips them (it returns the last
// table whose range starts at or before the CTA).  The two-launch fix-up is update_fixup_mp_kernel's: it reads no
// position.
template <int VEC, int NCH, int THREADS, typename RowT, bool INLINE, bool SCALE>
__global__ void __launch_bounds__(THREADS, (NCH <= 1) ? 3 : ((NCH <= 2) ? 2 : 1))
update_tiles_jagged_kernel(const TableDesc* __restrict__ desc, const uint32_t* __restrict__ keys,
                           const uint32_t* __restrict__ bags, const uint32_t* __restrict__ wts, const float* __restrict__ dT,
                           float lr, float* __restrict__ partial, uint8_t* __restrict__ flags,
                           uint32_t* __restrict__ head_list, uint32_t* __restrict__ head_count, UpdateGeom gm0,
                           const __grid_constant__ MpGeom g, unsigned long long* clk) {
    const uint32_t lin = blockIdx.x;
    const int k = mp_find(g.pre, g.ntab, lin);
    UpdateGeom gm = update_geom_mp(gm0, g, k);
    gm.P = 1;
    update_tiles_body<VEC, NCH, THREADS, RowT, INLINE, SCALE>(desc, keys, bags, dT, lr, partial, flags, head_list, head_count,
                                                              gm, k, (int)(lin - g.pre[k]), lin, (uint32_t)gm.chunks, clk,
                                                              lin, wts);
}

static int lanes_per_row_log2(int C) {
    int l = 0;
    while ((1 << l) < C && l < 5) ++l;
    return l;
}

// Entries per lane-group tile: the smallest multiple of 4 (the keys of a batch are one 16-byte load) up to
// 32 with which the whole batch is ONE wave of resident CTAs (`resident_threads` per SM follow from the
// kernel's launch bound).  At DLRM batch sizes a second wave costs a full dependent key -> row -> store
// latency chain, and a longer tile costs one such chain per 4 entries; measured on B200 (26 tables x 2048
// lookups): D = 128 tile 4 / 8 / 16 -> 24.2 / 17.8 / 16.0 us, D = 64 -> 14.9 / 11.3 / 12.2 us, i.e. the
// first tile that fits one wave wins.  (Round 1 only tried powers of two: an owner with 4 tables x 16384
// lookups -- 8 GPUs -- then jumped from 16 to 32 entries, 37 us instead of 18 us for the 3-table owners.)
static int choose_update_tile(int64_t total_entries, int lpr, int sm_count, int resident_threads) {
    const int64_t capacity = (int64_t)sm_count * resident_threads / lpr;
    int64_t tile = (total_entries + capacity - 1) / capacity;
    tile = (tile + 3) / 4 * 4;
    if (tile < 4) tile = 4;
    if (tile > 32) tile = 32;
    return (int)tile;
}

// Upper bound on chunks (CTAs) per table for any batch with B*P <= max_lookups.
int64_t update_tiles_cap(int ntab, int D, int64_t max_lookups, int sm_count) {
    (void)ntab;
    (void)sm_count;
    const int vec = (D % 4 == 0) ? 4 : 1;
    const int C = D / vec;
    const int lpr = 1 << lanes_per_row_log2(C);
    const int nch = (C + lpr - 1) / lpr;
    const int G = (nch > 4 ? 128 : 256) / lpr;
    return ceil_div64(ceil_div64(max_lookups, 4), G) + 2;   // smallest tile (4) gives the most chunks
}

// Consumes the last sort (B and every table's P_k).  With equal P_k the tables share one geometry and the grid
// is two-dimensional (grid.y = table); otherwise one flat grid of sum_k chunks_k CTAs, g.pre mapping a CTA to
// (table, chunk).  The tile is chosen from the total entry count either way, so equal P_k take the same tiles
// and chunks on both grids, hence the same bits.  A jagged sort (g.B = 1, P_k = L_k) takes the flat grid with
// update_tiles_jagged_kernel over the bag ids (and, for mean or weighted pooling, the weights) that launch_jagged_bags wrote into
// pos / keys [sorted_buf ^ 1]; the fix-up kernel is the same for both, it reads no position.
template <int VEC, int NCH, typename RowT>
static int launch_update_t(dlrmb_tables* t, const float* dT, int slots, int slot0, float lr, cudaStream_t s) {
    constexpr int THREADS = (NCH > 4) ? 128 : 256;   // keeps the two partial arrays within 48 KB
    const int32_t* P = t->h_sorted_P;
    bool equal = true;
    int64_t total = 0, maxL = 0;
    for (int k = 0; k < t->ntab; ++k) {
        const int64_t L = (int64_t)t->sorted_B * P[k];
        total += L;
        maxL = L > maxL ? L : maxL;
        equal = equal && P[k] == P[0];
    }
    UpdateGeom gm;
    gm.C = t->D / VEC;
    gm.lpr_log2 = lanes_per_row_log2(gm.C);
    const int lpr = 1 << gm.lpr_log2;
    const int G = THREADS / lpr;
    gm.G = G;
    gm.tile = choose_update_tile(total, lpr, t->sm_count, THREADS * ((NCH <= 1) ? 3 : ((NCH <= 2) ? 2 : 1)));
    {   // tuning aid (dlrmb_set_option("update_tile", v)): 4, 8, 16 or 32 entries per lane group
        const int v = g_opt.update_tile.load(std::memory_order_relaxed);
        if (v >= 4 && v <= 32 && v % 4 == 0) gm.tile = v;
    }
    gm.slots = slots;
    gm.slot0 = slot0;
    gm.cap = t->cap;
    gm.pcap = t->partial_tiles_cap;
    const uint32_t* keys = t->keys[t->sorted_buf];
    const uint32_t* pos = t->pos[t->sorted_buf];
    // DLRM-sized batches: level 3 runs inside the same launch (see the header comment)
    const bool inline_fixup = total <= kUpdateInlineMaxEntries &&
                              g_opt.update_two_launches.load(std::memory_order_relaxed) == 0;
    const int jagged = t->sorted_jagged;   // -1: uniform or _mp sort, 0 / 1 / 2: jagged sum / mean / weighted sum
    if (equal && jagged < 0) {
        gm.L = (int)maxL;
        gm.P = P[0];
        gm.tiles = (gm.L + gm.tile - 1) / gm.tile;
        gm.chunks = (gm.tiles + G - 1) / G;
        DLRMB_REQUIRE(gm.chunks <= gm.pcap, "internal: update chunk capacity exceeded (%d > %lld)",
                      gm.chunks, (long long)gm.pcap);
        DLRMB_REQUIRE((int64_t)t->ntab * gm.chunks < (1ll << 31), "batch too large for one update launch");
        dim3 grid((unsigned)gm.chunks, (unsigned)t->ntab);
        const int64_t total_chunks = (int64_t)t->ntab * gm.chunks;
        if (inline_fixup) {
            update_tiles_kernel<VEC, NCH, THREADS, RowT, true><<<grid, THREADS, 0, s>>>(
                t->d_desc, keys, pos, dT, lr, t->partial, t->tile_flags, t->head_list, t->head_count, gm, clock_slot(CLK_UPDATE));
            DLRMB_LAUNCH_CHECK();
            return DLRMB_OK;
        }
        DLRMB_CUDA(cudaMemsetAsync(t->head_count, 0, sizeof(uint32_t), s));
        update_tiles_kernel<VEC, NCH, THREADS, RowT, false><<<grid, THREADS, 0, s>>>(
            t->d_desc, keys, pos, dT, lr, t->partial, t->tile_flags, t->head_list, t->head_count, gm, clock_slot(CLK_UPDATE));
        DLRMB_LAUNCH_CHECK();
        unsigned fgrid = (unsigned)(total_chunks < (int64_t)t->sm_count * 8 ? total_chunks : (int64_t)t->sm_count * 8);
        update_fixup_kernel<VEC, NCH, RowT><<<fgrid, 256, 0, s>>>(t->d_desc, keys, lr, t->partial, t->tile_flags,
                                                                 t->head_list, t->head_count, gm, clock_slot(CLK_FIXUP));
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    }
    // mixed P_k or jagged: only the `_mp` and jagged sorts, at most kMpMaxTables tables
    MpGeom g;
    g.ntab = t->ntab;
    g.B = (uint32_t)t->sorted_B;
    g.nlist = 0;
    gm.L = (int)maxL;
    gm.P = 1;
    gm.tiles = 0;
    gm.chunks = 0;
    int64_t chunks_total = 0;
    for (int k = 0; k < t->ntab; ++k) {
        g.P[k] = (uint32_t)P[k];
        g.off[k] = 0;   // unused by the update
        const int64_t tiles = ceil_div64((int64_t)g.B * g.P[k], gm.tile);
        const int64_t chunks = ceil_div64(tiles, G);
        DLRMB_REQUIRE(chunks <= gm.pcap, "internal: update chunk capacity exceeded (%lld > %lld)", (long long)chunks,
                      (long long)gm.pcap);
        g.units[k] = (uint32_t)tiles;
        g.pre[k] = (uint32_t)chunks_total;
        chunks_total += chunks;
    }
    g.pre[t->ntab] = (uint32_t)chunks_total;
    DLRMB_REQUIRE(chunks_total < (1ll << 31), "batch too large for one update launch");
    if (chunks_total == 0) return DLRMB_OK;   // a jagged batch without lookups
    const uint32_t* bags = t->pos[t->sorted_buf ^ 1];
    const uint32_t* wts = t->keys[t->sorted_buf ^ 1];
    auto tiles = [&](auto inl) {
        constexpr bool INL = decltype(inl)::value;
        const unsigned n = (unsigned)chunks_total;
        if (jagged >= 1)   // mean or per-sample weights: one weight per sorted entry
            update_tiles_jagged_kernel<VEC, NCH, THREADS, RowT, INL, true><<<n, THREADS, 0, s>>>(
                t->d_desc, keys, bags, wts, dT, lr, t->partial, t->tile_flags, t->head_list, t->head_count, gm, g,
                clock_slot(CLK_UPDATE));
        else if (jagged == 0)
            update_tiles_jagged_kernel<VEC, NCH, THREADS, RowT, INL, false><<<n, THREADS, 0, s>>>(
                t->d_desc, keys, bags, wts, dT, lr, t->partial, t->tile_flags, t->head_list, t->head_count, gm, g,
                clock_slot(CLK_UPDATE));
        else
            update_tiles_mp_kernel<VEC, NCH, THREADS, RowT, INL><<<n, THREADS, 0, s>>>(
                t->d_desc, keys, pos, dT, lr, t->partial, t->tile_flags, t->head_list, t->head_count, gm, g,
                clock_slot(CLK_UPDATE));
    };
    if (inline_fixup) {
        tiles(std::true_type{});
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    }
    DLRMB_CUDA(cudaMemsetAsync(t->head_count, 0, sizeof(uint32_t), s));
    tiles(std::false_type{});
    DLRMB_LAUNCH_CHECK();
    unsigned fgrid = (unsigned)(chunks_total < (int64_t)t->sm_count * 8 ? chunks_total : (int64_t)t->sm_count * 8);
    update_fixup_mp_kernel<VEC, NCH, RowT><<<fgrid, 256, 0, s>>>(t->d_desc, keys, lr, t->partial, t->tile_flags,
                                                                t->head_list, t->head_count, gm, g, clock_slot(CLK_FIXUP));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <typename RowT>
static int launch_update_r(dlrmb_tables* t, const float* dT, int slots, int slot0, float lr, cudaStream_t s) {
    const bool vec4 = (t->D % 4 == 0) && ((reinterpret_cast<uintptr_t>(dT) & 15) == 0);
    if (t->D % 4 == 0 && !vec4) {
        set_error("dT must be 16-byte aligned when D is a multiple of 4");
        return DLRMB_EINVAL;
    }
    const int C = vec4 ? t->D / 4 : t->D;
    const int lpr = 1 << lanes_per_row_log2(C);
    const int nch = (C + lpr - 1) / lpr;
    if (vec4) {
        if (nch == 1) return launch_update_t<4, 1, RowT>(t, dT, slots, slot0, lr, s);
        if (nch == 2) return launch_update_t<4, 2, RowT>(t, dT, slots, slot0, lr, s);
        if (nch <= 4) return launch_update_t<4, 4, RowT>(t, dT, slots, slot0, lr, s);
        if (nch <= 8) return launch_update_t<4, 8, RowT>(t, dT, slots, slot0, lr, s);
    } else {
        if (nch == 1) return launch_update_t<1, 1, RowT>(t, dT, slots, slot0, lr, s);
        if (nch == 2) return launch_update_t<1, 2, RowT>(t, dT, slots, slot0, lr, s);
        if (nch <= 4) return launch_update_t<1, 4, RowT>(t, dT, slots, slot0, lr, s);
        if (nch <= 8) return launch_update_t<1, 8, RowT>(t, dT, slots, slot0, lr, s);
    }
    set_error("embedding dim %d unsupported by the update kernel", t->D);
    return DLRMB_EINVAL;
}

int launch_update(dlrmb_tables* t, const float* dT, int slots, int slot0, float lr, cudaStream_t s) {
    if (t->elem_bytes == 2) return launch_update_r<__nv_bfloat16>(t, dT, slots, slot0, lr, s);
    return launch_update_r<float>(t, dT, slots, slot0, lr, s);
}

}  // namespace dlrmb
