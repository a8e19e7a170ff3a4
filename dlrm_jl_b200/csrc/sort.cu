// Index sort / dedup for the sparse-gradient update.
//
// Role in the reference: EmbeddingTables.SparseIndexer, the per-table dictionary that
// compacts duplicate row ids before EmbeddingTables.update! (DLRM.jl src/train/train.jl:107-115,
// 276-290).  Here the dictionary is replaced by a stable sort of (row id, flat position) pairs per
// table, which makes duplicates adjacent and fixes their accumulation order (ascending flat
// position) so the update is deterministic without floating-point atomics.
//
// Two paths, chosen per table from L_k = B*P_k (one batch can use both):
//   * L_k <= kSmemSortMax: one CTA per table runs the whole LSD radix sort in shared memory
//     (digits of up to 9 bits, as many passes as that table's row count needs); a single launch
//     covers all such tables.  Training steps do not even pay that launch: dlrmb_embedding_fwd_sort runs
//     the same sort in extra CTAs of the lookup launch (lookup.cu), hidden behind the gather.
//   * larger L_k: least-significant-digit radix sort, digits of up to 9 bits, tiles of 4096 keys, all such
//     tables batched through grid.y.  Per pass: per-tile digit histogram -> exclusive scan over
//     (digit, tile), one CTA per digit -> stable scatter whose in-tile ranks come from warp match_any + per-warp
//     digit counters in shared memory and whose keys are reordered in shared memory first, so each
//     digit's keys leave the CTA as one contiguous run.  The sort arrays of a whole batch fit L2 (126 MB), so the
//     passes run at L2 rather than HBM speed.
// Output: keys[sorted_buf] (ascending 0-based row ids) and pos[sorted_buf] (the stable
// permutation), both [ntab][max_lookups].
#include "common.cuh"
#include "sort_small.cuh"

namespace dlrmb {

// ---------------------------------------------------------------------------------------------
// large path: LSD radix sort over global memory (device bodies; the kernels are below)
// ---------------------------------------------------------------------------------------------
constexpr int RT = 256;        // threads per CTA
constexpr int RI = 16;         // keys per thread
constexpr int RTILE = RT * RI; // keys per tile

// exclusive prefix of `v` over the 256 threads of the CTA (thread order); wsum is 8 words of smem
__device__ __forceinline__ uint32_t block_excl_scan_256(uint32_t v, uint32_t* wsum, uint32_t* total_out) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    uint32_t run = inc - v, tot = 0;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) {
        const uint32_t s = wsum[ww];
        if (ww < w) run += s;
        tot += s;
    }
    if (total_out) *total_out = tot;
    __syncthreads();
    return run;
}

// The first pass reads the caller's index array directly (FIRST): no separate conversion pass.
template <typename IdxT, bool FIRST>
__device__ __forceinline__ uint32_t radix_load_key(const IdxT* __restrict__ idx, int idx_base,
                                                   const uint32_t* __restrict__ keys, int e) {
    if (FIRST) return (uint32_t)((int64_t)idx[e] - idx_base);
    return keys[e];
}

// Digits are up to 9 bits wide (NB = 512 bins max): the pass count is ceil(bits / 9) and the bits
// are spread evenly over the passes, so 1e8 rows (27 bits) take 3 passes and 1e5 rows (17 bits) 2.
constexpr int NB = 512;

// One tile's digit histogram: `ik` / `kin` are the table's index list and key stream, `hist` its [NB][tiles]
template <typename IdxT, bool FIRST>
__device__ __forceinline__ void radix_hist_body(const IdxT* __restrict__ ik, int idx_base, const uint32_t* __restrict__ kin,
                                                int L, int shift, uint32_t mask, uint32_t* __restrict__ hist, int tiles,
                                                int tile) {
    __shared__ uint32_t h[NB];
    const int tid = threadIdx.x;
    h[tid] = 0;
    h[tid + RT] = 0;
    __syncthreads();
    const int base = tile * RTILE;
    uint32_t kk[RI];
#pragma unroll
    for (int i = 0; i < RI; ++i) {
        const int e = base + i * RT + tid;
        kk[i] = e < L ? radix_load_key<IdxT, FIRST>(ik, idx_base, kin, e) : 0u;
    }
#pragma unroll
    for (int i = 0; i < RI; ++i)
        if (base + i * RT + tid < L) atomicAdd(&h[(kk[i] >> shift) & mask], 1u);
    __syncthreads();
    for (uint32_t d = tid; d <= mask; d += RT) hist[(size_t)d * tiles + tile] = h[d];
}

// One CTA per (digit, table): exclusive scan over that digit's per-tile counts (contiguous, so
// the loads coalesce), in place, plus the digit's total.
__device__ __forceinline__ void radix_scan_body(uint32_t* __restrict__ h, uint32_t* __restrict__ total, int tiles) {
    __shared__ uint32_t wsum[8];
    uint32_t running = 0;
    for (int c = 0; c < tiles; c += RT) {
        const int i = c + threadIdx.x;
        const uint32_t v = i < tiles ? h[i] : 0u;
        uint32_t tot;
        const uint32_t ex = block_excl_scan_256(v, wsum, &tot);
        if (i < tiles) h[i] = running + ex;
        running += tot;
    }
    if (threadIdx.x == 0) *total = running;
}

// Scatter with a shared-memory reorder: the tile's keys are first placed in digit order in shared
// memory, then written out in that order, so the keys of one digit leave as one contiguous run
// (coalesced) instead of one 4-byte store per key.
// (`ik`, `kin`, `pin`, `ko`, `po`, `hist` [NB][tiles], `dtot` [NB]: this table's streams and counts)
template <typename IdxT, bool FIRST>
__device__ __forceinline__ void radix_scatter_body(const IdxT* __restrict__ ik, int idx_base, const uint32_t* __restrict__ kin,
                                                   const uint32_t* __restrict__ pin, uint32_t* __restrict__ ko,
                                                   uint32_t* __restrict__ po, int L, int shift, uint32_t mask,
                                                   const uint32_t* __restrict__ hist, const uint32_t* __restrict__ dtot,
                                                   int tiles, int tile) {
    __shared__ uint16_t wc[RT / 32][NB];      // per-warp digit counts, then exclusive prefix over warps
    __shared__ uint32_t lstart[NB];           // first slot of each digit inside the sorted tile
    __shared__ uint32_t gdst[NB];             // global position of slot 0 of each digit, minus lstart
    __shared__ uint32_t skeys[RTILE];
    __shared__ uint32_t svals[RTILE];
    __shared__ uint32_t wsum[8];
    const int tid = threadIdx.x;
    const int w = tid >> 5, lane = tid & 31;
    for (int i = tid; i < (RT / 32) * NB; i += RT) (&wc[0][0])[i] = 0;
    __syncthreads();

    const int tile_base = tile * RTILE;
    const int base = tile_base + w * (32 * RI);
    const int n_valid = min(RTILE, L - tile_base);
    uint32_t key[RI], val[RI], rank[RI];
    const uint32_t lt_mask = (1u << lane) - 1u;
#pragma unroll
    for (int i = 0; i < RI; ++i) {
        const int e = base + i * 32 + lane;
        const bool valid = e < L;
        key[i] = valid ? radix_load_key<IdxT, FIRST>(ik, idx_base, kin, e) : 0xffffffffu;
        val[i] = FIRST ? (uint32_t)e : (valid ? pin[e] : 0u);
    }
#pragma unroll
    for (int i = 0; i < RI; ++i) {
        const bool valid = (base + i * 32 + lane) < L;
        const uint32_t dig = valid ? ((key[i] >> shift) & mask) : (NB + lane);
        const uint32_t peers = __match_any_sync(0xffffffffu, dig);
        const uint32_t lt = peers & lt_mask;
        const uint32_t b = valid ? wc[w][dig] : 0u;
        __syncwarp();
        if (valid && lt == 0) wc[w][dig] = (uint16_t)(b + __popc(peers));
        __syncwarp();
        rank[i] = b + __popc(lt);
    }
    __syncthreads();
    {
        // thread t owns digits 2t and 2t+1
        const uint32_t d0 = 2 * tid, d1 = 2 * tid + 1;
        uint32_t c0 = 0, c1 = 0;
        if (d0 <= mask) {
#pragma unroll
            for (int ww = 0; ww < RT / 32; ++ww) {
                const uint32_t c = wc[ww][d0];
                wc[ww][d0] = (uint16_t)c0;
                c0 += c;
            }
        }
        if (d1 <= mask) {
#pragma unroll
            for (int ww = 0; ww < RT / 32; ++ww) {
                const uint32_t c = wc[ww][d1];
                wc[ww][d1] = (uint16_t)c1;
                c1 += c;
            }
        }
        const uint32_t lex = block_excl_scan_256(c0 + c1, wsum, nullptr);       // slots inside the tile
        const uint32_t t0 = d0 <= mask ? dtot[d0] : 0u;
        const uint32_t t1 = d1 <= mask ? dtot[d1] : 0u;
        const uint32_t gex = block_excl_scan_256(t0 + t1, wsum, nullptr);       // buckets in the stream
        if (d0 <= mask) {
            lstart[d0] = lex;
            gdst[d0] = gex + hist[(size_t)d0 * tiles + tile] - lex;
        }
        if (d1 <= mask) {
            lstart[d1] = lex + c0;
            gdst[d1] = gex + t0 + hist[(size_t)d1 * tiles + tile] - (lex + c0);
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < RI; ++i) {
        if ((base + i * 32 + lane) < L) {
            const uint32_t dig = (key[i] >> shift) & mask;
            const uint32_t slot = lstart[dig] + wc[w][dig] + rank[i];
            skeys[slot] = key[i];
            svals[slot] = val[i];
        }
    }
    __syncthreads();
    for (int j = tid; j < n_valid; j += RT) {
        const uint32_t kk = skeys[j];
        const uint32_t dst = gdst[(kk >> shift) & mask] + (uint32_t)j;
        ko[dst] = kk;
        po[dst] = svals[j];
    }
}

static int key_bits(int64_t max_rows) {
    int bits = 1;
    while (bits < 32 && (1ll << bits) < max_rows) ++bits;
    return bits;
}

// ---------------------------------------------------------------------------------------------
// Every regime in one batch.  Table k has L_k = B * P_k keys at g.off[k].
//   L_k <= kSmemSortMax: one shared-memory launch, one CTA per listed table (sized for the longest list;
//                        body in sort_small.cuh, which the fused lookup + sort launches also run)
//   larger L_k:          the radix passes above, grid.y over the listed tables, grid.x over the largest
//                        table's tiles (CTAs past their own table's tile count return at once)
// The radix pass count follows the largest table of the handle, so the radix tables finish in half
// passes % 2; the shared-memory sorts write there directly.
// ---------------------------------------------------------------------------------------------
template <typename IdxT, int ITEMS, int THREADS>
__global__ void __launch_bounds__(THREADS)
sort_small_mp_kernel(const IdxT* __restrict__ idx, int idx_base, const __grid_constant__ MpGeom g,
                     const TableDesc* __restrict__ desc, uint32_t* __restrict__ keys_out, uint32_t* __restrict__ pos_out,
                     int64_t cap, unsigned long long* clk) {
    extern __shared__ uint32_t sort_smem[];
    const int k = g.list[blockIdx.x];
    clock_in(clk, blockIdx.x);
    sort_small_body<IdxT, ITEMS, THREADS>(idx + g.off[k], idx_base, (int)(g.B * g.P[k]), desc[k].rows,
                                          keys_out + (size_t)k * cap, pos_out + (size_t)k * cap, sort_smem);
    clock_out(clk, blockIdx.x);
}

template <typename IdxT, int ITEMS, int THREADS>
static int launch_sort_small_mp(dlrmb_tables* t, const IdxT* idx, int idx_base, const MpGeom& g, int half,
                                cudaStream_t s) {
    constexpr size_t smem = SmallSortGeom<ITEMS, THREADS>::smem_bytes();
    static unsigned long long attr_done = 0;
    int rc = ensure_smem_attr((const void*)sort_small_mp_kernel<IdxT, ITEMS, THREADS>, (int)smem, &attr_done);
    if (rc) return rc;
    sort_small_mp_kernel<IdxT, ITEMS, THREADS><<<g.nlist, THREADS, smem, s>>>(idx, idx_base, g, t->d_desc, t->keys[half],
                                                                             t->pos[half], t->cap, clock_slot(CLK_SORT));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <typename IdxT, bool FIRST>
__global__ void __launch_bounds__(RT)
radix_hist_mp_kernel(const IdxT* __restrict__ idx, int idx_base, const uint32_t* __restrict__ keys, int64_t cap,
                     const __grid_constant__ MpGeom g, int shift, uint32_t mask, uint32_t* __restrict__ tile_hist,
                     int64_t hist_stride) {
    const int k = g.list[blockIdx.y];
    const int tiles = (int)g.units[k];
    if ((int)blockIdx.x >= tiles) return;
    radix_hist_body<IdxT, FIRST>(idx + g.off[k], idx_base, keys + (size_t)k * cap, (int)(g.B * g.P[k]), shift, mask,
                                 tile_hist + (size_t)k * hist_stride, tiles, blockIdx.x);
}

__global__ void __launch_bounds__(RT)
radix_scan_mp_kernel(uint32_t* __restrict__ tile_hist, uint32_t* __restrict__ digit_total, const __grid_constant__ MpGeom g,
                     int64_t hist_stride) {
    const int d = blockIdx.x, k = g.list[blockIdx.y];
    const int tiles = (int)g.units[k];
    radix_scan_body(tile_hist + (size_t)k * hist_stride + (size_t)d * tiles, digit_total + k * NB + d, tiles);
}

template <typename IdxT, bool FIRST>
__global__ void __launch_bounds__(RT)
radix_scatter_mp_kernel(const IdxT* __restrict__ idx, int idx_base, const uint32_t* __restrict__ keys_in,
                        const uint32_t* __restrict__ pos_in, uint32_t* __restrict__ keys_out,
                        uint32_t* __restrict__ pos_out, int64_t cap, const __grid_constant__ MpGeom g, int shift,
                        uint32_t mask, const uint32_t* __restrict__ tile_hist, const uint32_t* __restrict__ digit_total,
                        int64_t hist_stride) {
    const int k = g.list[blockIdx.y];
    const int tiles = (int)g.units[k];
    if ((int)blockIdx.x >= tiles) return;
    const size_t o = (size_t)k * cap;
    radix_scatter_body<IdxT, FIRST>(idx + g.off[k], idx_base, keys_in + o, pos_in + o, keys_out + o, pos_out + o,
                                    (int)(g.B * g.P[k]), shift, mask, tile_hist + (size_t)k * hist_stride,
                                    digit_total + k * NB, tiles, blockIdx.x);
}

static int radix_passes(const dlrmb_tables* t) {
    const int bits = key_bits(t->max_rows);
    return (bits + 8) / 9;
}

int sort_mp_final_half(const dlrmb_tables* t, const MpGeom& g) {
    for (int k = 0; k < g.ntab; ++k)
        if ((int64_t)g.B * g.P[k] > kSmemSortMax) return radix_passes(t) & 1;
    return 0;
}

template <typename IdxT>
static int launch_sort_mp_t(dlrmb_tables* t, const IdxT* idx, int idx_base, const MpGeom& g0, int64_t skip_max,
                            int half, cudaStream_t s) {
    MpGeom g = g0;
    // shared-memory regime
    g.nlist = 0;
    int64_t lmax = 0;
    for (int k = 0; k < g.ntab; ++k) {
        const int64_t L = (int64_t)g.B * g.P[k];
        if (L > skip_max && L <= kSmemSortMax) {
            g.list[g.nlist++] = (uint16_t)k;
            lmax = L > lmax ? L : lmax;
        }
    }
    int rc = DLRMB_OK;
    if (g.nlist > 0) {
        if (lmax <= 1024) rc = launch_sort_small_mp<IdxT, 4, 256>(t, idx, idx_base, g, half, s);
        else if (lmax <= 2048) rc = launch_sort_small_mp<IdxT, 8, 256>(t, idx, idx_base, g, half, s);
        else if (lmax <= 4096) rc = launch_sort_small_mp<IdxT, 16, 256>(t, idx, idx_base, g, half, s);
        else if (lmax <= 8192) rc = launch_sort_small_mp<IdxT, 8, 1024>(t, idx, idx_base, g, half, s);
        else rc = launch_sort_small_mp<IdxT, 16, 1024>(t, idx, idx_base, g, half, s);
        if (rc) return rc;
    }
    // radix regime
    g.nlist = 0;
    int max_tiles = 0;
    for (int k = 0; k < g.ntab; ++k) {
        const int64_t L = (int64_t)g.B * g.P[k];
        if (L > kSmemSortMax) {
            g.list[g.nlist++] = (uint16_t)k;
            g.units[k] = (uint32_t)ceil_div64(L, RTILE);
            max_tiles = (int)g.units[k] > max_tiles ? (int)g.units[k] : max_tiles;
        }
    }
    if (g.nlist > 0) {
        DLRMB_REQUIRE(max_tiles <= t->radix_tiles_cap, "internal: radix tile capacity exceeded");
        const int bits = key_bits(t->max_rows);
        const int passes = radix_passes(t);
        const int per_pass = (bits + passes - 1) / passes;     // <= 9
        DLRMB_REQUIRE((passes & 1) == half, "internal: radix passes end in the other half");
        const int64_t cap = t->cap, hs = (int64_t)NB * t->radix_tiles_cap;
        dim3 grid((unsigned)max_tiles, (unsigned)g.nlist);
        int cur = 0, shift = 0;
        for (int p = 0; p < passes; ++p) {
            const int nb = (bits - shift) < per_pass ? (bits - shift) : per_pass;
            const uint32_t mask = (1u << nb) - 1u;
            dim3 sgrid(mask + 1u, (unsigned)g.nlist);
            if (p == 0)
                radix_hist_mp_kernel<IdxT, true><<<grid, RT, 0, s>>>(idx, idx_base, t->keys[cur], cap, g, shift, mask, t->tile_hist, hs);
            else
                radix_hist_mp_kernel<IdxT, false><<<grid, RT, 0, s>>>(idx, idx_base, t->keys[cur], cap, g, shift, mask, t->tile_hist, hs);
            DLRMB_LAUNCH_CHECK();
            radix_scan_mp_kernel<<<sgrid, RT, 0, s>>>(t->tile_hist, t->digit_total, g, hs);
            DLRMB_LAUNCH_CHECK();
            if (p == 0)
                radix_scatter_mp_kernel<IdxT, true><<<grid, RT, 0, s>>>(idx, idx_base, t->keys[cur], t->pos[cur], t->keys[cur ^ 1],
                                                                       t->pos[cur ^ 1], cap, g, shift, mask, t->tile_hist,
                                                                       t->digit_total, hs);
            else
                radix_scatter_mp_kernel<IdxT, false><<<grid, RT, 0, s>>>(idx, idx_base, t->keys[cur], t->pos[cur], t->keys[cur ^ 1],
                                                                        t->pos[cur ^ 1], cap, g, shift, mask, t->tile_hist,
                                                                        t->digit_total, hs);
            DLRMB_LAUNCH_CHECK();
            cur ^= 1;
            shift += nb;
        }
    }
    t->sorted_buf = half;
    return DLRMB_OK;
}

int launch_sort_mp(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g, int64_t skip_max,
                   int half, cudaStream_t s) {
    if (idx_bytes == 4) return launch_sort_mp_t<uint32_t>(t, static_cast<const uint32_t*>(idx), idx_base, g, skip_max, half, s);
    return launch_sort_mp_t<int64_t>(t, static_cast<const int64_t*>(idx), idx_base, g, skip_max, half, s);
}

// ---------------------------------------------------------------------------------------------
// jagged bags: position -> bag of every sorted entry.  Table k's sorted positions are relative to its block
// (element g.off[k] of `values`); the bag of x = g.off[k] + pos is the largest b with offsets[k*B + b] <= x,
// found by binary search over the table's B offsets (L1-resident: B * 4 or 8 bytes).  Written in sorted order
// so that the update reads a bag id where it reads a position, four per 16-byte load.  MEAN also writes the
// bag's weight fl(1 / n) as f32 bits; WEIGHTED writes the entry's own weight, weights[x], in its place.  Table k
// owns CTAs [g.pre[k], g.pre[k+1]) (none when L_k = 0).
// ---------------------------------------------------------------------------------------------
template <typename IdxT>
__device__ __forceinline__ uint32_t jagged_bag_of(const IdxT* __restrict__ ok, uint32_t B, int64_t x) {
    uint32_t lo = 0, hi = B - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if ((int64_t)__ldg(ok + mid) <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

template <typename IdxT, bool MEAN>
__global__ void __launch_bounds__(256)
jagged_bags_kernel(const IdxT* __restrict__ offsets, uint32_t B, const __grid_constant__ MpGeom g,
                   const uint32_t* __restrict__ pos, uint32_t* __restrict__ bags, uint32_t* __restrict__ wts, int64_t cap) {
    const int k = mp_find(g.pre, g.ntab, blockIdx.x);
    const uint32_t L = g.P[k];
    const IdxT* __restrict__ ok = offsets + (size_t)k * B;
    const size_t o = (size_t)k * cap;
    const uint32_t step = (g.pre[k + 1] - g.pre[k]) * blockDim.x;
    for (uint32_t i = (blockIdx.x - g.pre[k]) * blockDim.x + threadIdx.x; i < L; i += step) {
        const int64_t x = g.off[k] + (int64_t)pos[o + i];
        const uint32_t lo = jagged_bag_of(ok, B, x);
        bags[o + i] = lo;
        if (MEAN) wts[o + i] = __float_as_uint(__fdiv_rn(1.0f, (float)((int64_t)__ldg(ok + lo + 1) - (int64_t)__ldg(ok + lo))));
    }
}

// WEIGHTED: the same pass, the weight gathered from the entry's position in `values`
template <typename IdxT>
__global__ void __launch_bounds__(256)
jagged_bags_weighted_kernel(const IdxT* __restrict__ offsets, const float* __restrict__ weights, uint32_t B,
                            const __grid_constant__ MpGeom g, const uint32_t* __restrict__ pos,
                            uint32_t* __restrict__ bags, uint32_t* __restrict__ wts, int64_t cap) {
    const int k = mp_find(g.pre, g.ntab, blockIdx.x);
    const uint32_t L = g.P[k];
    const IdxT* __restrict__ ok = offsets + (size_t)k * B;
    const size_t o = (size_t)k * cap;
    const uint32_t step = (g.pre[k + 1] - g.pre[k]) * blockDim.x;
    for (uint32_t i = (blockIdx.x - g.pre[k]) * blockDim.x + threadIdx.x; i < L; i += step) {
        const int64_t x = g.off[k] + (int64_t)pos[o + i];
        const uint32_t lo = jagged_bag_of(ok, B, x);
        bags[o + i] = lo;
        wts[o + i] = __float_as_uint(__ldg(weights + x));
    }
}

template <typename IdxT>
static int launch_jagged_bags_t(dlrmb_tables* t, const IdxT* offsets, const float* weights, const MpGeom& g0, int B,
                                int pooling, int half, cudaStream_t s) {
    MpGeom g = g0;
    int64_t total = 0;
    for (int k = 0; k < g.ntab; ++k) {
        g.pre[k] = (uint32_t)total;
        total += ceil_div64(g.P[k], 256 * 4);
    }
    g.pre[g.ntab] = (uint32_t)total;
    if (total == 0) return DLRMB_OK;
    const uint32_t* pos = t->pos[half];
    uint32_t* bags = t->pos[half ^ 1];
    uint32_t* wts = t->keys[half ^ 1];
    if (pooling == kJaggedWeighted)
        jagged_bags_weighted_kernel<IdxT><<<(unsigned)total, 256, 0, s>>>(offsets, weights, (uint32_t)B, g, pos, bags,
                                                                          wts, t->cap);
    else if (pooling == 1)
        jagged_bags_kernel<IdxT, true><<<(unsigned)total, 256, 0, s>>>(offsets, (uint32_t)B, g, pos, bags, wts, t->cap);
    else
        jagged_bags_kernel<IdxT, false><<<(unsigned)total, 256, 0, s>>>(offsets, (uint32_t)B, g, pos, bags, wts, t->cap);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

int launch_jagged_bags(dlrmb_tables* t, const void* offsets, const float* weights, int idx_bytes, const MpGeom& g,
                       int B, int pooling, int half, cudaStream_t s) {
    if (idx_bytes == 4)
        return launch_jagged_bags_t<uint32_t>(t, static_cast<const uint32_t*>(offsets), weights, g, B, pooling, half, s);
    return launch_jagged_bags_t<int64_t>(t, static_cast<const int64_t*>(offsets), weights, g, B, pooling, half, s);
}

// ---------------------------------------------------------------------------------------------
// parity export: unique ids + segment offsets of one table's sorted stream (single CTA)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
dedup_export_kernel(const uint32_t* __restrict__ keys, int L, int64_t* __restrict__ uniq,
                    int32_t* __restrict__ seg, int32_t* __restrict__ n_uniq) {
    __shared__ int warp_cnt[32];
    __shared__ int running;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) running = 0;
    __syncthreads();
    for (int base = 0; base < L; base += 1024) {
        int i = base + tid;
        bool head = i < L && (i == 0 || keys[i] != keys[i - 1]);
        uint32_t bal = __ballot_sync(0xffffffffu, head);
        if (lane == 0) warp_cnt[w] = __popc(bal);
        __syncthreads();
        int before = running;
        for (int ww = 0; ww < w; ++ww) before += warp_cnt[ww];
        int total = 0;
        for (int ww = 0; ww < 32; ++ww) total += warp_cnt[ww];
        if (head) {
            int o = before + __popc(bal & ((1u << lane) - 1u));
            uniq[o] = (int64_t)keys[i];
            seg[o] = i;
        }
        __syncthreads();
        if (tid == 0) running += total;
        __syncthreads();
    }
    if (tid == 0) {
        seg[running] = L;
        *n_uniq = running;
    }
}

int launch_dedup_export(dlrmb_tables* t, int k, cudaStream_t s) {
    const int L = (int)sorted_lookups(t, k);
    dedup_export_kernel<<<1, 1024, 0, s>>>(t->keys[t->sorted_buf] + (size_t)k * t->cap, L,
                                           t->d_uniq, t->d_seg, t->d_nuniq);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

}  // namespace dlrmb
