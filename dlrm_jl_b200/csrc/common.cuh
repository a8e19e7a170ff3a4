// Internal declarations shared by the translation units of libdlrm_b200.so.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>

#include <atomic>

#include "dlrm_b200.h"

namespace dlrmb {

// ---- error plumbing ----------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define DLRMB_CUDA(expr)                                                                    \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ::dlrmb::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,         \
                               cudaGetErrorString(_e));                                     \
            return (_e == cudaErrorMemoryAllocation) ? DLRMB_ENOMEM : DLRMB_ECUDA;          \
        }                                                                                   \
    } while (0)

#define DLRMB_REQUIRE(cond, ...)                                                            \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            ::dlrmb::set_error(__VA_ARGS__);                                                \
            return DLRMB_EINVAL;                                                            \
        }                                                                                   \
    } while (0)

#define DLRMB_LAUNCH_CHECK()                                                                \
    do {                                                                                    \
        ::dlrmb::g_launches.fetch_add(1, std::memory_order_relaxed);                        \
        DLRMB_CUDA(cudaGetLastError());                                                     \
    } while (0)

// RAII: make `dev` current for the scope of an entry point, restore the caller's device on every
// return path.
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// ---- optional device-side kernel stamps (dlrmb_clock_enable) ---------------------------------
// When a clock buffer is registered, thread 0 of every CTA of the main kernels stores %globaltimer
// (32 ns steps on B200) at entry (atomic min) and exit (atomic max) into [kernel][cta % kClockCtas][2]; the
// host pre-fills the slots and takes min(entry), max(exit).
// This times a kernel where it really runs -- inside the multi-stream CUDA graph of a training step --
// without the several microseconds a CUDA-event pair adds around a 10 us kernel.  A null pointer
// (the default) costs one predicated branch.
constexpr int kClockCtas = 4096;     // stamp slots per kernel; CTA c folds into slot c % 4096 (earliest entry, latest exit)
enum ClockKernel { CLK_LOOKUP = 0, CLK_SORT, CLK_UPDATE, CLK_FIXUP, CLK_IFWD, CLK_IBWD, CLK_BCE, CLK_COUNT };
unsigned long long* clock_slot(int which);       // host: device pointer of that kernel's stamps, or nullptr

__device__ __forceinline__ unsigned long long clock_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void clock_in(unsigned long long* c, unsigned cta) {
    if (c != nullptr && threadIdx.x == 0) atomicMin(&c[2 * (cta % (unsigned)kClockCtas)], clock_now());
}
__device__ __forceinline__ void clock_out(unsigned long long* c, unsigned cta) {
    if (c != nullptr && threadIdx.x == 0) atomicMax(&c[2 * (cta % (unsigned)kClockCtas) + 1], clock_now());
}

// ---- table storage -----------------------------------------------------------------------
struct TableDesc {
    float* base;   // [rows][D] in HBM, 256-byte aligned; f32, or bf16 when the tables store bf16
    int64_t rows;
};

// Row storage access.  Tables are f32 (the reference default) or bf16 (its `embedding_eltype`
// option, DLRM.jl src/model/model.jl:187 and the BF16 load/store hooks of src/cachedarrays.jl:5-19):
// all arithmetic stays fp32, only the stored rows are rounded (to nearest even).
template <typename RowT> struct RowIO;
template <> struct RowIO<float> {
    static __device__ __forceinline__ const float* row(const float* base, size_t r, size_t D) { return base + r * D; }
    static __device__ __forceinline__ float* row(float* base, size_t r, size_t D) { return base + r * D; }
    static __device__ __forceinline__ float4 load4(const float* row, int c) { return reinterpret_cast<const float4*>(row)[c]; }
    static __device__ __forceinline__ float4 ldg4(const float* row, int c) { return __ldg(reinterpret_cast<const float4*>(row) + c); }
    static __device__ __forceinline__ void store4(float* row, int c, float4 v) { reinterpret_cast<float4*>(row)[c] = v; }
    static __device__ __forceinline__ float load1(const float* row, int c) { return row[c]; }
    static __device__ __forceinline__ float ldg1(const float* row, int c) { return __ldg(row + c); }
    static __device__ __forceinline__ void store1(float* row, int c, float v) { row[c] = v; }
};
template <> struct RowIO<__nv_bfloat16> {
    using B = __nv_bfloat16;
    static __device__ __forceinline__ const B* row(const float* base, size_t r, size_t D) { return reinterpret_cast<const B*>(base) + r * D; }
    static __device__ __forceinline__ B* row(float* base, size_t r, size_t D) { return reinterpret_cast<B*>(base) + r * D; }
    static __device__ __forceinline__ float4 unpack(uint2 q) {
        return make_float4(__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xffff0000u),
                           __uint_as_float(q.y << 16), __uint_as_float(q.y & 0xffff0000u));
    }
    static __device__ __forceinline__ float4 load4(const B* row, int c) { return unpack(reinterpret_cast<const uint2*>(row)[c]); }
    static __device__ __forceinline__ float4 ldg4(const B* row, int c) { return unpack(__ldg(reinterpret_cast<const uint2*>(row) + c)); }
    static __device__ __forceinline__ void store4(B* row, int c, float4 v) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 q;
        q.x = *reinterpret_cast<unsigned int*>(&lo);
        q.y = *reinterpret_cast<unsigned int*>(&hi);
        reinterpret_cast<uint2*>(row)[c] = q;
    }
    static __device__ __forceinline__ float load1(const B* row, int c) { return __bfloat162float(row[c]); }
    static __device__ __forceinline__ float ldg1(const B* row, int c) { return __bfloat162float(row[c]); }
    static __device__ __forceinline__ void store1(B* row, int c, float v) { row[c] = __float2bfloat16_rn(v); }
};

// Geometry of the sorted-stream reduction (update.cu): every lane group walks TILE
// consecutive entries of the per-table sorted (row id, position) stream.
constexpr int kUpdateTile = 16;
// Largest per-table lookup count the single-CTA shared-memory sort handles (sort.cu).
constexpr int kSmemSortMax = 16384;
// Largest per-table lookup count whose sort rides in the lookup launch (256-thread sort CTAs).
constexpr int kFusedSortMax = 4096;

// Per-table pooling factors (the `_mp` entry points).  Table k's indices are the [B][P_k] block at
// element off[k] = B * (P_0 + .. + P_{k-1}).  The geometry reaches the kernels by value as one
// kernel-parameter struct (about 7 KB at kMpMaxTables; sm_100 accepts up to 32 KB), so a call needs no
// device copy and stays graph-capturable.  `pre` is a prefix over tables of the CTAs (lookup) or chunks
// (update) each table owns; a CTA finds its table by binary search in it.  `list` names the tables of
// one sort launch, `units` counts per-table radix tiles or update tiles.
constexpr int kMpMaxTables = 256;
struct MpGeom {
    int ntab;
    uint32_t B;
    int nlist;                          // entries of `list` used by this launch
    uint32_t P[kMpMaxTables];
    int64_t off[kMpMaxTables];
    uint32_t pre[kMpMaxTables + 1];
    uint16_t list[kMpMaxTables];
    uint32_t units[kMpMaxTables];
};

// the table k whose range [pre[k], pre[k+1]) holds x (pre strictly increasing, pre[0] = 0)
__device__ __forceinline__ int mp_find(const uint32_t* pre, int ntab, uint32_t x) {
    int lo = 0, hi = ntab - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (pre[mid] <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// Process-wide tuning / test switches (dlrmb_set_option); read by the launchers, never from the
// environment.
struct Options {
    std::atomic<int> interact_general{0};     // 1: general tiled interaction kernels even for the specialised shapes
    std::atomic<int> update_two_launches{0};  // 1: separate fix-up launch at every batch size
    std::atomic<int> update_tile{0};          // 4, 8, .. 32 entries per lane group (0 = chosen per batch)
    std::atomic<int> bwd_variant{0};          // one-sample-per-warp backward (d = 128): 0 = by batch size, 1 = FFMA2 at 144 registers,
                                              // 2 = FFMA2 at 128 registers, 3 = S stored once at 144, 5 / 6 = streaming kernels (T
                                              // rows through a cp.async ring; 6 = S stored once, row-paired FFMA2)
    std::atomic<int> fwd_tb{0};               // tiled forward register block 3 | 6 | 9 (0 = default)
    std::atomic<int> fwd_ks{0};               // tiled forward k-split log2
    std::atomic<int> fwd_ksplit{1};           // tensor-core forward: 0 = one warp per sample always, 1 = two warps per sample for
                                              // one-wave batches (default), 2 = two warps per sample always
};
extern Options g_opt;

}  // namespace dlrmb

struct dlrmb_tables {
    int device = 0;
    int ntab = 0;
    int D = 0;
    int elem_bytes = 4;        // 4 = f32 rows, 2 = bf16 rows
    int sm_count = 148;
    int64_t max_lookups = 0;   // max B*P per table
    int64_t cap = 0;           // max_lookups rounded up to 4: stride of the per-table streams
    int64_t total_rows = 0;
    int64_t max_rows = 0;
    int64_t* h_rows = nullptr;       // host copy
    int64_t* h_offsets = nullptr;    // element offsets of each table inside `slab`
    float* slab = nullptr;           // all tables, one allocation (f32 or bf16 elements)
    dlrmb::TableDesc* d_desc = nullptr;
    int32_t* d_slotmap = nullptr;    // sharded use: element offset of each local table in a destination sample row
                                     // (slot * dest_D + col0, dlrmb_tables_set_slot_map / _set_dest_map)
    int slotmap_max = -1;            // largest slot of the map
    int dest_D = 0;                  // floats per slot of the destination rows
    bool dest_vec4 = false;          // dest_D and every col0 are multiples of 4 (16-byte peer stores possible)
    cudaStream_t own_stream = nullptr;

    // sort / update workspace (all [ntab][max_lookups] unless noted)
    uint32_t* keys[2] = {nullptr, nullptr};   // 0-based row ids, ping-pong
    uint32_t* pos[2] = {nullptr, nullptr};    // flat position b*P+p, ping-pong
    uint32_t* tile_hist = nullptr;            // radix: [ntab][256][tiles]
    uint32_t* digit_total = nullptr;          // radix: [ntab][256]
    int sorted_buf = 0;                       // which ping-pong half holds the sorted stream
    int64_t radix_tiles_cap = 0;
    float* partial = nullptr;                 // [ntab][tiles][2][D] boundary partial sums
    uint8_t* tile_flags = nullptr;            // [ntab][tiles] boundary flags
    int64_t partial_tiles_cap = 0;
    uint32_t* head_list = nullptr;            // [ntab * tiles] tiles whose last run continues
    uint32_t* head_count = nullptr;           // [1 + ntab]: listed heads (two-launch path), CTAs done per table
    // dedup export scratch
    int32_t* d_seg = nullptr;                 // [max_lookups + 1]
    int64_t* d_uniq = nullptr;                // [max_lookups]
    int32_t* d_nuniq = nullptr;

    // state of the last sort
    bool sorted_valid = false;
    int sorted_B = 0;
    int32_t* h_sorted_P = nullptr;            // [ntab], host: P_k of every table (L_k after a jagged sort, sorted_B = 1)
    int sorted_jagged = -1;                   // -1: uniform or _mp sort; 0 / 1 / 2: jagged sort with sum / mean /
                                              // per-sample-weighted sum pooling, bag ids (and the entries' weights
                                              // in modes 1 and 2) in pos / keys [sorted_buf ^ 1]

    // host-entry-point staging (device side), grown on demand
    void* stage_idx = nullptr;  size_t stage_idx_bytes = 0;
    float* stage_a = nullptr;   size_t stage_a_bytes = 0;
    float* stage_b = nullptr;   size_t stage_b_bytes = 0;
    float* stage_c = nullptr;   size_t stage_c_bytes = 0;
    float* stage_d = nullptr;   size_t stage_d_bytes = 0;
};

namespace dlrmb {

// kernels' host-side launchers (each returns a dlrmb_status)
int launch_interaction_fwd(float* T, const float* x, int B, int F, int d, int pad_to_mul,
                           float* out, int sm_count, cudaStream_t s);
int launch_interaction_bwd(const float* dOut, const float* T, int B, int F, int d, int pad_to_mul,
                           float* dT, float* dx, int sm_count, cudaStream_t s);
int launch_interaction_bwd_ex(const float* dOut, const float* T, int B, int F, int d, int pad_to_mul,
                              float* dT, float* dx, const void* dests, long long sample_offset, int qlog,
                              int sm_count, cudaStream_t s);
int launch_interaction_bwd_dx(const float* dOut, const float* T, int B, int F, int d, int pad_to_mul, float* dx,
                              int sm_count, cudaStream_t s);
bool interaction_has_warp_path(int F, int d);
int launch_update(dlrmb_tables* t, const float* dT, int slots, int slot0, float lr, cudaStream_t s);
int launch_dedup_export(dlrmb_tables* t, int k, cudaStream_t s);
int launch_init_uniform(dlrmb_tables* t, uint64_t seed, cudaStream_t s);
int launch_convert_rows(dlrmb_tables* t, int k, float* f32_buf, bool to_table, cudaStream_t s);
int launch_check_indices(dlrmb_tables* t, const void* d_idx, int idx_bytes, int idx_base, int B,
                         int P, cudaStream_t s, long long* bad_table, long long* bad_pos,
                         long long* bad_val);
int launch_bce_sigmoid(const float* z, const float* y, int B, float* prob, float* dz, float* loss,
                       float* scratch, cudaStream_t s);
int launch_dense_fwd_bias_act(float* z, const float* bias, int B, int N, int relu, int sm_count, cudaStream_t s);
int64_t dense_bwd_scratch_floats(int N);
int launch_dense_bwd_act_bias(const float* dy, const float* y, int B, int N, float* dz, float* db,
                              float* scratch, cudaStream_t s);
// lookup / sort launchers: `g` carries ntab, B, P and off filled in; the launchers fill the rest of their copy
int launch_lookup_mp(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g,
                     float* out, int slots, int slot0, cudaStream_t s);
int launch_lookup_sort_mp(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g,
                          float* out, int slots, int slot0, cudaStream_t s);
// sort of every table with L_k > skip_max (0 = all tables); keys[] / pos[] half `half` receives the result
int launch_sort_mp(dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, const MpGeom& g, int64_t skip_max,
                   int half, cudaStream_t s);
int sort_mp_final_half(const dlrmb_tables* t, const MpGeom& g);
int launch_update_mp(dlrmb_tables* t, const float* dT, int slots, int slot0, float lr, cudaStream_t s);
int launch_check_indices_mp(dlrmb_tables* t, const void* d_idx, int idx_bytes, int idx_base, const MpGeom& g,
                            cudaStream_t s, long long* bad_table, long long* bad_pos, long long* bad_val);
// argument checks of the `_mp` entry points at batch B; fills ntab, B, P and off of `g`
int check_mp_args(const dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, int B, const int32_t* P,
                  MpGeom* g);
// record tables [k0, k0 + g.ntab) of the sort that just ran (dlrmb_embedding_update_sorted and the dedup export
// read it); the sort is valid once its last table is recorded
void mark_sorted(dlrmb_tables* t, const MpGeom& g, int k0);
// tables [k0, k0 + n) of `t` as a handle of their own: the same tables and workspaces from table k0 on.
// max_rows stays the handle's, so the radix sort of every group ends in the same ping-pong half.
dlrmb_tables table_group(const dlrmb_tables& t, int k0, int n);
// gather CTAs per table of an `_mp` lookup (fills g.pre); returns the total
int64_t lookup_grid_mp(const dlrmb_tables* t, MpGeom& g, uint32_t C, int* cshift);
// Jagged (variable-length) bags, the `_jagged` entry points.  The sort geometry is the `_mp` one with B = 1,
// P[k] = L_k and off[k] = L_0 + .. + L_{k-1}: a table's block is sorted as one bag of L_k lookups.  The lookup
// and the position -> bag pass also read the batch's B and the offsets [ntab * B + 1] (element offsets into
// `values`, same width as the indices).
int check_jagged_args(const dlrmb_tables* t, const void* values, const void* offsets, int idx_bytes, int idx_base,
                      int B, const int64_t* L, int pooling, MpGeom* g);
// `pooling` of the launchers below: 0 sum, 1 mean, or kJaggedWeighted for sum pooling with per-sample weights
// (`weights`, one f32 per entry of values; null otherwise).
constexpr int kJaggedWeighted = 2;
int launch_lookup_jagged(dlrmb_tables* t, const void* values, const void* offsets, const float* weights, int idx_bytes,
                         int idx_base, const MpGeom& g, int B, int pooling, float* out, int slots, int slot0,
                         cudaStream_t s);
// CTAs per table of a jagged lookup over B bags per table (fills g.pre from g.P = L); returns the total
int64_t lookup_grid_jagged(const dlrmb_tables* t, MpGeom& g, uint32_t B, uint32_t C);
// after a jagged sort into half `half`: bag id (and, with mean pooling, weight 1/n as f32 bits; with per-sample
// weights, the entry's weight) of every sorted entry into pos[half ^ 1] (and keys[half ^ 1])
int launch_jagged_bags(dlrmb_tables* t, const void* offsets, const float* weights, int idx_bytes, const MpGeom& g,
                       int B, int pooling, int half, cudaStream_t s);
// dw[j] = dT[b(j)][slot0 + k] . table_k[values[j]] for every entry of the batch (order: lookup.cu, the header)
int launch_weight_grad_jagged(dlrmb_tables* t, const void* values, const void* offsets, int idx_bytes, int idx_base,
                              int B, const float* dT, int slots, int slot0, float* dw, cudaStream_t s);
// lookups of table k in the last sort
static inline int64_t sorted_lookups(const dlrmb_tables* t, int k) { return (int64_t)t->sorted_B * t->h_sorted_P[k]; }

// A batch with one pooling factor P for every table, through the launchers above (MpGeom holds kMpMaxTables
// tables): launch(v, idx, g, slot0) runs once per group of at most kMpMaxTables consecutive tables, where v is
// table_group of the group, idx and slot0 are moved to its first table and g has P_k = P.  With `sorts` the
// launches sort the indices, and the batch is recorded as the last sort.
template <typename Launch>
int run_uniform(dlrmb_tables* t, const void* idx, int idx_bytes, int B, int P, int slot0, bool sorts, Launch&& launch) {
    MpGeom g;
    g.B = (uint32_t)B;
    g.nlist = 0;
    for (int k = 0; k < kMpMaxTables; ++k) {
        g.P[k] = (uint32_t)P;
        g.off[k] = (int64_t)k * B * P;
    }
    for (int k0 = 0; k0 < t->ntab; k0 += kMpMaxTables) {
        g.ntab = t->ntab - k0 < kMpMaxTables ? t->ntab - k0 : kMpMaxTables;
        dlrmb_tables v = table_group(*t, k0, g.ntab);
        int rc = launch(&v, static_cast<const char*>(idx) + (size_t)k0 * B * P * idx_bytes, g, slot0 + k0);
        if (rc) return rc;
        if (sorts) {
            t->sorted_buf = v.sorted_buf;
            mark_sorted(t, g, k0);
        }
    }
    return DLRMB_OK;
}
int device_sm_count(int device);
int64_t update_tiles_cap(int ntab, int D, int64_t max_lookups, int sm_count);
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device)
int ensure_smem_attr(const void* func, int bytes, unsigned long long* done_mask);

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace dlrmb
