// C-ABI surface of libdlrm_b200.so: handle management, argument validation, host-buffer
// entry points.  The kernels live in lookup.cu / interact.cu / sort.cu / update.cu.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace dlrmb {

static thread_local char tl_error[512] = "";
std::atomic<long long> g_launches{0};
Options g_opt;
static std::atomic<unsigned long long*> g_clock_buf{nullptr};
unsigned long long* clock_slot(int which) {
    unsigned long long* b = g_clock_buf.load(std::memory_order_relaxed);
    return b ? b + (size_t)which * 2 * kClockCtas : nullptr;
}

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tl_error, sizeof(tl_error), fmt, ap);
    va_end(ap);
}

int device_sm_count(int device) {
    static std::mutex mu;
    static int cache[64];
    std::lock_guard<std::mutex> lock(mu);
    if (device < 0 || device >= 64) return 148;
    if (cache[device] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0)
            n = 148;
        cache[device] = n;
    }
    return cache[device];
}

static int grow(void** p, size_t* have, size_t need) {
    if (*have >= need) return DLRMB_OK;
    if (*p) DLRMB_CUDA(cudaFree(*p));
    *p = nullptr;
    *have = 0;
    size_t want = need + need / 4 + 256;
    DLRMB_CUDA(cudaMalloc(p, want));
    *have = want;
    return DLRMB_OK;
}

}  // namespace dlrmb

using namespace dlrmb;

// sort / update workspaces, sized for `max_lookups` = max B*P per table (nothing else in the library
// allocates per call)
static void free_workspace(dlrmb_tables* t) {
    for (int i = 0; i < 2; ++i) {
        cudaFree(t->keys[i]);
        cudaFree(t->pos[i]);
        t->keys[i] = t->pos[i] = nullptr;
    }
    cudaFree(t->tile_hist);
    cudaFree(t->digit_total);
    cudaFree(t->partial);
    cudaFree(t->tile_flags);
    cudaFree(t->head_list);
    cudaFree(t->head_count);
    cudaFree(t->d_seg);
    cudaFree(t->d_uniq);
    cudaFree(t->d_nuniq);
    t->tile_hist = t->digit_total = t->head_list = t->head_count = nullptr;
    t->partial = nullptr;
    t->tile_flags = nullptr;
    t->d_seg = nullptr;
    t->d_uniq = nullptr;
    t->d_nuniq = nullptr;
    t->sorted_valid = false;
}

static int alloc_workspace(dlrmb_tables* t, int64_t max_lookups) {
    const int ntab = t->ntab;
    t->max_lookups = max_lookups;
    t->cap = (max_lookups + 3) / 4 * 4;
    size_t nl = (size_t)ntab * (size_t)t->cap + 8;
    for (int i = 0; i < 2; ++i) {
        DLRMB_CUDA(cudaMalloc((void**)&t->keys[i], sizeof(uint32_t) * nl));
        DLRMB_CUDA(cudaMalloc((void**)&t->pos[i], sizeof(uint32_t) * nl));
    }
    t->radix_tiles_cap = ceil_div64(max_lookups, 4096);
    DLRMB_CUDA(cudaMalloc((void**)&t->tile_hist, sizeof(uint32_t) * (size_t)ntab * 512 * (size_t)t->radix_tiles_cap));
    DLRMB_CUDA(cudaMalloc((void**)&t->digit_total, sizeof(uint32_t) * (size_t)ntab * 512));
    t->partial_tiles_cap = update_tiles_cap(ntab, t->D, max_lookups, t->sm_count);
    DLRMB_CUDA(cudaMalloc((void**)&t->partial, sizeof(float) * (size_t)ntab * (size_t)t->partial_tiles_cap * 2 * (size_t)t->D));
    DLRMB_CUDA(cudaMalloc((void**)&t->tile_flags, (size_t)ntab * (size_t)t->partial_tiles_cap));
    DLRMB_CUDA(cudaMalloc((void**)&t->head_list, sizeof(uint32_t) * (size_t)ntab * (size_t)t->partial_tiles_cap));
    DLRMB_CUDA(cudaMalloc((void**)&t->head_count, (1 + (size_t)ntab) * sizeof(uint32_t)));   // listed heads; CTAs done per table
    DLRMB_CUDA(cudaMemset(t->head_count, 0, (1 + (size_t)ntab) * sizeof(uint32_t)));
    DLRMB_CUDA(cudaMalloc((void**)&t->d_seg, sizeof(int32_t) * ((size_t)max_lookups + 1)));
    DLRMB_CUDA(cudaMalloc((void**)&t->d_uniq, sizeof(int64_t) * (size_t)max_lookups));
    DLRMB_CUDA(cudaMalloc((void**)&t->d_nuniq, sizeof(int32_t)));
    return DLRMB_OK;
}

#define GUARD(t)                                                     \
    DLRMB_REQUIRE((t) != nullptr, "null tables handle");             \
    DeviceGuard _guard((t)->device);                                 \
    DLRMB_REQUIRE(_guard.ok, "cudaSetDevice(%d) failed", (t)->device)

extern "C" {

int32_t dlrmb_abi_version(void) { return DLRMB_ABI_VERSION; }
const char* dlrmb_last_error(void) { return tl_error; }
int64_t dlrmb_launch_count(void) { return g_launches.load(); }

static std::atomic<int>* find_option(const char* name) {
    if (!name) return nullptr;
    if (!strcmp(name, "interact_general")) return &g_opt.interact_general;
    if (!strcmp(name, "update_two_launches")) return &g_opt.update_two_launches;
    if (!strcmp(name, "update_tile")) return &g_opt.update_tile;
    if (!strcmp(name, "bwd_variant")) return &g_opt.bwd_variant;
    if (!strcmp(name, "fwd_tb")) return &g_opt.fwd_tb;
    if (!strcmp(name, "fwd_ks")) return &g_opt.fwd_ks;
    if (!strcmp(name, "fwd_ksplit")) return &g_opt.fwd_ksplit;
    return nullptr;
}

int32_t dlrmb_set_option(const char* name, int64_t value) {
    std::atomic<int>* o = find_option(name);
    DLRMB_REQUIRE(o != nullptr, "unknown option '%s'", name ? name : "(null)");
    o->store((int)value);
    return DLRMB_OK;
}

int64_t dlrmb_clock_buffer_bytes(void) { return (int64_t)CLK_COUNT * 2 * kClockCtas * sizeof(unsigned long long); }
int32_t dlrmb_clock_kernels(void) { return CLK_COUNT; }
int32_t dlrmb_clock_enable(void* device_buffer) {
    g_clock_buf.store(static_cast<unsigned long long*>(device_buffer));
    return DLRMB_OK;
}

int32_t dlrmb_get_option(const char* name, int64_t* value) {
    std::atomic<int>* o = find_option(name);
    DLRMB_REQUIRE(o != nullptr && value != nullptr, "unknown option '%s'", name ? name : "(null)");
    *value = o->load();
    return DLRMB_OK;
}

int32_t dlrmb_tables_create(int32_t device, int32_t ntab, const int64_t* rows, int32_t D,
                            int64_t max_lookups, dlrmb_tables** out) {
    return dlrmb_tables_create_ex(device, ntab, rows, D, max_lookups, 4, out);
}

int32_t dlrmb_tables_create_ex(int32_t device, int32_t ntab, const int64_t* rows, int32_t D,
                               int64_t max_lookups, int32_t elem_bytes, dlrmb_tables** out) {
    DLRMB_REQUIRE(out != nullptr, "out is null");
    *out = nullptr;
    DLRMB_REQUIRE(elem_bytes == 4 || elem_bytes == 2, "elem_bytes must be 4 (f32) or 2 (bf16), got %d", elem_bytes);
    DLRMB_REQUIRE(ntab > 0 && ntab <= 65535, "ntab must be in 1..65535 (got %d)", ntab);
    DLRMB_REQUIRE(rows != nullptr, "rows is null");
    DLRMB_REQUIRE(D > 0 && ((D % 4 == 0 && D <= 1024) || D <= 256),
                  "D must be in 1..256, or a multiple of 4 up to 1024 (got %d)", D);
    DLRMB_REQUIRE(max_lookups > 0 && max_lookups < (1ll << 30),
                  "max_lookups must be in 1..2^30 (got %lld)", (long long)max_lookups);
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);

    dlrmb_tables* t = new dlrmb_tables();
    t->device = device;
    t->ntab = ntab;
    t->D = D;
    t->elem_bytes = elem_bytes;
    t->max_lookups = max_lookups;
    t->cap = (max_lookups + 3) / 4 * 4;
    t->sm_count = device_sm_count(device);
    t->h_rows = (int64_t*)malloc(sizeof(int64_t) * ntab);
    t->h_sorted_P = (int32_t*)malloc(sizeof(int32_t) * ntab);
    t->h_offsets = (int64_t*)malloc(sizeof(int64_t) * (ntab + 1));
    int64_t off = 0;
    for (int k = 0; k < ntab; ++k) {
        if (rows[k] <= 0 || rows[k] >= (1ll << 32)) {
            set_error("rows[%d] = %lld outside 1..2^32-1", k, (long long)rows[k]);
            dlrmb_tables_destroy(t);
            return DLRMB_EINVAL;
        }
        t->h_rows[k] = rows[k];
        t->h_offsets[k] = off;
        int64_t elems = rows[k] * (int64_t)D;
        off += (elems + 127) / 128 * 128;  // keep every table 256-byte aligned (f32 and bf16)
        t->total_rows += rows[k];
        if (rows[k] > t->max_rows) t->max_rows = rows[k];
    }
    t->h_offsets[ntab] = off;

    auto fail = [&](int code) {
        dlrmb_tables_destroy(t);
        return code;
    };
#define TRY_CUDA(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                       \
            return fail(_e == cudaErrorMemoryAllocation ? DLRMB_ENOMEM : DLRMB_ECUDA);       \
        }                                                                                    \
    } while (0)

    TRY_CUDA(cudaStreamCreateWithFlags(&t->own_stream, cudaStreamNonBlocking));
    TRY_CUDA(cudaMalloc((void**)&t->slab, (size_t)elem_bytes * (size_t)off));
    TRY_CUDA(cudaMalloc((void**)&t->d_desc, sizeof(TableDesc) * ntab));
    {
        TableDesc* h = (TableDesc*)malloc(sizeof(TableDesc) * ntab);
        for (int k = 0; k < ntab; ++k) {
            h[k].base = reinterpret_cast<float*>(reinterpret_cast<char*>(t->slab) + (size_t)t->h_offsets[k] * elem_bytes);
            h[k].rows = t->h_rows[k];
        }
        cudaError_t e = cudaMemcpy(t->d_desc, h, sizeof(TableDesc) * ntab, cudaMemcpyHostToDevice);
        free(h);
        TRY_CUDA(e);
    }
    {
        int rc = alloc_workspace(t, max_lookups);
        if (rc) return fail(rc);
    }
#undef TRY_CUDA
    *out = t;
    return DLRMB_OK;
}

int32_t dlrmb_tables_destroy(dlrmb_tables* t) {
    if (!t) return DLRMB_OK;
    DeviceGuard guard(t->device);
    if (t->own_stream) cudaStreamSynchronize(t->own_stream);
    cudaFree(t->slab);
    cudaFree(t->d_desc);
    cudaFree(t->d_slotmap);
    free_workspace(t);
    cudaFree(t->stage_idx);
    cudaFree(t->stage_a);
    cudaFree(t->stage_b);
    cudaFree(t->stage_c);
    cudaFree(t->stage_d);
    if (t->own_stream) cudaStreamDestroy(t->own_stream);
    free(t->h_rows);
    free(t->h_sorted_P);
    free(t->h_offsets);
    delete t;
    return DLRMB_OK;
}

int32_t dlrmb_tables_elem_bytes(const dlrmb_tables* t) { return t ? t->elem_bytes : 0; }

int32_t dlrmb_tables_info(const dlrmb_tables* t, int32_t* ntab, int32_t* D, int64_t* max_lookups,
                          int64_t* total_rows) {
    DLRMB_REQUIRE(t != nullptr, "null tables handle");
    if (ntab) *ntab = t->ntab;
    if (D) *D = t->D;
    if (max_lookups) *max_lookups = t->max_lookups;
    if (total_rows) *total_rows = t->total_rows;
    return DLRMB_OK;
}

int32_t dlrmb_tables_reserve(dlrmb_tables* t, int64_t max_lookups) {
    GUARD(t);
    DLRMB_REQUIRE(max_lookups > 0 && max_lookups < (1ll << 30), "max_lookups must be in 1..2^30 (got %lld)",
                  (long long)max_lookups);
    if (max_lookups <= t->max_lookups) return DLRMB_OK;
    DLRMB_CUDA(cudaDeviceSynchronize());     // earlier launches may still use the old workspaces
    free_workspace(t);
    return alloc_workspace(t, max_lookups);
}

static inline char* table_ptr(dlrmb_tables* t, int k) {
    return reinterpret_cast<char*>(t->slab) + (size_t)t->h_offsets[k] * t->elem_bytes;
}

int32_t dlrmb_tables_upload(dlrmb_tables* t, int32_t k, const float* host) {
    GUARD(t);
    DLRMB_REQUIRE(k >= 0 && k < t->ntab, "table index %d outside 0..%d", k, t->ntab - 1);
    DLRMB_REQUIRE(host != nullptr, "host buffer is null");
    size_t bytes = sizeof(float) * (size_t)t->h_rows[k] * (size_t)t->D;
    if (t->elem_bytes == 4) {
        DLRMB_CUDA(cudaMemcpyAsync(table_ptr(t, k), host, bytes, cudaMemcpyHostToDevice, t->own_stream));
    } else {   // bf16 storage: stage the f32 rows on the device, round to nearest even there
        int rc = grow((void**)&t->stage_a, &t->stage_a_bytes, bytes);
        if (rc) return rc;
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, host, bytes, cudaMemcpyHostToDevice, t->own_stream));
        rc = launch_convert_rows(t, k, t->stage_a, true, t->own_stream);
        if (rc) return rc;
    }
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_tables_download(dlrmb_tables* t, int32_t k, float* host) {
    GUARD(t);
    DLRMB_REQUIRE(k >= 0 && k < t->ntab, "table index %d outside 0..%d", k, t->ntab - 1);
    DLRMB_REQUIRE(host != nullptr, "host buffer is null");
    size_t bytes = sizeof(float) * (size_t)t->h_rows[k] * (size_t)t->D;
    // the caller's compute streams may still be updating the table: drain the device first
    DLRMB_CUDA(cudaDeviceSynchronize());
    if (t->elem_bytes == 4) {
        DLRMB_CUDA(cudaMemcpyAsync(host, table_ptr(t, k), bytes, cudaMemcpyDeviceToHost, t->own_stream));
    } else {
        int rc = grow((void**)&t->stage_a, &t->stage_a_bytes, bytes);
        if (rc) return rc;
        rc = launch_convert_rows(t, k, t->stage_a, false, t->own_stream);
        if (rc) return rc;
        DLRMB_CUDA(cudaMemcpyAsync(host, t->stage_a, bytes, cudaMemcpyDeviceToHost, t->own_stream));
    }
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_tables_device_ptr(dlrmb_tables* t, int32_t k, float** dev) {
    DLRMB_REQUIRE(t != nullptr && dev != nullptr, "null argument");
    DLRMB_REQUIRE(k >= 0 && k < t->ntab, "table index %d outside 0..%d", k, t->ntab - 1);
    *dev = reinterpret_cast<float*>(table_ptr(t, k));
    return DLRMB_OK;
}

int32_t dlrmb_tables_init_uniform(dlrmb_tables* t, uint64_t seed, dlrmb_stream stream) {
    GUARD(t);
    return launch_init_uniform(t, seed, (cudaStream_t)stream);
}

int32_t dlrmb_tables_sync(dlrmb_tables* t) {
    GUARD(t);
    DLRMB_CUDA(cudaDeviceSynchronize());
    return DLRMB_OK;
}

static int check_idx_args(const dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, int B, int P) {
    DLRMB_REQUIRE(idx != nullptr, "idx is null");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(idx_base == 0 || idx_base == 1, "idx_base must be 0 or 1 (got %d)", idx_base);
    DLRMB_REQUIRE(B > 0 && P > 0, "B and P must be positive (got %d, %d)", B, P);
    DLRMB_REQUIRE((int64_t)B * P <= t->max_lookups, "B*P = %lld exceeds max_lookups = %lld",
                  (long long)B * P, (long long)t->max_lookups);
    return DLRMB_OK;
}

int32_t dlrmb_embedding_fwd(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                            int32_t B, int32_t P, float* out, int32_t slots, int32_t slot0,
                            dlrmb_stream stream) {
    GUARD(t);
    int rc = check_idx_args(t, idx, idx_bytes, idx_base, B, P);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    return run_uniform(t, idx, idx_bytes, B, P, slot0, false, [&](dlrmb_tables* v, const void* gidx, const MpGeom& g, int gslot0) {
        return launch_lookup_mp(v, gidx, idx_bytes, idx_base, g, out, slots, gslot0, (cudaStream_t)stream);
    });
}

int32_t dlrmb_embedding_fwd_sort(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                 int32_t B, int32_t P, float* out, int32_t slots, int32_t slot0,
                                 dlrmb_stream stream) {
    GUARD(t);
    int rc = check_idx_args(t, idx, idx_bytes, idx_base, B, P);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    t->sorted_valid = false;
    return run_uniform(t, idx, idx_bytes, B, P, slot0, true, [&](dlrmb_tables* v, const void* gidx, const MpGeom& g, int gslot0) {
        return launch_lookup_sort_mp(v, gidx, idx_bytes, idx_base, g, out, slots, gslot0, (cudaStream_t)stream);
    });
}

static int check_interaction_args(int B, int F, int d, int pad_to_mul) {
    DLRMB_REQUIRE(B > 0 && F >= 1 && d >= 1, "B, F, d must be positive (got %d, %d, %d)", B, F, d);
    DLRMB_REQUIRE(F <= 255, "F = %d exceeds 255 feature slots", F);
    DLRMB_REQUIRE(pad_to_mul >= 1, "pad_to_mul must be >= 1 (got %d)", pad_to_mul);
    return DLRMB_OK;
}

int32_t dlrmb_interaction_fwd(int32_t device, float* T, const float* x, int32_t B, int32_t F,
                              int32_t d, int32_t pad_to_mul, float* out, dlrmb_stream stream) {
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(T != nullptr && out != nullptr, "T / out is null");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_interaction_fwd(T, x, B, F, d, pad_to_mul, out, device_sm_count(device), (cudaStream_t)stream);
}

int32_t dlrmb_interaction_bwd(int32_t device, const float* dOut, const float* T, int32_t B,
                              int32_t F, int32_t d, int32_t pad_to_mul, float* dT, float* dx,
                              dlrmb_stream stream) {
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(dOut && T && dT && dx, "null buffer");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_interaction_bwd(dOut, T, B, F, d, pad_to_mul, dT, dx, device_sm_count(device), (cudaStream_t)stream);
}

int32_t dlrmb_dense_fwd_bias_act(int32_t device, float* z, const float* bias, int32_t B, int32_t N, int32_t relu,
                                 dlrmb_stream stream) {
    DLRMB_REQUIRE(B > 0 && N > 0, "B and N must be positive (got %d, %d)", B, N);
    DLRMB_REQUIRE(z && bias, "null buffer");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_dense_fwd_bias_act(z, bias, B, N, relu, device_sm_count(device), (cudaStream_t)stream);
}

int64_t dlrmb_dense_bwd_scratch_floats(int32_t N) { return dense_bwd_scratch_floats(N); }

int32_t dlrmb_dense_bwd_act_bias(int32_t device, const float* dy, const float* y, int32_t B, int32_t N,
                                 float* dz, float* db, float* scratch, dlrmb_stream stream) {
    DLRMB_REQUIRE(B > 0 && N > 0, "B and N must be positive (got %d, %d)", B, N);
    DLRMB_REQUIRE(dy && dz && db && scratch, "null buffer");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_dense_bwd_act_bias(dy, y, B, N, dz, db, scratch, (cudaStream_t)stream);
}

int32_t dlrmb_interaction_has_warp_path(int32_t F, int32_t d) { return interaction_has_warp_path(F, d) ? 1 : 0; }

int32_t dlrmb_interaction_bwd_scatter(int32_t device, const float* dOut, const float* T, int32_t B,
                                      int32_t F, int32_t d, int32_t pad_to_mul,
                                      const dlrmb_slot_dest* dests, int64_t sample_offset, float* dx,
                                      dlrmb_stream stream) {
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(dOut && T && dests && dx, "null buffer");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_interaction_bwd_ex(dOut, T, B, F, d, pad_to_mul, const_cast<float*>(T) /* unused */, dx, dests,
                                     (long long)sample_offset, 0, device_sm_count(device), (cudaStream_t)stream);
}

int32_t dlrmb_interaction_bwd_scatter_cols(int32_t device, const float* dOut, const float* T, int32_t B,
                                           int32_t F, int32_t d, int32_t pad_to_mul, const dlrmb_slot_dest* dests,
                                           int32_t Q, int64_t sample_offset, float* dx, dlrmb_stream stream) {
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(dOut && T && dests && dx, "null buffer");
    DLRMB_REQUIRE(Q >= 1 && Q <= 32 && (Q & (Q - 1)) == 0, "Q must be a power of two in 1..32 (got %d)", Q);
    DLRMB_REQUIRE(d % Q == 0 && (d / Q) % 4 == 0, "d / Q must be a multiple of 4 (d = %d, Q = %d)", d, Q);
    int qlog = 0;
    while ((1 << qlog) < Q) ++qlog;
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_interaction_bwd_ex(dOut, T, B, F, d, pad_to_mul, const_cast<float*>(T) /* unused */, dx, dests,
                                     (long long)sample_offset, qlog, device_sm_count(device), (cudaStream_t)stream);
}

int32_t dlrmb_interaction_bwd_dx(int32_t device, const float* dOut, const float* T, int32_t B, int32_t F, int32_t d,
                                 int32_t pad_to_mul, float* dx, dlrmb_stream stream) {
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(dOut && T && dx, "null buffer");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_interaction_bwd_dx(dOut, T, B, F, d, pad_to_mul, dx, device_sm_count(device), (cudaStream_t)stream);
}

int32_t dlrmb_embedding_sort(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                             int32_t B, int32_t P, dlrmb_stream stream) {
    GUARD(t);
    int rc = check_idx_args(t, idx, idx_bytes, idx_base, B, P);
    if (rc) return rc;
    t->sorted_valid = false;
    return run_uniform(t, idx, idx_bytes, B, P, 0, true, [&](dlrmb_tables* v, const void* gidx, const MpGeom& g, int) {
        return launch_sort_mp(v, gidx, idx_bytes, idx_base, g, 0, sort_mp_final_half(v, g), (cudaStream_t)stream);
    });
}

int32_t dlrmb_embedding_update_sorted(dlrmb_tables* t, const float* dT, int32_t slots,
                                      int32_t slot0, float lr, dlrmb_stream stream) {
    GUARD(t);
    if (!t->sorted_valid) {
        set_error("dlrmb_embedding_update_sorted called without a preceding dlrmb_embedding_sort");
        return DLRMB_ESTATE;
    }
    DLRMB_REQUIRE(dT != nullptr, "dT is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    return launch_update(t, dT, slots, slot0, lr, (cudaStream_t)stream);
}

int32_t dlrmb_embedding_bwd_sgd(dlrmb_tables* t, const void* idx, int32_t idx_bytes,
                                int32_t idx_base, int32_t B, int32_t P, const float* dT,
                                int32_t slots, int32_t slot0, float lr, dlrmb_stream stream) {
    int rc = dlrmb_embedding_sort(t, idx, idx_bytes, idx_base, B, P, stream);
    if (rc) return rc;
    return dlrmb_embedding_update_sorted(t, dT, slots, slot0, lr, stream);
}

int32_t dlrmb_sort_dedup_export(dlrmb_tables* t, int32_t k, int64_t* uniq, int32_t* seg_offsets,
                                int32_t* perm, int32_t* n_uniq) {
    GUARD(t);
    if (!t->sorted_valid) {
        set_error("dlrmb_sort_dedup_export called without a preceding dlrmb_embedding_sort");
        return DLRMB_ESTATE;
    }
    DLRMB_REQUIRE(k >= 0 && k < t->ntab, "table index %d outside 0..%d", k, t->ntab - 1);
    DLRMB_REQUIRE(uniq && seg_offsets && perm && n_uniq, "null output buffer");
    DLRMB_CUDA(cudaDeviceSynchronize());
    int rc = launch_dedup_export(t, k, t->own_stream);
    if (rc) return rc;
    int64_t L = sorted_lookups(t, k);
    int32_t n = 0;
    DLRMB_CUDA(cudaMemcpyAsync(&n, t->d_nuniq, sizeof(int32_t), cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    *n_uniq = n;
    DLRMB_CUDA(cudaMemcpyAsync(uniq, t->d_uniq, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaMemcpyAsync(seg_offsets, t->d_seg, sizeof(int32_t) * (n + 1), cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaMemcpyAsync(perm, t->pos[t->sorted_buf] + (size_t)k * t->cap, sizeof(uint32_t) * L,
                               cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_check_indices(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                            int32_t B, int32_t P, int32_t idx_on_host) {
    GUARD(t);
    int rc = check_idx_args(t, idx, idx_bytes, idx_base, B, P);
    if (rc) return rc;
    const void* d_idx = idx;
    size_t bytes = (size_t)t->ntab * B * P * idx_bytes;
    if (idx_on_host) {
        rc = grow(&t->stage_idx, &t->stage_idx_bytes, bytes);
        if (rc) return rc;
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_idx, idx, bytes, cudaMemcpyHostToDevice, t->own_stream));
        d_idx = t->stage_idx;
    } else {
        DLRMB_CUDA(cudaDeviceSynchronize());
    }
    long long bt = -1, bp = -1, bv = 0;
    rc = launch_check_indices(t, d_idx, idx_bytes, idx_base, B, P, t->own_stream, &bt, &bp, &bv);
    if (rc) return rc;
    if (bt >= 0) {
        set_error("index out of range: table %lld, flat position %lld, value %lld not in [%d, %lld]",
                  bt, bp, bv, idx_base, (long long)t->h_rows[bt] - 1 + idx_base);
        return DLRMB_EOOB;
    }
    return DLRMB_OK;
}

int32_t dlrmb_bce_sigmoid_fwd_bwd(int32_t device, const float* logits, const float* labels, int32_t B,
                                  float* prob, float* dlogits, float* loss, float* scratch,
                                  dlrmb_stream stream) {
    DLRMB_REQUIRE(B > 0, "B must be positive (got %d)", B);
    DLRMB_REQUIRE(logits && labels && dlogits && loss && scratch, "null buffer");
    DeviceGuard guard(device);
    DLRMB_REQUIRE(guard.ok, "cudaSetDevice(%d) failed", device);
    return launch_bce_sigmoid(logits, labels, B, prob, dlogits, loss, scratch, (cudaStream_t)stream);
}

// ---- host-buffer entry points --------------------------------------------------------------
static int stage_indices(dlrmb_tables* t, const void* idx, int idx_bytes, int B, int P) {
    size_t bytes = (size_t)t->ntab * B * P * idx_bytes;
    int rc = grow(&t->stage_idx, &t->stage_idx_bytes, bytes);
    if (rc) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_idx, idx, bytes, cudaMemcpyHostToDevice, t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_embedding_fwd_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes,
                                 int32_t idx_base, int32_t B, int32_t P, float* out,
                                 int32_t slots, int32_t slot0) {
    GUARD(t);
    int rc = check_idx_args(t, idx, idx_bytes, idx_base, B, P);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab, "slots too small");
    size_t obytes = sizeof(float) * (size_t)B * slots * t->D;
    if ((rc = stage_indices(t, idx, idx_bytes, B, P))) return rc;
    if ((rc = grow((void**)&t->stage_a, &t->stage_a_bytes, obytes))) return rc;
    if (slot0 > 0)  // reserved slots are the caller's (x); keep whatever the host buffer holds
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, out, obytes, cudaMemcpyHostToDevice, t->own_stream));
    rc = run_uniform(t, t->stage_idx, idx_bytes, B, P, slot0, false, [&](dlrmb_tables* v, const void* gidx, const MpGeom& g, int gslot0) {
        return launch_lookup_mp(v, gidx, idx_bytes, idx_base, g, t->stage_a, slots, gslot0, t->own_stream);
    });
    if (rc) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(out, t->stage_a, obytes, cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

static int interaction_width(int F, int d, int pad_to_mul) {
    int unpadded = d + F * (F - 1) / 2;
    return (unpadded + pad_to_mul - 1) / pad_to_mul * pad_to_mul;
}

int32_t dlrmb_interaction_fwd_host(dlrmb_tables* t, float* T, const float* x, int32_t B, int32_t F,
                                   int32_t d, int32_t pad_to_mul, float* out) {
    GUARD(t);
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(T != nullptr && out != nullptr, "T / out is null");
    int width = interaction_width(F, d, pad_to_mul);
    size_t tb = sizeof(float) * (size_t)B * F * d, xb = sizeof(float) * (size_t)B * d,
           ob = sizeof(float) * (size_t)B * width;
    if ((rc = grow((void**)&t->stage_a, &t->stage_a_bytes, tb))) return rc;
    if ((rc = grow((void**)&t->stage_b, &t->stage_b_bytes, ob))) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, T, tb, cudaMemcpyHostToDevice, t->own_stream));
    const float* dx = nullptr;
    if (x) {
        if ((rc = grow((void**)&t->stage_c, &t->stage_c_bytes, xb))) return rc;
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_c, x, xb, cudaMemcpyHostToDevice, t->own_stream));
        dx = t->stage_c;
    }
    rc = launch_interaction_fwd(t->stage_a, dx, B, F, d, pad_to_mul, t->stage_b, t->sm_count, t->own_stream);
    if (rc) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(out, t->stage_b, ob, cudaMemcpyDeviceToHost, t->own_stream));
    if (x)  // fast_vcat wrote x into slot 0 of T
        DLRMB_CUDA(cudaMemcpyAsync(T, t->stage_a, tb, cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_interaction_bwd_host(dlrmb_tables* t, const float* dOut, const float* T, int32_t B,
                                   int32_t F, int32_t d, int32_t pad_to_mul, float* dT, float* dx) {
    GUARD(t);
    int rc = check_interaction_args(B, F, d, pad_to_mul);
    if (rc) return rc;
    DLRMB_REQUIRE(dOut && T && dT && dx, "null buffer");
    int width = interaction_width(F, d, pad_to_mul);
    size_t tb = sizeof(float) * (size_t)B * F * d, xb = sizeof(float) * (size_t)B * d,
           ob = sizeof(float) * (size_t)B * width;
    if ((rc = grow((void**)&t->stage_a, &t->stage_a_bytes, tb))) return rc;
    if ((rc = grow((void**)&t->stage_b, &t->stage_b_bytes, ob))) return rc;
    if ((rc = grow((void**)&t->stage_c, &t->stage_c_bytes, xb))) return rc;
    if ((rc = grow((void**)&t->stage_d, &t->stage_d_bytes, tb))) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, T, tb, cudaMemcpyHostToDevice, t->own_stream));
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_b, dOut, ob, cudaMemcpyHostToDevice, t->own_stream));
    rc = launch_interaction_bwd(t->stage_b, t->stage_a, B, F, d, pad_to_mul, t->stage_d, t->stage_c,
                                t->sm_count, t->own_stream);
    if (rc) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(dT, t->stage_d, tb, cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaMemcpyAsync(dx, t->stage_c, xb, cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_embedding_bwd_sgd_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes,
                                     int32_t idx_base, int32_t B, int32_t P, const float* dT,
                                     int32_t slots, int32_t slot0, float lr) {
    GUARD(t);
    int rc = check_idx_args(t, idx, idx_bytes, idx_base, B, P);
    if (rc) return rc;
    DLRMB_REQUIRE(dT != nullptr, "dT is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab, "slots too small");
    size_t gb = sizeof(float) * (size_t)B * slots * t->D;
    if ((rc = stage_indices(t, idx, idx_bytes, B, P))) return rc;
    if ((rc = grow((void**)&t->stage_a, &t->stage_a_bytes, gb))) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, dT, gb, cudaMemcpyHostToDevice, t->own_stream));
    t->sorted_valid = false;
    rc = run_uniform(t, t->stage_idx, idx_bytes, B, P, 0, true, [&](dlrmb_tables* v, const void* gidx, const MpGeom& g, int) {
        return launch_sort_mp(v, gidx, idx_bytes, idx_base, g, 0, sort_mp_final_half(v, g), t->own_stream);
    });
    if (rc) return rc;
    if ((rc = launch_update(t, t->stage_a, slots, slot0, lr, t->own_stream))) return rc;
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

}  // extern "C"

// ---- per-table pooling factors (`_mp`) -----------------------------------------------------------
namespace dlrmb {

int check_mp_args(const dlrmb_tables* t, const void* idx, int idx_bytes, int idx_base, int B, const int32_t* P,
                  MpGeom* g) {
    DLRMB_REQUIRE(idx != nullptr, "idx is null");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(idx_base == 0 || idx_base == 1, "idx_base must be 0 or 1 (got %d)", idx_base);
    DLRMB_REQUIRE(P != nullptr, "P (per-table pooling factors) is null");
    DLRMB_REQUIRE(t->ntab <= kMpMaxTables, "per-table pooling factors support up to %d tables (handle has %d)",
                  kMpMaxTables, t->ntab);
    DLRMB_REQUIRE(B > 0, "B must be positive (got %d)", B);
    int64_t off = 0;
    int32_t maxP = 0;
    for (int k = 0; k < t->ntab; ++k) {
        DLRMB_REQUIRE(P[k] >= 1, "P[%d] = %d: every pooling factor must be >= 1", k, P[k]);
        maxP = P[k] > maxP ? P[k] : maxP;
        g->P[k] = (uint32_t)P[k];
        g->off[k] = off;
        off += (int64_t)B * P[k];
    }
    DLRMB_REQUIRE((int64_t)B * maxP <= t->max_lookups, "B*max(P) = %lld exceeds max_lookups = %lld",
                  (long long)B * maxP, (long long)t->max_lookups);
    g->ntab = t->ntab;
    g->B = (uint32_t)B;
    g->nlist = 0;
    return DLRMB_OK;
}

static int64_t mp_index_count(const MpGeom& g) { return (int64_t)g.off[g.ntab - 1] + (int64_t)g.B * g.P[g.ntab - 1]; }

void mark_sorted(dlrmb_tables* t, const MpGeom& g, int k0) {
    t->sorted_B = (int)g.B;
    for (int k = 0; k < g.ntab; ++k) t->h_sorted_P[k0 + k] = (int32_t)g.P[k];
    t->sorted_jagged = -1;
    t->sorted_valid = k0 + g.ntab == t->ntab;
}

// Host-only checks (no CUDA call, so they also refuse bad arguments on a machine without a GPU).
int check_jagged_args(const dlrmb_tables* t, const void* values, const void* offsets, int idx_bytes, int idx_base,
                      int B, const int64_t* L, int pooling, MpGeom* g) {
    DLRMB_REQUIRE(offsets != nullptr, "offsets is null");
    DLRMB_REQUIRE(L != nullptr, "L (per-table lookup counts) is null");
    DLRMB_REQUIRE(idx_bytes == 4 || idx_bytes == 8, "idx_bytes must be 4 or 8 (got %d)", idx_bytes);
    DLRMB_REQUIRE(idx_base == 0 || idx_base == 1, "idx_base must be 0 or 1 (got %d)", idx_base);
    DLRMB_REQUIRE(pooling == 0 || pooling == 1, "pooling must be 0 (sum) or 1 (mean) (got %d)", pooling);
    DLRMB_REQUIRE(B > 0, "B must be positive (got %d)", B);
    DLRMB_REQUIRE(t != nullptr, "null tables handle");
    DLRMB_REQUIRE(t->ntab <= kMpMaxTables, "jagged batches support up to %d tables (handle has %d)", kMpMaxTables,
                  t->ntab);
    int64_t off = 0;
    for (int k = 0; k < t->ntab; ++k) {
        DLRMB_REQUIRE(L[k] >= 0, "L[%d] = %lld: lookup counts must be >= 0", k, (long long)L[k]);
        DLRMB_REQUIRE(L[k] <= t->max_lookups, "L[%d] = %lld exceeds max_lookups = %lld", k, (long long)L[k],
                      (long long)t->max_lookups);
        g->P[k] = (uint32_t)L[k];
        g->off[k] = off;
        off += L[k];
    }
    DLRMB_REQUIRE(values != nullptr || off == 0, "values is null");
    DLRMB_REQUIRE(idx_bytes == 8 || off <= INT32_MAX, "%lld lookups need 8-byte offsets", (long long)off);
    g->ntab = t->ntab;
    g->B = 1;
    g->nlist = 0;
    return DLRMB_OK;
}

dlrmb_tables table_group(const dlrmb_tables& t, int k0, int n) {
    dlrmb_tables v = t;
    v.ntab = n;
    v.d_desc += k0;
    if (v.d_slotmap) v.d_slotmap += k0;
    for (int i = 0; i < 2; ++i) {
        v.keys[i] += (size_t)k0 * t.cap;
        v.pos[i] += (size_t)k0 * t.cap;
    }
    v.tile_hist += (size_t)k0 * 512 * t.radix_tiles_cap;
    v.digit_total += (size_t)k0 * 512;
    return v;
}

}  // namespace dlrmb

extern "C" {

int32_t dlrmb_mp_max_tables(void) { return kMpMaxTables; }

int32_t dlrmb_embedding_fwd_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                               const int32_t* P, float* out, int32_t slots, int32_t slot0, dlrmb_stream stream) {
    GUARD(t);
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B, P, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    return launch_lookup_mp(t, idx, idx_bytes, idx_base, g, out, slots, slot0, (cudaStream_t)stream);
}

int32_t dlrmb_embedding_fwd_sort_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                    const int32_t* P, float* out, int32_t slots, int32_t slot0, dlrmb_stream stream) {
    GUARD(t);
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B, P, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    t->sorted_valid = false;
    rc = launch_lookup_sort_mp(t, idx, idx_bytes, idx_base, g, out, slots, slot0, (cudaStream_t)stream);
    if (rc) return rc;
    mark_sorted(t, g, 0);
    return DLRMB_OK;
}

int32_t dlrmb_embedding_sort_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                const int32_t* P, dlrmb_stream stream) {
    GUARD(t);
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B, P, &g);
    if (rc) return rc;
    t->sorted_valid = false;
    rc = launch_sort_mp(t, idx, idx_bytes, idx_base, g, 0, sort_mp_final_half(t, g), (cudaStream_t)stream);
    if (rc) return rc;
    mark_sorted(t, g, 0);
    return DLRMB_OK;
}

int32_t dlrmb_embedding_bwd_sgd_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                   const int32_t* P, const float* dT, int32_t slots, int32_t slot0, float lr,
                                   dlrmb_stream stream) {
    int rc = dlrmb_embedding_sort_mp(t, idx, idx_bytes, idx_base, B, P, stream);
    if (rc) return rc;
    return dlrmb_embedding_update_sorted(t, dT, slots, slot0, lr, stream);
}

int32_t dlrmb_check_indices_mp(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                               const int32_t* P, int32_t idx_on_host) {
    GUARD(t);
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B, P, &g);
    if (rc) return rc;
    const void* d_idx = idx;
    size_t bytes = (size_t)mp_index_count(g) * idx_bytes;
    if (idx_on_host) {
        rc = grow(&t->stage_idx, &t->stage_idx_bytes, bytes);
        if (rc) return rc;
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_idx, idx, bytes, cudaMemcpyHostToDevice, t->own_stream));
        d_idx = t->stage_idx;
    } else {
        DLRMB_CUDA(cudaDeviceSynchronize());
    }
    long long bt = -1, bp = -1, bv = 0;
    rc = launch_check_indices_mp(t, d_idx, idx_bytes, idx_base, g, t->own_stream, &bt, &bp, &bv);
    if (rc) return rc;
    if (bt >= 0) {
        set_error("index out of range: table %lld, flat position %lld, value %lld not in [%d, %lld]",
                  bt, bp, bv, idx_base, (long long)t->h_rows[bt] - 1 + idx_base);
        return DLRMB_EOOB;
    }
    return DLRMB_OK;
}

// ---- jagged (variable-length) bags -----------------------------------------------------------------------------
// `weighted`: the `_weighted` calls, sum pooling with per-sample `weights`; the launchers take it as pooling
// kJaggedWeighted.  Otherwise `pooling` is the caller's (0 sum or 1 mean, checked by check_jagged_args).
static int check_jagged_call(const dlrmb_tables* t, const void* values, const void* offsets, const float* weights,
                             bool weighted, int idx_bytes, int idx_base, int B, const int64_t* L, int* pooling,
                             MpGeom* g) {
    int rc = check_jagged_args(t, values, offsets, idx_bytes, idx_base, B, L, weighted ? 0 : *pooling, g);
    if (rc || !weighted) return rc;
    DLRMB_REQUIRE(weights != nullptr || g->off[g->ntab - 1] + g->P[g->ntab - 1] == 0, "weights is null");
    *pooling = kJaggedWeighted;
    return DLRMB_OK;
}

static int jagged_sort(dlrmb_tables* t, const void* values, const void* offsets, const float* weights, bool weighted,
                       int idx_bytes, int idx_base, int B, const int64_t* L, int pooling, dlrmb_stream stream) {
    MpGeom g;
    int rc = check_jagged_call(t, values, offsets, weights, weighted, idx_bytes, idx_base, B, L, &pooling, &g);
    if (rc) return rc;
    GUARD(t);
    t->sorted_valid = false;
    const int half = sort_mp_final_half(t, g);
    rc = launch_sort_mp(t, values, idx_bytes, idx_base, g, 0, half, (cudaStream_t)stream);
    if (rc) return rc;
    rc = launch_jagged_bags(t, offsets, weights, idx_bytes, g, B, pooling, half, (cudaStream_t)stream);
    if (rc) return rc;
    mark_sorted(t, g, 0);
    t->sorted_jagged = pooling;
    return DLRMB_OK;
}

static int jagged_fwd(dlrmb_tables* t, const void* values, const void* offsets, const float* weights, bool weighted,
                      int idx_bytes, int idx_base, int B, const int64_t* L, int pooling, float* out, int slots,
                      int slot0, dlrmb_stream stream, bool sort) {
    MpGeom g;
    int rc = check_jagged_call(t, values, offsets, weights, weighted, idx_bytes, idx_base, B, L, &pooling, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    GUARD(t);
    if (sort) t->sorted_valid = false;
    rc = launch_lookup_jagged(t, values, offsets, weights, idx_bytes, idx_base, g, B, pooling, out, slots, slot0,
                              (cudaStream_t)stream);
    if (rc || !sort) return rc;
    return jagged_sort(t, values, offsets, weights, weighted, idx_bytes, idx_base, B, L, pooling, stream);
}

int32_t dlrmb_embedding_fwd_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                   int32_t idx_base, int32_t B, const int64_t* L, int32_t pooling, float* out,
                                   int32_t slots, int32_t slot0, dlrmb_stream stream) {
    return jagged_fwd(t, values, offsets, nullptr, false, idx_bytes, idx_base, B, L, pooling, out, slots, slot0, stream,
                      false);
}

int32_t dlrmb_embedding_fwd_sort_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                        int32_t idx_base, int32_t B, const int64_t* L, int32_t pooling, float* out,
                                        int32_t slots, int32_t slot0, dlrmb_stream stream) {
    return jagged_fwd(t, values, offsets, nullptr, false, idx_bytes, idx_base, B, L, pooling, out, slots, slot0, stream,
                      true);
}

int32_t dlrmb_embedding_sort_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                    int32_t idx_base, int32_t B, const int64_t* L, int32_t pooling, dlrmb_stream stream) {
    return jagged_sort(t, values, offsets, nullptr, false, idx_bytes, idx_base, B, L, pooling, stream);
}

int32_t dlrmb_embedding_fwd_jagged_weighted(dlrmb_tables* t, const void* values, const void* offsets,
                                            const float* weights, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                            const int64_t* L, float* out, int32_t slots, int32_t slot0,
                                            dlrmb_stream stream) {
    return jagged_fwd(t, values, offsets, weights, true, idx_bytes, idx_base, B, L, 0, out, slots, slot0, stream, false);
}

int32_t dlrmb_embedding_fwd_sort_jagged_weighted(dlrmb_tables* t, const void* values, const void* offsets,
                                                 const float* weights, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                                 const int64_t* L, float* out, int32_t slots, int32_t slot0,
                                                 dlrmb_stream stream) {
    return jagged_fwd(t, values, offsets, weights, true, idx_bytes, idx_base, B, L, 0, out, slots, slot0, stream, true);
}

int32_t dlrmb_embedding_sort_jagged_weighted(dlrmb_tables* t, const void* values, const void* offsets,
                                             const float* weights, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                             const int64_t* L, dlrmb_stream stream) {
    return jagged_sort(t, values, offsets, weights, true, idx_bytes, idx_base, B, L, 0, stream);
}

int32_t dlrmb_embedding_weight_grad_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                           int32_t idx_base, int32_t B, const int64_t* L, const float* dT, int32_t slots,
                                           int32_t slot0, float* dw, dlrmb_stream stream) {
    MpGeom g;
    int rc = check_jagged_args(t, values, offsets, idx_bytes, idx_base, B, L, 0, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(dw != nullptr || g.off[g.ntab - 1] + g.P[g.ntab - 1] == 0, "dw is null");
    DLRMB_REQUIRE(dT != nullptr, "dT is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab,
                  "slots = %d too small for slot0 = %d + %d tables", slots, slot0, t->ntab);
    DLRMB_REQUIRE(t->D % 4 != 0 || (reinterpret_cast<uintptr_t>(dT) & 15) == 0,
                  "dT must be 16-byte aligned when D is a multiple of 4");
    GUARD(t);
    return launch_weight_grad_jagged(t, values, offsets, idx_bytes, idx_base, B, dT, slots, slot0, dw,
                                     (cudaStream_t)stream);
}

int32_t dlrmb_check_indices_jagged(dlrmb_tables* t, const void* values, const void* offsets, int32_t idx_bytes,
                                   int32_t idx_base, int32_t B, const int64_t* L, int32_t on_host) {
    MpGeom g;
    int rc = check_jagged_args(t, values, offsets, idx_bytes, idx_base, B, L, 0, &g);
    if (rc) return rc;
    GUARD(t);
    const int64_t noff = (int64_t)t->ntab * B + 1;
    const int64_t nval = g.off[t->ntab - 1] + g.P[t->ntab - 1];
    // the offsets on the host, widened to int64
    std::vector<char> raw;
    const void* src = offsets;
    if (!on_host) {
        DLRMB_CUDA(cudaDeviceSynchronize());
        raw.resize((size_t)noff * idx_bytes);
        DLRMB_CUDA(cudaMemcpy(raw.data(), offsets, raw.size(), cudaMemcpyDeviceToHost));
        src = raw.data();
    }
    std::vector<int64_t> ho((size_t)noff);
    for (int64_t i = 0; i < noff; ++i)
        ho[i] = idx_bytes == 4 ? (int64_t)static_cast<const uint32_t*>(src)[i] : static_cast<const int64_t*>(src)[i];
    DLRMB_REQUIRE(ho[0] == 0, "offsets[0] = %lld: the first offset must be 0", (long long)ho[0]);
    for (int64_t i = 0; i + 1 < noff; ++i)
        DLRMB_REQUIRE(ho[i] <= ho[i + 1], "offsets decrease at table %lld, bag %lld: offsets[%lld] = %lld > offsets[%lld] = %lld",
                      (long long)(i / B), (long long)(i % B), (long long)i, (long long)ho[i], (long long)(i + 1),
                      (long long)ho[i + 1]);
    for (int k = 0; k < t->ntab; ++k) {
        const int64_t n = ho[(int64_t)(k + 1) * B] - ho[(int64_t)k * B];
        DLRMB_REQUIRE(n == (int64_t)g.P[k], "table %d: offsets give %lld lookups, L[%d] = %lld", k, (long long)n, k,
                      (long long)g.P[k]);
    }
    const void* d_val = values;
    if (on_host && nval > 0) {
        rc = grow(&t->stage_idx, &t->stage_idx_bytes, (size_t)nval * idx_bytes);
        if (rc) return rc;
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_idx, values, (size_t)nval * idx_bytes, cudaMemcpyHostToDevice, t->own_stream));
        d_val = t->stage_idx;
    }
    long long bt = -1, bp = -1, bv = 0;
    if (nval > 0) {
        rc = launch_check_indices_mp(t, d_val, idx_bytes, idx_base, g, t->own_stream, &bt, &bp, &bv);
        if (rc) return rc;
    }
    if (bt >= 0) {
        // the bag of the offender: the last bag of table bt that starts at or before it
        const int64_t x = g.off[bt] + bp;
        int64_t b = 0;
        while (b + 1 < B && ho[bt * B + b + 1] <= x) ++b;
        set_error("index out of range: table %lld, bag %lld, position %lld of the table's values, value %lld not in [%d, %lld]",
                  bt, (long long)b, bp, bv, idx_base, (long long)t->h_rows[bt] - 1 + idx_base);
        return DLRMB_EOOB;
    }
    return DLRMB_OK;
}

int32_t dlrmb_embedding_fwd_mp_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base, int32_t B,
                                    const int32_t* P, float* out, int32_t slots, int32_t slot0) {
    GUARD(t);
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B, P, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(out != nullptr, "out is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab, "slots too small");
    size_t ibytes = (size_t)mp_index_count(g) * idx_bytes;
    size_t obytes = sizeof(float) * (size_t)B * slots * t->D;
    if ((rc = grow(&t->stage_idx, &t->stage_idx_bytes, ibytes))) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_idx, idx, ibytes, cudaMemcpyHostToDevice, t->own_stream));
    if ((rc = grow((void**)&t->stage_a, &t->stage_a_bytes, obytes))) return rc;
    if (slot0 > 0)  // reserved slots are the caller's (x); keep whatever the host buffer holds
        DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, out, obytes, cudaMemcpyHostToDevice, t->own_stream));
    rc = launch_lookup_mp(t, t->stage_idx, idx_bytes, idx_base, g, t->stage_a, slots, slot0, t->own_stream);
    if (rc) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(out, t->stage_a, obytes, cudaMemcpyDeviceToHost, t->own_stream));
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

int32_t dlrmb_embedding_bwd_sgd_mp_host(dlrmb_tables* t, const void* idx, int32_t idx_bytes, int32_t idx_base,
                                        int32_t B, const int32_t* P, const float* dT, int32_t slots, int32_t slot0,
                                        float lr) {
    GUARD(t);
    MpGeom g;
    int rc = check_mp_args(t, idx, idx_bytes, idx_base, B, P, &g);
    if (rc) return rc;
    DLRMB_REQUIRE(dT != nullptr, "dT is null");
    DLRMB_REQUIRE(slot0 >= 0 && slots >= slot0 + t->ntab, "slots too small");
    size_t ibytes = (size_t)mp_index_count(g) * idx_bytes;
    size_t gb = sizeof(float) * (size_t)B * slots * t->D;
    if ((rc = grow(&t->stage_idx, &t->stage_idx_bytes, ibytes))) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_idx, idx, ibytes, cudaMemcpyHostToDevice, t->own_stream));
    if ((rc = grow((void**)&t->stage_a, &t->stage_a_bytes, gb))) return rc;
    DLRMB_CUDA(cudaMemcpyAsync(t->stage_a, dT, gb, cudaMemcpyHostToDevice, t->own_stream));
    t->sorted_valid = false;
    if ((rc = launch_sort_mp(t, t->stage_idx, idx_bytes, idx_base, g, 0, sort_mp_final_half(t, g), t->own_stream)))
        return rc;
    mark_sorted(t, g, 0);
    if ((rc = launch_update(t, t->stage_a, slots, slot0, lr, t->own_stream))) return rc;
    DLRMB_CUDA(cudaStreamSynchronize(t->own_stream));
    return DLRMB_OK;
}

}  // extern "C"
