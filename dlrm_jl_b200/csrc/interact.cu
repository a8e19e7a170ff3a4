// Dot-product feature interaction, forward and backward, as batched small-Gram kernels.
//
// Replaces DotInteraction forward (DLRM.jl src/model/interact.jl:394-411: fast_vcat :271-281,
// process_batches :449-467, process_slice! :338-362, gemmavx! :318-326,
// triangular_slice_kernel! :64-75) and its pullback (dot_back :424-436, process_batches_back
// :469-489, triangular_slice_back_fuse_add_transpose_kernel! :154-173, sumavx :329-336).
//
// Forward, per sample b:  out[b] = [ x_b ; <T_b[i], T_b[j]> for j = 1..F-1, i = 0..j-1 ; 0-pad ]
//   flat position of pair i<j is d + j(j-1)/2 + i.
// Backward, per sample b: S symmetric F x F with zero diagonal from dOut[b][d:], then
//   dT_b[f] = sum_j S[j][f] * T_b[j],  dx_b = dOut[b][:d] + dT_b[0].
//
// Both are HBM-bound at DLRM shapes (5-12 flop/byte, below the fp32 FMA ridge), so the work
// stays on the FP32 FMA pipe (TF32 tensor cores would break the 1e-5 tolerance) and the design
// goal is one read of T and one write of the result per sample:
//   - a CTA owns NS consecutive samples; their T rows are staged into shared memory by TMA 1-D
//     bulk copies (cp.async.bulk, one per feature row, completion on an mbarrier), row stride
//     padded by 4 floats so the 128-bit operand reads of different rows spread across the bank
//     groups;
//   - forward: each thread owns a TB x TB register block of the Gram lower triangle (TB = 3 by
//     default; 6 and 9, and a k-split across adjacent lanes combined with warp shuffles, are
//     compiled in but measured slower at DLRM shapes) and walks k in float4 steps; results are
//     staged in shared memory so that the CTA's output, which is again one contiguous global
//     range, is written fully coalesced;
//   - backward: each thread owns 4 features x one float4 of k, reads one float4 of T and one
//     float4 of S per j (16 FMAs per two 128-bit shared loads) and writes dT as float4.
#include <stdlib.h>

#include "common.cuh"

namespace dlrmb {

// ---- TMA 1-D bulk copy (cp.async.bulk, SASS UBLKCP) completing on an mbarrier ----------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

static inline int interaction_width(int F, int d, int pad_to_mul) {
    int unpadded = d + F * (F - 1) / 2;
    return (unpadded + pad_to_mul - 1) / pad_to_mul * pad_to_mul;
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int TB>
__global__ void __launch_bounds__(256)
interaction_fwd_kernel(float* __restrict__ T, const float* __restrict__ x, int B, int F, int d,
                       int width, float* __restrict__ out, int NS, int nblk, int ks_log2) {
    extern __shared__ float4 smem4[];
    const int d4 = d >> 2;
    const int ldt4 = d4 + 1;              // row stride in float4 (4 floats of padding)
    const int Fp = nblk * TB;             // rows incl. zero padding
    const int nt = nblk * (nblk + 1) / 2; // register-block tasks per sample
    float4* Ts = smem4;                                   // [NS][Fp][ldt4]
    float* Os = reinterpret_cast<float*>(Ts + (size_t)NS * Fp * ldt4);  // [NS][width]
    unsigned char* pr = reinterpret_cast<unsigned char*>(Os + (size_t)NS * width);  // [nt][2]

    const int tid = threadIdx.x;
    const int s0 = blockIdx.x * NS;
    const int ns = min(NS, B - s0);

    __shared__ unsigned long long bar;
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_arrive_expect_tx(&bar, (unsigned)(ns * F * d * sizeof(float)));
    }
    __syncthreads();
    // stage T: one TMA bulk copy per feature row (slot 0 from x when given)
    for (int r = tid; r < ns * F; r += blockDim.x) {
        const int s = r / F, f = r - s * F;
        const float* src = (x != nullptr && f == 0) ? x + (size_t)(s0 + s) * d
                                                    : T + ((size_t)(s0 + s) * F + f) * d;
        bulk_g2s(Ts + ((size_t)s * Fp + f) * ldt4, src, (unsigned)(d * sizeof(float)), &bar);
    }
    // meanwhile: block-pair table (task q -> bi >= bj) and zeroed padding rows
    for (int q = tid; q < nt; q += blockDim.x) {
        int bi = (int)((sqrtf(8.f * q + 1.f) - 1.f) * 0.5f);
        while ((bi + 1) * (bi + 2) / 2 <= q) ++bi;
        while (bi * (bi + 1) / 2 > q) --bi;
        pr[2 * q] = (unsigned char)bi;
        pr[2 * q + 1] = (unsigned char)(q - bi * (bi + 1) / 2);
    }
    if (Fp > F) {
        const int padrows = Fp - F;
        for (int i = tid; i < ns * padrows * d4; i += blockDim.x) {
            const int c = i % d4, r = i / d4;
            const int s = r / padrows, f = F + (r - s * padrows);
            Ts[((size_t)s * Fp + f) * ldt4 + c] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    mbar_wait(&bar, 0);
    __syncthreads();

    // x passthrough: out[b][0:d] = T[b][0]; also fast_vcat into T when x came separately
    for (int i = tid; i < ns * d4; i += blockDim.x) {
        int c = i % d4, s = i / d4;
        float4 v = Ts[(size_t)s * Fp * ldt4 + c];
        float* o = Os + (size_t)s * width + 4 * c;
        o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
        if (x != nullptr) reinterpret_cast<float4*>(T + (size_t)(s0 + s) * F * d)[c] = v;
    }
    const int npair = F * (F - 1) / 2;
    for (int i = tid; i < ns * (width - d - npair); i += blockDim.x) {
        int padw = width - d - npair;
        int s = i / padw, c = i % padw;
        Os[(size_t)s * width + d + npair + c] = 0.f;
    }

    // Gram blocks.  A task is (sample, block pair, k-slice): KS = 2^ks_log2 adjacent lanes can split
    // the k range of one TB x TB block and combine their partial dot products with warp shuffles
    // (KS = 1 by default).
    const int KS = 1 << ks_log2;
    const int tps = nt * KS;              // tasks per sample
    const int kper = d4 >> ks_log2;       // float4 k-steps per task
    const int total_tasks = ns * tps;
    for (int base_task = 0; base_task < total_tasks; base_task += blockDim.x) {
        const int task = base_task + tid;
        const bool live = task < total_tasks;
        const int s = live ? task / tps : 0;
        const int rem = live ? task - s * tps : 0;
        const int q = rem >> ks_log2;
        const int ks = rem & (KS - 1);
        const int bi = pr[2 * q], bj = pr[2 * q + 1];
        const float4* A = Ts + ((size_t)s * Fp + bi * TB) * ldt4 + ks * kper;
        const float4* Bm = Ts + ((size_t)s * Fp + bj * TB) * ldt4 + ks * kper;
        float acc[TB][TB];
#pragma unroll
        for (int r = 0; r < TB; ++r)
#pragma unroll
            for (int c = 0; c < TB; ++c) acc[r][c] = 0.f;
        if (live) {
            for (int k = 0; k < kper; ++k) {
                float4 a[TB];
#pragma unroll
                for (int r = 0; r < TB; ++r) a[r] = A[r * ldt4 + k];
#pragma unroll
                for (int c = 0; c < TB; ++c) {
                    const float4 b = Bm[c * ldt4 + k];
#pragma unroll
                    for (int r = 0; r < TB; ++r) {
                        float v = acc[r][c];
                        v = fmaf(a[r].x, b.x, v);
                        v = fmaf(a[r].y, b.y, v);
                        v = fmaf(a[r].z, b.z, v);
                        v = fmaf(a[r].w, b.w, v);
                        acc[r][c] = v;
                    }
                }
            }
        }
        for (int o = 1; o < KS; o <<= 1) {   // uniform across the warp
#pragma unroll
            for (int r = 0; r < TB; ++r)
#pragma unroll
                for (int c = 0; c < TB; ++c) acc[r][c] += __shfl_xor_sync(0xffffffffu, acc[r][c], o);
        }
        if (live && ks == 0) {
            float* o = Os + (size_t)s * width + d;
#pragma unroll
            for (int r = 0; r < TB; ++r)
#pragma unroll
                for (int c = 0; c < TB; ++c) {
                    int j = bi * TB + r, i = bj * TB + c;
                    if (i < j && j < F) o[j * (j - 1) / 2 + i] = acc[r][c];
                }
        }
    }
    __syncthreads();

    // coalesced store of the CTA's contiguous output range
    float* og = out + (size_t)s0 * width;
    const int total = ns * width;
    for (int i = tid; i < total; i += blockDim.x) og[i] = Os[i];
}

// Any shape (d not a multiple of 4, unaligned buffers): one thread per output element.
__global__ void __launch_bounds__(256)
interaction_fwd_generic_kernel(float* __restrict__ T, const float* __restrict__ x, int B, int F,
                               int d, int width, float* __restrict__ out) {
    const int npair = F * (F - 1) / 2;
    const int64_t total = (int64_t)B * width;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (int64_t)gridDim.x * blockDim.x) {
        int b = (int)(e / width);
        int c = (int)(e - (int64_t)b * width);
        const float* Tb = T + (size_t)b * F * d;
        const float* r0 = x ? x + (size_t)b * d : Tb;
        float v = 0.f;
        if (c < d) {
            v = r0[c];
        } else if (c < d + npair) {
            int m = c - d;
            int j = (int)((sqrtf(8.f * m + 1.f) + 1.f) * 0.5f);
            while (j * (j - 1) / 2 > m) --j;
            while ((j + 1) * j / 2 <= m) ++j;
            int i = m - j * (j - 1) / 2;
            const float* ri = (i == 0) ? r0 : Tb + (size_t)i * d;
            const float* rj = Tb + (size_t)j * d;
            for (int k = 0; k < d; ++k) v = fmaf(ri[k], rj[k], v);
        }
        out[e] = v;
    }
}

__global__ void __launch_bounds__(256)
copy_x_into_slot0_kernel(float* __restrict__ T, const float* __restrict__ x, int B, int F, int d) {
    const int64_t total = (int64_t)B * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (int64_t)gridDim.x * blockDim.x) {
        int64_t b = e / d;
        T[b * F * d + (e - b * d)] = x[e];
    }
}

int ensure_smem_attr(const void* func, int bytes, unsigned long long* done_mask) {
    int dev = 0;
    DLRMB_CUDA(cudaGetDevice(&dev));
    const unsigned long long bit = 1ull << (dev & 63);
    if (!(*done_mask & bit)) {
        DLRMB_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        *done_mask |= bit;
    }
    return DLRMB_OK;
}

struct TilePlan {
    int ns, threads;
    size_t smem;
};

// Pick samples-per-CTA and CTA size.  These kernels are latency-bound at DLRM batch sizes, so the
// plan keeps CTAs small (shared memory <= ~40 KB: at least 5 resident CTAs per SM, whose load /
// compute / store phases then overlap), fills whole rounds of the CTA with tasks, and among
// equals prefers more samples per CTA (fewer, fuller CTAs).
static TilePlan plan_tiles(int B, int tasks_per_sample, size_t smem_per_sample, size_t smem_fixed,
                           int sm_count) {
    TilePlan best{1, 128, smem_per_sample + smem_fixed};
    double best_score = -1.0;
    const size_t budget = 40 * 1024;
    for (int ns = 1; ns <= 16; ++ns) {
        size_t smem = ns * smem_per_sample + smem_fixed;
        if (smem > budget && ns > 1) break;
        for (int threads = 96; threads <= 256; threads += 32) {
            int tasks = ns * tasks_per_sample;
            int rounds = (tasks + threads - 1) / threads;
            double eff = (double)tasks / ((double)rounds * threads);
            int64_t ctas = (B + ns - 1) / ns;
            double fill = ctas >= 4 * (int64_t)sm_count ? 1.0 : (double)ctas / (4.0 * sm_count);
            double score = eff * (0.6 + 0.4 * fill) - 0.01 * (rounds - 1) + 0.001 * ns;
            if (score > best_score) {
                best_score = score;
                best = TilePlan{ns, threads, smem};
            }
        }
    }
    (void)sm_count;
    return best;
}

template <int TB>
static int launch_fwd_tb(float* T, const float* x, int B, int F, int d, int width, float* out,
                         int sm_count, cudaStream_t s) {
    const int nblk = (F + TB - 1) / TB;
    const int nt = nblk * (nblk + 1) / 2;
    const int Fp = nblk * TB;
    const int d4 = d / 4;
    // k-split (KS = 2^ks_log2 lanes per block): off by default, see launch_interaction_fwd
    int ks_log2 = 0;
    {   // tuning aid: dlrmb_set_option("fwd_ks", v)
        const int v = g_opt.fwd_ks.load(std::memory_order_relaxed);
        if (v >= 0 && v <= 3 && d4 % (1 << v) == 0) ks_log2 = v;
    }
    size_t per_sample = ((size_t)Fp * (d4 + 1) * 4 + width) * sizeof(float);
    size_t fixed = (size_t)nt * 2 + 16;
    TilePlan p = plan_tiles(B, nt << ks_log2, per_sample, fixed, sm_count);
    DLRMB_REQUIRE(p.smem <= 200 * 1024, "interaction tile needs %zu bytes of shared memory", p.smem);
    static unsigned long long attr_done = 0;
    int rc = ensure_smem_attr((const void*)interaction_fwd_kernel<TB>, 200 * 1024, &attr_done);
    if (rc) return rc;
    int grid = (B + p.ns - 1) / p.ns;
    interaction_fwd_kernel<TB><<<grid, p.threads, p.smem, s>>>(T, x, B, F, d, width, out, p.ns, nblk, ks_log2);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

// interact_warp.cu: warp-per-sample FFMA2 kernels for the DLRM shapes (-1 = no specialisation)
int try_interaction_fwd_warp(float* T, const float* x, int B, int F, int d, int width, float* out,
                             cudaStream_t s);
int try_interaction_bwd_warp(const float* dOut, const float* T, int B, int F, int d, int width,
                             float* dT, float* dx, const void* dests, long long sample_offset, int qlog,
                             cudaStream_t s);

int launch_interaction_fwd(float* T, const float* x, int B, int F, int d, int pad_to_mul,
                           float* out, int sm_count, cudaStream_t s) {
    const int width = interaction_width(F, d, pad_to_mul);
    const bool aligned = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(T) & 15) == 0) &&
                         (x == nullptr || (reinterpret_cast<uintptr_t>(x) & 15) == 0);
    if (aligned) {
        int rc = try_interaction_fwd_warp(T, x, B, F, d, width, out, s);
        if (rc >= 0) return rc;
    }
    if (!aligned || F < 2) {
        int64_t total = (int64_t)B * width;
        int64_t blocks = ceil_div64(total, 256);
        if (blocks > sm_count * 16) blocks = sm_count * 16;
        interaction_fwd_generic_kernel<<<(unsigned)blocks, 256, 0, s>>>(T, x, B, F, d, width, out);
        DLRMB_LAUNCH_CHECK();
        if (x != nullptr) {
            int64_t b2 = ceil_div64((int64_t)B * d, 256);
            if (b2 > sm_count * 16) b2 = sm_count * 16;
            copy_x_into_slot0_kernel<<<(unsigned)b2, 256, 0, s>>>(T, x, B, F, d);
            DLRMB_LAUNCH_CHECK();
        }
        return DLRMB_OK;
    }
    // Register-block edge TB and k-split KS.  Measured on B200 (benchmarks/tune_interaction_fwd.py,
    // F = 27, B = 2048): TB = 3 with no k-split is the fastest plan at d = 64 and d = 128 (18.2 us vs
    // 21.4 us for TB = 6 and 20.3-29.8 us for TB = 9; every k-split variant loses to its shuffle
    // reduction), so it is the default; the larger blocks stay selectable for tuning.
    int tb = 3;
    {   // tuning aid: dlrmb_set_option("fwd_tb", v)
        const int v = g_opt.fwd_tb.load(std::memory_order_relaxed);
        if (v == 3 || v == 6 || v == 9) tb = v;
    }
    if (tb == 3) return launch_fwd_tb<3>(T, x, B, F, d, width, out, sm_count, s);
    if (tb == 6) return launch_fwd_tb<6>(T, x, B, F, d, width, out, sm_count, s);
    return launch_fwd_tb<9>(T, x, B, F, d, width, out, sm_count, s);
}

// ------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------
// SCATTER: instead of dT[b][f][:], the gradient row of feature slot f >= 1 is stored at
// dests[f].base + (sample_offset + b) * dests[f].sample_stride + dests[f].offset -- the gradient
// buffer of the rank that owns that table, mapped over NVLink (table-wise sharded embeddings: the
// interaction backward and the gradient all-to-all in one kernel).  Slot 0 (x) only feeds dx.
struct SlotDest {
    float* base;
    long long sample_stride;   // floats between consecutive samples in the destination
    long long offset;          // floats: position of this table inside a destination sample
};

// COLS: column pieces, dests[f * Q + q] for columns [q * d / Q, (q + 1) * d / Q) of slot f (Q = 1 << qlog, d / Q a
// multiple of 4): chunk k goes to piece k / (d / 4Q) at chunk k % (d / 4Q) (column-wise sharded tables).
template <bool SCATTER, bool COLS>
__device__ __forceinline__ void
interaction_bwd_body(const float* __restrict__ dOut, const float* __restrict__ T, int B, int F,
                     int d, int width, float* __restrict__ dT, float* __restrict__ dx, int NS,
                     const SlotDest* __restrict__ dests, long long sample_offset, int qlog) {
    extern __shared__ float4 smem4[];
    const int d4 = d >> 2;
    const int ldt4 = d4 + 1;
    const int Fp = (F + 3) & ~3;   // S rows padded to a float4 multiple
    const int nfb = Fp >> 2;
    float4* Ts = smem4;                                           // [NS][F][ldt4]
    float4* Ss = Ts + (size_t)NS * F * ldt4;                      // [NS][F][Fp/4]
    float* Gs = reinterpret_cast<float*>(Ss + (size_t)NS * F * nfb);  // [NS][width]

    const int tid = threadIdx.x;
    const int s0 = blockIdx.x * NS;
    const int ns = min(NS, B - s0);
    const int npair = F * (F - 1) / 2;

    __shared__ unsigned long long bar;
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_arrive_expect_tx(&bar, (unsigned)(ns * F * d * sizeof(float)));
    }
    __syncthreads();
    // stage T: one TMA bulk copy per feature row into the padded-stride tile
    for (int r = tid; r < ns * F; r += blockDim.x)
        bulk_g2s(Ts + (size_t)r * ldt4, T + ((size_t)s0 * F + r) * d, (unsigned)(d * sizeof(float)), &bar);
    // dOut tile: contiguous but only 4-byte aligned (odd row width) -> coalesced scalar loads
    const float* gg = dOut + (size_t)s0 * width;
    for (int i = tid; i < ns * width; i += blockDim.x) Gs[i] = __ldg(gg + i);
    // pair table m -> (hi, lo), and S zeroed (diagonal and padding columns stay zero)
    unsigned char* pr = reinterpret_cast<unsigned char*>(Gs + (size_t)NS * width);
    for (int m = tid; m < npair; m += blockDim.x) {
        int j = (int)((sqrtf(8.f * m + 1.f) + 1.f) * 0.5f);
        while (j * (j - 1) / 2 > m) --j;
        while ((j + 1) * j / 2 <= m) ++j;
        pr[2 * m] = (unsigned char)j;
        pr[2 * m + 1] = (unsigned char)(m - j * (j - 1) / 2);
    }
    for (int i = tid; i < ns * F * nfb; i += blockDim.x) Ss[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    // S[hi][lo] = S[lo][hi] = g[d + m]
    float* Sf = reinterpret_cast<float*>(Ss);
    for (int i = tid; i < ns * npair; i += blockDim.x) {
        const int s = i / npair, m = i - s * npair;
        const int hi = pr[2 * m], lo = pr[2 * m + 1];
        const float v = Gs[(size_t)s * width + d + m];
        float* Sb = Sf + (size_t)s * F * Fp;
        Sb[hi * Fp + lo] = v;
        Sb[lo * Fp + hi] = v;
    }
    mbar_wait(&bar, 0);
    __syncthreads();

    const int per_sample = nfb * d4;
    for (int task = tid; task < ns * per_sample; task += blockDim.x) {
        const int s = task / per_sample;
        const int rem = task - s * per_sample;
        const int fb = rem / d4;
        const int k = rem - fb * d4;
        const float4* Tp = Ts + (size_t)s * F * ldt4 + k;
        const float4* Sp = Ss + (size_t)s * F * nfb + fb;
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll 3
        for (int j = 0; j < F; ++j) {
            const float4 t = Tp[(size_t)j * ldt4];
            const float4 sv = Sp[(size_t)j * nfb];
            a0.x = fmaf(sv.x, t.x, a0.x); a0.y = fmaf(sv.x, t.y, a0.y); a0.z = fmaf(sv.x, t.z, a0.z); a0.w = fmaf(sv.x, t.w, a0.w);
            a1.x = fmaf(sv.y, t.x, a1.x); a1.y = fmaf(sv.y, t.y, a1.y); a1.z = fmaf(sv.y, t.z, a1.z); a1.w = fmaf(sv.y, t.w, a1.w);
            a2.x = fmaf(sv.z, t.x, a2.x); a2.y = fmaf(sv.z, t.y, a2.y); a2.z = fmaf(sv.z, t.z, a2.z); a2.w = fmaf(sv.z, t.w, a2.w);
            a3.x = fmaf(sv.w, t.x, a3.x); a3.y = fmaf(sv.w, t.y, a3.y); a3.z = fmaf(sv.w, t.z, a3.z); a3.w = fmaf(sv.w, t.w, a3.w);
        }
        const int f0 = fb * 4;
        if (SCATTER && COLS) {
            const float4 av[4] = {a0, a1, a2, a3};
            const int qw = d4 >> qlog;                 // chunks per piece
            const int piece = k / qw, kc = k - piece * qw;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int f = f0 + q;
                if (f >= 1 && f < F) {
                    const SlotDest dd = dests[(f << qlog) + piece];
                    float* row = dd.base + (sample_offset + s0 + s) * dd.sample_stride + dd.offset;
                    reinterpret_cast<float4*>(row)[kc] = av[q];
                }
            }
        } else if (SCATTER) {
            const float4 av[4] = {a0, a1, a2, a3};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int f = f0 + q;
                if (f >= 1 && f < F) {
                    const SlotDest dd = dests[f];
                    float* row = dd.base + (sample_offset + s0 + s) * dd.sample_stride + dd.offset;
                    reinterpret_cast<float4*>(row)[k] = av[q];
                }
            }
        } else {
            float4* o = reinterpret_cast<float4*>(dT + ((size_t)(s0 + s) * F + f0) * d) + k;
            o[0] = a0;
            if (f0 + 1 < F) o[d4] = a1;
            if (f0 + 2 < F) o[2 * d4] = a2;
            if (f0 + 3 < F) o[3 * d4] = a3;
        }
        if (fb == 0) {
            const float* g = Gs + (size_t)s * width + 4 * k;
            float4 r = make_float4(__fadd_rn(g[0], a0.x), __fadd_rn(g[1], a0.y), __fadd_rn(g[2], a0.z), __fadd_rn(g[3], a0.w));
            reinterpret_cast<float4*>(dx + (size_t)(s0 + s) * d)[k] = r;
        }
    }
}

template <bool SCATTER>
__global__ void __launch_bounds__(256)
interaction_bwd_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B, int F,
                       int d, int width, float* __restrict__ dT, float* __restrict__ dx, int NS,
                       const SlotDest* __restrict__ dests, long long sample_offset) {
    interaction_bwd_body<SCATTER, false>(dOut, T, B, F, d, width, dT, dx, NS, dests, sample_offset, 0);
}

__global__ void __launch_bounds__(256)
interaction_bwd_cols_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B, int F, int d, int width,
                            float* __restrict__ dx, int NS, const SlotDest* __restrict__ dests, long long sample_offset,
                            int qlog) {
    interaction_bwd_body<true, true>(dOut, T, B, F, d, width, nullptr, dx, NS, dests, sample_offset, qlog);
}

__global__ void __launch_bounds__(256)
interaction_bwd_generic_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B,
                               int F, int d, int width, float* __restrict__ dT, float* __restrict__ dx) {
    const int64_t total = (int64_t)B * F * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (int64_t)gridDim.x * blockDim.x) {
        int k = (int)(e % d);
        int64_t r = e / d;
        int f = (int)(r % F);
        int64_t b = r / F;
        const float* g = dOut + b * width;
        const float* Tb = T + b * F * d;
        float acc = 0.f;
        for (int j = 0; j < F; ++j) {
            if (j == f) continue;
            int hi = max(j, f), lo = min(j, f);
            acc = fmaf(g[d + hi * (hi - 1) / 2 + lo], Tb[(size_t)j * d + k], acc);
        }
        dT[e] = acc;
        if (f == 0) dx[b * d + k] = __fadd_rn(g[k], acc);
    }
}

// dx alone: dx[b] = dOut[b][:d] + sum_j S[0][j] T[b][j]  (S[0][j] = the gradient of pair (j, 0), j >= 1).
// The sharded step launches it in front of the scattering backward: the bottom MLP's backward only needs
// dx, so it can start while the full pullback is still pushing its 24 MB of gradient rows over NVLink.
// One thread per (sample, 16-byte chunk); terms are accumulated in ascending j with one fused
// multiply-add each -- the order of the full kernels, so the bits agree with their dx.
__global__ void __launch_bounds__(256)
interaction_bwd_dx_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B, int F, int d4, int width,
                          float* __restrict__ dx) {
    const int64_t n = (int64_t)B * d4;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    const int d = d4 * 4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const int64_t b = i / d4;
        const int c = (int)(i - b * d4);
        const float* g = dOut + (size_t)b * width;
        const float4* Tb = reinterpret_cast<const float4*>(T) + (size_t)b * F * d4 + c;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        {   // j = 0: S[0][0] = 0 (kept so that signed zeros match the full kernels)
            const float4 t = __ldg(Tb);
            acc.x = fmaf(0.f, t.x, acc.x); acc.y = fmaf(0.f, t.y, acc.y); acc.z = fmaf(0.f, t.z, acc.z); acc.w = fmaf(0.f, t.w, acc.w);
        }
        for (int j = 1; j < F; ++j) {
            const float sj = __ldg(g + d + j * (j - 1) / 2);
            const float4 t = __ldg(Tb + (size_t)j * d4);
            acc.x = fmaf(sj, t.x, acc.x); acc.y = fmaf(sj, t.y, acc.y); acc.z = fmaf(sj, t.z, acc.z); acc.w = fmaf(sj, t.w, acc.w);
        }
        const float* gx = g + 4 * c;      // row width is odd in general: 4-byte aligned only
        reinterpret_cast<float4*>(dx)[i] = make_float4(__fadd_rn(__ldg(gx), acc.x), __fadd_rn(__ldg(gx + 1), acc.y),
                                                       __fadd_rn(__ldg(gx + 2), acc.z), __fadd_rn(__ldg(gx + 3), acc.w));
    }
}

int launch_interaction_bwd_dx(const float* dOut, const float* T, int B, int F, int d, int pad_to_mul, float* dx,
                              int sm_count, cudaStream_t s) {
    const int width = interaction_width(F, d, pad_to_mul);
    DLRMB_REQUIRE(d % 4 == 0 && (reinterpret_cast<uintptr_t>(T) & 15) == 0 && (reinterpret_cast<uintptr_t>(dx) & 15) == 0,
                  "dlrmb_interaction_bwd_dx needs d %% 4 == 0 and 16-byte aligned T / dx");
    int64_t blocks = ceil_div64((int64_t)B * (d / 4), 256);
    if (blocks > (int64_t)sm_count * 16) blocks = (int64_t)sm_count * 16;
    interaction_bwd_dx_kernel<<<(unsigned)blocks, 256, 0, s>>>(dOut, T, B, F, d / 4, width, dx);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

int launch_interaction_bwd(const float* dOut, const float* T, int B, int F, int d, int pad_to_mul,
                           float* dT, float* dx, int sm_count, cudaStream_t s) {
    return launch_interaction_bwd_ex(dOut, T, B, F, d, pad_to_mul, dT, dx, nullptr, 0, 0, sm_count, s);
}

int launch_interaction_bwd_ex(const float* dOut, const float* T, int B, int F, int d, int pad_to_mul,
                              float* dT, float* dx, const void* dests, long long sample_offset, int qlog,
                              int sm_count, cudaStream_t s) {
    const int width = interaction_width(F, d, pad_to_mul);
    const bool aligned = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(T) & 15) == 0) &&
                         ((reinterpret_cast<uintptr_t>(dT) & 15) == 0) &&
                         ((reinterpret_cast<uintptr_t>(dx) & 15) == 0);
    if (dests != nullptr && !aligned) {
        set_error("the scattered interaction backward needs d % 4 == 0 and 16-byte aligned buffers");
        return DLRMB_EINVAL;
    }
    if (!aligned) {
        int64_t blocks = ceil_div64((int64_t)B * F * d, 256);
        if (blocks > sm_count * 16) blocks = sm_count * 16;
        interaction_bwd_generic_kernel<<<(unsigned)blocks, 256, 0, s>>>(dOut, T, B, F, d, width, dT, dx);
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    }
    {
        int rc = try_interaction_bwd_warp(dOut, T, B, F, d, width, dT, dx, dests, sample_offset, qlog, s);
        if (rc >= 0) return rc;
    }
    const int d4 = d / 4;
    const int Fp = (F + 3) & ~3;
    size_t per_sample = ((size_t)F * (d4 + 1) * 4 + (size_t)F * Fp + width) * sizeof(float);
    TilePlan p = plan_tiles(B, (Fp / 4) * d4, per_sample, (size_t)F * (F - 1) + 16, sm_count);
    DLRMB_REQUIRE(p.smem <= 200 * 1024, "interaction tile needs %zu bytes of shared memory", p.smem);
    static unsigned long long attr_done = 0;
    static unsigned long long attr_done2 = 0;
    static unsigned long long attr_done3 = 0;
    int rc = (dests && qlog > 0) ? ensure_smem_attr((const void*)interaction_bwd_cols_kernel, 200 * 1024, &attr_done3)
             : dests             ? ensure_smem_attr((const void*)interaction_bwd_kernel<true>, 200 * 1024, &attr_done2)
                                 : ensure_smem_attr((const void*)interaction_bwd_kernel<false>, 200 * 1024, &attr_done);
    if (rc) return rc;
    int grid = (B + p.ns - 1) / p.ns;
    if (dests && qlog > 0)
        interaction_bwd_cols_kernel<<<grid, p.threads, p.smem, s>>>(dOut, T, B, F, d, width, dx, p.ns,
                                                                     static_cast<const SlotDest*>(dests), sample_offset, qlog);
    else if (dests)
        interaction_bwd_kernel<true><<<grid, p.threads, p.smem, s>>>(dOut, T, B, F, d, width, dT, dx, p.ns,
                                                                      static_cast<const SlotDest*>(dests), sample_offset);
    else
        interaction_bwd_kernel<false><<<grid, p.threads, p.smem, s>>>(dOut, T, B, F, d, width, dT, dx, p.ns, nullptr, 0);
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

}  // namespace dlrmb
