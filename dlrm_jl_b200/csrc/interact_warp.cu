// Dot-product feature interaction for the DLRM shapes: one WARP per sample, packed FP32 FMAs.
//
// Same contract as interact.cu (DLRM.jl src/model/interact.jl:394-411 forward, :424-436 and
// :469-489 backward), specialised at compile time for the (F, d) pairs the Criteo models use so
// every loop bound and shared-memory offset is an immediate.  What the tiled kernels of interact.cu
// lose at DLRM batch sizes -- CTA-wide barriers between load / compute / store phases, a shared-
// memory pipe saturated by 3x3 register blocks, and an issue stream that is half address
// arithmetic -- is what this design removes:
//
//   * a warp owns its samples from first load to last store; there is no __syncthreads and a CTA is
//     only a container of independent warps, so the warps of an SM drift into different phases and
//     the DRAM stream, the FMA pipe and the store stream overlap;
//   * all FMAs are FFMA2 (PTX fma.rn.f32x2, sm_100+): two IEEE fp32 FMAs per issue slot, operands
//     taken as the natural 64-bit halves of 128-bit loads;
//   * backward, d = 128 (interaction_bwd_ring2_kernel, the default): output-stationary and streaming -- the warp
//     keeps the accumulators of about half of the output rows and streams the rows of T through a ring in shared
//     memory filled by cp.async, consuming row j while the next twelve are in flight; S is stored once and an FFMA2
//     computes the same column of two output rows with the streamed T value as its SCALAR operand (the hardware
//     broadcasts it).  Other geometries and the peer-store epilogue (interaction_bwd_warp_kernel): a lane keeps its
//     float4 column slice of ALL F rows of T in registers (F LDG.128 in flight per lane, no shared-memory staging
//     of T at all); S in shared memory, stored once, one broadcast load of two S values feeding four FFMA2 (scalar
//     operand again).  The per-output summation order (j ascending, one fused multiply-add per term) is the tiled
//     kernel's in all of them, so they produce the same bits.  (Round 1 duplicated every S entry in shared memory
//     to build the (s, s) pair fma.rn.f32x2 asks for; ptxas folds that pair into FFMA2's scalar operand, so the
//     duplicate was never needed.  Measured and not kept in round 2: S stored once with the FFMA2 halves carrying
//     two different j -- F*d/2 register moves per sample: 23.8 vs 16.2 us at B = 2048;
//     profiles/r02_interaction_variants.txt, r02_bwd_variants.txt.)
//   * forward: T rows arrive by TMA bulk copies (cp.async.bulk, one per row, one mbarrier per
//     warp) at bank-staggered row addresses and the Gram matrix is computed on the tensor cores in
//     3xTF32 form (see interaction_fwd_mma_kernel); the sample's output row is assembled in the dead
//     part of the tile and leaves as one contiguous coalesced range.  (The FP32 FFMA2 forward of
//     round 1 was bound by the shared-memory -> register path and has been removed.)
#include "common.cuh"

namespace dlrmb {

namespace {

__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// d = a * b + c on both halves (two independent round-to-nearest fp32 FMAs; SASS FFMA2)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra, rb, rc, rd;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
}

struct SlotDestW {   // same layout as SlotDest in interact.cu / dlrmb_slot_dest
    float* base;
    long long sample_stride;
    long long offset;
};

// ------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------
// flat pair index m = hi(hi-1)/2 + lo  ->  (hi << 8) | lo, for hi < 32 (constant-initialised)
struct PairTable {
    unsigned short v[496];
    constexpr PairTable() : v() {
        int m = 0;
        for (int hi = 1; hi < 32; ++hi)
            for (int lo = 0; lo < hi; ++lo) v[m++] = (unsigned short)((hi << 8) | lo);
    }
};
__device__ const PairTable kPairTable{};

template <int F, int D, int VAR = 0>
struct BwdGeom {
    static constexpr int LPS = D / 4;            // lanes per sample (one float4 of k each)
    static constexpr int LPS_LOG2 = LPS >= 32 ? 5 : LPS >= 16 ? 4 : LPS >= 8 ? 3 : LPS >= 4 ? 2 : LPS >= 2 ? 1 : 0;
    static constexpr int SPW = 32 / LPS;         // samples per warp
    static constexpr int FP2 = (F + 1) & ~1;     // S row length, even
    static constexpr int NPAIR = F * (F - 1) / 2;
    static constexpr int NI = (NPAIR + 31) / 32; // pair entries per lane
    static constexpr int SSTRIDE_DUP = F * FP2 * 2 + 4;   // floats per sample of duplicated S (+16 B bank stagger)
    static constexpr int NF0 = (F % 3 == 0) ? 3 : ((F % 2 == 0) ? 2 : 1);
    // Variants of this kernel for one sample per warp (d = 128), selected by `bwd_variant` (the default is the streaming
    // kernel further down; B = 2048 / 16384, cold inputs, profiles/r02_bwd_variants.txt):
    //   VAR 0  FFMA2, S duplicated in shared memory, NF0 output rows per pass, 144 registers (the round-1 kernel; also
    //          every geometry with several samples per warp): 18.0 / 100 us.
    //   VAR 1  the same at 128 registers with nine rows per pass (the compiler walks them one after another, nothing
    //          spills): 8 CTAs fit per SM -- registers are allocated per SM sub-partition (16384 each), so a 32-thread
    //          warp at 144 or 168 registers leaves room for 3 warps per sub-partition = 6 CTAs per SM, and 2048 samples
    //          (1024 CTAs) were 888 CTAs + a second wave of 136 that started when the first ended (per-CTA %globaltimer
    //          stamps, benchmarks/cta_timeline.py: 13 % of the CTAs entered 12 us late).  One wave: 16.2 us, but 105 us
    //          at B = 16384 (many waves either way).
    //   VAR 2  S stored ONCE: FFMA2 takes a scalar operand for both halves (SASS `FFMA2 Rd, Ra.F32, Rb.F32x2, Rc`), so
    //          the duplicate only ever existed to please the PTX form fma.rn.f32x2 -- ptxas folds the pair (s, s) into
    //          the scalar form.  Half the shared-memory loads per FMA: 14.9 / 84 us (0.64 / 0.91 of the HBM peak).  Also
    //          the kernel behind the peer-store epilogue (168 registers).
    // Same products in the same order in all of them: same bits (tests/test_gpu_parity.py).  Measured and not kept:
    // FFMA2 at 128 registers with NF0 rows (84 bytes of spills) or one row per pass, scalar FFMA instead of FFMA2 for
    // VAR 2 (17.0 / 93 us: twice the issue slots).
    static constexpr int NF = (VAR == 1 && F % 9 == 0) ? 9 : NF0;
    static constexpr bool DUP = (VAR == 1) || (VAR == 0 && SPW == 1);   // several samples per warp: S stored once as well
    static constexpr int SSTRIDE = DUP ? SSTRIDE_DUP : F * FP2 + 4;
    static constexpr int WARPS = 2;
    static constexpr int max_regs(bool scatter) { return (SPW == 1 && !scatter) ? (VAR == 1 ? 128 : 144) : 168; }
    static constexpr size_t smem_bytes() { return (size_t)WARPS * SPW * SSTRIDE * 4; }
    static_assert(F <= 32, "pair table covers F <= 32");
};

// COLS: the scatter destinations are column pieces, dests[f * Q + q] for columns [q * D / Q, (q + 1) * D / Q) of
// slot f (Q = 1 << qlog, D / Q a multiple of 4): lane kl stores its float4 into piece kl / (LPS / Q) at chunk
// kl % (LPS / Q) (column-wise sharded tables).
template <int F, int D, bool SCATTER, int VAR, bool COLS = false>
__global__ void __launch_bounds__(BwdGeom<F, D, VAR>::WARPS * 32) __maxnreg__((BwdGeom<F, D, VAR>::max_regs(SCATTER)))
interaction_bwd_warp_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B, int width,
                            float* __restrict__ dT, float* __restrict__ dx,
                            const SlotDestW* __restrict__ dests, long long sample_offset, unsigned long long* clk,
                            int qlog = 0) {
    using G = BwdGeom<F, D, VAR>;
    extern __shared__ float4 smem4[];
    clock_in(clk, blockIdx.x);
    float* Sd = reinterpret_cast<float*>(smem4);                                   // [WARPS][SPW][SSTRIDE]

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long group = (long long)blockIdx.x * G::WARPS + warp;     // SPW consecutive samples
    if (group * G::SPW >= B) {                                           // warp-uniform
        clock_out(clk, blockIdx.x);
        return;
    }
    const int sub = lane / G::LPS;
    const int kl = lane - sub * G::LPS;
    const long long b = group * G::SPW + sub;
    const bool valid = b < B;

    // the lane's share of the pair table and of the first sample's pair gradients: issued first so
    // that their latency hides behind the T loads
    unsigned short pv[G::NI];
    float gv[G::NI];
    {
        const float* gp = dOut + (size_t)(group * G::SPW) * width + D;
#pragma unroll
        for (int i = 0; i < G::NI; ++i) {
            const int m = lane + 32 * i;
            pv[i] = kPairTable.v[m < G::NPAIR ? m : 0];
            gv[i] = (m < G::NPAIR) ? __ldg(gp + m) : 0.f;
        }
    }

    // T column slices: F independent 16-byte loads per lane
    float4 t[F];
    {
        const float4* Tp = reinterpret_cast<const float4*>(T) + (size_t)(valid ? b : 0) * F * G::LPS + kl;
#pragma unroll
        for (int j = 0; j < F; ++j) t[j] = valid ? __ldg(Tp + (size_t)j * G::LPS) : make_float4(0.f, 0.f, 0.f, 0.f);
    }

    // duplicated S of the warp's samples: Sd[s][f][j] = (S[j][f], S[j][f]), zero diagonal / padding
    float* Sw = Sd + (size_t)warp * G::SPW * G::SSTRIDE;
#pragma unroll 1
    for (int s2 = 0; s2 < G::SPW; ++s2) {
        const long long bb = group * G::SPW + s2;
        if (bb >= B) break;                                  // warp-uniform
        float2* Sb = reinterpret_cast<float2*>(Sw + (size_t)s2 * G::SSTRIDE);
        float* Sb1 = Sw + (size_t)s2 * G::SSTRIDE;
        if (s2 > 0) {
            const float* gp = dOut + (size_t)bb * width + D;
#pragma unroll
            for (int i = 0; i < G::NI; ++i) {
                const int m = lane + 32 * i;
                gv[i] = (m < G::NPAIR) ? __ldg(gp + m) : 0.f;
            }
        }
#pragma unroll
        for (int i = 0; i < G::NI; ++i) {
            if (lane + 32 * i < G::NPAIR) {
                const int hi = pv[i] >> 8, lo = pv[i] & 0xff;
                if (G::DUP) {
                    Sb[hi * G::FP2 + lo] = make_float2(gv[i], gv[i]);
                    Sb[lo * G::FP2 + hi] = make_float2(gv[i], gv[i]);
                } else {
                    Sb1[hi * G::FP2 + lo] = gv[i];
                    Sb1[lo * G::FP2 + hi] = gv[i];
                }
            }
        }
        for (int f = lane; f < F; f += 32) {
            if (G::DUP) {
                Sb[f * G::FP2 + f] = make_float2(0.f, 0.f);
                if (G::FP2 > F) Sb[f * G::FP2 + F] = make_float2(0.f, 0.f);
            } else {
                Sb1[f * G::FP2 + f] = 0.f;
                if (G::FP2 > F) Sb1[f * G::FP2 + F] = 0.f;
            }
        }
    }
    __syncwarp();
    if (!valid) {
        clock_out(clk, blockIdx.x);
        return;
    }

    const float* Srow = Sw + (size_t)sub * G::SSTRIDE;
    const float* gb = dOut + (size_t)b * width;
#pragma unroll 1
    for (int f0 = 0; f0 < F; f0 += G::NF) {
        float2 lo2[G::NF], hi2[G::NF];
#pragma unroll
        for (int q = 0; q < G::NF; ++q) lo2[q] = hi2[q] = make_float2(0.f, 0.f);
        if (G::DUP) {
#pragma unroll
            for (int jp = 0; jp < G::FP2 / 2; ++jp) {
#pragma unroll
                for (int q = 0; q < G::NF; ++q) {
                    const float4 sv = *reinterpret_cast<const float4*>(Srow + ((f0 + q) * G::FP2 + 2 * jp) * 2);
                    lo2[q] = ffma2(make_float2(sv.x, sv.y), make_float2(t[2 * jp].x, t[2 * jp].y), lo2[q]);
                    hi2[q] = ffma2(make_float2(sv.x, sv.y), make_float2(t[2 * jp].z, t[2 * jp].w), hi2[q]);
                    if (2 * jp + 1 < F) {
                        lo2[q] = ffma2(make_float2(sv.z, sv.w), make_float2(t[2 * jp + 1].x, t[2 * jp + 1].y), lo2[q]);
                        hi2[q] = ffma2(make_float2(sv.z, sv.w), make_float2(t[2 * jp + 1].z, t[2 * jp + 1].w), hi2[q]);
                    }
                }
            }
        } else {
            // S[f][j] once: FFMA2 takes a scalar operand for both halves (SASS `FFMA2 Rd, Ra.F32, Rb.F32x2, Rc`; ptxas
            // emits it for the pair (s, s)), so a 64-bit broadcast load of two S values feeds four FFMA2 and nothing in
            // shared memory is duplicated (the S row pitch FP2 is even: the pair (2 jp, 2 jp + 1) is 8-byte aligned)
#pragma unroll
            for (int jp = 0; jp < G::FP2 / 2; ++jp) {
#pragma unroll
                for (int q = 0; q < G::NF; ++q) {
                    const float2 sv = *reinterpret_cast<const float2*>(Srow + (f0 + q) * G::FP2 + 2 * jp);
                    lo2[q] = ffma2(make_float2(sv.x, sv.x), make_float2(t[2 * jp].x, t[2 * jp].y), lo2[q]);
                    hi2[q] = ffma2(make_float2(sv.x, sv.x), make_float2(t[2 * jp].z, t[2 * jp].w), hi2[q]);
                    if (2 * jp + 1 < F) {
                        lo2[q] = ffma2(make_float2(sv.y, sv.y), make_float2(t[2 * jp + 1].x, t[2 * jp + 1].y), lo2[q]);
                        hi2[q] = ffma2(make_float2(sv.y, sv.y), make_float2(t[2 * jp + 1].z, t[2 * jp + 1].w), hi2[q]);
                    }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < G::NF; ++q) {
            const int f = f0 + q;
            const float4 r = make_float4(lo2[q].x, lo2[q].y, hi2[q].x, hi2[q].y);
            if (SCATTER && COLS) {
                if (f >= 1) {
                    const int lqlog = G::LPS_LOG2 - qlog;     // lanes per piece: 1 << lqlog
                    const SlotDestW dd = dests[(f << qlog) + (kl >> lqlog)];
                    float* row = dd.base + (sample_offset + b) * dd.sample_stride + dd.offset;
                    reinterpret_cast<float4*>(row)[kl & ((1 << lqlog) - 1)] = r;
                }
            } else if (SCATTER) {
                if (f >= 1) {
                    const SlotDestW dd = dests[f];
                    float* row = dd.base + (sample_offset + b) * dd.sample_stride + dd.offset;
                    reinterpret_cast<float4*>(row)[kl] = r;
                }
            } else {
                reinterpret_cast<float4*>(dT)[((size_t)b * F + f) * G::LPS + kl] = r;
            }
            if (f == 0) {
                const float* g = gb + 4 * kl;    // row width is odd in general: 4-byte aligned only
                reinterpret_cast<float4*>(dx)[(size_t)b * G::LPS + kl] =
                    make_float4(__fadd_rn(__ldg(g), r.x), __fadd_rn(__ldg(g + 1), r.y),
                                __fadd_rn(__ldg(g + 2), r.z), __fadd_rn(__ldg(g + 3), r.w));
            }
        }
    }
    clock_out(clk, blockIdx.x);
}

// ------------------------------------------------------------------------------------------
// forward on the tensor cores: 3xTF32 (error-compensated) warp-level MMA
// ------------------------------------------------------------------------------------------
// An FP32-FMA forward is bound by the shared-memory -> register path: a 4 x 4 register block
// reads 8 floats per 16 FMAs, and that path delivers 32 floats per clock per SM against 128 FMAs per
// clock (ncu: 1,090 shared wavefronts per sample, 7 us of shared-memory pipe per SM at B = 2048,
// above the 5 us the HBM traffic takes).  The k-reduction is what the tensor core does internally,
// so here a warp computes its sample's Gram matrix with mma.sync.m16n8k8 TF32 MMAs: every operand
// fragment of a k-step -- A and B are both rows of T -- comes from 2 * ceil(F / 8) conflict-free
// 32-bit loads (128 wavefronts per sample), and fp32 accuracy is kept by splitting each operand into
// a TF32 head and a TF32 tail and accumulating  a_lo*b_hi + a_hi*b_lo + a_hi*b_hi  in fp32 (the
// dropped a_lo*b_lo term is 2^-20 relative).  Integer-valued inputs stay exact.  Measured against a
// float64 Gram matrix (benchmarks/fwd_accuracy.py, B = 2048, F = 27, d = 128): relative L2 error
// 1.2e-6 (0.15e-6 for the FP32-FMA kernels), tolerance 1e-5.
template <int F, int D>
struct MmaGeom {
    static constexpr int LDF = D + 4;                  // row pitch in floats: (D + 4) / 4 is odd, so the 8 rows x 4 k of a
                                                       // fragment load fall into 32 different banks
    static constexpr int MT = (F + 15) / 16;           // 16-row tiles (M)
    static constexpr int RBP = 2 * MT;                 // 8-row blocks loaded per k-step
    static constexpr int NT = (F + 7) / 8;             // 8-column tiles (N)
    static constexpr int NPAIR = F * (F - 1) / 2;
    // (Measured and not kept: 2 or 4 feature rows per TMA bulk copy with the bank stagger after every 2 / 4 rows --
    // 12.0 us either way at B = 2048, so the forward is not bound by the number of bulk requests.)
    static __host__ __device__ constexpr int roff(int r) { return r * LDF; }
    static constexpr int SSZ = F * LDF;                // floats per sample
    static constexpr int OS_OFF = LDF;                 // output staging starts behind row 0
    static constexpr int WARPS = 2;
    // The last 8-column tile of the last 16-row tile holds only the pairs among the rows past 8 * (NT - 1): three
    // of its 128 entries at F = 27 (rows 24..26), a sixth of the sample's MMAs.  When there are at most three such
    // pairs they are plain FP32 dot products over the warp's lanes instead, and that tile is never issued.
    static constexpr int TAIL0 = 8 * (NT - 1);         // first row of the tail block
    static constexpr int TAILR = F - TAIL0;            // rows in it (1..8)
    static constexpr bool TAIL_FMA = (NT > 1) && (NT == 2 * MT) && (TAILR <= 3);
    static constexpr int TAILP = TAIL_FMA ? TAILR * (TAILR - 1) / 2 : 0;
    static __host__ __device__ constexpr bool tile_used(int i, int j) {
        return j <= 2 * i + 1 && !(TAIL_FMA && i == MT - 1 && j == NT - 1);
    }
    static constexpr size_t smem_bytes() { return (size_t)WARPS * SSZ * 4 + (size_t)WARPS * 8; }
    static_assert(F <= 32 && D % 8 == 0, "one warp covers F <= 32 rows; k-steps of 8");
    static_assert(((D + 4) / 4) % 2 == 1, "row pitch must stagger the banks");
    static_assert(NPAIR <= SSZ - OS_OFF || F == 1, "output staging must fit behind row 0");
};

__device__ __forceinline__ void mma_tf32(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// FP32 dot products of the tail block's row pairs over k in [kbeg, kend): lane-strided partial sums, then an
// xor-tree over the warp; every lane returns the totals.  Pair order: (r0+1, r0), (r0+2, r0), (r0+2, r0+1).
template <typename G>
__device__ __forceinline__ void tail_pairs_fma(const float* Ts, int lane, int kbeg, int kend, float (&tp)[3]) {
    tp[0] = tp[1] = tp[2] = 0.f;
    if (G::TAILP == 0) return;
    for (int k = kbeg + lane; k < kend; k += 32) {
        const float a = Ts[G::roff(G::TAIL0) + k], b = Ts[G::roff(G::TAIL0 + 1) + k];
        tp[0] = fmaf(b, a, tp[0]);
        if (G::TAILR == 3) {
            const float c = Ts[G::roff(G::TAIL0 + 2) + k];
            tp[1] = fmaf(c, a, tp[1]);
            tp[2] = fmaf(c, b, tp[2]);
        }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        if (q >= G::TAILP) break;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) tp[q] += __shfl_xor_sync(0xffffffffu, tp[q], off);
    }
}

// where the tail pairs go in the staged output row: pair (row, col) sits at row * (row - 1) / 2 + col
template <typename G>
__device__ __forceinline__ void tail_pairs_store(float* Os, int lane, const float (&tp)[3]) {
    if (G::TAILP == 0) return;
    constexpr int r1 = G::TAIL0 + 1, r2 = G::TAIL0 + 2;
    if (lane == 0) Os[r1 * (r1 - 1) / 2 + G::TAIL0] = tp[0];
    if (G::TAILR == 3) {
        if (lane == 1) Os[r2 * (r2 - 1) / 2 + G::TAIL0] = tp[1];
        if (lane == 2) Os[r2 * (r2 - 1) / 2 + G::TAIL0 + 1] = tp[2];
    }
}

template <int F, int D>
__global__ void __launch_bounds__(MmaGeom<F, D>::WARPS * 32)
interaction_fwd_mma_kernel(float* __restrict__ T, const float* __restrict__ x, int B, int width,
                           float* __restrict__ out, unsigned long long* clk) {
    using G = MmaGeom<F, D>;
    extern __shared__ float4 smem4[];
    clock_in(clk, blockIdx.x);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float* Ts = reinterpret_cast<float*>(smem4) + (size_t)warp * G::SSZ;
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(reinterpret_cast<float*>(smem4) + (size_t)G::WARPS * G::SSZ) + warp;

    const long long b = (long long)blockIdx.x * G::WARPS + warp;     // the warp's sample
    if (b >= B) {
        clock_out(clk, blockIdx.x);
        return;
    }

    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
                     ::"r"(smem_addr(bar)), "r"((unsigned)(F * D * sizeof(float))) : "memory");
    }
    __syncwarp();
    if (lane < F) {   // one TMA bulk copy per feature row (slot 0 from x when it is handed separately)
        const float* src = (x != nullptr && lane == 0) ? x + (size_t)b * D : T + ((size_t)b * F + lane) * D;
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                     ::"r"(smem_addr(Ts + lane * G::LDF)), "l"(src), "r"((unsigned)(D * sizeof(float))), "r"(smem_addr(bar))
                     : "memory");
    }

    const int g = lane >> 2, t = lane & 3;
    int roff[G::RBP];
#pragma unroll
    for (int rb = 0; rb < G::RBP; ++rb) roff[rb] = min(8 * rb + g, F - 1) * G::LDF + t;   // clamped rows are discarded below

    float acc[G::MT][G::NT][4];
#pragma unroll
    for (int i = 0; i < G::MT; ++i)
#pragma unroll
        for (int j = 0; j < G::NT; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;

    {   // wait for the tile
        unsigned done = 0;
        while (!done) {
            asm volatile(
                "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                : "=r"(done) : "r"(smem_addr(bar)), "r"(0) : "memory");
        }
    }
    if (x != nullptr) {   // fused fast_vcat: x also becomes slot 0 of T in global memory
        for (int c = lane; c < D / 4; c += 32)
            reinterpret_cast<float4*>(T + (size_t)b * F * D)[c] = reinterpret_cast<const float4*>(Ts)[c];
    }

#pragma unroll 2
    for (int k0 = 0; k0 < D; k0 += 8) {
        unsigned hi[G::RBP][2], lo[G::RBP][2];
#pragma unroll
        for (int rb = 0; rb < G::RBP; ++rb)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                // head = v truncated to TF32 (10 mantissa bits), tail = the exact remainder v - head
                // truncated to TF32: |v - head - tail| < 2^-20 |v|.  Rounding both to nearest instead
                // was measured: rel. L2 error 0.91e-6 instead of 1.24e-6 (the MMA's own fp32
                // accumulation dominates), 6 % slower at B = 16384 -- not taken.
                const float v = Ts[roff[rb] + k0 + 4 * h];
                const unsigned vh = __float_as_uint(v) & 0xffffe000u;
                hi[rb][h] = vh;
                lo[rb][h] = __float_as_uint(v - __uint_as_float(vh)) & 0xffffe000u;
            }
#pragma unroll
        for (int i = 0; i < G::MT; ++i) {
            const unsigned ah[4] = {hi[2 * i][0], hi[2 * i + 1][0], hi[2 * i][1], hi[2 * i + 1][1]};
            const unsigned al[4] = {lo[2 * i][0], lo[2 * i + 1][0], lo[2 * i][1], lo[2 * i + 1][1]};
#pragma unroll
            for (int j = 0; j < G::NT; ++j) {
                if (!G::tile_used(i, j)) continue;      // tile entirely above the diagonal, or the tail tile
                // small terms first.  (Measured and not taken: issuing the three passes tile-
                // interleaved so that no MMA waits for its predecessor, 14.3 vs 13.8 us at B = 2048;
                // delivering the tile as two column halves on two mbarriers so that the first half's
                // MMAs overlap the second half's loads, 13.5 vs 13.9 us at B = 2048 but 63 vs 59.5 us
                // at B = 16384.)
                mma_tf32(acc[i][j], al, hi[j][0], hi[j][1]);
                mma_tf32(acc[i][j], ah, lo[j][0], lo[j][1]);
                mma_tf32(acc[i][j], ah, hi[j][0], hi[j][1]);
            }
        }
    }
    float tp[3];
    tail_pairs_fma<G>(Ts, lane, 0, D, tp);
    __syncwarp();   // every lane is done reading rows >= 1: their space becomes the output staging

    float* Os = Ts + G::LDF;   // pair m at Os[m]; row 0 (x) stays at Ts[0, D)
#pragma unroll
    for (int i = 0; i < G::MT; ++i)
#pragma unroll
        for (int j = 0; j < G::NT; ++j) {
            if (!G::tile_used(i, j)) continue;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int row = 16 * i + g + ((e & 2) ? 8 : 0);
                const int col = 8 * j + 2 * t + (e & 1);
                if (col < row && row < F) Os[row * (row - 1) / 2 + col] = acc[i][j][e];
            }
        }
    tail_pairs_store<G>(Os, lane, tp);
    __syncwarp();

    float* og = out + (size_t)b * width;
    for (int c = lane; c < D; c += 32) og[c] = Ts[c];
    for (int c = lane; c < G::NPAIR; c += 32) og[D + c] = Os[c];
    for (int c = D + G::NPAIR + lane; c < width; c += 32) og[c] = 0.f;   // pad_to_mul padding
    clock_out(clk, blockIdx.x);
}

// Two warps per sample, for batches that are a single wave of the kernel above (B <= 4096 at d >= 64): the
// CTA (64 threads) owns ONE sample, warp h contracts the k range [h * D/2, (h+1) * D/2) of the same shared
// tile, warp 1 hands its partial accumulators to warp 0 through the dead part of the tile.  At one sample
// per warp the MMA phase is a dependent chain per accumulator tile on 14 warps per SM (tensor pipe 36 %
// active, ncu); splitting k halves that chain and doubles the warps that feed the pipe, for three
// 64-thread barriers and 3 KB of shared traffic.  At large batches (several waves, the load of one
// sample overlapping the MMAs of another) the one-warp kernel is the faster one and stays in charge.
template <int F, int D>
__global__ void __launch_bounds__(64)
interaction_fwd_mma_ksplit_kernel(float* __restrict__ T, const float* __restrict__ x, int B, int width,
                                  float* __restrict__ out, unsigned long long* clk) {
    using G = MmaGeom<F, D>;
    extern __shared__ float4 smem4[];
    clock_in(clk, blockIdx.x);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float* Ts = reinterpret_cast<float*>(smem4);
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(Ts + G::SSZ);
    const long long b = blockIdx.x;          // grid = B

    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
                     ::"r"(smem_addr(bar)), "r"((unsigned)(F * D * sizeof(float))) : "memory");
    }
    __syncthreads();
    if (warp == 0 && lane < F) {   // one TMA bulk copy per feature row (slot 0 from x when it is handed separately)
        const float* src = (x != nullptr && lane == 0) ? x + (size_t)b * D : T + ((size_t)b * F + lane) * D;
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                     ::"r"(smem_addr(Ts + lane * G::LDF)), "l"(src), "r"((unsigned)(D * sizeof(float))), "r"(smem_addr(bar))
                     : "memory");
    }

    const int g = lane >> 2, t = lane & 3;
    int roff[G::RBP];
#pragma unroll
    for (int rb = 0; rb < G::RBP; ++rb) roff[rb] = G::roff(min(8 * rb + g, F - 1)) + t;   // clamped rows are discarded below

    float acc[G::MT][G::NT][4];
#pragma unroll
    for (int i = 0; i < G::MT; ++i)
#pragma unroll
        for (int j = 0; j < G::NT; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;

    {   // wait for the tile (both warps poll the same barrier)
        unsigned done = 0;
        while (!done) {
            asm volatile(
                "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                : "=r"(done) : "r"(smem_addr(bar)), "r"(0) : "memory");
        }
    }
    if (x != nullptr && warp == 1) {   // fused fast_vcat: x also becomes slot 0 of T in global memory
        for (int c = lane; c < D / 4; c += 32)
            reinterpret_cast<float4*>(T + (size_t)b * F * D)[c] = reinterpret_cast<const float4*>(Ts)[c];
    }

    const int kbeg = warp * (D / 2);
#pragma unroll 2
    for (int k0 = kbeg; k0 < kbeg + D / 2; k0 += 8) {
        unsigned hi[G::RBP][2], lo[G::RBP][2];
#pragma unroll
        for (int rb = 0; rb < G::RBP; ++rb)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float v = Ts[roff[rb] + k0 + 4 * h];
                const unsigned vh = __float_as_uint(v) & 0xffffe000u;
                hi[rb][h] = vh;
                lo[rb][h] = __float_as_uint(v - __uint_as_float(vh)) & 0xffffe000u;
            }
#pragma unroll
        for (int i = 0; i < G::MT; ++i) {
            const unsigned ah[4] = {hi[2 * i][0], hi[2 * i + 1][0], hi[2 * i][1], hi[2 * i + 1][1]};
            const unsigned al[4] = {lo[2 * i][0], lo[2 * i + 1][0], lo[2 * i][1], lo[2 * i + 1][1]};
#pragma unroll
            for (int j = 0; j < G::NT; ++j) {
                if (!G::tile_used(i, j)) continue;      // tile entirely above the diagonal, or the tail tile
                mma_tf32(acc[i][j], al, hi[j][0], hi[j][1]);
                mma_tf32(acc[i][j], ah, lo[j][0], lo[j][1]);
                mma_tf32(acc[i][j], ah, hi[j][0], hi[j][1]);
            }
        }
    }
    float tp[3];
    tail_pairs_fma<G>(Ts, lane, kbeg, kbeg + D / 2, tp);
    __syncthreads();   // both warps are done reading rows >= 1: their space becomes scratch

    float* Os = Ts + G::OS_OFF;               // pair m at Os[m]; row 0 (x) stays at Ts[0, D)
    float* red = Os + ((G::NPAIR + 3) & ~3);  // warp 1's partial accumulators: [tile][e][lane], then its tail pairs
    float* red_tail = red + G::MT * G::NT * 4 * 32;
    static_assert(((G::NPAIR + 3) & ~3) + G::MT * G::NT * 4 * 32 + 4 <= G::SSZ - G::OS_OFF, "scratch must fit behind row 0");
    if (warp == 1) {
#pragma unroll
        for (int i = 0; i < G::MT; ++i)
#pragma unroll
            for (int j = 0; j < G::NT; ++j) {
                if (!G::tile_used(i, j)) continue;
#pragma unroll
                for (int e = 0; e < 4; ++e) red[((i * G::NT + j) * 4 + e) * 32 + lane] = acc[i][j][e];
            }
        if (G::TAILP > 0 && lane == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q)
                if (q < G::TAILP) red_tail[q] = tp[q];
        }
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < G::MT; ++i)
#pragma unroll
            for (int j = 0; j < G::NT; ++j) {
                if (!G::tile_used(i, j)) continue;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float v = acc[i][j][e] + red[((i * G::NT + j) * 4 + e) * 32 + lane];
                    const int row = 16 * i + g + ((e & 2) ? 8 : 0);
                    const int col = 8 * j + 2 * t + (e & 1);
                    if (col < row && row < F) Os[row * (row - 1) / 2 + col] = v;
                }
            }
        if (G::TAILP > 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q)
                if (q < G::TAILP) tp[q] += red_tail[q];
            tail_pairs_store<G>(Os, lane, tp);
        }
    }
    __syncthreads();

    float* og = out + (size_t)b * width;
    for (int c = threadIdx.x; c < D; c += 64) og[c] = Ts[c];
    for (int c = threadIdx.x; c < G::NPAIR; c += 64) og[D + c] = Os[c];
    for (int c = D + G::NPAIR + threadIdx.x; c < width; c += 64) og[c] = 0.f;   // pad_to_mul padding
    clock_out(clk, blockIdx.x);
}

template <int F, int D>
int launch_fwd_mma_ksplit(float* T, const float* x, int B, int width, float* out, cudaStream_t s) {
    using G = MmaGeom<F, D>;
    static unsigned long long attr_done = 0;
    const size_t smem = (size_t)G::SSZ * 4 + 16;
    int rc = ensure_smem_attr((const void*)interaction_fwd_mma_ksplit_kernel<F, D>, (int)smem, &attr_done);
    if (rc) return rc;
    interaction_fwd_mma_ksplit_kernel<F, D><<<(unsigned)B, 64, smem, s>>>(T, x, B, width, out, clock_slot(CLK_IFWD));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <int F, int D>
int launch_fwd_mma(float* T, const float* x, int B, int width, float* out, cudaStream_t s) {
    using G = MmaGeom<F, D>;
    static unsigned long long attr_done = 0;
    const size_t smem = G::smem_bytes();
    int rc = ensure_smem_attr((const void*)interaction_fwd_mma_kernel<F, D>, (int)smem, &attr_done);
    if (rc) return rc;
    const long long grid = ((long long)B + G::WARPS - 1) / G::WARPS;
    interaction_fwd_mma_kernel<F, D><<<(unsigned)grid, G::WARPS * 32, smem, s>>>(T, x, B, width, out, clock_slot(CLK_IFWD));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

template <int F, int D, int VAR>
int launch_bwd_warp_plain(const float* dOut, const float* T, int B, int width, float* dT, float* dx, cudaStream_t s) {
    using G = BwdGeom<F, D, VAR>;
    static unsigned long long attr_done = 0;
    const size_t smem = G::smem_bytes();
    const long long groups = ((long long)B + G::SPW - 1) / G::SPW;
    const long long grid = (groups + G::WARPS - 1) / G::WARPS;
    int rc = ensure_smem_attr((const void*)interaction_bwd_warp_kernel<F, D, false, VAR>, (int)smem, &attr_done);
    if (rc) return rc;
    interaction_bwd_warp_kernel<F, D, false, VAR><<<(unsigned)grid, G::WARPS * 32, smem, s>>>(
        dOut, T, B, width, dT, dx, nullptr, 0, clock_slot(CLK_IBWD));
    DLRMB_LAUNCH_CHECK();
    return DLRMB_OK;
}

// Output-stationary ("streaming") backward for one sample per warp (d = 128): the warp keeps the accumulators of about
// HALF of the output rows and streams the rows of T through a ring, consuming row j (one FMA per output row and
// column, j ascending -- the order of the kernels above, hence the same bits) while the next rows are in flight.
// Two passes over T, the second from L2.  What this buys over interaction_bwd_warp_kernel, whose warps hold ALL of T
// (108 registers) before the first FMA:
//   * 128 registers: 4 warps per SM sub-partition, so 2048 samples are ONE wave of CTAs (8 per SM);
//   * the FMAs of a pass run while its rows arrive, instead of after the last of the 27 loads has landed; the
//     stores of the first half leave while the second pass computes.
// The ring of T rows lives in SHARED memory, filled by asynchronous copies (cp.async: global -> shared without
// passing through registers; a ring in registers was measured first: ptxas spills it to local memory at 128
// registers, 25.8 us against 15.9 us at B = 2048).  Every lane copies and later reads back only its
// own 16-byte column slice, so the only synchronisation is the lane's own cp.async group count.  Registers hold
// the accumulators and little else: nothing spills at 128 registers, and the ring can be RS rows deep.
template <int F, int D, int RS>
struct BwdRingGeom {
    using G = BwdGeom<F, D>;
    static constexpr int RING = RS * D;                               // floats per warp
    static constexpr int PER_WARP = G::SSTRIDE_DUP + RING;            // S (duplicated) + ring; SSTRIDE_DUP * 4 is a multiple of 16
    static constexpr size_t smem_bytes() { return (size_t)G::WARPS * PER_WARP * 4; }
};

__device__ __forceinline__ void cp_async16(float* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_addr(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

template <int F, int D, int F0, int NFH, int RS, int SLOT0, bool REFILL>
__device__ __forceinline__ void bwd_ring_pass(const float4* __restrict__ Tp, float* ring, const float* Srow, int lane,
                                              float2 (&lo)[NFH], float2 (&hi)[NFH]) {
    using G = BwdGeom<F, D>;
#pragma unroll
    for (int q = 0; q < NFH; ++q) lo[q] = hi[q] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < F; ++j) {
        constexpr int dummy = 0;
        (void)dummy;
        const int slot = (SLOT0 + j) % RS;
        cp_async_wait<RS - 1>();                       // all but the RS - 1 youngest groups have landed: row j is here
        const float4 tj = *reinterpret_cast<const float4*>(ring + slot * D + 4 * lane);
#pragma unroll
        for (int q = 0; q < NFH / 2; ++q) {
            const int f = F0 + 2 * q;
            if (f >= F) continue;
            const float4 sv = *reinterpret_cast<const float4*>(Srow + (j * G::FP2 + f) * 2);
            lo[2 * q] = ffma2(make_float2(sv.x, sv.y), make_float2(tj.x, tj.y), lo[2 * q]);
            hi[2 * q] = ffma2(make_float2(sv.x, sv.y), make_float2(tj.z, tj.w), hi[2 * q]);
            if (f + 1 < F) {
                lo[2 * q + 1] = ffma2(make_float2(sv.z, sv.w), make_float2(tj.x, tj.y), lo[2 * q + 1]);
                hi[2 * q + 1] = ffma2(make_float2(sv.z, sv.w), make_float2(tj.z, tj.w), hi[2 * q + 1]);
            }
        }
        // the slot is free (tj is in registers and consumed): the row it holds next; past the end = the next pass
        if (j + RS < F) cp_async16(ring + slot * D + 4 * lane, Tp + (size_t)(j + RS) * G::LPS);
        else if (REFILL) cp_async16(ring + slot * D + 4 * lane, Tp + (size_t)(j + RS - F) * G::LPS);
        cp_async_commit();                             // one group per row consumed, empty at the end of the last pass
    }
}

template <int F, int D, int RS>
__global__ void __launch_bounds__(BwdGeom<F, D>::WARPS * 32, 8)
interaction_bwd_ring_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B, int width,
                            float* __restrict__ dT, float* __restrict__ dx, unsigned long long* clk) {
    using G = BwdGeom<F, D>;
    using RG = BwdRingGeom<F, D, RS>;
    static_assert(G::SPW == 1 && RS <= F, "one sample per warp; the ring is primed with RS rows");
    constexpr int H = G::FP2 / 2;
    static_assert(H % 2 == 0, "two output rows per S load");
    extern __shared__ float4 smem4[];
    clock_in(clk, blockIdx.x);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * G::WARPS + warp;
    if (b >= B) {                             // warp-uniform
        clock_out(clk, blockIdx.x);
        return;
    }
    float* Sw = reinterpret_cast<float*>(smem4) + (size_t)warp * RG::PER_WARP;
    float* ring = Sw + G::SSTRIDE_DUP;
    const float* gb = dOut + (size_t)b * width;
    const float4* Tp = reinterpret_cast<const float4*>(T) + (size_t)b * F * G::LPS + lane;
#pragma unroll
    for (int r = 0; r < RS; ++r) {            // prime the ring: RS rows in flight before anything else
        cp_async16(ring + r * D + 4 * lane, Tp + (size_t)r * G::LPS);
        cp_async_commit();
    }
    {   // duplicated S: Sd[j][f] = (S[j][f], S[j][f]), zero diagonal / padding
        float2* Sb = reinterpret_cast<float2*>(Sw);
#pragma unroll
        for (int i = 0; i < G::NI; ++i) {
            const int m = lane + 32 * i;
            if (m < G::NPAIR) {
                const unsigned short p = kPairTable.v[m];
                const float gvv = __ldg(gb + D + m);
                const int hi = p >> 8, lo = p & 0xff;
                Sb[hi * G::FP2 + lo] = make_float2(gvv, gvv);
                Sb[lo * G::FP2 + hi] = make_float2(gvv, gvv);
            }
        }
        for (int f = lane; f < F; f += 32) {
            Sb[f * G::FP2 + f] = make_float2(0.f, 0.f);
            if (G::FP2 > F) Sb[f * G::FP2 + F] = make_float2(0.f, 0.f);
        }
    }
    __syncwarp();

    float2 lo[H], hi[H];
    float4* dTp = reinterpret_cast<float4*>(dT) + (size_t)b * F * G::LPS + lane;
    bwd_ring_pass<F, D, 0, H, RS, 0, true>(Tp, ring, Sw, lane, lo, hi);
#pragma unroll
    for (int q = 0; q < H; ++q) {
        const float4 r = make_float4(lo[q].x, lo[q].y, hi[q].x, hi[q].y);
        dTp[(size_t)q * G::LPS] = r;
        if (q == 0) {
            const float* g = gb + 4 * lane;    // row width is odd in general: 4-byte aligned only
            reinterpret_cast<float4*>(dx)[(size_t)b * G::LPS + lane] =
                make_float4(__fadd_rn(__ldg(g), r.x), __fadd_rn(__ldg(g + 1), r.y),
                            __fadd_rn(__ldg(g + 2), r.z), __fadd_rn(__ldg(g + 3), r.w));
        }
    }
    bwd_ring_pass<F, D, H, H, RS, F % RS, false>(Tp, ring, Sw, lane, lo, hi);
#pragma unroll
    for (int q = 0; q < H; ++q) {
        if (H + q >= F) continue;
        dTp[(size_t)(H + q) * G::LPS] = make_float4(lo[q].x, lo[q].y, hi[q].x, hi[q].y);
    }
    clock_out(clk, blockIdx.x);
}

// Row-paired form of the ring kernel: an FFMA2 computes the SAME column of TWO output rows,
//     (acc[f][c], acc[f+1][c]) += (S[j][f], S[j][f+1]) * (T[j][c], T[j][c]),
// so S is stored once (consecutive f are consecutive in memory: one LDS.128 = four output rows, no duplicated
// entries) and the broadcast operand is the streamed value of T: FFMA2 takes a scalar for both halves (SASS
// `FFMA2 Rd, Ra.F32x2, Rb.F32, Rc`; ptxas emits it for the pair (t, t)), so nothing is duplicated anywhere.
// 243 instead of 432 shared-memory loads per sample; the same products in the same order (j ascending), hence
// the same bits.
template <int F, int D, int F0, int NFH, int RS, int SLOT0, bool REFILL>
__device__ __forceinline__ void bwd_ring2_pass(const float4* __restrict__ Tp, float* ring, const float* S1, int lane,
                                               float2 (&acc)[NFH / 2][4]) {
    using G = BwdGeom<F, D>;
    constexpr int FP4 = (F + 3) & ~3;
    static_assert(NFH % 4 == 0 && F0 % 4 == 0 && F0 + NFH <= FP4, "four output rows per S load");
#pragma unroll
    for (int p = 0; p < NFH / 2; ++p)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[p][c] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < F; ++j) {
        const int slot = (SLOT0 + j) % RS;
        cp_async_wait<RS - 1>();                       // row j has landed (see bwd_ring_pass)
        const float4 tj = *reinterpret_cast<const float4*>(ring + slot * D + 4 * lane);
        const float2 tx = make_float2(tj.x, tj.x), ty = make_float2(tj.y, tj.y);
        const float2 tz = make_float2(tj.z, tj.z), tw = make_float2(tj.w, tj.w);
#pragma unroll
        for (int q = 0; q < NFH / 4; ++q) {
            const int f = F0 + 4 * q;
            if (f >= F) continue;
            const float4 sv = *reinterpret_cast<const float4*>(S1 + j * FP4 + f);
            const float2 s01 = make_float2(sv.x, sv.y);
            acc[2 * q][0] = ffma2(s01, tx, acc[2 * q][0]);
            acc[2 * q][1] = ffma2(s01, ty, acc[2 * q][1]);
            acc[2 * q][2] = ffma2(s01, tz, acc[2 * q][2]);
            acc[2 * q][3] = ffma2(s01, tw, acc[2 * q][3]);
            if (f + 2 < F) {
                const float2 s23 = make_float2(sv.z, sv.w);
                acc[2 * q + 1][0] = ffma2(s23, tx, acc[2 * q + 1][0]);
                acc[2 * q + 1][1] = ffma2(s23, ty, acc[2 * q + 1][1]);
                acc[2 * q + 1][2] = ffma2(s23, tz, acc[2 * q + 1][2]);
                acc[2 * q + 1][3] = ffma2(s23, tw, acc[2 * q + 1][3]);
            }
        }
        if (j + RS < F) cp_async16(ring + slot * D + 4 * lane, Tp + (size_t)(j + RS) * G::LPS);
        else if (REFILL) cp_async16(ring + slot * D + 4 * lane, Tp + (size_t)(j + RS - F) * G::LPS);
        cp_async_commit();
    }
}

template <int F, int D, int RS>
__global__ void __launch_bounds__(BwdGeom<F, D>::WARPS * 32, 8)
interaction_bwd_ring2_kernel(const float* __restrict__ dOut, const float* __restrict__ T, int B, int width,
                             float* __restrict__ dT, float* __restrict__ dx, unsigned long long* clk) {
    using G = BwdGeom<F, D>;
    static_assert(G::SPW == 1 && RS <= F, "one sample per warp; the ring is primed with RS rows");
    constexpr int FP4 = (F + 3) & ~3;                      // S row pitch
    constexpr int H1 = ((FP4 / 2) + 3) & ~3;               // output rows of the first pass (16 of 27)
    constexpr int H2 = FP4 - H1;                           // second pass, padding rows included (12)
    constexpr int SSZ1 = F * FP4 + 4;                      // floats of S per warp (+16 B: keeps the ring 16-byte aligned)
    constexpr int PER_WARP = SSZ1 + RS * D;
    extern __shared__ float4 smem4[];
    clock_in(clk, blockIdx.x);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * G::WARPS + warp;
    if (b >= B) {                             // warp-uniform
        clock_out(clk, blockIdx.x);
        return;
    }
    float* S1 = reinterpret_cast<float*>(smem4) + (size_t)warp * PER_WARP;
    float* ring = S1 + SSZ1;
    const float* gb = dOut + (size_t)b * width;
    const float4* Tp = reinterpret_cast<const float4*>(T) + (size_t)b * F * G::LPS + lane;
#pragma unroll
    for (int r = 0; r < RS; ++r) {            // prime the ring
        cp_async16(ring + r * D + 4 * lane, Tp + (size_t)r * G::LPS);
        cp_async_commit();
    }
    {   // S1[j][f] = S[j][f], zero diagonal and padding columns
#pragma unroll
        for (int i = 0; i < G::NI; ++i) {
            const int m = lane + 32 * i;
            if (m < G::NPAIR) {
                const unsigned short p = kPairTable.v[m];
                const float gvv = __ldg(gb + D + m);
                const int hi = p >> 8, lo = p & 0xff;
                S1[hi * FP4 + lo] = gvv;
                S1[lo * FP4 + hi] = gvv;
            }
        }
        for (int f = lane; f < F; f += 32) {
            S1[f * FP4 + f] = 0.f;
#pragma unroll
            for (int c = F; c < FP4; ++c) S1[f * FP4 + c] = 0.f;
        }
    }
    __syncwarp();

    float4* dTp = reinterpret_cast<float4*>(dT) + (size_t)b * F * G::LPS + lane;
    {
        float2 acc[H1 / 2][4];
        bwd_ring2_pass<F, D, 0, H1, RS, 0, true>(Tp, ring, S1, lane, acc);
#pragma unroll
        for (int p = 0; p < H1 / 2; ++p) {
            const float4 r0 = make_float4(acc[p][0].x, acc[p][1].x, acc[p][2].x, acc[p][3].x);
            const float4 r1 = make_float4(acc[p][0].y, acc[p][1].y, acc[p][2].y, acc[p][3].y);
            if (2 * p < F) dTp[(size_t)(2 * p) * G::LPS] = r0;
            if (2 * p + 1 < F) dTp[(size_t)(2 * p + 1) * G::LPS] = r1;
            if (p == 0) {
                const float* g = gb + 4 * lane;    // row width is odd in general: 4-byte aligned only
                reinterpret_cast<float4*>(dx)[(size_t)b * G::LPS + lane] =
                    make_float4(__fadd_rn(__ldg(g), r0.x), __fadd_rn(__ldg(g + 1), r0.y),
                                __fadd_rn(__ldg(g + 2), r0.z), __fadd_rn(__ldg(g + 3), r0.w));
            }
        }
    }
    {
        float2 acc[H2 / 2][4];
        bwd_ring2_pass<F, D, H1, H2, RS, F % RS, false>(Tp, ring, S1, lane, acc);
#pragma unroll
        for (int p = 0; p < H2 / 2; ++p) {
            const int f = H1 + 2 * p;
            if (f < F) dTp[(size_t)f * G::LPS] = make_float4(acc[p][0].x, acc[p][1].x, acc[p][2].x, acc[p][3].x);
            if (f + 1 < F) dTp[(size_t)(f + 1) * G::LPS] = make_float4(acc[p][0].y, acc[p][1].y, acc[p][2].y, acc[p][3].y);
        }
    }
    clock_out(clk, blockIdx.x);
}

template <int F, int D>
int launch_bwd_ring2(const float* dOut, const float* T, int B, int width, float* dT, float* dx, cudaStream_t s) {
    using G = BwdGeom<F, D>;
    if constexpr (G::SPW == 1 && F >= 12) {
        constexpr int RS = 12;
        constexpr int FP4 = (F + 3) & ~3;
        static unsigned long long attr_done = 0;
        const size_t smem = (size_t)G::WARPS * (F * FP4 + 4 + RS * D) * 4;
        const long long grid = ((long long)B + G::WARPS - 1) / G::WARPS;
        int rc = ensure_smem_attr((const void*)interaction_bwd_ring2_kernel<F, D, RS>, (int)smem, &attr_done);
        if (rc) return rc;
        interaction_bwd_ring2_kernel<F, D, RS><<<(unsigned)grid, G::WARPS * 32, smem, s>>>(dOut, T, B, width, dT, dx,
                                                                                          clock_slot(CLK_IBWD));
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    } else {
        return -1;
    }
}

template <int F, int D>
int launch_bwd_ring(const float* dOut, const float* T, int B, int width, float* dT, float* dx, cudaStream_t s) {
    using G = BwdGeom<F, D>;
    if constexpr (G::SPW == 1 && F >= 12) {
        constexpr int RS = 12;
        static unsigned long long attr_done = 0;
        const size_t smem = BwdRingGeom<F, D, RS>::smem_bytes();
        const long long grid = ((long long)B + G::WARPS - 1) / G::WARPS;
        int rc = ensure_smem_attr((const void*)interaction_bwd_ring_kernel<F, D, RS>, (int)smem, &attr_done);
        if (rc) return rc;
        interaction_bwd_ring_kernel<F, D, RS><<<(unsigned)grid, G::WARPS * 32, smem, s>>>(dOut, T, B, width, dT, dx,
                                                                                         clock_slot(CLK_IBWD));
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    } else {
        return -1;
    }
}

template <int F, int D>
int launch_bwd_warp(const float* dOut, const float* T, int B, int width, float* dT, float* dx,
                    const void* dests, long long sample_offset, int qlog, cudaStream_t s) {
    using G = BwdGeom<F, D>;
    if (dests && qlog > 0) {   // column pieces: the peer-store kernel below with the piece-wise epilogue
        constexpr int SV = (G::SPW == 1) ? 2 : 0;
        static unsigned long long attr_done = 0;
        const size_t smem = BwdGeom<F, D, SV>::smem_bytes();
        const long long groups = ((long long)B + G::SPW - 1) / G::SPW;
        const long long grid = (groups + G::WARPS - 1) / G::WARPS;
        int rc = ensure_smem_attr((const void*)interaction_bwd_warp_kernel<F, D, true, SV, true>, (int)smem, &attr_done);
        if (rc) return rc;
        interaction_bwd_warp_kernel<F, D, true, SV, true><<<(unsigned)grid, G::WARPS * 32, smem, s>>>(
            dOut, T, B, width, nullptr, dx, static_cast<const SlotDestW*>(dests), sample_offset, clock_slot(CLK_IBWD), qlog);
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    }
    if (dests) {   // peer-store epilogue: the resident kernel, with S stored once (VAR 2) for one sample per warp
        constexpr int SV = (G::SPW == 1) ? 2 : 0;
        static unsigned long long attr_done = 0;
        const size_t smem = BwdGeom<F, D, SV>::smem_bytes();
        const long long groups = ((long long)B + G::SPW - 1) / G::SPW;
        const long long grid = (groups + G::WARPS - 1) / G::WARPS;
        int rc = ensure_smem_attr((const void*)interaction_bwd_warp_kernel<F, D, true, SV>, (int)smem, &attr_done);
        if (rc) return rc;
        interaction_bwd_warp_kernel<F, D, true, SV><<<(unsigned)grid, G::WARPS * 32, smem, s>>>(
            dOut, T, B, width, dT, dx, static_cast<const SlotDestW*>(dests), sample_offset, clock_slot(CLK_IBWD));
        DLRMB_LAUNCH_CHECK();
        return DLRMB_OK;
    }
    if (G::SPW == 1) {   // one sample per warp: see BwdGeom
        int v = g_opt.bwd_variant.load(std::memory_order_relaxed);
        // default: the streaming kernel with S stored once (fastest at every batch size measured, 2048 .. 16384:
        // profiles/r02_bwd_variants.txt); the others stay selectable for the parity tests and A/B runs
        if (v < 1 || v > 6) v = 6;
        if (v == 5 || v == 6) {
            const int rc = (v == 5) ? launch_bwd_ring<F, D>(dOut, T, B, width, dT, dx, s)
                                    : launch_bwd_ring2<F, D>(dOut, T, B, width, dT, dx, s);
            if (rc != -1) return rc;
            v = 3;   // no streaming kernel for this F: the resident kernel with S stored once
        }
        if (v == 2) return launch_bwd_warp_plain<F, D, (G::SPW == 1) ? 1 : 0>(dOut, T, B, width, dT, dx, s);
        if (v == 3) return launch_bwd_warp_plain<F, D, (G::SPW == 1) ? 2 : 0>(dOut, T, B, width, dT, dx, s);
    }
    return launch_bwd_warp_plain<F, D, 0>(dOut, T, B, width, dT, dx, s);
}

constexpr int kKsplitMaxBatch = 4096;   // up to here the forward is one wave of CTAs on 148 SMs

// dlrmb_set_option("interact_general", 1) sends the specialised shapes through the general tiled kernels
// of interact.cu (parity tests compare the two); default = the specialised kernels.
bool warp_path_enabled() { return g_opt.interact_general.load(std::memory_order_relaxed) == 0; }

}  // namespace

// Shapes with a compiled warp-per-sample specialisation: the Criteo models (26 tables + the dense
// slot, d = 16..128) and the geometry of the reference's golden files (7 tables, d = 16).
#define DLRMB_WARP_SHAPES(X) X(27, 128) X(27, 64) X(27, 32) X(27, 16) X(8, 16)

bool interaction_has_warp_path(int F, int d) {
#define X(FF, DD) if (F == FF && d == DD) return true;
    DLRMB_WARP_SHAPES(X)
#undef X
    return false;
}

// Returns DLRMB_OK after launching, or -1 when there is no specialisation for (F, d) and the caller
// must take the general path.
int try_interaction_fwd_warp(float* T, const float* x, int B, int F, int d, int width, float* out,
                             cudaStream_t s) {
    if (!warp_path_enabled()) return -1;
    {   // one-wave batches of the wide Criteo shapes: two warps per sample ("fwd_ksplit" = 0 keeps one warp per sample)
        const int mode = g_opt.fwd_ksplit.load(std::memory_order_relaxed);
        if (mode != 0 && (mode == 2 || B <= kKsplitMaxBatch)) {
            if (F == 27 && d == 128) return launch_fwd_mma_ksplit<27, 128>(T, x, B, width, out, s);
            if (F == 27 && d == 64) return launch_fwd_mma_ksplit<27, 64>(T, x, B, width, out, s);
        }
    }
#define X(FF, DD) if (F == FF && d == DD) return launch_fwd_mma<FF, DD>(T, x, B, width, out, s);
    DLRMB_WARP_SHAPES(X)
#undef X
    return -1;
}

int try_interaction_bwd_warp(const float* dOut, const float* T, int B, int F, int d, int width,
                             float* dT, float* dx, const void* dests, long long sample_offset, int qlog,
                             cudaStream_t s) {
    if (!warp_path_enabled()) return -1;
#define X(FF, DD) \
    if (F == FF && d == DD) return launch_bwd_warp<FF, DD>(dOut, T, B, width, dT, dx, dests, sample_offset, qlog, s);
    DLRMB_WARP_SHAPES(X)
#undef X
    return -1;
}

}  // namespace dlrmb
