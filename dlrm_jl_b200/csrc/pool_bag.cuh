// The pooling loop shared by the jagged lookups of lookup.cu and the fused jagged lookup + exchange of p2p.cu, so
// that both pool a bag with the same instructions (and hence the same bits).
#pragma once
#include "common.cuh"

namespace dlrmb {

template <int VEC> struct Vec;
template <> struct Vec<4> {
    using type = float4;
    template <typename RowT>
    static __device__ __forceinline__ float4 ldrow(const float* base, size_t r, size_t D, int c) {
        return RowIO<RowT>::ldg4(RowIO<RowT>::row(base, r, D), c);
    }
    static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ float4 add(float4 a, float4 b) {
        return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
    }
    static __device__ __forceinline__ float4 scale(float4 a, float w) {
        return make_float4(__fmul_rn(a.x, w), __fmul_rn(a.y, w), __fmul_rn(a.z, w), __fmul_rn(a.w, w));
    }
};
template <> struct Vec<1> {
    using type = float;
    template <typename RowT>
    static __device__ __forceinline__ float ldrow(const float* base, size_t r, size_t D, int c) {
        return RowIO<RowT>::ldg1(RowIO<RowT>::row(base, r, D), c);
    }
    static __device__ __forceinline__ float zero() { return 0.f; }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float scale(float a, float w) { return __fmul_rn(a, w); }
};

// Sum of chunk c of the rows ip[0 .. n) (fp32, from +0.0f, ascending), four row loads in flight: the loop of
// lookup.cu's lookup_pool_body (which keeps its own copy: calling this helper there changes the VEC = 1 kernels' SASS).
// WEIGHTED multiplies row p by wp[p] before it is added: acc = fl(acc + fl(w * row)), never contracted.
template <typename IdxT, int VEC, typename RowT, bool WEIGHTED = false>
__device__ __forceinline__ typename Vec<VEC>::type pool_bag(const float* __restrict__ tb, const IdxT* __restrict__ ip,
                                                            uint32_t n, int idx_base, size_t D, uint32_t c,
                                                            const float* __restrict__ wp = nullptr) {
    using V = typename Vec<VEC>::type;
    V acc = Vec<VEC>::zero();
    uint32_t p = 0;
    for (; p + 4 <= n; p += 4) {
        int64_t r0 = (int64_t)__ldg(ip + p) - idx_base;
        int64_t r1 = (int64_t)__ldg(ip + p + 1) - idx_base;
        int64_t r2 = (int64_t)__ldg(ip + p + 2) - idx_base;
        int64_t r3 = (int64_t)__ldg(ip + p + 3) - idx_base;
        V v0 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r0, D, c);
        V v1 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r1, D, c);
        V v2 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r2, D, c);
        V v3 = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r3, D, c);
        if (WEIGHTED) {
            v0 = Vec<VEC>::scale(v0, __ldg(wp + p));
            v1 = Vec<VEC>::scale(v1, __ldg(wp + p + 1));
            v2 = Vec<VEC>::scale(v2, __ldg(wp + p + 2));
            v3 = Vec<VEC>::scale(v3, __ldg(wp + p + 3));
        }
        acc = Vec<VEC>::add(acc, v0);
        acc = Vec<VEC>::add(acc, v1);
        acc = Vec<VEC>::add(acc, v2);
        acc = Vec<VEC>::add(acc, v3);
    }
    for (; p < n; ++p) {
        int64_t r = (int64_t)__ldg(ip + p) - idx_base;
        V v = Vec<VEC>::template ldrow<RowT>(tb, (size_t)r, D, c);
        if (WEIGHTED) v = Vec<VEC>::scale(v, __ldg(wp + p));
        acc = Vec<VEC>::add(acc, v);
    }
    return acc;
}

}  // namespace dlrmb
