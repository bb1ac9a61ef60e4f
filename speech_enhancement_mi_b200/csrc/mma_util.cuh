// Warp-level tensor-core helpers shared by the per-stream kernels of the small-channel layers (front_mma.cu, back_mma.cu):
// ldmatrix / mma.sync.m16n8k16 wrappers, flush-to-zero MUFU forms, cp.async, fp16 packing, the in-CTA GlobalLayerNorm
// reduction.  Fragment roles (g = lane / 4, tg = lane % 4): A rows g, g + 8; B column g; C rows g, g + 8, columns 2 tg,
// 2 tg + 1.  The C fragments of two adjacent n-tiles ARE the A fragment of a k-step (registers are reused as operands).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include "se_internal.h"

namespace se {
namespace mma_util {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
// not volatile: a pure register function, so that the compiler may move the dependent HMMA behind the NEXT ldmatrix (two
// volatile statements keep their order, which serialised every ldmatrix -> mma pair on the ~30-cycle shared-memory latency)
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(float x, float y) {
    const __half2 h = __floats2half2_rn(x, y);
    return *reinterpret_cast<const uint32_t*>(&h);
}
// MUFU forms with flush-to-zero: without .ftz the compiler wraps every ex2 / rcp in a denormal range check (FSETP + two
// predicated FMULs), which tripled the instruction count of the epilogues (ncu: FMUL 14 %, FSETP 6 % of the kernel)
__device__ __forceinline__ float ex2_ftz(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_ftz(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float kLog2e = 1.4426950408889634f;
// gate: the caller passes z = -log2(e) * (pre-activation); the factor is folded into the gate weights and bias
__device__ __forceinline__ float sigmoid_from_neg_log2(float z) { return rcp_ftz(1.0f + ex2_ftz(z)); }
__device__ __forceinline__ float fast_elu(float x) { return x > 0.f ? x : ex2_ftz(x * kLog2e) - 1.0f; }
// Contiguous tile range of a warp such that the four SM sub-partitions (warp w issues on sub-partition w % 4, and the
// tensor pipe of a sub-partition is what bounds the mma.sync passes) get equal shares: sub-partition sp owns the sp-th
// quarter of the tiles and its warps (w / 4 = 0 .. nwarps / 4 - 1) split that quarter.  Sizes differ by at most one tile
// between sub-partitions and between the warps of one (warp * n / nwarps let one sub-partition collect all the
// rounded-up ranges: 36 tiles against 32 in the first encoder level).
__device__ __forceinline__ void warp_tile_range(int warp, int nwarps, int ntiles, int& lo, int& hi) {
    const int sp = warp & 3, k = warp >> 2, per = nwarps >> 2;
    const int s0 = (sp * ntiles) >> 2, n = (((sp + 1) * ntiles) >> 2) - s0;
    lo = s0 + (k * n) / per;
    hi = s0 + ((k + 1) * n) / per;
}
// exact quotient r / d for r < 65536 with magic = ceil(2^32 / d)
__device__ __forceinline__ int div_magic(int r, uint32_t magic) { return (int)__umulhi((uint32_t)r, magic); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void unpack8(const uint4& u, float* v) {
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(h[i]);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ uint4 pack8(const float* o) {
    uint4 u;
    u.x = pack_h2(o[0], o[1]);
    u.y = pack_h2(o[2], o[3]);
    u.z = pack_h2(o[4], o[5]);
    u.w = pack_h2(o[6], o[7]);
    return u;
}

// GlobalLayerNorm coefficients of one stream from the per-thread partial sums (CRN_ELU.py:40-51 /
// distillation_crn.py:51): every thread calls this; returns after a __syncthreads with s_co = {mean, 1/den}
template <int NWARPS = kWarps>
__device__ __forceinline__ void block_gln(float psum, float psq, double count, int student, double* s_red, float* s_co) {
    double ds = psum, dq = psq;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        ds += __shfl_xor_sync(0xffffffffu, ds, off);
        dq += __shfl_xor_sync(0xffffffffu, dq, off);
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_red[warp] = ds;
        s_red[NWARPS + warp] = dq;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, q = 0.0;
        for (int w = 0; w < NWARPS; ++w) {
            a += s_red[w];
            q += s_red[NWARPS + w];
        }
        gln_mean_inv(a, q, count, student, s_co[0], s_co[1]);
    }
    __syncthreads();
}

}  // namespace mma_util
}  // namespace se
