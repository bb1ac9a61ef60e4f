// Dedicated kernels for the two layer shapes that the 128-row tcgen05 tiles serve badly (fp16 operand mode):
//   * the last transposed convolution (CRN_ELU.py:352-358, 16 -> 2 channels): the GEMM has N = 4 useful columns of a
//     16-wide tile and gathers 9 taps x 16 channels per row -- 0.6 % of the tensor peak, 194 us per step;
//   * the 1x1 mask / residual pair on a 16- (or 8-) channel skip tensor (CRN_ELU.py:305-306): K = 16 is padded to a
//     64-element k-block, so 3/4 of the operand traffic and of the MMA work is zeros -- 151 us per step.
// Both read their data once.  Default: warp-level mma.sync kernels whose A fragments come straight from global memory
// (second half of this file; 0.074 / 0.064 ms).  SE_B200_SMALL_MMA=0 selects the first generation kept for A/B runs:
// one thread per position on the CUDA cores, weights broadcast from shared memory (0.112 / 0.110 ms, bound by the
// shared-memory operand fetches).  Per-stream GlobalLayerNorm statistics are reduced per block in both.
#include <cuda_fp16.h>

#include <cstdlib>

#include "se_internal.h"

namespace se {
namespace {

constexpr int T = kFramesPerChunk;

__device__ __forceinline__ float elu_fast(float x) {  // ex2.approx.ftz: one MUFU, no range fix-up (see gemm_tc.cu)
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(1.4426950408889634f * x));
    return x > 0.f ? x : y - 1.0f;
}

template <int N>
__device__ __forceinline__ void load_halves(const __half* p, float* v) {  // N = 8 or 16 halves, 16-byte aligned
#pragma unroll
    for (int u = 0; u < N / 8; ++u) {
        const uint4 q = __ldg(reinterpret_cast<const uint4*>(p) + u);
        const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(h[i]);
            v[8 * u + 2 * i] = f.x;
            v[8 * u + 2 * i + 1] = f.y;
        }
    }
}

__device__ __forceinline__ void block_stats(float s, float ss, double* stats, int b) {
    __shared__ float red[2][8];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        ss += __shfl_xor_sync(0xffffffffu, ss, off);
    }
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = s;
        red[1][threadIdx.x >> 5] = ss;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, c = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            a += red[0][w];
            c += red[1][w];
        }
        atomicAdd(stats + 2 * b, (double)a);
        atomicAdd(stats + 2 * b + 1, (double)c);
    }
}

// grid (ceil(Fin / 32), B), 256 threads: lane = input bin f' inside the block's 32-bin slab, warp w = frames w, w+8, w+16
template <int CIN>
__global__ void __launch_bounds__(256) deconv_last_kernel(DeconvLastParams p) {
    __shared__ __align__(16) float sw[9 * CIN * 4];  // [kt][j][ci][n], n = parity * 2 + co
    __shared__ float sb[4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 9 * CIN * 4; i += 256) {
        const int n = i & 3, k = i >> 2;  // k = (kt * 3 + j) * CIN + ci
        sw[i] = __ldg(p.w + (long long)n * p.Kp + k);
    }
    if (tid < 4) sb[tid] = __ldg(p.bias + tid);
    __syncthreads();
    const int b = blockIdx.y;
    const int f = blockIdx.x * 32 + lane;
    const bool valid = f < p.Fin;
    const int fl = valid ? f : p.Fin - 1;  // clamped: out-of-range lanes compute on valid memory and store nothing
    const __half* base = p.in + (long long)b * p.sB + (long long)fl * p.sF;
    const int Fy = 2 * p.Fin - 1;
    float s = 0.f, ss = 0.f;
    // the warp's (up to) three frames are processed together: one weight fetch feeds 12 FMAs and three independent
    // load streams are in flight
    int tt[3];
    bool tv[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        tv[i] = warp + 8 * i < T;
        tt[i] = tv[i] ? warp + 8 * i : warp;  // clamped: computed, not stored
    }
    float acc[3][4];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int n = 0; n < 4; ++n) acc[i][n] = sb[n];
#pragma unroll
    for (int kt = 0; kt < 3; ++kt) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float x[3][CIN];
#pragma unroll
            for (int i = 0; i < 3; ++i)
                load_halves<CIN>(base + (long long)(tt[i] + (2 - kt) * p.d) * p.sT + (long long)(2 - j) * p.sF, x[i]);
            const float4* w = reinterpret_cast<const float4*>(sw + (kt * 3 + j) * CIN * 4);
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci) {
                const float4 q = w[ci];
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    acc[i][0] = fmaf(x[i][ci], q.x, acc[i][0]);
                    acc[i][1] = fmaf(x[i][ci], q.y, acc[i][1]);
                    acc[i][2] = fmaf(x[i][ci], q.z, acc[i][2]);
                    acc[i][3] = fmaf(x[i][ci], q.w, acc[i][3]);
                }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        if (valid && tv[i]) {
            float2* y = reinterpret_cast<float2*>(p.y) + ((long long)b * T + tt[i]) * Fy + 2 * f;
            const float e0 = elu_fast(acc[i][0]), e1 = elu_fast(acc[i][1]);
            y[0] = make_float2(e0, e1);
            s += e0 + e1;
            ss += e0 * e0 + e1 * e1;
            if (f < p.Fin - 1) {  // bin 2 f' + 1 exists
                const float o0 = elu_fast(acc[i][2]), o1 = elu_fast(acc[i][3]);
                y[1] = make_float2(o0, o1);
                s += o0 + o1;
                ss += o0 * o0 + o1 * o1;
            }
        }
    }
    block_stats(s, ss, p.stats, b);
}

// grid (ceil(T * Fs / 256), B), one thread per position
template <int C>
__global__ void __launch_bounds__(256) skip_small_kernel(SkipSmallParams p) {
    __shared__ __align__(16) float sw[2 * C * C];  // [n][ci], n = 2 co (mask) / 2 co + 1 (residual)
    __shared__ float sb[2 * C];
    const int tid = threadIdx.x;
    for (int i = tid; i < 2 * C * C; i += 256) sw[i] = __ldg(p.w + (long long)(i / C) * p.Kp + i % C);
    if (tid < 2 * C) sb[tid] = __ldg(p.bias + tid);
    __syncthreads();
    const int b = blockIdx.y;
    const int r = blockIdx.x * 256 + tid;
    float s = 0.f, ss = 0.f;
    if (r < T * p.Fs) {
        const int t = r / p.Fs, f = r - t * p.Fs;
        float x[C];
        load_halves<C>(p.in + (long long)b * p.sB + (long long)t * p.sT + (long long)f * p.sF, x);
        uint32_t pm[C / 2], pr[C / 2];  // packed half2 pairs (kept in registers: no local-memory staging)
#pragma unroll
        for (int cp = 0; cp < C / 2; ++cp) {
            float a[4] = {sb[4 * cp], sb[4 * cp + 1], sb[4 * cp + 2], sb[4 * cp + 3]};  // mask, residual of 2 channels
            const float4* w0 = reinterpret_cast<const float4*>(sw + (4 * cp) * C);      // 4 consecutive weight rows
#pragma unroll
            for (int c4 = 0; c4 < C / 4; ++c4) {
#pragma unroll
                for (int r4 = 0; r4 < 4; ++r4) {
                    const float4 q = w0[r4 * (C / 4) + c4];
                    a[r4] = fmaf(q.x, x[4 * c4], a[r4]);
                    a[r4] = fmaf(q.y, x[4 * c4 + 1], a[r4]);
                    a[r4] = fmaf(q.z, x[4 * c4 + 2], a[r4]);
                    a[r4] = fmaf(q.w, x[4 * c4 + 3], a[r4]);
                }
            }
            const __half2 hm = __floats2half2_rn(a[0], a[2]);
            const __half2 hr = __floats2half2_rn(elu_fast(a[1]), elu_fast(a[3]));
            pm[cp] = *reinterpret_cast<const uint32_t*>(&hm);
            pr[cp] = *reinterpret_cast<const uint32_t*>(&hr);
            s += a[0] + a[2];
            ss += a[0] * a[0] + a[2] * a[2];
        }
        const long long o = (((long long)b * T + t) * p.Fs + f) * C;
#pragma unroll
        for (int u = 0; u < C / 8; ++u) {
            reinterpret_cast<uint4*>(p.rm + o)[u] = make_uint4(pm[4 * u], pm[4 * u + 1], pm[4 * u + 2], pm[4 * u + 3]);
            reinterpret_cast<uint4*>(p.rr + o)[u] = make_uint4(pr[4 * u], pr[4 * u + 1], pr[4 * u + 2], pr[4 * u + 3]);
        }
    }
    block_stats(s, ss, p.stats, b);
}

// ---- warp-level tensor-core versions (mma.sync m16n8k16, fp16 operands, fp32 accumulate) ------------------------------
// The CUDA-core kernels above are bound by the shared-memory operand fetches (one LDS per 1-3 FMAs: 110 us each, three
// times their FMA and HBM bounds).  Both layers are tiny GEMMs over positions whose A rows are 16 consecutive fp16
// channels in memory, so a warp loads the m16k16 A fragment of 16 consecutive positions straight from global memory
// (4-byte loads, every 32-byte sector used whole), keeps the B fragments (weights, rounded to fp16 like every other
// GEMM operand of this mode) in registers for its lifetime, and never touches shared memory.
__device__ __forceinline__ void mma16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
    asm(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// D = A B + (c0, c1, c0, c1): the bias pair of the lane's two columns is the C operand, no accumulator initialisation
__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1, float c0, float c1) {
    asm(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%10,%11};"
        : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(c0), "f"(c1));
}
__device__ __forceinline__ uint32_t pack_h2(float x, float y) {
    const __half2 h = __floats2half2_rn(x, y);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t ld_u32(const __half* q) { return __ldg(reinterpret_cast<const unsigned int*>(q)); }
__device__ __forceinline__ uint2 ld_u64(const __half* q) { return __ldg(reinterpret_cast<const uint2*>(q)); }
// The order of the 16 k slots of a step is free as long as A and B agree: with 16 channels per row, lane t supplies
// channels 4t .. 4t+3 (slots 2t, 2t+1 <- channels 4t, 4t+1; slots 2t+8, 2t+9 <- channels 4t+2, 4t+3), one 8-byte load
// per row; with 8 channels the upper slots are zero and lane t supplies channels 2t, 2t+1.

// grid (gx, B): the warps of a stream's blocks stride over its groups of 16 positions.  Fragment roles (g = lane / 4,
// t = lane % 4): A rows g, g + 8 = positions, B column g = output channel of the n-tile, C columns 2t, 2t + 1.
// n-tiles [0, C/8) are the mask channels, [C/8, C/4) the residual channels.  Lane t supplies the CPL = C/4 consecutive
// channels CPL t .. CPL t + CPL - 1 of its rows (one 4 / 8 byte load per row); k-step s consumes elements
// 4s .. 4s+3 of that chunk.  NSPLIT > 1 splits the n-tiles over neighbouring warps that read the same rows; measured for
// C = 64 (NSPLIT = 2, 64 registers of B fragments): 0.148 ms against 0.094 ms of the tcgen05 GEMM, whose 128-wide tile is
// full at that width.  In fp16 inference 32 and 64 channels run fused with the blend (skip_blend_tc.cu); the dispatch
// below serves 8 and 16.
template <int C, int NSPLIT, int GQ>
__global__ void __launch_bounds__(256) skip_small_mma_kernel(SkipSmallParams p) {
    static_assert(C == 8 || C == 16, "skip_small_mma: 8 or 16 channels (one 4- or 8-byte A load per row)");
    constexpr int NT = C / 4, HT = NT / 2;          // n-tiles, n-tiles per kind
    constexpr int KS = C >= 16 ? C / 16 : 1;        // k-steps
    constexpr int CPL = C >= 16 ? C / 4 : 2;        // channels per lane and row
    constexpr int NTW = NT / NSPLIT;                // n-tiles of this warp
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const int ns = warp % NSPLIT, wg = warp / NSPLIT;  // n-split index, group-worker index
    uint32_t bf[NTW][KS][2];
    float bs[NTW][2];
#pragma unroll
    for (int jj = 0; jj < NTW; ++jj) {
        const int j = ns * NTW + jj;
        const int kind = j / HT, ch0 = 8 * (j % HT);
        const float* wr = p.w + (long long)(2 * (ch0 + g) + kind) * p.Kp + CPL * t;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            if (C >= 16) {  // 16-byte aligned: Kp and the arena offsets are multiples of 4 floats
                const float4 w4 = __ldg(reinterpret_cast<const float4*>(wr) + ks);
                bf[jj][ks][0] = pack_h2(w4.x, w4.y);
                bf[jj][ks][1] = pack_h2(w4.z, w4.w);
            } else {
                bf[jj][ks][0] = pack_h2(__ldg(wr), __ldg(wr + 1));
                bf[jj][ks][1] = 0u;
            }
        }
        bs[jj][0] = __ldg(p.bias + 2 * (ch0 + 2 * t) + kind);
        bs[jj][1] = __ldg(p.bias + 2 * (ch0 + 2 * t + 1) + kind);
    }
    const int b = blockIdx.y;
    const int total = T * p.Fs;
    const int ngroups = (total + 15) >> 4;
    const int stride = gridDim.x * (8 / NSPLIT);
    // everything below a stream's base pointers is 32-bit element arithmetic (a stream's buffers are far below 2^31)
    const __half* in = p.in + (long long)b * p.sB + CPL * t;
    const int sT = (int)p.sT, sF = (int)p.sF, Fs = p.Fs;
    const bool odd = t & 1;  // even lanes store row g (their own pair + the neighbour's), odd lanes row g + 8
    __half* rm = p.rm + (long long)b * total * C + 2 * (t & 2) + (odd ? 8 * C : 0);
    __half* rr = p.rr + (long long)b * total * C + 2 * (t & 2) + (odd ? 8 * C : 0);
    float s = 0.f, ss = 0.f;
    // GQ groups per pass (their loads are in flight together); the weights are fetched once per warp
    for (int g0 = blockIdx.x * (8 / NSPLIT) + wg; g0 < ngroups; g0 += GQ * stride) {
        int row0[GQ];
        uint32_t a[GQ][KS][4];
#pragma unroll
        for (int q = 0; q < GQ; ++q) {
            const int rb = (g0 + q * stride) * 16;  // warp-uniform: one division per group
            const int tb = rb / Fs, fb = rb - tb * Fs;
            row0[q] = rb + g;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                int tt = tb, f = fb + g + 8 * h;
                if (f >= Fs) {  // Fs >= 16 (checked by the launcher): at most one wrap
                    f -= Fs;
                    ++tt;
                }
                if (tt >= T) {  // beyond the last position: computed on valid memory, never stored
                    tt = T - 1;
                    f = Fs - 1;
                }
                const __half* src = in + (tt * sT + f * sF);
                if (C == 16) {
                    const uint2 u = ld_u64(src);
                    a[q][0][h] = u.x;
                    a[q][0][2 + h] = u.y;
                } else {
                    a[q][0][h] = ld_u32(src);
                    a[q][0][2 + h] = 0u;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < GQ; ++q) {
            const bool v0 = row0[q] < total, v1 = row0[q] + 8 < total;
            const bool ov = odd ? v1 : v0;
            const int o = row0[q] * C;
#pragma unroll
            for (int jj = 0; jj < NTW; ++jj) {
                const int j = ns * NTW + jj;
                float c[4];
                mma16816(c, a[q][0][0], a[q][0][1], a[q][0][2], a[q][0][3], bf[jj][0][0], bf[jj][0][1], bs[jj][0], bs[jj][1]);
#pragma unroll
                for (int ks = 1; ks < KS; ++ks)
                    mma16816(c, a[q][ks][0], a[q][ks][1], a[q][ks][2], a[q][ks][3], bf[jj][ks][0], bf[jj][ks][1]);
                const bool mask = j < HT;  // warp-uniform
                if (mask) {
                    if (v0) {
                        s += c[0] + c[1];
                        ss = fmaf(c[0], c[0], fmaf(c[1], c[1], ss));
                    }
                    if (v1) {
                        s += c[2] + c[3];
                        ss = fmaf(c[2], c[2], fmaf(c[3], c[3], ss));
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) c[k] = elu_fast(c[k]);
                }
                const uint32_t p0 = pack_h2(c[0], c[1]), p1 = pack_h2(c[2], c[3]);
                const uint32_t got = __shfl_xor_sync(0xffffffffu, odd ? p0 : p1, 1);
                const uint2 v = odd ? make_uint2(got, p1) : make_uint2(p0, got);
                if (ov) *reinterpret_cast<uint2*>((mask ? rm : rr) + (o + 8 * (j % HT))) = v;
            }
        }
    }
    block_stats(s, ss, p.stats, b);
}

// grid (1, B): the warps of a stream's block stride over its (16 input bins f' = the rows of the fragment, frame) tasks.
// K = 9 taps x CIN (one k-step per tap), N = 4 (n = parity * 2 + co) of an 8-wide tile: lanes t = 0 / 1 hold the even /
// odd output bin of rows g, g + 8.
template <int CIN>
__global__ void __launch_bounds__(256) deconv_last_mma_kernel(DeconvLastParams p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    uint32_t bf[9][2];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        bf[tap][0] = bf[tap][1] = 0u;
        if (g < 4) {
            const float* wr = p.w + (long long)g * p.Kp + tap * CIN;
            if (CIN == 16) {
                bf[tap][0] = pack_h2(__ldg(wr + 4 * t), __ldg(wr + 4 * t + 1));
                bf[tap][1] = pack_h2(__ldg(wr + 4 * t + 2), __ldg(wr + 4 * t + 3));
            } else {
                bf[tap][0] = pack_h2(__ldg(wr + 2 * t), __ldg(wr + 2 * t + 1));
            }
        }
    }
    const float b0 = t < 2 ? __ldg(p.bias + 2 * t) : 0.f, b1 = t < 2 ? __ldg(p.bias + 2 * t + 1) : 0.f;
    const int b = blockIdx.y;
    const int Fy = 2 * p.Fin - 1;
    const int ntasks = ((p.Fin + 15) >> 4) * T;  // task = (group of 16 bins, frame), frame fastest: the warps of a
    float s = 0.f, ss = 0.f;                      // block work on neighbouring frames of one group (shared input rows)
    // everything below the stream's base pointer is 32-bit element arithmetic (a stream's buffer is far below 2^31)
    const __half* in = p.in + (long long)b * p.sB + (CIN == 16 ? 4 : 2) * t;
    const int sT = (int)p.sT, sF = (int)p.sF;
    const int step = gridDim.x * 8;
    auto fetch = [&](uint32_t (&a)[9][4], int task) {
        if (task >= ntasks) return;
        const int grp = task / T, tt = task - grp * T;
        int ro[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int f = grp * 16 + g + 8 * h;
            const int fl = f < p.Fin ? f : p.Fin - 1;  // clamped: computed on valid memory, never stored
            ro[h] = fl * sF + tt * sT;
        }
#pragma unroll
        for (int kt = 0; kt < 3; ++kt) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int off = (2 - kt) * p.d * sT + (2 - j) * sF;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (CIN == 16) {
                        const uint2 u = ld_u64(in + (ro[h] + off));
                        a[kt * 3 + j][h] = u.x;
                        a[kt * 3 + j][2 + h] = u.y;
                    } else {
                        a[kt * 3 + j][h] = ld_u32(in + (ro[h] + off));
                        a[kt * 3 + j][2 + h] = 0u;
                    }
                }
            }
        }
    };
    auto compute = [&](const uint32_t (&a)[9][4], int task) {
        const int grp = task / T, tt = task - grp * T;
        // two accumulation chains (even / odd taps) halve the dependent-mma latency
        float c[4] = {b0, b1, b0, b1}, c2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            if (tap & 1) mma16816(c2, a[tap][0], a[tap][1], a[tap][2], a[tap][3], bf[tap][0], bf[tap][1]);
            else mma16816(c, a[tap][0], a[tap][1], a[tap][2], a[tap][3], bf[tap][0], bf[tap][1]);
        }
        if (t < 2) {  // t = parity of the output bin
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int f = grp * 16 + g + 8 * h;
                if (f < p.Fin && (t == 0 || f < p.Fin - 1)) {
                    const float e0 = elu_fast(c[2 * h] + c2[2 * h]), e1 = elu_fast(c[2 * h + 1] + c2[2 * h + 1]);
                    reinterpret_cast<float2*>(p.y)[((long long)b * T + tt) * Fy + 2 * f + t] = make_float2(e0, e1);
                    s += e0 + e1;
                    ss += e0 * e0 + e1 * e1;
                }
            }
        }
    };
    // software pipeline over the warp's tasks: the fragments of the next task are requested before the current one is
    // multiplied (two register sets, ping-pong), so the DRAM latency of a task hides behind its predecessor
    uint32_t fa[9][4], fb[9][4];
    int task = blockIdx.x * 8 + warp;
    fetch(fa, task);
    while (task < ntasks) {
        fetch(fb, task + step);
        compute(fa, task);
        task += step;
        if (task >= ntasks) break;
        fetch(fa, task + step);
        compute(fb, task);
        task += step;
    }
    block_stats(s, ss, p.stats, b);
}

}  // namespace

bool deconv_last_supported(int Cin) { return Cin == 8 || Cin == 16; }
bool skip_small_supported(int C) { return C == 8 || C == 16; }

int launch_deconv_last(const DeconvLastParams& p, int Cin, cudaStream_t st) {
    if (p.B <= 0) return 0;
    SE_REQUIRE(p.B <= 65535, "deconv_last: at most 65535 streams per launch");
    const bool cuda_cores = getenv("SE_B200_SMALL_MMA") && atoi(getenv("SE_B200_SMALL_MMA")) == 0;  // A/B switch
    const dim3 grid(cuda_cores ? (p.Fin + 31) / 32 : 1, p.B);  // one block per stream: fewer, longer blocks measured fastest
    if (cuda_cores && Cin == 16) deconv_last_kernel<16><<<grid, 256, 0, st>>>(p);
    else if (cuda_cores && Cin == 8) deconv_last_kernel<8><<<grid, 256, 0, st>>>(p);
    else if (Cin == 16) deconv_last_mma_kernel<16><<<grid, 256, 0, st>>>(p);
    else if (Cin == 8) deconv_last_mma_kernel<8><<<grid, 256, 0, st>>>(p);
    else SE_REQUIRE(false, "deconv_last: input channels must be 8 or 16");
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_skip_small(const SkipSmallParams& p, int C, cudaStream_t st) {
    if (p.B <= 0) return 0;
    SE_REQUIRE(p.B <= 65535, "skip_small: at most 65535 streams per launch");
    SE_REQUIRE(p.Fs >= 16, "skip_small: at least 16 bins");
    const bool cuda_cores = getenv("SE_B200_SMALL_MMA") && atoi(getenv("SE_B200_SMALL_MMA")) == 0;  // A/B switch
    const bool cc = cuda_cores && C <= 16;
    const dim3 grid(cc ? (T * p.Fs + 255) / 256 : (C <= 16 ? 2 : 1), p.B);
    if (cc && C == 16) skip_small_kernel<16><<<grid, 256, 0, st>>>(p);
    else if (cc && C == 8) skip_small_kernel<8><<<grid, 256, 0, st>>>(p);
    else if (C == 16) skip_small_mma_kernel<16, 1, 2><<<grid, 256, 0, st>>>(p);
    else if (C == 8) skip_small_mma_kernel<8, 1, 2><<<grid, 256, 0, st>>>(p);
    else SE_REQUIRE(false, "skip_small: channels must be 8 or 16");
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace se
