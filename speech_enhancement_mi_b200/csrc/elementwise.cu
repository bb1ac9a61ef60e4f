// HBM-bound elementwise kernels of the CRN path: GlobalLayerNorm application fused with the residual add / gated
// skip blend that follows it, the fp32-path GRU cell update, the causal-state roll, framing and overlap-add.
#include <cuda_fp16.h>

#include "se_internal.h"

namespace se {

namespace {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__device__ __forceinline__ void gln_coeffs(const double* stats, int b, double count, int student, float& mean,
                                           float& inv) {
    gln_mean_inv(stats[2 * b], stats[2 * b + 1], count, student, mean, inv);
}

__device__ __forceinline__ float4 load4(const float* base, long long idx, bool is_half) {
    if (!is_half) return *reinterpret_cast<const float4*>(base + idx);
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(base) + idx);
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

// grid (ceil(T / kNormFrames), B): one block per group of frames of one stream, one thread per 4 channels (C % 4 == 0).
// The per-stream coefficients (double arithmetic) are computed once per block; no 64-bit division per element.
constexpr int kNormFrames = 7;
__global__ void __launch_bounds__(256) norm_apply_kernel(NormApplyParams p) {
    const int t0 = blockIdx.x * kNormFrames;
    const int b = p.b0 + blockIdx.y;
    __shared__ float s_co[4];
    if (threadIdx.x == 0) {
        gln_coeffs(p.stats, b, p.count, p.student, s_co[0], s_co[1]);
        if (p.mode == 2) gln_coeffs(p.stats_r, b, p.count_r, p.student, s_co[2], s_co[3]);
    }
    __syncthreads();
    const float mean = s_co[0], inv = s_co[1];
    const int C4 = p.C >> 2;
    const int n4 = p.F * C4;
    const bool ih = p.in_half != 0;
    const int nt = min(kNormFrames, p.T - t0);
    for (int i = threadIdx.x; i < n4 * nt; i += blockDim.x) {
        const int tl = i / n4;
        const int j = i - tl * n4;
        const int t = t0 + tl;
        const int f = j / C4;
        const int c = (j - f * C4) * 4;
        const long long yrow = ((long long)b * p.T + t) * p.Fy * p.C;
        float* orow = p.out + b * p.oB + t * p.oT;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (f < p.Fy) {
            const float4 y = load4(p.y, yrow + f * p.C + c, ih);
            const int wi = p.per_feature ? (f * p.C + c) : c;
            const float4 w = *reinterpret_cast<const float4*>(p.w + wi);
            const float4 bb = *reinterpret_cast<const float4*>(p.b + wi);
            // same operation order as the reference: (x - mean) / den * w + b; the division is done as a multiply by
            // the reciprocal (<= 1 ulp difference, inside the stated fp tolerance)
            o.x = (y.x - mean) * inv * w.x + bb.x;
            o.y = (y.y - mean) * inv * w.y + bb.y;
            o.z = (y.z - mean) * inv * w.z + bb.z;
            o.w = (y.w - mean) * inv * w.w + bb.w;
        }
        if (p.mode == 1) {
            const float4 x = *reinterpret_cast<const float4*>(p.res + b * p.rB + t * p.rT + f * p.rF + c);
            o.x += x.x;
            o.y += x.y;
            o.z += x.z;
            o.w += x.w;
        } else if (p.mode == 2) {
            const float mr = s_co[2], ir = s_co[3];
            const long long ri = (((long long)b * p.T + t) * p.F + f) * p.C + c;
            const float4 rm = load4(p.rm, ri, ih);
            const float4 rr = load4(p.rr, ri, ih);
            const float4 w = *reinterpret_cast<const float4*>(p.wr + c);
            const float4 bb = *reinterpret_cast<const float4*>(p.br + c);
            const float m0 = sigmoidf_((rm.x - mr) * ir * w.x + bb.x);
            const float m1 = sigmoidf_((rm.y - mr) * ir * w.y + bb.y);
            const float m2 = sigmoidf_((rm.z - mr) * ir * w.z + bb.z);
            const float m3 = sigmoidf_((rm.w - mr) * ir * w.w + bb.w);
            o.x = m0 * rr.x + (1.0f - m0) * o.x;
            o.y = m1 * rr.y + (1.0f - m1) * o.y;
            o.z = m2 * rr.z + (1.0f - m2) * o.z;
            o.w = m3 * rr.w + (1.0f - m3) * o.w;
        }
        if (p.out_half) {
            __half* oh = reinterpret_cast<__half*>(p.out) + b * p.oB + t * p.oT + f * p.oF + c;
            const __half2 lo = __floats2half2_rn(o.x, o.y), hi = __floats2half2_rn(o.z, o.w);
            uint2 u;
            u.x = *reinterpret_cast<const unsigned*>(&lo);
            u.y = *reinterpret_cast<const unsigned*>(&hi);
            *reinterpret_cast<uint2*>(oh) = u;
        } else {
            *reinterpret_cast<float4*>(orow + f * p.oF + c) = o;
        }
    }
}

// fp16 storage fast path: 8 channels (16 bytes) per thread and access, twice the bytes in flight of the float4 path.
// Same arithmetic; needs C % 8 == 0, fp16 inputs and outputs.
__device__ __forceinline__ void unpack8(const uint4& u, float* v) {
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(h[i]);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ void load8(const float* __restrict__ q, float* v) {
    const float4 lo = __ldg(reinterpret_cast<const float4*>(q)), hi = __ldg(reinterpret_cast<const float4*>(q) + 1);
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
}
// A thread keeps ONE (bin, 8-channel) unit for all frames of the block: the affine terms are loaded once and folded with
// the stream's statistics into one FMA per value (x * a + d, a = w / den, d = b - mean * a), the index arithmetic is
// done once per unit instead of once per access, and the frame loop is unrolled so that up to 3 x kNormFrames 16-byte
// loads are in flight per thread.  The outputs are rounded to fp16, which hides the re-association and the fast
// reciprocal / exponential of the mask sigmoid (the exact-order fp32 path is norm_apply_kernel above).
template <int MODE>
__global__ void __launch_bounds__(256, MODE == 2 ? 3 : 4) norm_apply_h8_kernel(NormApplyParams p) {
    constexpr int FB = MODE == 2 ? 2 : kNormFrames;  // frames per batch: all loads of a batch are issued before its first use
    const int t0 = blockIdx.x * kNormFrames;
    const int b = p.b0 + blockIdx.y;
    __shared__ float s_co[4];
    const int C8 = p.C >> 3;
    const int n8 = p.F * C8;
    const int nt = min(kNormFrames, p.T - t0);
    const __half* yh = reinterpret_cast<const __half*>(p.y) + ((long long)b * p.T + t0) * p.Fy * p.C;
    const __half* rmh = reinterpret_cast<const __half*>(p.rm) + ((long long)b * p.T + t0) * p.F * p.C;
    const __half* rrh = reinterpret_cast<const __half*>(p.rr) + ((long long)b * p.T + t0) * p.F * p.C;
    __half* oh = reinterpret_cast<__half*>(p.out) + b * p.oB + t0 * p.oT;
    const int ystep = p.Fy * p.C, rstep = p.F * p.C;
    bool first = true;
    for (int j = threadIdx.x; first || j < n8; j += blockDim.x) {
        const bool live = j < n8;  // only the first pass can be dead (every thread has to reach the barrier below)
        const int f = j / C8;
        const int c = (j - f * C8) * 8;
        const bool has_y = live && f < p.Fy;
        const int yo = f * p.C + c, ro = yo;  // offsets inside a frame (y rows hold Fy bins, the skip rows F bins)
        float a[8], d[8], ar[8], dr[8];
        uint4 uy[FB], um[FB], ur[FB];
        auto issue = [&](int tb) {
#pragma unroll
            for (int q = 0; q < FB; ++q) {
                const int tl = tb + q;
                uy[q] = make_uint4(0, 0, 0, 0);
                if (tl < kNormFrames && tl < nt && live) {
                    if (has_y) uy[q] = *reinterpret_cast<const uint4*>(yh + tl * ystep + yo);
                    if (MODE == 2) {
                        um[q] = *reinterpret_cast<const uint4*>(rmh + tl * rstep + ro);
                        ur[q] = *reinterpret_cast<const uint4*>(rrh + tl * rstep + ro);
                    }
                }
            }
        };
        // everything this unit reads is requested before the stream's statistics are needed
        issue(0);
        if (live) {
            const int wi = p.per_feature ? (f * p.C + c) : c;
            load8(p.w + wi, a);
            load8(p.b + wi, d);
            if (MODE == 2) {
                load8(p.wr + c, ar);
                load8(p.br + c, dr);
            }
        }
        if (first) {
            if (threadIdx.x == 0) gln_coeffs(p.stats, b, p.count, p.student, s_co[0], s_co[1]);
            if (MODE == 2 && threadIdx.x == 32) gln_coeffs(p.stats_r, b, p.count_r, p.student, s_co[2], s_co[3]);
            __syncthreads();
            first = false;
        }
        if (!live) break;
        {
            const float mean = s_co[0], inv = s_co[1];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                a[k] *= inv;
                d[k] = fmaf(-mean, a[k], d[k]);
            }
        }
        if (MODE == 2) {
            // the mask is 1 / (1 + 2^(-(x * ar + dr) * log2 e)): fold the sign and log2 e into the affine terms
            const float mr = s_co[2], ir = s_co[3] * -1.4426950408889634f;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                ar[k] *= ir;
                dr[k] = fmaf(-mr, ar[k], -1.4426950408889634f * dr[k]);
            }
        }
#pragma unroll
        for (int tb = 0; tb < kNormFrames; tb += FB) {
            if (tb > 0) issue(tb);
#pragma unroll
            for (int q = 0; q < FB; ++q) {
                const int tl = tb + q;
                if (tl < kNormFrames && tl < nt) {
                    float o[8];
                    if (has_y) {
                        unpack8(uy[q], o);
#pragma unroll
                        for (int k = 0; k < 8; ++k) o[k] = fmaf(o[k], a[k], d[k]);
                    } else {
#pragma unroll
                        for (int k = 0; k < 8; ++k) o[k] = 0.f;
                    }
                    if (MODE == 2) {
                        float rm[8], rr[8];
                        unpack8(um[q], rm);
                        unpack8(ur[q], rr);
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            // one MUFU each (exp2f / __fdividef add range fix-ups around theirs; flushed results are exact)
                            float e2, m;
                            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2) : "f"(fmaf(rm[k], ar[k], dr[k])));
                            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(m) : "f"(1.0f + e2));
                            o[k] = fmaf(m, rr[k] - o[k], o[k]);
                        }
                    }
                    uint4 uo;
                    __half2* ho = reinterpret_cast<__half2*>(&uo);
#pragma unroll
                    for (int k = 0; k < 4; ++k) ho[k] = __floats2half2_rn(o[2 * k], o[2 * k + 1]);
                    *reinterpret_cast<uint4*>(oh + tl * p.oT + f * p.oF + c) = uo;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) gru_pointwise_kernel(const float* __restrict__ gi, long long giB,
                                                            const float* __restrict__ gh,
                                                            const float* __restrict__ hprev, long long hB,
                                                            float* __restrict__ hout, int B, int H) {
    const long long total = (long long)B * H;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(i % H);
        const int b = (int)(i / H);
        const float* g = gi + b * giB;
        const float* h = gh + (long long)b * 3 * H;
        const float r = sigmoidf_(g[j] + h[j]);
        const float z = sigmoidf_(g[H + j] + h[H + j]);
        const float n = tanhf(g[2 * H + j] + r * h[2 * H + j]);
        const float hp = hprev[b * hB + j];
        hout[b * hB + j] = (1.0f - z) * n + z * hp;
    }
}

// grid (slices, B): a block moves one slice of kRollSlice floats of one entry of one stream; the launcher lays the
// entries' slices end to end (no empty blocks), four 16-byte loads per thread are in flight before the first store
constexpr int kRollSlice = 4096;
__global__ void __launch_bounds__(256) roll_kernel(RollTable tab, int first, int zero) {
    int ei = 0;
    while (ei + 1 < tab.n && (int)blockIdx.x >= tab.first_block[ei + 1]) ++ei;
    const RollEntry e = tab.e[ei];
    const int b = first + blockIdx.y;
    float* base = e.base + b * e.sB;
    const int n4 = e.count >> 2;
    const int i0 = ((int)blockIdx.x - tab.first_block[ei]) * (kRollSlice / 4) + threadIdx.x;
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int i = i0 + 256 * k;
        if (!zero && i < n4) v[k] = *reinterpret_cast<const float4*>(base + e.src_off + 4 * i);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = i0 + 256 * k;
        if (i < n4) *reinterpret_cast<float4*>(base + e.dst_off + 4 * i) = v[k];
    }
}

__global__ void set_io_kernel(IoDesc* dst, IoDesc v) { *dst = v; }

__global__ void __launch_bounds__(256) fill_noise_kernel(float* __restrict__ x, long long n, float amp) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        uint32_t h = (uint32_t)i * 2654435761u + (uint32_t)(i >> 32) * 40503u;
        h ^= h >> 15;
        h *= 2246822519u;
        h ^= h >> 13;
        x[i] = amp * ((float)(h >> 8) * (1.0f / 8388608.0f) - 1.0f);
    }
}

// utility.py:339-370 -- chunk n of stream b is row b*N+n = padded[n*P : n*P+K], padded = [P zeros | x | gap | P zeros]
__global__ void __launch_bounds__(256) segmentation_kernel(const float* __restrict__ x, int B, int C, long long L,
                                                           int K, int N, float* __restrict__ out) {
    const int P = K / 2;
    const long long total = (long long)B * N * C * K;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i % K);
        long long r = i / K;
        const int c = (int)(r % C);
        r /= C;
        const int n = (int)(r % N);
        const int b = (int)(r / N);
        const long long src = (long long)n * P + k - P;
        out[i] = (src >= 0 && src < L) ? x[((long long)b * C + c) * L + src] : 0.f;
    }
}

// utility.py:373-403 -- y[q] = (even(q) + odd(q)) / 2 for q in [P, N*P), then drop `gap` samples of tail
__global__ void __launch_bounds__(256) over_add_kernel(const float* __restrict__ chunks, int C, int N, int K, int gap,
                                                       float* __restrict__ out) {
    const int P = K / 2;
    const long long Lout = (long long)N * P - P - gap;
    const long long total = (long long)C * Lout;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long q = i % Lout + P;
        const int c = (int)(i / Lout);
        const int n1 = (int)(q / P);  // chunk starting at n1*P: offset q - n1*P in [0,P)
        const int n0 = n1 - 1;        // chunk starting at n0*P: offset in [P, K)
        const float a = chunks[((long long)c * N + n0) * K + (q - (long long)n0 * P)];
        const float b = chunks[((long long)c * N + n1) * K + (q - (long long)n1 * P)];
        // reference adds input1 (even chunks) + input2 (odd chunks): fp add is commutative, so order is immaterial
        out[i] = (a + b) / 2;
    }
}

inline int grid_for(long long n, int block = 256) {
    long long g = (n + block - 1) / block;
    const long long cap = 148LL * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

int launch_norm_apply(const NormApplyParams& p, cudaStream_t st) {
    SE_REQUIRE(p.C % 4 == 0, "norm_apply: C must be a multiple of 4");
    if (p.B <= 0 || p.T <= 0 || p.F <= 0) return 0;
    SE_REQUIRE(p.B <= 65535, "norm_apply: at most 65535 streams per launch");
    const dim3 grid((p.T + kNormFrames - 1) / kNormFrames, p.B);
    if (p.in_half && p.out_half && p.mode != 1 && p.C % 8 == 0 && p.oF % 8 == 0 && p.oT % 8 == 0 && p.oB % 8 == 0) {
        if (p.mode == 2) norm_apply_h8_kernel<2><<<grid, 256, 0, st>>>(p);
        else norm_apply_h8_kernel<0><<<grid, 256, 0, st>>>(p);
    } else {
        const int n4 = p.F * (p.C / 4);
        const int threads = n4 >= 256 ? 256 : (n4 >= 128 ? 128 : 64);
        norm_apply_kernel<<<grid, threads, 0, st>>>(p);
    }
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_gru_pointwise(const float* gi, long long giB, const float* gh, const float* hprev, long long hB,
                         float* hout, int B, int H, cudaStream_t st) {
    if (B == 0) return 0;
    gru_pointwise_kernel<<<grid_for((long long)B * H), 256, 0, st>>>(gi, giB, gh, hprev, hB, hout, B, H);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

static int roll_or_zero(const RollTable& tab_in, int first, int B, int zero, cudaStream_t st) {
    if (B == 0 || tab_in.n == 0) return 0;
    RollTable tab = tab_in;
    int blocks = 0;
    for (int i = 0; i < tab.n; ++i) {
        tab.first_block[i] = blocks;
        blocks += (tab.e[i].count + kRollSlice - 1) / kRollSlice;
    }
    tab.first_block[tab.n] = blocks;
    if (blocks == 0) return 0;
    // gridDim.y is limited to 65535 streams per launch
    for (int off = 0; off < B; off += 65535) {
        const int nb = (B - off) < 65535 ? (B - off) : 65535;
        roll_kernel<<<dim3(blocks, nb), 256, 0, st>>>(tab, first + off, zero);
        SE_CUDA_OK(cudaGetLastError());
    }
    return 0;
}
int launch_roll(const RollTable& tab, int first, int B, cudaStream_t st) { return roll_or_zero(tab, first, B, 0, st); }
int launch_zero(const RollTable& tab, int first, int B, cudaStream_t st) { return roll_or_zero(tab, first, B, 1, st); }

int launch_fill_noise(float* x, long long n, float amp, cudaStream_t st) {
    if (n <= 0) return 0;
    long long blocks = (n + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    fill_noise_kernel<<<(int)blocks, 256, 0, st>>>(x, n, amp);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_set_io(IoDesc* dst, const IoDesc& v, cudaStream_t st) {
    set_io_kernel<<<1, 1, 0, st>>>(dst, v);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_segmentation(const float* x, int B, int C, long long L, int K, int gap, int N, float* out,
                        cudaStream_t st) {
    (void)gap;
    const long long total = (long long)B * N * C * K;
    if (total == 0) return 0;
    segmentation_kernel<<<grid_for(total), 256, 0, st>>>(x, B, C, L, K, N, out);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_over_add(const float* chunks, int C, int N, int K, int gap, float* out, cudaStream_t st) {
    const long long total = (long long)C * ((long long)N * (K / 2) - K / 2 - gap);
    if (total <= 0) return 0;
    over_add_kernel<<<grid_for(total), 256, 0, st>>>(chunks, C, N, K, gap, out);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace se
