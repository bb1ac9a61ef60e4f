// STFT framing + Hamming window + real FFT-400 + input features, and its inverse: cIRM mask application + inverse
// real FFT-400 + window + intra-chunk overlap-add + envelope division + 50 % chunk overlap-add with a carried half.
//
// n_fft = 400 = 20 x 20 is not a power of two: both transforms are four-step (20-point DFT, twiddle, 20-point DFT)
// Cooley-Tukey factorizations staged entirely in shared memory, exploiting the Hermitian symmetry of a real signal.
//   forward : n = 20*n1 + n2, k = k1 + 20*k2 :  X[k] = sum_n2 W20^(n2 k2) * W400^(n2 k1) * sum_n1 x[n] W20^(n1 k1)
//   inverse : same indices, conjugate twiddles, X[400-k] = conj X[k], imag of DC / Nyquist ignored (C2R semantics
//             of torch.fft.irfft inside torch.istft).
// Reference call sites: CRN_ELU.py:417-424 (stft_trans), :369-373 (features), :401-405 + utility.py:439-442 (mask),
// CRN_ELU.py:426-432 (istft_trans), utility.py:393-403 (over_add).
#include <cuda_fp16.h>
#include <math.h>

#include <cstdlib>
#include <type_traits>
#include <vector>

#include "se_internal.h"

namespace se {

namespace {

constexpr int NFFT = 400;
constexpr int HOP = 160;
constexpr int NBIN = 201;
constexpr int T = kFramesPerChunk;  // 21
constexpr int K = 3200;             // chunk
constexpr int GROUP = 7;            // frames handled per pass
constexpr int ROW = 21;             // padded row length (float2) of the 20x20 intermediate

__constant__ float2 c_w20[20];    // exp(-2 pi i j / 20)
// tables indexed per thread live in global memory: a warp reading 32 different words of a __constant__ array is served
// one word at a time (the constant cache broadcasts, it does not gather)
__device__ __align__(16) float2 c_w400[400];  // exp(-2 pi i j / 400)  (16-byte aligned: cp.async source)
__device__ __align__(16) float c_window[NFFT];
__device__ float c_env[K];  // sum_t w^2 at output positions (istft window envelope, trimmed)

// 16-byte asynchronous copy into shared memory; src_bytes < 16 zero-fills the rest (0: nothing is read)
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(src), "r"(src_bytes)
                 : "memory");
}
__device__ __forceinline__ void cp_async_wait_all_groups() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// Branch-free atan2 for the fp16 feature layout (the result is rounded to fp16, 11 significant bits: absolute error
// >= 5e-4 for |phase| >= 1).  Odd minimax polynomial of degree 9 on [0, 1] (Hastings; |error| <= 1.1e-5 rad), octant
// folding by selects.  atan2(+-0, x < 0) = +-pi and atan2(0, 0) = 0 as in the exact function.
__device__ __forceinline__ float fast_atan2(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float a = __fdividef(mn, fmaxf(mx, 1e-37f));
    const float q = a * a;
    float r = fmaf(q, 0.0208351f, -0.0851330f);
    r = fmaf(q, r, 0.1801410f);
    r = fmaf(q, r, -0.3302995f);
    r = fmaf(q, r, 0.9998660f);
    r *= a;
    r = ay > ax ? 1.57079632679f - r : r;
    r = x < 0.f ? 3.14159265359f - r : r;
    return copysignf(r, y);
}
__device__ __forceinline__ float fast_sqrt(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b) {  // a * conj(b)
    return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}

// ------------------------------------------------------------------------------------------------------------
// STFT + features.  Work item (b, g) = frames [7g, 7g+7) of all microphones of stream b; a persistent grid of two blocks
// per SM walks the items, and the samples of a block's NEXT item are in flight (cp.async into the other half of a double
// buffer) while it transforms the current one.
// ------------------------------------------------------------------------------------------------------------
constexpr int SPAN = (GROUP - 1) * HOP + NFFT;  // 1360 padded samples cover 7 frames

struct StftSmem {
    alignas(16) float xs[2][3][SPAN];  // raw samples (zero outside the chunk), up to 3 mics per pass set; double buffer
    alignas(16) float win[NFFT];
    float2 w20[20];
    alignas(16) float2 w400[400];
    float2 y[3][GROUP][11][ROW];    // stage-1 output rows k1 = 0..10 (the rest by Hermitian symmetry), before the twiddle
    float2 spec[3][GROUP][NBIN + 1];
};

__global__ void __launch_bounds__(448, 2) stft_features_kernel(StftParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    StftSmem& s = *reinterpret_cast<StftSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int M = p.M;  // <= 3 per pass set (host guarantees M == 3 for the feature path)
    const int nitems = p.B * (T / GROUP);

    // Everything a block needs arrives by cp.async (16-byte units, zero fill where the frame window leaves the chunk or
    // the caller's signal): element-wise loads through registers exposed a DRAM round trip per loop iteration -- half of
    // the kernel's time in round 1 (profiles/r02_stft_regions.txt).
    for (int i = tid; i < NFFT / 4; i += blockDim.x) cp_async16_zfill(&s.win[4 * i], &c_window[4 * i], 16u);
    for (int i = tid; i < NFFT / 2; i += blockDim.x) cp_async16_zfill(&s.w400[2 * i], &c_w400[2 * i], 16u);
    if (tid < 20) s.w20[tid] = c_w20[tid];
    const long long stream_stride = p.io->in_stream_stride, mic_stride = p.io->in_mic_stride, in_len = p.io->in_len;
    const float* in_base = p.io->in;
    const long long in_offset = p.io->in_offset;
    // sample i of the span is chunk sample n = t0*HOP + i - NFFT/2 (center=True zero padding outside [0, K)) = signal
    // sample j = in_off + n (segmentation zero padding outside [0, in_len)); n of a 4-sample unit starts at a multiple of 4
    auto fetch = [&](int item, int buf) {
        const int b = item / (T / GROUP), t0 = (item % (T / GROUP)) * GROUP;
        const int brow = p.nb > 0 ? b % p.nb : b;  // training layout: stream = chunk * nb + utterance
        const float* in = in_base + brow * stream_stride;
        const long long in_off = in_offset + (p.nb > 0 ? (long long)(b / p.nb) * p.hop_chunk : 0);
        const bool vec_ok =
            ((reinterpret_cast<uintptr_t>(in) | (uintptr_t)(mic_stride * 4) | (uintptr_t)(in_off * 4)) & 15) == 0;
        if (vec_ok) {
            for (int u = tid; u < M * (SPAN / 4); u += blockDim.x) {
                const int m = u / (SPAN / 4), i = 4 * (u - m * (SPAN / 4));
                const int n = t0 * HOP + i - NFFT / 2;
                const long long j = in_off + n;
                long long left = (n >= 0 && n < K && j >= 0) ? in_len - j : 0;  // valid samples from j on
                left = left < 0 ? 0 : (left > 4 ? 4 : left);
                cp_async16_zfill(&s.xs[buf][m][i], in + m * mic_stride + (left > 0 ? j : 0), (uint32_t)left * 4u);
            }
        } else {
            for (int m = 0; m < M; ++m) {
                for (int i = tid; i < SPAN; i += blockDim.x) {
                    const int n = t0 * HOP + i - NFFT / 2;
                    const long long j = in_off + n;
                    s.xs[buf][m][i] = (n >= 0 && n < K && j >= 0 && j < in_len) ? in[m * mic_stride + j] : 0.f;
                }
            }
        }
    };
    if ((int)blockIdx.x < nitems) fetch(blockIdx.x, 0);
    int buf = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, buf ^= 1) {
    const int b = item / (T / GROUP), t0 = (item % (T / GROUP)) * GROUP;
    // this item's samples have landed; every thread is past the previous item's output phase (s.spec, s.y reusable) and
    // past its stage 1 (the other sample buffer is free for the prefetch)
    cp_async_wait_all_groups();
    __syncthreads();
    if (item + (int)gridDim.x < nitems) fetch(item + gridDim.x, buf ^ 1);

    // exp(-2 pi i j / 20) = (kC20[j], kS20[j]); both DFT stages are fully unrolled so that every twiddle is an immediate
    constexpr float kC20[20] = {1.0f, 0.951056516f, 0.809016994f, 0.587785252f, 0.309016994f, 0.0f, -0.309016994f, -0.587785252f, -0.809016994f, -0.951056516f, -1.0f, -0.951056516f, -0.809016994f, -0.587785252f, -0.309016994f, 0.0f, 0.309016994f, 0.587785252f, 0.809016994f, 0.951056516f};
    constexpr float kS20[20] = {0.0f, -0.309016994f, -0.587785252f, -0.809016994f, -0.951056516f, -1.0f, -0.951056516f, -0.809016994f, -0.587785252f, -0.309016994f, 0.0f, 0.309016994f, 0.587785252f, 0.809016994f, 0.951056516f, 1.0f, 0.951056516f, 0.809016994f, 0.587785252f, 0.309016994f};
    // ---- stage 1: per (mic, frame, n2) the 20-point DFT over n1 of the windowed real samples, k1 = 0..10 (the rest by
    //      Hermitian symmetry), then the twiddle W400^(n2 k1).  20 loads feed 200 FMAs held in registers.
    for (int u = tid; u < M * GROUP * 20; u += blockDim.x) {
        const int n2 = u % 20;
        const int fr = (u / 20) % GROUP;
        const int m = u / (20 * GROUP);
        const float* x = &s.xs[buf][m][fr * HOP];
        float v[20];
#pragma unroll
        for (int n1 = 0; n1 < 20; ++n1) v[n1] = x[20 * n1 + n2] * s.win[20 * n1 + n2];
        // W^((20-n) k) = conj(W^(n k)): inputs n and 20-n share a twiddle, so the sums run over their sum / difference
        float sp[10], dm[10];
#pragma unroll
        for (int n1 = 1; n1 <= 9; ++n1) {
            sp[n1] = v[n1] + v[20 - n1];
            dm[n1] = v[n1] - v[20 - n1];
        }
#pragma unroll
        for (int k1 = 0; k1 <= 10; ++k1) {
            float re = (k1 & 1) ? v[0] - v[10] : v[0] + v[10], im = 0.f;
#pragma unroll
            for (int n1 = 1; n1 <= 9; ++n1) {
                re = fmaf(sp[n1], kC20[(n1 * k1) % 20], re);
                im = fmaf(dm[n1], kS20[(n1 * k1) % 20], im);
            }
            s.y[m][fr][k1][n2] = make_float2(re, im);
        }
    }
    __syncthreads();
    // ---- stage 2: per (mic, frame, k1) the 20-point DFT over n2 -> bins k = k1 + 20 k2 <= 200 -------------------------
    for (int u = tid; u < M * GROUP * 20; u += blockDim.x) {
        const int k1 = u % 20;
        const int fr = (u / 20) % GROUP;
        const int m = u / (20 * GROUP);
        float2 yr[20];
        const int kr = k1 <= 10 ? k1 : 20 - k1;  // row 20-k1 is the conjugate of row k1 (real input)
        const float sg = k1 <= 10 ? 1.f : -1.f;
#pragma unroll
        for (int n2 = 0; n2 < 20; ++n2) {
            const float2 v = s.y[m][fr][kr][n2];
            yr[n2] = cmul(make_float2(v.x, sg * v.y), s.w400[n2 * k1]);  // twiddle W400^(n2 k1)
        }
        float2 sp2[10], dm2[10];
#pragma unroll
        for (int n2 = 1; n2 <= 9; ++n2) {
            sp2[n2] = make_float2(yr[n2].x + yr[20 - n2].x, yr[n2].y + yr[20 - n2].y);
            dm2[n2] = make_float2(yr[n2].x - yr[20 - n2].x, yr[n2].y - yr[20 - n2].y);
        }
#pragma unroll
        for (int k2 = 0; k2 <= 10; ++k2) {
            const int k = k1 + 20 * k2;
            if (k < NBIN) {
                // y[n] W + y[20-n] conj(W) = (sp.x c - dm.y s, dm.x s + sp.y c), sp / dm = sum / difference of the pair
                float re = (k2 & 1) ? yr[0].x - yr[10].x : yr[0].x + yr[10].x;
                float im = (k2 & 1) ? yr[0].y - yr[10].y : yr[0].y + yr[10].y;
#pragma unroll
                for (int n2 = 1; n2 <= 9; ++n2) {
                    const float wc = kC20[(n2 * k2) % 20], ws = kS20[(n2 * k2) % 20];
                    re = fmaf(sp2[n2].x, wc, re);
                    re = fmaf(-dm2[n2].y, ws, re);
                    im = fmaf(dm2[n2].x, ws, im);
                    im = fmaf(sp2[n2].y, wc, im);
                }
                // DC and Nyquist bins of a real signal are exactly real (pocketfft r2c returns +0 there)
                if (k == 0 || k == NBIN - 1) im = 0.f;
                s.spec[m][fr][k] = make_float2(re, im);
            }
        }
    }
    __syncthreads();

    // ---- outputs ---------------------------------------------------------------------------------------------
    if (p.spec_ref != nullptr) {  // reference layout [R][M][F][T][2]
        for (int o = tid; o < M * GROUP * NBIN; o += blockDim.x) {
            const int fr = o % GROUP;
            const int k = (o / GROUP) % NBIN;
            const int m = o / (GROUP * NBIN);
            const float2 v = s.spec[m][fr][k];
            float2* dst = reinterpret_cast<float2*>(p.spec_ref) + (((long long)b * M + m) * NBIN + k) * T + t0 + fr;
            *dst = v;
        }
    }
    if (p.feat != nullptr || p.feat_h8 != nullptr) {
        for (int o = tid; o < GROUP * NBIN; o += blockDim.x) {
            const int k = o % NBIN;
            const int fr = o / NBIN;
            const int t = t0 + fr;
            float mag[3], ph[3];
            if (p.feat_h8 != nullptr && !p.student) {  // fp16 feature layout: approximations far below the fp16 rounding
#pragma unroll
                for (int m = 0; m < 3; ++m) {
                    const float2 v = s.spec[m][fr][k];
                    mag[m] = fast_sqrt(fmaf(v.x, v.x, fmaf(v.y, v.y, 1e-10f)));
                    ph[m] = fast_atan2(v.y, v.x);
                }
            } else {
#pragma unroll
                for (int m = 0; m < 3; ++m) {
                    const float2 v = s.spec[m][fr][k];
                    mag[m] = sqrtf(v.x * v.x + v.y * v.y + 1e-10f);  // CRN_ELU.py:372
                    ph[m] = p.student ? atanf(v.y / (v.x + 1e-8f) + 1e-8f)  // distillation_crn.py:340
                                      : atan2f(v.y, v.x);                   // CRN_ELU.py:370
                }
            }
            if (p.feat_h8 != nullptr) {
                const __half2 h0 = __floats2half2_rn(mag[0], mag[1]), h1 = __floats2half2_rn(mag[2], ph[0] - ph[1]),
                              h2 = __floats2half2_rn(ph[0] - ph[2], 0.f);
                uint4 u;
                u.x = *reinterpret_cast<const unsigned*>(&h0);
                u.y = *reinterpret_cast<const unsigned*>(&h1);
                u.z = *reinterpret_cast<const unsigned*>(&h2);
                u.w = 0u;
                *reinterpret_cast<uint4*>(p.feat_h8 + b * p.fB + t * p.fT + k * p.fF) = u;
            } else {
                float* f = p.feat + b * p.fB + t * p.fT + k * p.fF;
                f[0] = mag[0];
                f[p.fC] = mag[1];
                f[2 * p.fC] = mag[2];
                f[3 * p.fC] = ph[0] - ph[1];
                f[4 * p.fC] = ph[0] - ph[2];
            }
            reinterpret_cast<float2*>(p.noisy)[((long long)b * T + t) * NBIN + k] = s.spec[0][fr][k];
        }
    }
    }  // items
}

// features from a reference-layout spectrum (TemporalCRN.forward entry, CRN_ELU.py:369-373)
__global__ void __launch_bounds__(256) features_from_spec_kernel(const float* __restrict__ spec, int B, int M,
                                                                 int student, float* __restrict__ feat, long long fB,
                                                                 long long fC, long long fT, long long fF,
                                                                 float* __restrict__ noisy, __half* feat_h8) {
    const long long total = (long long)B * T * NBIN;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i % NBIN);
        const int t = (int)((i / NBIN) % T);
        const int b = (int)(i / ((long long)NBIN * T));
        float mag[3], ph[3];
        float2 v0 = make_float2(0.f, 0.f);
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const float2 v = reinterpret_cast<const float2*>(spec)[(((long long)b * M + m) * NBIN + k) * T + t];
            if (m == 0) v0 = v;
            mag[m] = sqrtf(v.x * v.x + v.y * v.y + 1e-10f);
            ph[m] = student ? atanf(v.y / (v.x + 1e-8f) + 1e-8f) : atan2f(v.y, v.x);
        }
        if (feat_h8 != nullptr) {
            const __half2 h0 = __floats2half2_rn(mag[0], mag[1]), h1 = __floats2half2_rn(mag[2], ph[0] - ph[1]),
                          h2 = __floats2half2_rn(ph[0] - ph[2], 0.f);
            uint4 u;
            u.x = *reinterpret_cast<const unsigned*>(&h0);
            u.y = *reinterpret_cast<const unsigned*>(&h1);
            u.z = *reinterpret_cast<const unsigned*>(&h2);
            u.w = 0u;
            *reinterpret_cast<uint4*>(feat_h8 + b * fB + t * fT + k * fF) = u;
        } else {
            float* f = feat + b * fB + t * fT + k * fF;
            f[0] = mag[0];
            f[fC] = mag[1];
            f[2 * fC] = mag[2];
            f[3 * fC] = ph[0] - ph[1];
            f[4 * fC] = ph[0] - ph[2];
        }
        reinterpret_cast<float2*>(noisy)[((long long)b * T + t) * NBIN + k] = v0;
    }
}

// ------------------------------------------------------------------------------------------------------------
// mask + iSTFT + overlap-add.  grid = B, one block per stream; frames processed in 3 groups of 7.
// ------------------------------------------------------------------------------------------------------------
constexpr int ISTFT_STAGE_UNITS = (GROUP * NBIN * 8 + 15) / 16 + 1;  // 16-byte units covering 7 frames of float2 bins from an 8-byte aligned start
struct IstftSmem {
    union {  // the spectrum is dead once stage A has produced z; the windowed frames are written after that
        float2 spec[GROUP][NBIN + 1];
        float frames[GROUP][NFFT];
    };
    float2 z[GROUP][11][ROW];
    float ola[NFFT + HOP * (T - 1)];  // 3600
    alignas(16) float win[NFFT];     // cp.async destinations: 16-byte aligned
    float2 w20[20];
    alignas(16) float2 w400[400];
    // staging of one frame group of the mask pre-activation and of the noisy spectrum (cp.async; the next group is in
    // flight while the current one is transformed), and of the carried half chunk
    uint4 stage_y[ISTFT_STAGE_UNITS];
    uint4 stage_x[ISTFT_STAGE_UNITS];
    alignas(16) float carry[K / 2];
    float co[2];  // mean and 1 / denominator of the GlobalLayerNorm in front of the mask
};

__device__ __forceinline__ float decompress_cirm(float m) {  // utility.py:439-442
    const float limit = 9.9f;
    const float ge = (m >= limit) ? 1.f : 0.f;
    const float le = (m <= -limit) ? 1.f : 0.f;
    const float in = (fabsf(m) < limit) ? 1.f : 0.f;
    m = limit * ge - limit * le + m * in;
    return -10.f * logf((10.f - m) / (10.f + m));
}

// The same function for the tensor-core precisions: log(a / b) = ln2 (lg2 a - lg2 b) with two MUFU.LG2 (absolute error of
// the mask ~1e-6, three orders below the tf32 / fp16 operand rounding); the clamp is the same selection written as min / max.
__device__ __forceinline__ float decompress_cirm_fast(float m) {
    m = fminf(fmaxf(m, -9.9f), 9.9f);
    float la, lb;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(la) : "f"(10.f - m));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lb) : "f"(10.f + m));
    return -6.93147180560f * (la - lb);
}

// 3 CTAs per SM (80 registers): the unrolled inverse stages want 110 registers, which left 2 CTAs per SM (0.157 vs 0.128 ms)
__global__ void __launch_bounds__(256, 3) mask_istft_kernel(MaskIstftParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    IstftSmem& s = *reinterpret_cast<IstftSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int b = blockIdx.x;

    // Global data arrives by cp.async and is awaited once per frame group: the per-bin loads of the mask / spectrum and
    // the carried half chunk used to expose a DRAM round trip per loop iteration (55 % of the kernel's samples).
    const bool staged = p.spec_in == nullptr;
    const float2* gy = reinterpret_cast<const float2*>(p.y) + (long long)b * T * NBIN;
    const float2* gx = reinterpret_cast<const float2*>(p.noisy) + (long long)b * T * NBIN;
    // group g = float2 elements [g*7*201, (g+1)*7*201) of the stream: copied in 16-byte units from the aligned address
    // at or below its first element (`skew` = 0 or 1 float2 of lead-in; the unit after the last element stays inside
    // the stream's block or the next stream's -- the last stream of the buffer is clamped)
    auto stage_group = [&](int g) {
        const float2* y0 = gy + g * GROUP * NBIN;
        const float2* x0 = gx + g * GROUP * NBIN;
        const int sky = (int)((reinterpret_cast<uintptr_t>(y0) >> 3) & 1), skx = (int)((reinterpret_cast<uintptr_t>(x0) >> 3) & 1);
        const int need_y = (GROUP * NBIN + sky + 1) / 2, need_x = (GROUP * NBIN + skx + 1) / 2;  // units holding data
        for (int i = tid; i < need_y; i += blockDim.x) {
            // the last unit may reach one float2 past the group: only past the END OF THE TENSOR is that out of bounds
            const bool tail = (i == need_y - 1) && (((GROUP * NBIN + sky) & 1) != 0) && b == p.B - 1 && g == T / GROUP - 1;
            cp_async16_zfill(&s.stage_y[i], reinterpret_cast<const uint4*>(y0 - sky) + i, tail ? 8u : 16u);
        }
        for (int i = tid; i < need_x; i += blockDim.x) {
            const bool tail = (i == need_x - 1) && (((GROUP * NBIN + skx) & 1) != 0) && b == p.B - 1 && g == T / GROUP - 1;
            cp_async16_zfill(&s.stage_x[i], reinterpret_cast<const uint4*>(x0 - skx) + i, tail ? 8u : 16u);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int i = tid; i < NFFT / 4; i += blockDim.x) cp_async16_zfill(&s.win[4 * i], &c_window[4 * i], 16u);
    for (int i = tid; i < NFFT / 2; i += blockDim.x) cp_async16_zfill(&s.w400[2 * i], &c_w400[2 * i], 16u);
    if (staged) stage_group(0);
    const bool carry_vec = p.carry != nullptr && (reinterpret_cast<uintptr_t>(p.carry) & 15) == 0;
    if (carry_vec) {
        const float* c = p.carry + (long long)b * (K / 2);
        for (int i = tid; i < K / 8; i += blockDim.x) cp_async16_zfill(&s.carry[4 * i], c + 4 * i, 16u);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    if (tid < 20) s.w20[tid] = c_w20[tid];
    for (int i = tid; i < NFFT + HOP * (T - 1); i += blockDim.x) s.ola[i] = 0.f;

    float mean = 0.f, inv = 0.f, w0 = 0.f, w1 = 0.f, b0 = 0.f, b1 = 0.f;
    if (p.spec_in == nullptr) {
        if (tid == 0) {  // one thread does the double-precision arithmetic (it was 15 % of the samples on all 256)
            const double sum = p.stats[2 * b], ssq = p.stats[2 * b + 1];
            const double mu = sum / p.count;
            double var = ssq / p.count - mu * mu;
            if (var < 0.0) var = 0.0;
            const float varf = (float)var;
            const float den = p.student ? (sqrtf(varf) + 1e-8f) : (sqrtf(varf + 1e-8f) + 1e-8f);
            s.co[0] = (float)mu;
            s.co[1] = 1.f / den;
        }
        w0 = p.w[0];
        w1 = p.w[1];
        b0 = p.b[0];
        b1 = p.b[1];
    }

    for (int g = 0; g < T / GROUP; ++g) {
        const int t0 = g * GROUP;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();  // staged group g (and, the first time, tables / carry) visible; previous group's frames consumed
        mean = s.co[0];
        inv = s.co[1];
        const float2* sy = reinterpret_cast<const float2*>(s.stage_y) +
                           ((reinterpret_cast<uintptr_t>(gy + g * GROUP * NBIN) >> 3) & 1);
        const float2* sx = reinterpret_cast<const float2*>(s.stage_x) +
                           ((reinterpret_cast<uintptr_t>(gx + g * GROUP * NBIN) >> 3) & 1);
        // ---- enhanced spectrum of this frame group -----------------------------------------------------------
        for (int o = tid; o < GROUP * NBIN; o += blockDim.x) {
            const int k = o % NBIN;
            const int fr = o / NBIN;
            const int t = t0 + fr;
            float2 e;
            if (p.spec_in != nullptr) {
                e = reinterpret_cast<const float2*>(p.spec_in)[((long long)b * NBIN + k) * T + t];
                if (p.adjoint) {  // sum_k Re(D_k e^{+2 pi i k n / N}) = C2R inverse of (N D_0, N/2 D_1 .. N/2 D_199, N D_200)
                    const float sc = (k == 0 || k == NBIN - 1) ? (float)NFFT : (float)(NFFT / 2);
                    e.x *= sc;
                    e.y *= sc;
                }
            } else {
                const float2 y = sy[o];  // element (t0 + fr, k) of the stream = o-th of the staged group
                const float2 x = sx[o];
                const float ar = (y.x - mean) * inv * w0 + b0, ai = (y.y - mean) * inv * w1 + b1;
                const float mr = p.fast ? decompress_cirm_fast(ar) : decompress_cirm(ar);
                const float mi = p.fast ? decompress_cirm_fast(ai) : decompress_cirm(ai);
                e = make_float2(mr * x.x - mi * x.y, mi * x.x + mr * x.y);  // CRN_ELU.py:402-403
                if (p.spec_ref != nullptr)
                    reinterpret_cast<float2*>(p.spec_ref)[((long long)b * NBIN + k) * T + t] = e;
            }
            if (k == 0 || k == NBIN - 1) e.y = 0.f;  // C2R: imaginary parts of DC / Nyquist are ignored
            s.spec[fr][k] = e;
        }
        __syncthreads();  // spectrum complete; the staging buffers are free for the next group
        if (staged && g + 1 < T / GROUP) stage_group(g + 1);
        if (p.spec_ref != nullptr && p.out_chunk == nullptr && p.carry == nullptr) continue;  // forward(): no iSTFT

        // exp(-2 pi i j / 20) = (kC20[j], kS20[j]); both stages are fully unrolled so that every twiddle is an immediate
        constexpr float kC20[20] = {1.0f, 0.951056516f, 0.809016994f, 0.587785252f, 0.309016994f, 0.0f, -0.309016994f, -0.587785252f, -0.809016994f, -0.951056516f, -1.0f, -0.951056516f, -0.809016994f, -0.587785252f, -0.309016994f, 0.0f, 0.309016994f, 0.587785252f, 0.809016994f, 0.951056516f};
        constexpr float kS20[20] = {0.0f, -0.309016994f, -0.587785252f, -0.809016994f, -0.951056516f, -1.0f, -0.951056516f, -0.809016994f, -0.587785252f, -0.309016994f, 0.0f, 0.309016994f, 0.587785252f, 0.809016994f, 0.951056516f, 1.0f, 0.951056516f, 0.809016994f, 0.587785252f, 0.309016994f};
        // ---- stage A: z[k1][n2] = sum_k2 Xfull[k1 + 20 k2] * conj(W20)^(n2 k2), then * conj(W400)^(n2 k1) -------
        // register-blocked like the forward transform: a thread loads the 20 inputs of one (frame, k1) once and produces
        // 10 of the 20 outputs with immediate twiddles (40 loads feed 360 FMAs; the loop version spent 40 shared-memory
        // loads per 80 FMAs)
        for (int o = tid; o < GROUP * 11 * 2; o += blockDim.x) {
            const int half = o & 1;
            const int k1 = (o >> 1) % 11;
            const int fr = o / 22;
            float2 v[20];
#pragma unroll
            for (int k2 = 0; k2 < 20; ++k2) {
                const int k = k1 + 20 * k2;
                if (k <= 200) {
                    v[k2] = s.spec[fr][k];
                } else {
                    v[k2] = s.spec[fr][NFFT - k];
                    v[k2].y = -v[k2].y;
                }
            }
            // v[k] conj(w) + v[20-k] w = (sp.x c + dm.y s, sp.y c - dm.x s), sp / dm = sum / difference of the pair
            float2 sp[10], dm[10];
#pragma unroll
            for (int k2 = 1; k2 <= 9; ++k2) {
                sp[k2] = make_float2(v[k2].x + v[20 - k2].x, v[k2].y + v[20 - k2].y);
                dm[k2] = make_float2(v[k2].x - v[20 - k2].x, v[k2].y - v[20 - k2].y);
            }
            auto emit = [&](auto n2c) {
                constexpr int n2 = decltype(n2c)::value;
                float re = (n2 & 1) ? v[0].x - v[10].x : v[0].x + v[10].x;
                float im = (n2 & 1) ? v[0].y - v[10].y : v[0].y + v[10].y;
#pragma unroll
                for (int k2 = 1; k2 <= 9; ++k2) {  // w = (kC20, kS20)[(n2 k2) % 20]
                    const float wc = kC20[(n2 * k2) % 20], ws = kS20[(n2 * k2) % 20];
                    re = fmaf(sp[k2].x, wc, re);
                    re = fmaf(dm[k2].y, ws, re);
                    im = fmaf(sp[k2].y, wc, im);
                    im = fmaf(-dm[k2].x, ws, im);
                }
                s.z[fr][k1][n2] = cmul_conj(make_float2(re, im), s.w400[n2 * k1]);
            };
            if (half == 0) {
                emit(std::integral_constant<int, 0>{}); emit(std::integral_constant<int, 1>{}); emit(std::integral_constant<int, 2>{});
                emit(std::integral_constant<int, 3>{}); emit(std::integral_constant<int, 4>{}); emit(std::integral_constant<int, 5>{});
                emit(std::integral_constant<int, 6>{}); emit(std::integral_constant<int, 7>{}); emit(std::integral_constant<int, 8>{});
                emit(std::integral_constant<int, 9>{});
            } else {
                emit(std::integral_constant<int, 10>{}); emit(std::integral_constant<int, 11>{}); emit(std::integral_constant<int, 12>{});
                emit(std::integral_constant<int, 13>{}); emit(std::integral_constant<int, 14>{}); emit(std::integral_constant<int, 15>{});
                emit(std::integral_constant<int, 16>{}); emit(std::integral_constant<int, 17>{}); emit(std::integral_constant<int, 18>{});
                emit(std::integral_constant<int, 19>{});
            }
        }
        __syncthreads();
        // ---- stage C: x[20 n1 + n2] = (z0 + (-1)^n1 z10 + 2 sum_{k1=1..9} Re(z[k1] conj(W20)^(n1 k1))) / 400 ----
        // one thread per (frame, n2): 11 inputs in registers, all 20 outputs n1 with immediate twiddles
        for (int o = tid; o < GROUP * 20; o += blockDim.x) {
            const int n2 = o % 20;
            const int fr = o / 20;
            float2 zv[11];
#pragma unroll
            for (int k1 = 0; k1 <= 10; ++k1) zv[k1] = s.z[fr][k1][n2];
            // outputs n1 and 20 - n1 share the cosine sum and differ in the sign of the sine sum
#pragma unroll
            for (int n1 = 0; n1 <= 10; ++n1) {
                float ac = 0.f, as = 0.f;
#pragma unroll
                for (int k1 = 1; k1 <= 9; ++k1) {  // Re(z * conj(w)), w = (kC20, kS20)[(n1 k1) % 20]
                    ac = fmaf(zv[k1].x, kC20[(n1 * k1) % 20], ac);
                    as = fmaf(zv[k1].y, kS20[(n1 * k1) % 20], as);
                }
                const float base = zv[0].x + ((n1 & 1) ? -zv[10].x : zv[10].x);
                const int n = 20 * n1 + n2;
                s.frames[fr][n] = (base + 2.f * (ac + as)) * (1.0f / NFFT) * s.win[n];
                if (n1 >= 1 && n1 <= 9) {
                    const int m = 20 * (20 - n1) + n2;
                    s.frames[fr][m] = (base + 2.f * (ac - as)) * (1.0f / NFFT) * s.win[m];
                }
            }
        }
        __syncthreads();
        // ---- overlap-add of this group's frames (deterministic order: ascending frame) ---------------------------
        // only the SPAN positions this group's frames reach, and per position only the <= 3 frames that cover it
        for (int rel = tid; rel < SPAN; rel += blockDim.x) {
            const int pos = t0 * HOP + rel;
            float acc = s.ola[pos];
            const int hi = min(GROUP - 1, rel / HOP);
            const int lo = rel < NFFT ? 0 : (rel - NFFT) / HOP + 1;
            for (int fr = lo; fr <= hi; ++fr) acc += s.frames[fr][rel - fr * HOP];
            s.ola[pos] = acc;
        }
        __syncthreads();
    }
    if (p.spec_ref != nullptr && p.out_chunk == nullptr && p.carry == nullptr) return;

    // ---- envelope division, trim n_fft/2, chunk-level 50 % overlap-add with the carried half ---------------------
    constexpr int P = K / 2;
    if (p.out_chunk != nullptr) {
        for (int n = tid; n < K; n += blockDim.x)
            p.out_chunk[(long long)b * K + n] = p.adjoint ? s.ola[NFFT / 2 + n] : s.ola[NFFT / 2 + n] / c_env[n];
    }
    if (p.carry != nullptr) {
        float* out = p.io->out + b * p.io->out_stream_stride;
        const int n_valid = p.io->n_valid;
        float* carry = p.carry + (long long)b * P;
        for (int n = tid; n < P; n += blockDim.x) {
            const float first = s.ola[NFFT / 2 + n] / c_env[n];
            const float second = s.ola[NFFT / 2 + P + n] / c_env[P + n];
            if (n < n_valid) out[n] = (first + (carry_vec ? s.carry[n] : carry[n])) / 2;  // utility.py:397-399
            carry[n] = second;
        }
    }
}


// ------------------------------------------------------------------------------------------------------------
// training layout (stream s = n*nb + i = chunk n of utterance i): chunk-level overlap-add and the adjoints of
// over_add / iSTFT / mask (the adjoint of the iSTFT is the STFT of dchunk / envelope scaled by c_k / n_fft)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) over_add_cm_kernel(const float* __restrict__ chunks, int nb, int N, int front,
                                                          long long L, float scale, float* __restrict__ pred) {
    constexpr int P = K / 2;
    const long long total = (long long)nb * L;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int u = (int)(i / L);
        const long long q = i - (long long)u * L + P + front;  // position on the padded grid (utility.py:393-403)
        const int n1 = (int)(q / P);
        float a = 0.f, b = 0.f;
        if (n1 >= 1 && n1 - 1 < N) a = chunks[((long long)(n1 - 1) * nb + u) * K + (q - (long long)(n1 - 1) * P)];
        if (n1 < N) b = chunks[((long long)n1 * nb + u) * K + (q - (long long)n1 * P)];
        pred[i] = (a + b) * scale;
    }
}

__global__ void __launch_bounds__(256) over_add_cm_bwd_kernel(const float* __restrict__ dpred, int nb, int N, int front,
                                                              long long L, float* __restrict__ dchunks) {
    constexpr int P = K / 2;
    const long long total = (long long)nb * N * K;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(i % K);
        const long long s = i / K;
        const int u = (int)(s % nb), n = (int)(s / nb);
        const long long q = (long long)n * P + j;
        const long long jj = q - P - front;
        float v = 0.f;
        if (q >= P && q < (long long)N * P && jj >= 0 && jj < L) v = 0.5f * dpred[(long long)u * L + jj] / c_env[j];
        dchunks[i] = v;
    }
}

__device__ __forceinline__ float decompress_cirm_grad(float m) {  // d/dm of utility.py:439-442
    return fabsf(m) < 9.9f ? 200.f / (100.f - m * m) : 0.f;
}

__global__ void __launch_bounds__(256) mask_bwd_kernel(MaskBwdParams p) {
    const long long per = (long long)T * NBIN;
    const long long total = per * p.B;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / per);
        const int r = (int)(i - b * per);
        const int t = r / NBIN, k = r - t * NBIN;
        const double sum = p.stats[2 * b], ssq = p.stats[2 * b + 1];
        const double mu = sum / p.count;
        double var = ssq / p.count - mu * mu;
        if (var < 0.0) var = 0.0;
        const float varf = (float)var;
        const float den = p.student ? (sqrtf(varf) + 1e-8f) : (sqrtf(varf + 1e-8f) + 1e-8f);
        const float mean = (float)mu, inv = 1.f / den;
        float2 d = reinterpret_cast<const float2*>(p.dspec)[((long long)b * NBIN + k) * T + t];
        const bool edge = (k == 0 || k == NBIN - 1);
        const float ck = (edge ? 1.f : 2.f) / NFFT;  // adjoint of the C2R transform
        d.x *= ck;
        d.y = edge ? 0.f : d.y * ck;
        const float2 y = reinterpret_cast<const float2*>(p.y)[i];
        const float2 x = reinterpret_cast<const float2*>(p.noisy)[i];
        const float m0 = (y.x - mean) * inv * p.w[0] + p.b[0];
        const float m1 = (y.y - mean) * inv * p.w[1] + p.b[1];
        const float dmr = d.x * x.x + d.y * x.y;   // E = M * X (complex): dM = dE * conj(X)
        const float dmi = -d.x * x.y + d.y * x.x;
        reinterpret_cast<float2*>(p.g)[i] = make_float2(dmr * decompress_cirm_grad(m0), dmi * decompress_cirm_grad(m1));
        if (p.dnoisy != nullptr) {  // E = M * X: dX = dE * conj(M), M the decompressed mask
            const float mr = decompress_cirm(m0), mi = decompress_cirm(m1);
            reinterpret_cast<float2*>(p.dnoisy)[i] = make_float2(d.x * mr + d.y * mi, -d.x * mi + d.y * mr);
        }
    }
}

// Adjoint of the input features (CRN_ELU.py:369-373; student phase distillation_crn.py:340), following torch's autograd
// of the reference expressions: mag_m = sqrt(re^2 + im^2 + 1e-10), ipd_m = angle_0 - angle_m (m = 1, 2); the mic-0
// spectrum also receives `dnoisy` (the mask multiply).  One thread per (stream, bin, frame), frames fastest.
__global__ void __launch_bounds__(256) features_bwd_kernel(FeatBwdParams p) {
    const long long per = (long long)NBIN * T;
    const long long total = per * p.B;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / per);
        const int r = (int)(i - b * per);
        const int k = r / T, t = r - k * T;
        const float* g = p.dfeat + b * p.fB + t * p.fT + k * p.fF;
        const float g3 = g[3 * p.fC], g4 = g[4 * p.fC];
        const float dang[3] = {g3 + g4, -g3, -g4};
        const float2* spec = reinterpret_cast<const float2*>(p.spec) + (long long)b * 3 * per;
        float2* dspec = reinterpret_cast<float2*>(p.dspec) + (long long)b * 3 * per;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const float2 v = spec[m * per + r];
            const float re = v.x, im = v.y;
            const float gm = g[m * p.fC] / sqrtf(re * re + im * im + 1e-10f);
            float dre = gm * re, dim = gm * im;
            if (p.student) {  // arctan(u), u = im / (re + 1e-8) + 1e-8
                const float den = re + 1e-8f;
                const float u = im / den + 1e-8f;
                const float du = dang[m] / (1.f + u * u);
                dim += du / den;
                dre += -du * im / (den * den);
            } else {  // atan2(im, re): (re, -im) / |X|^2, exactly 0 at re = im = 0 as torch.atan2's backward
                const float r2 = re * re + im * im;
                if (r2 > 0.f) {
                    const float rc = 1.f / r2;
                    dim += dang[m] * re * rc;
                    dre += -dang[m] * im * rc;
                }
            }
            if (m == 0) {
                const float2 dn = reinterpret_cast<const float2*>(p.dnoisy)[((long long)b * T + t) * NBIN + k];
                dre += dn.x;
                dim += dn.y;
            }
            dspec[m * per + r] = make_float2(dre, dim);
        }
    }
}

}  // namespace

int init_fft_tables() {
    std::vector<float2> w20(20), w400(400);
    std::vector<float> win(NFFT), env(K);
    const double pi = 3.14159265358979323846;
    for (int j = 0; j < 20; ++j) w20[j] = make_float2((float)cos(2 * pi * j / 20), (float)(-sin(2 * pi * j / 20)));
    for (int j = 0; j < 400; ++j) w400[j] = make_float2((float)cos(2 * pi * j / 400), (float)(-sin(2 * pi * j / 400)));
    // exact quadrant values (avoid 6e-17 residues turning into sign noise)
    w20[0] = make_float2(1.f, 0.f);
    w20[5] = make_float2(0.f, -1.f);
    w20[10] = make_float2(-1.f, 0.f);
    w20[15] = make_float2(0.f, 1.f);
    w400[0] = make_float2(1.f, 0.f);
    w400[100] = make_float2(0.f, -1.f);
    w400[200] = make_float2(-1.f, 0.f);
    w400[300] = make_float2(0.f, 1.f);
    for (int n = 0; n < NFFT; ++n) win[n] = (float)(0.54 - 0.46 * cos(2 * pi * n / NFFT));  // periodic Hamming
    std::vector<double> full(NFFT + HOP * (T - 1), 0.0);
    for (int t = 0; t < T; ++t)
        for (int n = 0; n < NFFT; ++n) full[t * HOP + n] += (double)win[n] * (double)win[n];
    for (int n = 0; n < K; ++n) env[n] = (float)full[NFFT / 2 + n];
    SE_CUDA_OK(cudaMemcpyToSymbol(c_w20, w20.data(), sizeof(float2) * 20));
    SE_CUDA_OK(cudaMemcpyToSymbol(c_w400, w400.data(), sizeof(float2) * 400));
    SE_CUDA_OK(cudaMemcpyToSymbol(c_window, win.data(), sizeof(float) * NFFT));
    SE_CUDA_OK(cudaMemcpyToSymbol(c_env, env.data(), sizeof(float) * K));
    SE_CUDA_OK(cudaFuncSetAttribute(stft_features_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(StftSmem)));
    SE_CUDA_OK(cudaFuncSetAttribute(mask_istft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(IstftSmem)));
    return 0;
}

int launch_stft_features(const StftParams& p, cudaStream_t st) {
    SE_REQUIRE(p.M >= 1 && p.M <= 3, "stft: at most 3 microphones per launch");
    SE_REQUIRE((p.feat == nullptr && p.feat_h8 == nullptr) || p.M == 3,
               "stft features need exactly 3 microphones (CRN_ELU.py:369-373)");
    if (p.B == 0) return 0;
    // 420 (mic, frame, n2) units per stage: one round of a block's 448 threads; two blocks per SM (28 warps) walk the
    // B x 3 items, stream-major (the three frame groups of a stream share 240 + 240 input samples through L2)
    int num_sms = 0;
    if (num_sms_current_device(&num_sms)) return 1;
    const int nitems = p.B * (T / GROUP);
    const int grid = nitems < 2 * num_sms ? nitems : 2 * num_sms;
    stft_features_kernel<<<grid, 448, sizeof(StftSmem), st>>>(p);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_features_from_spec(const float* spec, int B, int M, int student, float* feat, long long fB, long long fC,
                              long long fT, long long fF, float* noisy, cudaStream_t st, __half* feat_h8) {
    SE_REQUIRE(M == 3, "features need exactly 3 microphones (CRN_ELU.py:369-373)");
    if (B == 0) return 0;
    const long long total = (long long)B * T * NBIN;
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    features_from_spec_kernel<<<grid, 256, 0, st>>>(spec, B, M, student, feat, fB, fC, fT, fF, noisy, feat_h8);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_mask_istft(const MaskIstftParams& p, cudaStream_t st) {
    if (p.B == 0) return 0;
    mask_istft_kernel<<<p.B, 256, sizeof(IstftSmem), st>>>(p);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_over_add_cm(const float* chunks, int nb, int N, int Kc, int front, long long L, float* pred, cudaStream_t st,
                       float scale) {
    SE_REQUIRE(Kc == K, "over_add_cm: chunk length must be 3200");
    const long long total = (long long)nb * L;
    if (total <= 0) return 0;
    long long g = (total + 255) / 256;
    over_add_cm_kernel<<<(int)(g > 2368 ? 2368 : g), 256, 0, st>>>(chunks, nb, N, front, L, scale, pred);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_over_add_cm_bwd(const float* dpred, int nb, int N, int Kc, int front, long long L, float* dchunks,
                           cudaStream_t st) {
    SE_REQUIRE(Kc == K, "over_add_cm_bwd: chunk length must be 3200");
    const long long total = (long long)nb * N * K;
    if (total <= 0) return 0;
    long long g = (total + 255) / 256;
    over_add_cm_bwd_kernel<<<(int)(g > 2368 ? 2368 : g), 256, 0, st>>>(dpred, nb, N, front, L, dchunks);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_features_bwd(const FeatBwdParams& p, cudaStream_t st) {
    if (p.B <= 0) return 0;
    const long long total = (long long)p.B * T * NBIN;
    long long g = (total + 255) / 256;
    features_bwd_kernel<<<(int)(g > 2368 ? 2368 : g), 256, 0, st>>>(p);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_mask_bwd(const MaskBwdParams& p, cudaStream_t st) {
    if (p.B <= 0) return 0;
    const long long total = (long long)p.B * T * NBIN;
    long long g = (total + 255) / 256;
    mask_bwd_kernel<<<(int)(g > 2368 ? 2368 : g), 256, 0, st>>>(p);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace se
