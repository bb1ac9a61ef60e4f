// Gated skip path of the 32- and 64-channel decoder levels (CRN_ELU.py:297-306), fp16 operand mode, as ONE launch:
//   o   = GLN_norm(y) (zero on the bins past Fy, as F.pad)          y = ELU(deconv), statistics from its GEMM's epilogue
//   m   = sigmoid(GLN_residualnorm(residualmask(skip)))
//   r   = ELU(residual(skip))
//   out = m r + (1 - m) o                                            -> the next level's zero-bordered input interior
// One stream per CTA at a time.  The mask GlobalLayerNorm needs whole-stream statistics before any output can be formed,
// which the two-launch form (1x1 pair GEMM + blend kernel) paid for with an fp16 round trip of the mask pre-activation
// and of elu(residual) through HBM.  Here the stream's skip tensor (T x Fs positions, C channels) is one TMA box in
// shared memory (canonical K-major layout, SWIZZLE_128B rows for C = 64, SWIZZLE_64B for C = 32), and
//   pass 1: the mask MMAs of every 128-row tile go to TMEM and STAY there (NT x C columns); the epilogue reduces their
//           statistics (per thread in fp32, across the CTA in fp64 in a fixed order: no atomics, deterministic);
//   pass 2: the residual MMAs run tile by tile into a double-buffered 2 x C column region, and the epilogue forms `out`
//           from both accumulators and y and stores it with 16-byte stores.
// y arrives as a second TMA box per stream (one buffer, issued when the stream starts so that it lands during pass 1;
// swizzled like the skip rows, so the epilogue's row-per-thread reads are conflict-free).  The tiles start at
// min(128 m, roundup8(P) - 128), so the last one overlaps its predecessor instead of running past the buffer; its
// overlapped rows are neither counted nor stored twice.  The next stream's skip box (double-buffered) and an L2 prefetch
// of its y slab are issued when a stream starts, so HBM streams while the tensor pipe and the epilogue work.  The
// epilogue costs two MUFU ops per output (ex2 for the ELU, tanh for the sigmoid), 16 warps of it.
//
// Roles: warps 0-15 = epilogue (warp (q, cg): TMEM lanes 32 q .. 32 q + 31, channel quarter cg), warp 16 = TMA and MMA
// issuer (warp-uniform loop, one elected lane issues).
#include <cuda_fp16.h>
#include <stdint.h>

#include "mma_util.cuh"
#include "se_internal.h"

namespace se {
namespace {

using namespace mma_util;
constexpr int T = kFramesPerChunk;  // 21
constexpr int BM = 128;
constexpr int kEpiWarps = 16;
constexpr int kMmaWarp = kEpiWarps;
constexpr int kSbWarps = kEpiWarps + 1;
constexpr int kSbThreads = kSbWarps * 32;  // 544
constexpr int kMaxTiles = 16;
constexpr uint32_t kTmemCols = 512;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    uint64_t t0 = 0;
    for (uint32_t spins = 1;; ++spins) {
        if (mbar_try_wait(bar, parity)) return;
        if ((spins & 1023u) == 0) {  // protocol bug: fail loudly (after ~2 s) instead of hanging the GPU
            const uint64_t t = global_ns();
            if (t0 == 0) t0 = t;
            else if (t - t0 > 2000000000ull) __trap();
        }
    }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
template <int N>
__device__ __forceinline__ void tmem_ld_nowait(uint32_t taddr, uint32_t* r) {
    if (N == 16) tmem_ld16_nowait(taddr, r);
    else tmem_ld8_nowait(taddr, r);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// canonical no-swizzle K-major descriptor (the weights): 8-row core matrices of 16-byte rows, SBO bytes between core
// matrices along the rows, LBO bytes between the two 16-byte K chunks of one MMA
__device__ __forceinline__ uint64_t desc_nosw(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

template <int C>
struct SbCfg {
    static_assert(C == 32 || C == 64, "skip_blend_tc: 32 or 64 channels");
    static constexpr int ROWB = 2 * C;               // bytes of one position row of the skip operand (= swizzle span)
    static constexpr uint32_t SBO = 8 * ROWB;        // bytes between 8-row groups
    static constexpr uint64_t LAYOUT = C == 64 ? 2 : 4;  // UMMA layout type: SWIZZLE_128B / SWIZZLE_64B
    static constexpr int KS = C / 16;                // MMAs (K = 16) per tile and matrix
    static constexpr int CW = C / 4;                 // channels per epilogue thread
    static constexpr int W_BYTES = C * C * 2;        // one of the two weight matrices
    static constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
};

// K-major swizzled descriptor of the skip operand (rows of ROWB bytes, as the TMA box lands them)
template <int C>
__device__ __forceinline__ uint64_t desc_skip(uint32_t addr) {
    using S = SbCfg<C>;
    return (uint64_t)((addr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)(S::SBO >> 4) << 32) | (1ull << 46) |
           (S::LAYOUT << 61);
}

constexpr int kBars = 3 + kMaxTiles + 4;  // skip full x 2, y full, mask full per tile, residual full / free x 2
struct SbLayout {  // byte offsets into the 1024-aligned dynamic shared memory
    int P, Pr, NT;
    int a_bytes, off_y, off_w, off_par, off_red, off_bar, bytes;
};
__host__ __device__ inline SbLayout sb_layout(int C, int Fs, int Fy) {
    SbLayout l;
    l.P = T * Fs;
    l.Pr = (l.P + 7) / 8 * 8;
    l.NT = (l.Pr + BM - 1) / BM;
    l.a_bytes = (l.Pr * 2 * C + 1023) / 1024 * 1024;
    l.off_y = 2 * l.a_bytes;
    l.off_w = l.off_y + (T * Fy * 2 * C + 1023) / 1024 * 1024;
    l.off_par = l.off_w + 2 * C * C * 2;
    l.off_red = l.off_par + 10 * C * 4;                 // 6 per-channel constants, 4 per-stream coefficients
    l.off_bar = l.off_red + 2 * kSbWarps * 8 + 16;      // fp64 partials, 4 floats of coefficients
    l.bytes = l.off_bar + kBars * 8 + 16 + 1024;        // barriers, TMEM slot, alignment slack
    return l;
}

template <int C>
__global__ void __launch_bounds__(kSbThreads, 1) skip_blend_tc_kernel(const __grid_constant__ SkipBlendParams p) {
    using S = SbCfg<C>;
    constexpr int CW = S::CW, KS = S::KS;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // swizzle atoms: 1024-aligned
    const SbLayout L = sb_layout(C, p.Fs, p.Fy);
    const int P = L.P, NT = L.NT;
    float* par = reinterpret_cast<float*>(smem + L.off_par);
    float *s_bm = par, *s_br = par + C, *s_nw = par + 2 * C, *s_nb = par + 3 * C, *s_nwr = par + 4 * C,
          *s_nbr = par + 5 * C;
    float4* coef = reinterpret_cast<float4*>(par + 6 * C);  // per stream and channel: mask a, d; y a, d
    double* s_red = reinterpret_cast<double*>(smem + L.off_red);
    float* s_co = reinterpret_cast<float*>(s_red + 2 * kSbWarps);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L.off_bar + kBars * 8);
    const uint32_t a_smem = smem_u32(smem), w_smem = a_smem + (uint32_t)L.off_w;
    const uint32_t bar0 = a_smem + (uint32_t)L.off_bar;
    auto full_bar = [&](int s) { return bar0 + 8u * s; };                          // skip box of buffer s has landed
    const uint32_t y_full = bar0 + 16u;                                            // the stream's y box has landed
    auto mask_full = [&](int m) { return bar0 + 8u * (3 + m); };                   // mask MMAs of tile m done
    auto res_full = [&](int k) { return bar0 + 8u * (3 + kMaxTiles + k); };        // residual accumulator k ready
    auto res_free = [&](int k) { return bar0 + 8u * (3 + kMaxTiles + 2 + k); };    // ... and drained
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);

    // ---- one-time set-up -----------------------------------------------------------------------------------------
    // weights: the skip pair's packed fp16 rows (2 co = residualmask, 2 co + 1 = residual) -> two no-swizzle K-major
    // B operands [k chunk j][n][8 halves], mask matrix first
    for (int i = tid; i < 2 * C * (C / 8); i += kSbThreads) {
        const int mat = i / (C * (C / 8)), rem = i % (C * (C / 8)), j = rem / C, n = rem % C;
        const uint2* src = reinterpret_cast<const uint2*>(p.w + (long long)(2 * n + mat) * p.Kp + 8 * j);  // 8-byte aligned
        uint2* dst = reinterpret_cast<uint2*>(smem + L.off_w + mat * S::W_BYTES + (j * C + n) * 16);
        dst[0] = __ldg(src);
        dst[1] = __ldg(src + 1);
    }
    for (int c = tid; c < C; c += kSbThreads) {
        s_bm[c] = __ldg(p.bias + 2 * c);
        s_br[c] = __ldg(p.bias + 2 * c + 1);
        s_nw[c] = __ldg(p.nw + c);
        s_nb[c] = __ldg(p.nb + c);
        s_nwr[c] = __ldg(p.nwr + c);
        s_nbr[c] = __ldg(p.nbr + c);
    }
    // rows [P, Pr) of both skip buffers are never written by the box, only read by discarded accumulator rows: keep
    // them finite
    for (int i = tid; i < 2 * (L.Pr - P) * (C / 8); i += kSbThreads) {
        const int s = i / ((L.Pr - P) * (C / 8)), u = i % ((L.Pr - P) * (C / 8));
        *reinterpret_cast<uint4*>(smem + s * L.a_bytes + P * S::ROWB + 16 * u) = make_uint4(0, 0, 0, 0);
    }
    if (tid == 0) {
        for (int i = 0; i < 2; ++i) mbar_init(full_bar(i), 1);
        mbar_init(y_full, 1);
        for (int m = 0; m < kMaxTiles; ++m) mbar_init(mask_full(m), 1);
        for (int k = 0; k < 2; ++k) {
            mbar_init(res_full(k), 1);
            mbar_init(res_free(k), kEpiWarps * 32);  // every epilogue thread takes its share out of every tile
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // weights, zero rows: generic proxy -> MMA reads
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(s_tmem);
    const int res_col = NT * C;  // residual accumulators k = 0, 1 at res_col + k C; mask of tile m at m C

    const double count_m = (double)C * P, count_y = (double)C * p.Fy * T;
    const long long y_stream = (long long)T * p.Fy * C;  // halves of one stream's y slab
    auto tile_start = [&](int m) { return min(BM * m, L.Pr - BM); };
    uint32_t u = 0;  // residual tiles issued / drained so far by this CTA (accumulator u & 1, phase (u >> 1) & 1)
    int it = 0;
    if (warp_u == kMmaWarp && elect_one() && (int)blockIdx.x < p.B) {
        mbar_arrive_expect_tx(full_bar(0), (uint32_t)(P * S::ROWB));
        tma_load_4d(a_smem, &p.skip, full_bar(0), 0, p.f_org, p.t_org, blockIdx.x);
    }
    for (int b = blockIdx.x; b < p.B; b += gridDim.x, ++it) {
        const int s = it & 1;
        const uint32_t abuf = a_smem + (uint32_t)(s * L.a_bytes);
        float psum = 0.f, psq = 0.f;
        if (warp_u == kMmaWarp) {
            // ============================ TMA + MMA issuer ============================
            const int nb = b + gridDim.x;
            // buffer s ^ 1 was last read by the MMAs of the previous stream, all of which the epilogue has seen complete
            if (nb < p.B && elect_one()) {
                mbar_arrive_expect_tx(full_bar(s ^ 1), (uint32_t)(P * S::ROWB));
                tma_load_4d(a_smem + (uint32_t)((s ^ 1) * L.a_bytes), &p.skip, full_bar(s ^ 1), 0, p.f_org, p.t_org, nb);
                prefetch_l2(p.y + (long long)nb * y_stream, (uint32_t)(y_stream * 2));
            }
            // y has one buffer: the previous stream's pass 2 is over; it lands while pass 1 runs
            if (elect_one()) {
                mbar_arrive_expect_tx(y_full, (uint32_t)(T * p.Fy * S::ROWB));
                tma_load_4d(a_smem + (uint32_t)L.off_y, &p.ymap, y_full, 0, 0, 0, b);
            }
            __syncwarp();
            mbar_wait(full_bar(s), (uint32_t)(it >> 1) & 1u);
            tc_fence_after();
            if (elect_one()) {
                for (int m = 0; m < NT; ++m) {
                    const uint32_t a0 = abuf + (uint32_t)(tile_start(m) * S::ROWB);
#pragma unroll
                    for (int ks = 0; ks < KS; ++ks)
                        tc_mma_f16(tmem_base + (uint32_t)(m * C), desc_skip<C>(a0 + 32u * ks),
                                   desc_nosw(w_smem + (uint32_t)(ks * 2 * C * 16), C * 16, 128u), S::IDESC, ks ? 1u : 0u);
                    tc_commit(mask_full(m));
                }
            }
            __syncwarp();
            auto issue_res = [&](int m) {
                const int k = (int)(u & 1u);
                mbar_wait(res_free(k), ((u >> 1) & 1u) ^ 1u);  // use u waits for the drain of use u - 2
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a0 = abuf + (uint32_t)(tile_start(m) * S::ROWB);
#pragma unroll
                    for (int ks = 0; ks < KS; ++ks)
                        tc_mma_f16(tmem_base + (uint32_t)(res_col + k * C), desc_skip<C>(a0 + 32u * ks),
                                   desc_nosw(w_smem + (uint32_t)(S::W_BYTES + ks * 2 * C * 16), C * 16, 128u), S::IDESC,
                                   ks ? 1u : 0u);
                    tc_commit(res_full(k));
                }
                __syncwarp();
                ++u;
            };
            // the first two residual tiles find their accumulators drained by the previous stream; the rest wait for
            // pass 2, which starts only after the statistics barrier this warp takes part in below
            issue_res(0);
            issue_res(1);
            block_gln<kSbWarps>(0.f, 0.f, count_m, p.student, s_red, s_co);
            __syncthreads();  // per-stream coefficients
            for (int m = 2; m < NT; ++m) issue_res(m);
        } else {
            // ============================ epilogue ============================
            const int q = warp & 3, cg = warp >> 2;
            const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
            // ---- pass 1: statistics of the mask pre-activation (accumulator + bias) over exactly P x C values ----
            for (int m = 0; m < NT; ++m) {
                const int g = tile_start(m) + q * 32 + lane;
                if (lane == 0) mbar_wait(mask_full(m), (uint32_t)it & 1u);
                __syncwarp();
                tc_fence_after();
                uint32_t v[CW];
                tmem_ld_nowait<CW>(tq + (uint32_t)(m * C + cg * CW), v);
                tmem_ld_wait();
                if (g >= BM * m && g < P) {  // the last tile's rows below 128 m were counted by its predecessor
#pragma unroll
                    for (int c = 0; c < CW; ++c) {
                        const float x = __uint_as_float(v[c]) + s_bm[cg * CW + c];
                        psum += x;
                        psq = fmaf(x, x, psq);
                    }
                }
            }
            block_gln<kSbWarps>(psum, psq, count_m, p.student, s_red, s_co);
            if (tid < C) {
                // both GlobalLayerNorms with their affines folded into one FMA per value; the mask's carries the 1/2 of
                // sigmoid(x) = 1/2 + 1/2 tanh(x / 2) and its 1x1 bias
                float ym, yi;
                gln_mean_inv(p.stats[2 * b], p.stats[2 * b + 1], count_y, p.student, ym, yi);
                const float ma = s_nwr[tid] * s_co[1], ya = s_nw[tid] * yi;
                coef[tid] = make_float4(0.5f * ma, 0.5f * fmaf(s_bm[tid] - s_co[0], ma, s_nbr[tid]), ya,
                                        fmaf(-ym, ya, s_nb[tid]));
            }
            __syncthreads();
            // ---- pass 2: residual accumulators -> the blended block output ----
            if (lane == 0) mbar_wait(y_full, (uint32_t)it & 1u);
            __syncwarp();
            __half* ob = p.out + (long long)b * p.oB + cg * CW;
            for (int m = 0; m < NT; ++m, ++u) {
                const int g = tile_start(m) + q * 32 + lane;
                const bool valid = g >= BM * m && g < P;
                const int t = g / p.Fs, f = g - t * p.Fs;
                const bool has_y = valid && f < p.Fy;
                // y row t Fy + f of the swizzled box: 16-byte chunk j sits at chunk j ^ (row bits 7.. of the address)
                uint4 yr[CW / 8];
                const int yrow = t * p.Fy + f;
                const int swz = C == 64 ? (yrow & 7) : ((yrow >> 1) & 3);
#pragma unroll
                for (int o = 0; o < CW / 8; ++o)
                    yr[o] = has_y ? *reinterpret_cast<const uint4*>(smem + L.off_y + yrow * S::ROWB +
                                                                    16 * ((cg * (CW / 8) + o) ^ swz))
                                  : make_uint4(0, 0, 0, 0);
                const int k = (int)(u & 1u);
                if (lane == 0) mbar_wait(res_full(k), (u >> 1) & 1u);
                __syncwarp();
                tc_fence_after();
                uint32_t vm[CW], vr[CW];
                tmem_ld_nowait<CW>(tq + (uint32_t)(m * C + cg * CW), vm);
                tmem_ld_nowait<CW>(tq + (uint32_t)(res_col + k * C + cg * CW), vr);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(res_free(k));
                if (valid) {
                    float yv[CW];
#pragma unroll
                    for (int o = 0; o < CW / 8; ++o) unpack8(yr[o], yv + 8 * o);
                    float out[CW];
#pragma unroll
                    for (int c = 0; c < CW; ++c) {
                        const int ch = cg * CW + c;
                        const float4 k4 = coef[ch];
                        const float mk = fmaf(0.5f, tanh_approx(fmaf(__uint_as_float(vm[c]), k4.x, k4.y)), 0.5f);
                        const float r = fast_elu(__uint_as_float(vr[c]) + s_br[ch]);
                        const float o = has_y ? fmaf(yv[c], k4.z, k4.w) : 0.f;
                        out[c] = fmaf(mk, r - o, o);
                    }
                    uint4* dst = reinterpret_cast<uint4*>(ob + (long long)t * p.oT + (long long)f * p.oF);
#pragma unroll
                    for (int o = 0; o < CW / 8; ++o) dst[o] = pack8(out + 8 * o);
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // y reads (generic) before the next y box (async)
        tc_fence_before();
        __syncthreads();  // the mask columns, skip buffer s and the y buffer are free for the next streams
        tc_fence_after();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

template <int C>
int launch_t(const SkipBlendParams& p, cudaStream_t st) {
    const SbLayout L = sb_layout(C, p.Fs, p.Fy);
    SE_DYN_SMEM((skip_blend_tc_kernel<C>), (size_t)L.bytes);
    int num_sms = 0;
    if (num_sms_current_device(&num_sms)) return 1;
    skip_blend_tc_kernel<C><<<p.B < num_sms ? p.B : num_sms, kSbThreads, L.bytes, st>>>(p);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace

bool skip_blend_supported(int C, int Fs, int Fy) {
    if (C != 32 && C != 64) return false;
    if (Fy > Fs || T * Fs < BM) return false;
    const SbLayout L = sb_layout(C, Fs, Fy);
    // mask accumulators of every tile + the two residual accumulators in TMEM, the stream's skip box twice in SMEM
    return L.NT <= kMaxTiles && (L.NT + 2) * C <= (int)kTmemCols && L.bytes <= 227 * 1024 && Fs <= 256;
}

int make_skip_blend_maps(SkipBlendParams* p, const void* skip_base, int C, int Fp, int Tp, long long sT, long long sB,
                         int nB) {
    {  // the padded skip buffer [nB][Tp][Fp][C] fp16; one box = the interior of one stream (C x Fs x T), rows of 2 C bytes
        const long long dims[4] = {C, Fp, Tp, nB};
        const long long strides[3] = {(long long)C * 2, sT * 2, sB * 2};
        const int box[4] = {C, p->Fs, T, 1};
        if (make_tma_4d_f16(&p->skip, skip_base, dims, strides, box, 2 * C)) return 1;
    }
    // y [nB][T][Fy][C]; one box = one stream, swizzled like the skip rows so that the epilogue reads it conflict-free
    const long long dims[4] = {C, p->Fy, T, nB};
    const long long strides[3] = {(long long)C * 2, (long long)p->Fy * C * 2, (long long)T * p->Fy * C * 2};
    const int box[4] = {C, p->Fy, T, 1};
    return make_tma_4d_f16(&p->ymap, p->y, dims, strides, box, 2 * C);
}

int launch_skip_blend(const SkipBlendParams& p, int C, cudaStream_t st) {
    if (p.B <= 0) return 0;
    SE_REQUIRE(skip_blend_supported(C, p.Fs, p.Fy), "skip_blend_tc: unsupported shape");
    return C == 64 ? launch_t<64>(p, st) : launch_t<32>(p, st);
}

}  // namespace se
