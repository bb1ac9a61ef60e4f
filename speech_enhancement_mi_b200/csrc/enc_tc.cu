// Gated causal conv block of the encoder (CRN_ELU.py:230-247: k(5,3) conv, stride (2,1), time dilation 2^i, + ELU +
// gated 1x1 pair + GlobalLayerNorm) for the 16 -> 32 and 32 -> 64 channel levels, fp16 operand mode: one stream per CTA at
// a time, the stream's zero-bordered input resident in shared memory, the convolution an IMPLICIT GEMM on tcgen05.
//
// The input is held once, de-interleaved into (bin parity x channel octet) planes of 16-byte units [frame][bin / 2]
// (as enc_mma_kernel, front_mma.cu).  Output row r = frame * Jp + bin then reads, for tap (kt, kf) and octet h, the
// unit r + kt * dt * Jp + kf / 2 of plane (kf & 1, h): consecutive rows are consecutive units.  That is exactly the
// canonical NO-SWIZZLE K-major operand layout of a UMMA shared-memory descriptor (8-row core matrices of 16-byte rows,
// SBO = 128 bytes between them) with the second K chunk of a K = 16 MMA taken from the next octet's plane through the
// leading-dimension offset (LBO = plane pitch): every (tap, octet pair) is ONE tcgen05.mma over 128 output rows whose A
// descriptor points INTO the resident input (tools/micro/umma_im2col_test.cu checks the overlapped-descriptor
// arithmetic).  No im2col copy, no per-tap staging, 15 CIN / 16 MMAs per 128-row tile instead of 8 x that many
// mma.sync per warp.  The gate runs back to back: the epilogue writes the ELU tile as the fp16 A operand of a second
// MMA (N = 2 COUT: conv_trans | conv_gated) IN PLACE over the input units of the tile's own rows (a later tile only
// reads units at or above its first row; the COUT / 8 channel octets of a row = the 2 CIN / 8 input planes, so the same
// descriptor geometry addresses it), then gates that accumulator, counts it into the GlobalLayerNorm statistics and
// stores the pre-norm fp16 values over the same units again.  The pre-norm tensor never leaves the SM; pass 2 normalises
// into the next block's input interior.  The block is bound by its transcendentals (one ex2 for the ELU, one tanh for
// the sigmoid per output: 16 MUFU lanes per SM), so the epilogue runs on 16 warps = four accumulator groups.
//
// Roles in pass 1: warps 0-15 = four epilogue groups (one TMEM accumulator each, tiles round-robin), warp 16 = MMA
// issuer (warp-uniform loop, one elected lane issues); all 17 warps load, reduce the statistics and normalise.
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdlib.h>

#include "mma_util.cuh"
#include "se_internal.h"

#ifndef SE_ENC_PROFILE
#define SE_ENC_PROFILE 0  // -DSE_ENC_PROFILE=1: CTA 0 prints the cycles of its phases (load, pass 1, statistics, pass 2) and,
                          // for its third stream, the time line of every tile (issue, accumulator ready, epilogues)
#endif
#if SE_ENC_PROFILE
#include <stdio.h>
#define ENC_EV(slot) do { if (blockIdx.x == 0 && stream == 2 * (int)gridDim.x && lane == 0) s_ev[slot] = clock64() - tp1; } while (0)
#else
#define ENC_EV(slot) do { } while (0)
#endif

namespace se {
namespace {

using namespace mma_util;
constexpr int T = kFramesPerChunk;  // 21
constexpr int BM = 128;
constexpr int kGroups = 4;                 // epilogue groups = TMEM accumulators
constexpr int kMmaWarp = 4 * kGroups;      // 16
constexpr int kTcWarps = kMmaWarp + 1;
constexpr int kTcThreads = kTcWarps * 32;  // 544
constexpr int kTailUnits = 136;  // readable units behind the last plane (row overrun of the last tile + 2 bins)

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
// non-blocking phase test, warp-uniform result (lane 0 tests, the warp takes its answer)
__device__ __forceinline__ bool mbar_test_warp(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return __shfl_sync(0xffffffffu, ok, 0) != 0;
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
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// canonical no-swizzle K-major descriptor: 8-row core matrices of 16-byte rows, SBO bytes between core matrices along
// the rows, LBO bytes between the two 16-byte K chunks of one MMA
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

template <int CIN, int COUT>
struct TcCfg {
    static_assert(COUT == 2 * CIN && CIN % 16 == 0, "octet planes of the input are reused for the output");
    static constexpr int NH = CIN / 8;          // input channel octets
    static constexpr int NPL = 2 * NH;          // planes (bin parity x octet) = output octets
    static constexpr int HP = NH / 2;           // octet pairs = MMAs per tap
    static constexpr int KS = 15 * HP;          // conv MMAs per tile
    static constexpr int KS2 = COUT / 16;       // gate MMAs per tile
    static constexpr int W1_BYTES = KS * 2 * COUT * 16;
    static constexpr int W2_BYTES = KS2 * 2 * (2 * COUT) * 16;
    static constexpr int ACC_COLS = 2 * COUT;   // per group: trans | gated, the conv accumulator aliased on the first COUT
    static constexpr uint32_t TMEM_COLS = kGroups * ACC_COLS <= 256 ? 256 : 512;
    static_assert(kGroups * ACC_COLS <= 512, "TMEM has 512 columns");
};

template <int CIN, int COUT>
__global__ void __launch_bounds__(kTcThreads, 1) enc_tc_kernel(EncMmaParams p) {
    using S = TcCfg<CIN, COUT>;
    constexpr int NH = S::NH, NPL = S::NPL, HP = S::HP, KS = S::KS, KS2 = S::KS2;
    extern __shared__ __align__(128) unsigned char smem[];
    const int Jp = (p.Fp + 1) >> 1;
    const int plane = p.plane;  // units per plane (= 1 mod 8: the octets of one row sit in different bank groups)
    unsigned char* sw1 = smem + p.off_wf;
    unsigned char* sw2 = sw1 + S::W1_BYTES;
    float* spar = reinterpret_cast<float*>(sw2 + S::W2_BYTES);  // cb[COUT] | bt[COUT] | 0.5 bg[COUT]
    double* s_red = reinterpret_cast<double*>(spar + 3 * COUT);
    float* s_co = reinterpret_cast<float*>(s_red + 2 * kTcWarps);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_co + 2);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 2 * kGroups);
    const uint32_t x_smem = smem_u32(smem), w1_smem = smem_u32(sw1), w2_smem = smem_u32(sw2);
    const uint32_t bar0 = smem_u32(s_bar);
    auto acc_full = [&](int g) { return bar0 + 8u * g; };              // the MMAs into accumulator g have completed
    auto acc_free = [&](int g) { return bar0 + 8u * (kGroups + g); };  // its epilogue group has drained it
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
#if SE_ENC_PROFILE
    __shared__ long long s_ev[160];  // [0,32): MMA warp: conv issue / gate issue per tile; [32 + 8 i ...): tile i events
    for (int i = tid; i < 160; i += kTcThreads) s_ev[i] = 0;
    long long tp1 = 0;
#endif

    // ---- one-time set-up -----------------------------------------------------------------------------------------
    // B operands, packed once per weight upload (crn.cu) in exactly this layout:
    //   conv: MMA ks = (tap, octet pair hp); K chunk j = octet 2 hp + j of the tap; [ks][j][n] x 8 halves
    //   gate: [ks2][j][n2] x 8 halves, rows [0, COUT) conv_trans, [COUT, 2 COUT) conv_gated scaled by 1/2
    //         (sigmoid(z) = 1/2 + 1/2 tanh(z / 2))
    for (int i = tid; i < (S::W1_BYTES + S::W2_BYTES) / 16; i += kTcThreads) {
        const bool second = i >= S::W1_BYTES / 16;
        const uint4* src = reinterpret_cast<const uint4*>(second ? p.w2c : p.w1c) + (second ? i - S::W1_BYTES / 16 : i);
        cp_async16(w1_smem + 16u * (uint32_t)i, src);
    }
    cp_async_commit();
    for (int i = tid; i < COUT; i += kTcThreads) {
        spar[i] = __ldg(p.bias + i);
        spar[COUT + i] = __ldg(p.bias2 + 2 * i);
        spar[2 * COUT + i] = 0.5f * __ldg(p.bias2 + 2 * i + 1);
    }
    // the units the loads never write (odd-plane tail bin, plane padding, tail) are only read by discarded rows, but keep
    // them finite
    for (int i = tid; i < NPL * plane + kTailUnits; i += kTcThreads) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid == 0) {
        for (int g = 0; g < kGroups; ++g) {
            mbar_init(acc_full(g), 1);
            mbar_init(acc_free(g), kMmaWarp * 32);  // every epilogue thread takes its share out of every tile
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(S::TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    cp_async_wait_all();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // weights: generic-proxy writes -> MMA (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(s_tmem);

    auto issue_load = [&](int b) {  // global [Tp][Fp][NH] units -> planes
        const uint4* src = reinterpret_cast<const uint4*>(p.in + (long long)b * p.in_sB);
        const int total = p.Tp * p.Fp * NH;
        for (int u = tid; u < total; u += kTcThreads) {
            const int h = u & (NH - 1);
            const int pl = u / NH;
            const int tt = div_magic(pl, p.magic_Fp), pos = pl - tt * p.Fp;
            const int unit = ((pos & 1) * NH + h) * plane + tt * Jp + (pos >> 1);
            cp_async16(x_smem + 16u * unit, src + u);
        }
        cp_async_commit();
    };

    const int dtJ = p.dt * Jp;
    const int MT = (T * Jp + BM - 1) / BM;
    const int Fo = p.Fo;
    const double count = (double)COUT * Fo * T;

    for (int stream = blockIdx.x; stream < p.B; stream += gridDim.x) {
        const int b = p.b0 + stream;
#if SE_ENC_PROFILE
        const long long tp0 = clock64();
#endif
        issue_load(b);
        cp_async_wait_all();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // cp.async (generic proxy) -> MMA operand reads
        __syncthreads();
#if SE_ENC_PROFILE
        tp1 = clock64();
#endif
        float psum = 0.f, psq = 0.f;
        if (warp_u == kMmaWarp) {
            // ============================ MMA issuer ============================
            constexpr uint32_t idesc1 = (1u << 4) | ((uint32_t)(COUT >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            constexpr uint32_t idesc2 = (1u << 4) | ((uint32_t)((2 * COUT) >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
            // Phase A: the convolutions of all tiles, streaming through the four accumulators (an accumulator is free again
            // as soon as its ELU tile has been written); phase B, behind a CTA barrier: the gate MMAs over the ELU tiles.
            // Keeping the two apart makes each accumulator's round trip MMA -> one epilogue, not conv -> ELU -> gate -> gate
            // epilogue, so the tensor pipe and the epilogue warps overlap instead of waiting on one another per tile.
            for (int i = 0; i < MT; ++i) {
                const int g = i & (kGroups - 1);
                // use k of an accumulator waits for the drain of use k - 1; every stream goes through an even number of uses
                mbar_wait(acc_free(g), ((uint32_t)(i >> 2) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t a0 = x_smem + 16u * (uint32_t)(i * BM);
                const uint32_t tacc = tb + (uint32_t)(g * S::ACC_COLS);
                if (elect_one()) {
#pragma unroll
                    for (int ks = 0; ks < KS; ++ks) {
                        const int tap = ks / HP, hp = ks % HP, kt = tap / 5, kf = tap % 5;
                        const uint32_t unit = (uint32_t)(kt * dtJ + (kf >> 1) + ((kf & 1) * NH + 2 * hp) * plane);
                        const uint64_t ad = desc_nosw(a0 + 16u * unit, 16u * (uint32_t)plane, 128u);
                        const uint64_t bd = desc_nosw(w1_smem + (uint32_t)(ks * 2 * COUT * 16), COUT * 16, 128u);
                        tc_mma_f16(tacc, ad, bd, idesc1, ks ? 1u : 0u);
                    }
                    tc_commit(acc_full(g));
                }
                __syncwarp();
                ENC_EV(i);
            }
            __syncthreads();  // every ELU tile is written (and fenced towards the async proxy), every conv accumulator drained
            tc_fence_after();
            for (int j = 0; j < MT; ++j) {
                const int g = j & (kGroups - 1);
                const uint32_t k = (uint32_t)((MT - g + kGroups - 1) / kGroups + (j >> 2));
                mbar_wait(acc_free(g), (k & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t a0 = x_smem + 16u * (uint32_t)(j * BM);
                const uint32_t tacc = tb + (uint32_t)(g * S::ACC_COLS);
                if (elect_one()) {
#pragma unroll
                    for (int ks2 = 0; ks2 < KS2; ++ks2) {
                        const uint64_t ad = desc_nosw(a0 + 16u * (uint32_t)(2 * ks2 * plane), 16u * (uint32_t)plane, 128u);
                        const uint64_t bd = desc_nosw(w2_smem + (uint32_t)(ks2 * 2 * (2 * COUT) * 16), 2 * COUT * 16, 128u);
                        tc_mma_f16(tacc, ad, bd, idesc2, ks2 ? 1u : 0u);
                    }
                    tc_commit(acc_full(g));
                }
                __syncwarp();
                ENC_EV(16 + j);
            }
        } else if (warp_u < kMmaWarp) {
            // ============================ epilogue: thread = output row x a quarter of the channels ============================
            // All 16 warps work on every tile: warp (q, cg) owns TMEM lanes 32 q .. 32 q + 31 (rows) and the channel
            // quarter cg, so the tiles' epilogues are balanced whatever MT is.  Accumulator a = tile & 3.
            constexpr int CW = COUT / kGroups;  // channels per warp and tile: 16 (two octets) or 8 (one)
            const int q = warp & 3, cg = warp >> 2;
            const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
            // ---- phase A: conv accumulator -> bias, ELU -> fp16 A operand of the gate MMA, in place over the tile's rows ----
            for (int i = 0; i < MT; ++i) {
                const int a = i & (kGroups - 1);
                const int r = i * BM + q * 32 + lane;
                if (lane == 0) mbar_wait(acc_full(a), (uint32_t)(i >> 2) & 1u);
                __syncwarp();
                if (warp == 0) ENC_EV(32 + 8 * i + 1);
                tc_fence_after();
                uint32_t v[CW];
                if (CW == 16) tmem_ld16_nowait(tq + (uint32_t)(a * S::ACC_COLS + cg * CW), v);
                else tmem_ld8_nowait(tq + (uint32_t)(a * S::ACC_COLS + cg * CW), v);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(acc_free(a));  // this warp's share is out of the accumulator
                uint32_t h[CW / 2];
#pragma unroll
                for (int k = 0; k < CW / 2; ++k)
                    h[k] = pack_h2(fast_elu(__uint_as_float(v[2 * k]) + spar[cg * CW + 2 * k]),
                                   fast_elu(__uint_as_float(v[2 * k + 1]) + spar[cg * CW + 2 * k + 1]));
                // ELU channels of row r = unit r of plane (channel / 8): the row's own input is dead by now
#pragma unroll
                for (int o = 0; o < CW / 8; ++o)
                    *reinterpret_cast<uint4*>(smem + 16 * (size_t)((cg * (CW / 8) + o) * plane + r)) =
                        make_uint4(h[4 * o], h[4 * o + 1], h[4 * o + 2], h[4 * o + 3]);
                if (warp == 0) ENC_EV(32 + 8 * i + 2);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> gate MMAs (async proxy)
            __syncthreads();  // phase boundary (see the MMA issuer)
            // ---- phase B: gate accumulator -> y = trans * sigmoid(gated), statistics, fp16 in place over the same rows ----
            for (int i = 0; i < MT; ++i) {
                const int a = i & (kGroups - 1);
                const int r = i * BM + q * 32 + lane;
                const int t = div_magic(r, p.magic_Jp), fo = r - t * Jp;
                const bool valid = t < T && fo < Fo;
                const uint32_t k = (uint32_t)((MT - a + kGroups - 1) / kGroups + (i >> 2));  // uses of accumulator a so far
                if (lane == 0) mbar_wait(acc_full(a), k & 1u);
                __syncwarp();
                if (warp == 0) ENC_EV(32 + 8 * i + 3);
                tc_fence_after();
                uint32_t vt[CW], vg[CW];
                if (CW == 16) {
                    tmem_ld16_nowait(tq + (uint32_t)(a * S::ACC_COLS + cg * CW), vt);
                    tmem_ld16_nowait(tq + (uint32_t)(a * S::ACC_COLS + COUT + cg * CW), vg);
                } else {
                    tmem_ld8_nowait(tq + (uint32_t)(a * S::ACC_COLS + cg * CW), vt);
                    tmem_ld8_nowait(tq + (uint32_t)(a * S::ACC_COLS + COUT + cg * CW), vg);
                }
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(acc_free(a));
                const float m = valid ? 1.f : 0.f;
                float y[CW];
#pragma unroll
                for (int c = 0; c < CW; ++c) {
                    // trans * sigmoid(gated): the gated weights and bias carry the factor 1/2 of 1/2 + 1/2 tanh(z / 2)
                    const float th = tanh_approx(__uint_as_float(vg[c]) + spar[2 * COUT + cg * CW + c]);
                    y[c] = m * (__uint_as_float(vt[c]) + spar[COUT + cg * CW + c]) * fmaf(0.5f, th, 0.5f);
                    psum += y[c];
                    psq = fmaf(y[c], y[c], psq);
                }
                if (valid) {
#pragma unroll
                    for (int o = 0; o < CW / 8; ++o)
                        *reinterpret_cast<uint4*>(smem + 16 * (size_t)((cg * (CW / 8) + o) * plane + r)) =
                            make_uint4(pack_h2(y[8 * o], y[8 * o + 1]), pack_h2(y[8 * o + 2], y[8 * o + 3]),
                                       pack_h2(y[8 * o + 4], y[8 * o + 5]), pack_h2(y[8 * o + 6], y[8 * o + 7]));
                }
                if (warp == 0) ENC_EV(32 + 8 * i + 4);
            }
        } else {
            __syncthreads();  // (no such warp today: every warp is an epilogue warp or the issuer) phase boundary
        }
        __syncthreads();
#if SE_ENC_PROFILE
        const long long tp2 = clock64();
#endif
        block_gln<kTcWarps>(psum, psq, count, p.student, s_red, s_co);
#if SE_ENC_PROFILE
        const long long tp3 = clock64();
#endif
        // ---- pass 2: GlobalLayerNorm -> the next block's input interior ------------------------------------------------
        {
            const float mean = s_co[0], inv = s_co[1];
            const int o = tid % NPL;  // kTcThreads % NPL == 0: a thread always serves the same channel octet
            float na[8], nd[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                na[k] = __ldg(p.nw + 8 * o + k) * inv;
                nd[k] = fmaf(-mean, na[k], __ldg(p.nb + 8 * o + k));
            }
            __half* ob = p.out + (long long)b * p.oB + 8 * o;
            const unsigned char* yp = smem + 16 * (size_t)o * plane;
            const int total = T * Fo * NPL;
            for (int u = tid; u < total; u += kTcThreads) {
                const int row = u / NPL;
                const int t = div_magic(row, p.magic_Fo), f = row - t * Fo;
                const uint4 raw = *reinterpret_cast<const uint4*>(yp + 16 * (size_t)(t * Jp + f));
                float v[8];
                unpack8(raw, v);
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = fmaf(v[k], na[k], nd[k]);
                *reinterpret_cast<uint4*>(ob + t * p.oT + f * p.oF) = pack8(v);
            }
        }
        __syncthreads();  // the planes are free for the next stream's input
#if SE_ENC_PROFILE
        if (blockIdx.x == 0 && tid == 0 && stream < 3 * (int)gridDim.x) {
            printf("enc_tc<%d,%d> stream %d: load %lld  pass1 %lld  stats %lld  pass2 %lld cycles (MT %d)\n", CIN, COUT, stream,
                   tp1 - tp0, tp2 - tp1, tp3 - tp2, clock64() - tp3, MT);
            if (stream == 2 * (int)gridDim.x)
                for (int i = 0; i < MT; ++i)
                    printf("   tile %d: conv issued %lld gate issued %lld | epi1 start %lld conv done %lld ELU written %lld | gate done %lld y written %lld\n",
                           i, s_ev[i], s_ev[16 + i], s_ev[32 + 8 * i], s_ev[32 + 8 * i + 1], s_ev[32 + 8 * i + 2],
                           s_ev[32 + 8 * i + 3], s_ev[32 + 8 * i + 4]);
        }
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(S::TMEM_COLS) : "memory");
    }
}

// units per plane, = 1 (mod 8): the octets of one row then sit in different bank groups for pass 2.  (Core matrices that
// straddle 128-byte lines cost nothing: plane pitches = 0 (mod 8) measured the same MMA rate.)
int plane_units(int Tp, int Fp) {
    int plane = Tp * ((Fp + 1) / 2);
    while (plane % 8 != 1) ++plane;
    return plane;
}

template <int CIN, int COUT>
size_t enc_tc_bytes(int Tp, int Fp) {
    using S = TcCfg<CIN, COUT>;
    size_t off = ((size_t)S::NPL * plane_units(Tp, Fp) + kTailUnits) * 16;
    off += S::W1_BYTES + S::W2_BYTES + 3 * COUT * 4 + 2 * kTcWarps * 8 + 8 + 2 * kGroups * 8 + 16;
    return off;
}

template <int CIN, int COUT>
int launch_enc_tc_t(EncMmaParams p, cudaStream_t st) {
    using S = TcCfg<CIN, COUT>;
    const int Jp = (p.Fp + 1) / 2;
    p.plane = plane_units(p.Tp, p.Fp);
    p.off_wf = (int)(((size_t)S::NPL * p.plane + kTailUnits) * 16);
    const size_t bytes = enc_tc_bytes<CIN, COUT>(p.Tp, p.Fp);
    SE_REQUIRE(bytes <= 227 * 1024, "enc_tc: the stream does not fit in shared memory");
    auto magic = [](int d) { return (uint32_t)(((1ull << 32) + d - 1) / d); };  // exact for dividends < 65536
    SE_REQUIRE(p.Tp * p.Fp < 65536 && T * Jp + BM < 65536, "enc_tc: index range of the magic division");
    p.magic_Jp = magic(Jp);
    p.magic_Fo = magic(p.Fo);
    p.magic_Fp = magic(p.Fp);
    SE_DYN_SMEM((enc_tc_kernel<CIN, COUT>), bytes);
    int num_sms = 0;
    if (num_sms_current_device(&num_sms)) return 1;
    enc_tc_kernel<CIN, COUT><<<p.B < num_sms ? p.B : num_sms, kTcThreads, bytes, st>>>(p);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace

bool enc_tc_supported(int mode, int Cin, int Cout, int Tp, int Fp, int Fo) {
    if (mode == 0) return false;
    const int Jp = (Fp + 1) / 2;
    if (Fo > Jp || (Tp - T) % 2 != 0) return false;
    // 16 -> 32 runs too (SE_B200_ENC_TC=2) but only measures 117 us against 122 us for the mma.sync kernel, so it stays
    // there by default.  Measured with -DSE_ENC_PROFILE=1: a no-swizzle A operand is read at ~64 B/clk (65 cycles per
    // K = 16 MMA whatever N <= 64 is, twice the SWIZZLE_128B rate), so the conv phase costs 1,000 (16 ch) / 1,950 (32 ch)
    // cycles per 128-row tile, and the gate phase is paced by the ~900-cycle accumulator round trip per tile.
    if (Cin == 16 && Cout == 32) return mode == 2 && enc_tc_bytes<16, 32>(Tp, Fp) <= 227 * 1024;
    if (Cin == 32 && Cout == 64) return enc_tc_bytes<32, 64>(Tp, Fp) <= 227 * 1024;
    return false;
}

int launch_enc_tc(const EncMmaParams& p, int Cin, int Cout, cudaStream_t st) {
    if (p.B <= 0) return 0;
    SE_REQUIRE(enc_tc_supported(2, Cin, Cout, p.Tp, p.Fp, p.Fo), "enc_tc: unsupported shape");  // 2: every shape it has
    if (Cin == 16) return launch_enc_tc_t<16, 32>(p, st);
    return launch_enc_tc_t<32, 64>(p, st);
}

}  // namespace se
