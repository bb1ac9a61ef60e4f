// Tensor-core gathered GEMM for sm_100a: tcgen05.mma kind::tf32 (fp32 operands read as TF32, fp32 accumulation in
// TMEM).  Same GemmParams contract as gemm_fp32.cu -- C[m][n] = sum_k A(m,k) W[n][k] with A gathered through the koff
// table (implicit im2col over zero-bordered channels-last activations) -- plus the fused GRU-cell and small-gate
// epilogues.
//
// Persistent, warp-specialised kernel: one CTA per SM walks the 128 x BN output tiles round-robin.
//   warps 0-3        : producers.  Per 32-float k-block, 8 consecutive lanes issue the 8 x 16-byte cp.async gathers of
//                      one 128-byte tile row (a warp instruction touches 4 rows = 4 cache lines) into the canonical
//                      K-major SWIZZLE_128B layout (row r at (r/8)*1024 + (r%8)*128, 16-byte chunk j stored at
//                      j ^ (r%8)), the same for the weight rows, then arrive on the stage's "full" mbarrier through
//                      cp.async.mbarrier.arrive.noinc.  The stage ring runs on across tile boundaries.
//   warp 4           : allocates TMEM (NACC accumulators of BN columns); lane 0 issues the tcgen05.mma chain (4 MMAs of
//                      K=8 per k-block), commits each stage to its "empty" mbarrier and each finished tile to the
//                      accumulator's "tmem_full" mbarrier.
//   warps 5..5+4*NACC: NACC epilogue groups of 4 warps; group g owns accumulator g (tiles g, g+NACC, ... of this CTA), so
//                      the epilogue math of one tile overlaps the loads and MMAs of the next ones.  Thread = tile row:
//                      it reads its accumulator row from TMEM (tcgen05.ld 32x32b) in 32-column chunks, applies the
//                      epilogue function, parks the chunk in a warp-private staging buffer and the warp writes it out
//                      with coalesced 16-byte stores.
// Every mbarrier wait is bounded (trap after ~2 s) so that a protocol bug cannot hang the GPU.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdlib.h>

#include "se_internal.h"

namespace se {
namespace {

constexpr int BM = 128;
constexpr int BKB = 128;  // bytes per k-block row = one 128-byte swizzle atom: 32 tf32 (fp32 storage) or 64 fp16
constexpr int A_STAGE_BYTES = BM * BKB;
constexpr int kProducerThreads = 128;
constexpr int kFirstEpiWarp = 5;
constexpr int SPW = 36;  // pitch (floats) of a warp-private staging row: 32 columns + 4 (conflict-free float4 rows)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    // the suspend-time hint lets the hardware park the thread instead of returning at once
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
// SLEEP_NS > 0: back off between polls (waiters that are off the critical path must not eat issue slots)
template <int SLEEP_NS>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    uint64_t t0 = 0;
    for (uint32_t spins = 1;; ++spins) {
        if (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
        if (mbar_try_wait(bar, parity)) return;
        if ((spins & 1023u) == 0) {  // protocol bug: fail loudly (after ~2 s) instead of hanging the GPU
            const uint64_t t = global_ns();
            if (t0 == 0) t0 = t;
            else if (t - t0 > 2000000000ull) __trap();
        }
    }
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// TMA tile loads (cp.async.bulk.tensor, SASS: UTMALDG): box of the tensor map at the given coordinates -> shared memory,
// completion counted in bytes on the mbarrier
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// ---- CTA pair (cta_group::2): two CTAs of a cluster run ONE M256 MMA; the leader (cluster rank 0) issues it ---------
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local_addr, uint32_t rank) {  // same offset in CTA `rank`
    uint32_t a;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(local_addr), "r"(rank));
    return a;
}
// RELAXED: the arrive only hands a drained TMEM accumulator back (tcgen05.wait::ld + tcgen05.fence::before_thread_sync
// order the reads); .release at cluster scope compiles to MEMBAR.ALL.GPU, which made every epilogue thread wait for its
// own output stores once per tile
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// tile load whose completion is counted on an mbarrier that may live in the PEER CTA of the pair (the leader's)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* map, uint32_t bar_cluster, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const void* map, uint32_t bar_cluster, int c0, int c1, int c2,
                                                 int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar, uint16_t mask) {  // arrive on `bar` of the CTAs in `mask`
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// n / d by multiply-high with magic = ceil(2^32 / d) (exact for n < 2^32 / d); magic 0 encodes d = 1
__device__ __forceinline__ int div_mh(int n, uint32_t magic) { return magic ? (int)__umulhi((uint32_t)n, magic) : n; }
// One lane of the (converged) warp.  The single-thread roles run their loops WARP-UNIFORMLY and only predicate the issue
// on this: inside an `if (lane == 0)` region ptxas treats every operand as divergent and wraps each tcgen05.mma / TMA
// in an ELECT + R2UR.BROADCAST + BRA.U.ANY loop (about 100 cycles per MMA -- more than a 128 x 64 MMA takes to execute).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// one M128 x N x K(32 bytes) MMA; operands: fp32 storage read as TF32 (K = 8) or fp16 (K = 16), fp32 accumulate
template <typename AT>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                       uint32_t accumulate) {
    if (sizeof(AT) == 4) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// 16 / 8 consecutive fp32 accumulator columns of this thread's TMEM lane (issue only; tmem_ld_wait before use)
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

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO(16B)=1 @16 |
// SBO(1024B)=64 @32 | version=1 @46 | layout SWIZZLE_128B=2 @61
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

// Epilogue math of the tf32 path: MUFU-based exp / reciprocal (relative error ~1e-6, two orders below the TF32 operand
// rounding of 2^-11 that bounds this path's accuracy; the exact-mode kernels in gemm_fp32.cu keep expm1f / expf / tanhf).
// ex2.approx.ftz / rcp.approx.ftz: one MUFU each.  __expf / __fdividef (and exp2f) add a range check and a rescale for
// denormal results around their MUFU -- about ten instructions per sigmoid instead of four.  Flushed denormals are exact
// zeros here: sigmoid -> 0 / 1, elu -> -1, tanh -> +-1 at the ends of their ranges.
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
// tanh.approx.f32: ONE MUFU (max relative error 2^-11, the precision of the fp16 / tf32 operands these epilogues feed);
// sigmoid(x) = 1/2 + 1/2 tanh(x / 2).  The LSTM cell is bound by its transcendentals (3 sigmoids + 2 tanh per cell, 16
// MUFU lanes per SM): 5 MUFU per cell instead of 10 with ex2 + rcp.
__device__ __forceinline__ float fast_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_sigmoid(float x) { return fmaf(0.5f, fast_tanh(0.5f * x), 0.5f); }
__device__ __forceinline__ float fast_elu(float x) { return x > 0.f ? x : ex2_ftz(1.4426950408889634f * x) - 1.0f; }
// Epilogue math by form: X = true (3xTF32 split form, fp32-accurate products) keeps the exact-mode functions of
// gemm_fp32.cu -- the MUFU versions above are accurate to 2^-11 only and would bound the whole result there.
template <bool X>
__device__ __forceinline__ float epi_sigmoid(float x) { return X ? 1.f / (1.f + expf(-x)) : fast_sigmoid(x); }
template <bool X>
__device__ __forceinline__ float epi_tanh(float x) { return X ? tanhf(x) : fast_tanh(x); }
template <bool X>
__device__ __forceinline__ float epi_elu(float x) { return X ? (x > 0.f ? x : expm1f(x)) : fast_elu(x); }

// 3xTF32 operand split: x = hi + lo with hi = tf32(x), lo = tf32(x - hi) (|x - hi - lo| <= 2^-22 |x|).  Both halves are
// written as tf32 values (low 13 mantissa bits zero), so the products do not depend on how the tensor core reads the
// low bits of an fp32 word.
__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void split16(unsigned char* head, unsigned char* tail) {  // one 16-byte chunk in place
    const float4 v = *reinterpret_cast<const float4*>(head);
    uint4 h, l;
    h.x = to_tf32(v.x);
    h.y = to_tf32(v.y);
    h.z = to_tf32(v.z);
    h.w = to_tf32(v.w);
    l.x = to_tf32(v.x - __uint_as_float(h.x));
    l.y = to_tf32(v.y - __uint_as_float(h.y));
    l.z = to_tf32(v.z - __uint_as_float(h.z));
    l.w = to_tf32(v.w - __uint_as_float(h.w));
    *reinterpret_cast<uint4*>(head) = h;
    *reinterpret_cast<uint4*>(tail) = l;
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// per-stream (sum, sum of squares) of the rows a warp owns: rows are ordered by stream, so the warp holds a short
// monotone run of stream indices; one shuffle reduction and one pair of double atomics per distinct stream
__device__ __forceinline__ void stats_commit(double* stats, int stride, int b, float s, float ss) {
    const unsigned full = 0xffffffffu;
    int lo = b < 0 ? 0x7fffffff : b, hi = b;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        lo = min(lo, __shfl_xor_sync(full, lo, off));
        hi = max(hi, __shfl_xor_sync(full, hi, off));
    }
    for (int bb = lo; bb <= hi; ++bb) {  // no valid row: lo = INT_MAX > hi = -1, the loop does not run
        float a = b == bb ? s : 0.f, c = b == bb ? ss : 0.f;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            a += __shfl_xor_sync(full, a, off);
            c += __shfl_xor_sync(full, c, off);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(stats + (long long)stride * bb, (double)a);
            atomicAdd(stats + (long long)stride * bb + 1, (double)c);
        }
    }
}

// Cycle accounting of the warp roles (diagnostic; SE_B200_GEMM_PROFILE=1 at context creation turns it on through
// GemmTma::profile): [0] MMA thread waiting for operands (full), [1] for a drained accumulator (tempty), [2] total MMA-thread
// loop, [3] producer waiting for a free stage (empty), [4] producer total, [5] epilogue lead warps waiting for an
// accumulator (tfull), [6] epilogue lead warps total, [7] tiles.  Summed over CTAs; read with se_debug_gemm_counters.
__device__ unsigned long long g_gemm_prof[8];
#ifndef SE_GEMM_PROFILE
#define SE_GEMM_PROFILE 0  // build with -DSE_GEMM_PROFILE=1 (tools/gemm_roles.py does) to compile the accounting in
#endif
#ifndef SE_GEMM_TMA_FENCE
#define SE_GEMM_TMA_FENCE 0
#endif
constexpr bool kProf = SE_GEMM_PROFILE != 0;

constexpr int kW2Floats = 32 * 16 + 32;  // fused small gate: W2 [2*C2][16] + bias2 [2*C2], C2 <= 16

// B2B: the kernel instance carries the back-to-back gate GEMM (EPI_ELU_GATE): always for BN = 16 (first encoder conv),
// for BN = 32 / 64 only in the dedicated instances (fp16 operands) so that the plain GEMMs keep their deeper pipelines
// TMA: 0 = cp.async gather producers, 1 = TMA tile loads, 2 = TMA + CTA pair (cta_group::2: the two CTAs of a cluster run
// one M256 x BN MMA; each holds its own 128 rows of A and HALF of the weight tile, which halves the shared-memory reads of
// the tensor core and the fill traffic per SM -- these GEMMs run at the shared-memory bandwidth of their operand tiles)
// SPLIT: the 3xTF32 form (gemm_tc3x_kernel; gathered fp32 operands only).  A stage holds two operand planes, the tf32
// heads and the tf32 tails, so it is twice the size of a tf32 stage: the tile is capped at BN = 128 (two 64 KB stages
// beside the 72 KB of epilogue staging) and the narrower tiles get their own stage counts.
template <int BN, bool B2B = (BN == 16), int TMA = 0, bool SPLIT = false>
struct Cfg {
    // TMEM accumulators = epilogue groups.  Split form at BN = 128: 2 groups, so that the 13 warps get 128 registers
    // each (21 warps get 80, and the exact-mode LSTM cell spills at 80)
    static constexpr int NACC = (BN > 128 || (B2B && BN > 16) || (SPLIT && BN == 128)) ? 2 : 4;
    static constexpr int STAGES = SPLIT      ? (BN > 64 ? 2 : (BN > 16 ? 3 : 4))
                                  : TMA == 2 ? (BN > 128 ? 4 : (BN > 64 ? 5 : 6))
                                             : (BN > 128 ? 3 : (BN > 32 ? 4 : (B2B ? 4 : 6)));  // B2B: room for the gate tiles
    static constexpr int WARPS = kFirstEpiWarp + 4 * NACC;
    static constexpr int THREADS = WARPS * 32;
    // back-to-back gate (BN == 16, fp16 operands): a second accumulator of 32 columns per group, the ELU tile as an
    // fp16 A operand (128 rows x 128 B) per group and the 32 x 16 gate weights as a B operand (4 KB); the split form
    // (fp32 operands) keeps the register version of the gate and needs none of them
    static constexpr bool TC_GATE = B2B && !SPLIT;
    static constexpr int GATE_COLS = TC_GATE ? 2 * BN : 0;
    static constexpr int ETILE_BYTES = TC_GATE ? NACC * BM * BKB : 0;
    static constexpr int W2T_BYTES = TC_GATE ? 2 * BN * BKB : 0;
    static constexpr int TMEM_COLS_RAW = NACC * (BN + GATE_COLS);
    static constexpr uint32_t TMEM_COLS =
        TMEM_COLS_RAW <= 32 ? 32
                            : (TMEM_COLS_RAW <= 64 ? 64 : (TMEM_COLS_RAW <= 128 ? 128 : (TMEM_COLS_RAW <= 256 ? 256 : 512)));
    static constexpr int B_STAGE_BYTES = (TMA == 2 ? BN / 2 : BN) * BKB;
    static constexpr int PLANE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;  // one operand plane: A tile, then W tile
    static constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * PLANE_BYTES;     // split: heads, then tails
    static constexpr int TILE_BYTES = STAGES * STAGE_BYTES;
    static constexpr int KOFF_MAX = 512;  // K <= 2048
    static constexpr int OFF_ETILE = TILE_BYTES;               // 1024-aligned (SWIZZLE_128B atoms)
    static constexpr int OFF_W2T = OFF_ETILE + ETILE_BYTES;    // 1024-aligned
    static constexpr int OFF_KOFF = OFF_W2T + W2T_BYTES;
    static constexpr int OFF_BAR = OFF_KOFF + KOFF_MAX * 4;
    static constexpr int NBAR = 2 * STAGES + 2 * NACC + (B2B ? NACC : 0);
    static constexpr int OFF_TMEM = OFF_BAR + NBAR * 8;
    static constexpr int OFF_W2 = (OFF_TMEM + 8 + 15) / 16 * 16;  // float [kW2Floats]
    static constexpr int OFF_BIAS = OFF_W2 + kW2Floats * 4;       // float [4*NACC warps][BN]: warp-private bias row
    static constexpr int OFF_STG = OFF_BIAS + 4 * NACC * BN * 4;  // float [4*NACC warps][32][SPW]: staging
    static constexpr int BYTES = 1024 /*align slack*/ + OFF_STG + 4 * NACC * 32 * SPW * 4;
    static_assert(STAGE_BYTES % 1024 == 0, "stages must keep the 1024-byte swizzle alignment");
    static_assert(TMEM_COLS_RAW <= 512, "TMEM has 512 columns");
    static_assert(OFF_STG % 16 == 0 && OFF_BIAS % 16 == 0 && OFF_W2 % 16 == 0, "float4 alignment");
    static_assert(BYTES <= 227 * 1024, "shared memory budget");
    static_assert(!SPLIT || (TMA == 0 && BN <= 128), "the split form gathers fp32 operands into tiles of <= 128 columns");
};

// coalesced write-out of a staged chunk: W columns (8, 16 or 32) of the warp's 32 rows; consecutive lanes write
// consecutive float4 of a row.  `cnt` = valid columns of the chunk (<= W), `ooff` = this lane's row offset (-1: none)
template <int W, bool ROWCNT = false>
__device__ __forceinline__ void store_chunk(const float* stg, int col0, float* out, long long ooff, int cnt, bool vec4,
                                            int lane, bool out_half = false) {
    // ROWCNT: `cnt` is this lane's (= row's) own limit instead of a warp-uniform one
    const unsigned full = 0xffffffffu;
    if (out_half) {  // fp16 destination (operand of the next GEMM): `out` is a __half*, offsets are in halves
        __half* oh = reinterpret_cast<__half*>(out);
        if (vec4) {
            constexpr int C4 = W / 4;
            constexpr int RPI = 32 / C4;
            const int c4 = lane % C4;
#pragma unroll
            for (int i = 0; i < 32 / RPI; ++i) {
                const int r = i * RPI + lane / C4;
                const long long off = __shfl_sync(full, ooff, r);
                const int rc = ROWCNT ? __shfl_sync(full, cnt, r) : cnt;
                if (off >= 0 && 4 * c4 < rc) {
                    const float4 v = *reinterpret_cast<const float4*>(stg + r * SPW + col0 + 4 * c4);
                    const __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
                    uint2 u;
                    u.x = *reinterpret_cast<const uint32_t*>(&lo);
                    u.y = *reinterpret_cast<const uint32_t*>(&hi);
                    *reinterpret_cast<uint2*>(oh + off + 4 * c4) = u;
                }
            }
        } else {
            constexpr int RPI = 32 / W;
            const int c = lane % W;
#pragma unroll 4
            for (int i = 0; i < 32 / RPI; ++i) {
                const int r = i * RPI + lane / W;
                const long long off = __shfl_sync(full, ooff, r);
                const int rc = ROWCNT ? __shfl_sync(full, cnt, r) : cnt;
                if (off >= 0 && c < rc) oh[off + c] = __float2half_rn(stg[r * SPW + col0 + c]);
            }
        }
        return;
    }
    if (vec4) {
        constexpr int C4 = W / 4;     // float4 per row
        constexpr int RPI = 32 / C4;  // rows per warp instruction
        const int c4 = lane % C4;
#pragma unroll
        for (int i = 0; i < 32 / RPI; ++i) {
            const int r = i * RPI + lane / C4;
            const long long off = __shfl_sync(full, ooff, r);
            const int rc = ROWCNT ? __shfl_sync(full, cnt, r) : cnt;
            if (off >= 0 && 4 * c4 < rc)
                *reinterpret_cast<float4*>(out + off + 4 * c4) =
                    *reinterpret_cast<const float4*>(stg + r * SPW + col0 + 4 * c4);
        }
    } else {
        constexpr int RPI = 32 / W;
        const int c = lane % W;
#pragma unroll 4
        for (int i = 0; i < 32 / RPI; ++i) {
            const int r = i * RPI + lane / W;
            const long long off = __shfl_sync(full, ooff, r);
            const int rc = ROWCNT ? __shfl_sync(full, cnt, r) : cnt;
            if (off >= 0 && c < rc) out[off + c] = stg[r * SPW + col0 + c];
        }
    }
}

// gated 1x1 pair in registers (CRN_ELU.py:240): y[c] = (W2[2c].e + b2[2c]) * sigmoid(W2[2c+1].e + b2[2c+1]), c < C2
template <int KC, bool X>
__device__ __forceinline__ void small_gate(const float* s_w2, const float* e, int C2, float* y) {
    const float* b2 = s_w2 + 32 * 16;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        float a = 0.f;
        if (c < KC && c < C2) {
            float gt = b2[2 * c + 1];
            a = b2[2 * c];
            const float4* wa = reinterpret_cast<const float4*>(s_w2 + (2 * c) * 16);
            const float4* wg = reinterpret_cast<const float4*>(s_w2 + (2 * c + 1) * 16);
#pragma unroll
            for (int q = 0; q < KC / 4; ++q) {
                const float4 x = wa[q], z = wg[q];
                a += x.x * e[4 * q] + x.y * e[4 * q + 1] + x.z * e[4 * q + 2] + x.w * e[4 * q + 3];
                gt += z.x * e[4 * q] + z.y * e[4 * q + 1] + z.z * e[4 * q + 2] + z.w * e[4 * q + 3];
            }
            a *= epi_sigmoid<X>(gt);
        }
        y[c] = a;
    }
}

// The kernel body of both forms (gemm_tc_kernel, gemm_tc3x_kernel below)
template <int BN, typename AT, bool B2B, int TMA, bool SPLIT>
__device__ __forceinline__ void gemm_tc_body(const GemmParams& p, const GemmTma& tm) {
    constexpr int BKE = BKB / (int)sizeof(AT);  // elements per k-block
    constexpr int UE = 16 / (int)sizeof(AT);    // elements per 16-byte gather unit
    using S = Cfg<BN, B2B, TMA, SPLIT>;
    static_assert(!SPLIT || sizeof(AT) == 4, "the split form reads fp32 operands");
    constexpr int STAGES = S::STAGES;
    constexpr int NACC = S::NACC;
    constexpr bool PAIR = TMA == 2;
    constexpr int CS = PAIR ? 2 : 1;  // CTAs per tile row group
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t tiles = (raw + 1023u) & ~1023u;  // SWIZZLE_128B atoms need 1024-byte alignment
    unsigned char* tiles_ptr = smem_raw + (tiles - raw);
    int* s_koff = reinterpret_cast<int*>(tiles_ptr + S::OFF_KOFF);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(tiles_ptr + S::OFF_BAR);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tiles_ptr + S::OFF_TMEM);
    float* s_w2 = reinterpret_cast<float*>(tiles_ptr + S::OFF_W2);
    const uint32_t bar0 = smem_u32(s_bar);
    // barriers: [0,STAGES) full, [STAGES,2*STAGES) empty, then NACC tmem_full, NACC tmem_empty
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };
    auto tfull_bar = [&](int g) { return bar0 + 8u * (2 * STAGES + g); };
    auto tempty_bar = [&](int g) { return bar0 + 8u * (2 * STAGES + NACC + g); };

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);  // provably warp-uniform: role dispatch of the issuing warps
    const int lane = tid & 31;
    const int nkb = p.K / BKE;  // K and Npad are padded by the host (zero weights): no bounds checks on either operand
    const int ntn = (p.epi == EPI_GRU ? p.N : p.Npad) / BN;
    const int rowsPerStream = p.Tn * p.Fo;
    const int nstreams = p.M / rowsPerStream;
    // TMA: a tile is a rectangle of tm.bb streams x tm.bt frames x Fo bins (tm.rows of the 128 rows are real)
    const int ntiles_m = TMA ? ((nstreams + tm.bb - 1) / tm.bb) * tm.tgroups * tm.fsegs : (p.M + BM - 1) / BM;
    // CTA pair: the cluster walks "super-tiles" = two consecutive m-tiles x one n-tile; rank r owns m-tile 2 j + r (its
    // rows of A, its TMEM lanes, its epilogue).  An m-tile past the end is a dummy (out-of-range boxes are zero-filled,
    // every row masked): both CTAs of a pair run the same number of stages.
    const uint32_t crank = PAIR ? (uint32_t)(blockIdx.x & 1) : 0u;
    const int tfirst = (int)blockIdx.x / CS, tstep = (int)gridDim.x / CS;
    const int ntiles = ((ntiles_m + CS - 1) / CS) * ntn;

    if (TMA) {  // per k-block box origin (channel, bin, frame, -)
        for (int i = tid; i < 4 * nkb; i += S::THREADS) s_koff[i] = __ldg(reinterpret_cast<const int*>(tm.kcoord) + i);
    } else {
        for (int i = tid; i < p.K / UE; i += S::THREADS) s_koff[i] = __ldg(p.koff + i);
    }
    const AT* const Abase = reinterpret_cast<const AT*>(p.A);
    const AT* const Wbase = reinterpret_cast<const AT*>(p.W);
    const bool out_half = p.out_half != 0;
    // back-to-back gate on the tensor core: fp16 operands only (the ELU tile is rounded to fp16 exactly as the unfused
    // path rounds tmp_e); tf32 mode keeps the register version
    const bool b2b = B2B && p.epi == EPI_ELU_GATE && sizeof(AT) == 2;
    // gate bias: behind the fp32 weights of the register version (BN = 16), else at the start of the same region
    float* const s_b2 = BN == 16 ? s_w2 + 32 * 16 : s_w2;
    if (B2B && p.epi == EPI_ELU_GATE) {
        if (BN == 16)
            for (int i = tid; i < 2 * p.C2 * 16; i += S::THREADS) s_w2[i] = __ldg(p.W2 + i);
        for (int i = tid; i < 2 * p.C2; i += S::THREADS) s_b2[i] = __ldg(p.bias2 + i);
        if (b2b) {  // W2 [2 C2][BN] fp32, rows n = 2c (trans) / 2c+1 (gated): chunk j (8 halves) of row n, rows >= 2 C2 zero
            constexpr int CPR = BN / 8;  // 16-byte chunks per row
            for (int u = tid; u < 2 * BN * CPR; u += S::THREADS) {
                const int n = u / CPR, j = u % CPR;
                __align__(16) __half h[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) h[i] = __float2half_rn(n < 2 * p.C2 ? __ldg(p.W2 + n * BN + 8 * j + i) : 0.f);
                *reinterpret_cast<uint4*>(tiles_ptr + S::OFF_W2T + (n >> 3) * 1024 + (n & 7) * 128 + ((j ^ (n & 7)) << 4)) =
                    *reinterpret_cast<const uint4*>(h);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
    }
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), TMA ? 1 : kProducerThreads);  // pair: only the leader's is used (bytes of both CTAs)
            mbar_init(empty_bar(s), 1);
        }
        for (int g = 0; g < NACC; ++g) {
            mbar_init(tfull_bar(g), 1);
            // GRU tiles are read by every group; pair: the leader's barrier collects the epilogue threads of both CTAs
            mbar_init(tempty_bar(g), BN == 96 ? 128 * NACC : (PAIR ? 256 : 128));
            if (B2B) mbar_init(bar0 + 8u * (2 * STAGES + 2 * NACC + g), 1);  // gate MMA of group g finished
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        if (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                         "r"(S::TMEM_COLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                         "r"(S::TMEM_COLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();  // the peer's barriers and TMEM exist before anything is signalled at them
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(s_tmem);

    if (TMA && warp_u < 4) {
        // ============================ producer (TMA): warp 0, one elected lane issues ============================
        if (warp_u == 0) {
            uint32_t ps = 0, pphase = 0;
            // bytes that complete a stage: this CTA's two boxes; pair: the boxes of both CTAs land on the LEADER's barrier
            const uint32_t tx = (uint32_t)CS * ((uint32_t)tm.a_bytes + (uint32_t)S::B_STAGE_BYTES);
            constexpr int wrows = PAIR ? BN / 2 : BN;  // weight rows this CTA holds
            const bool prof = kProf && tm.profile != 0;
            long long w_empty = 0;
            const long long t_begin = kProf ? clock64() : 0;
            for (int tile = tfirst; tile < ntiles; tile += tstep) {
                // exact quotients by multiply-high (divisors <= 64, dividends < 2^26): a runtime division is ~50 instructions
                const int tdiv = div_mh(tile, tm.magic_ntn);
                const int tile_m = tdiv * CS + (int)crank, n0 = (tile - tdiv * ntn) * BN;
                const int tq = div_mh(tile_m, tm.magic_fsegs), fsg = tile_m - tq * tm.fsegs;
                const int bgrp = div_mh(tq, tm.magic_tgroups), tgrp = tq - bgrp * tm.tgroups;
                const int cb = p.b0 + bgrp * tm.bb, ct = tm.t_org + tgrp * tm.bt;
                const int cf = tm.f_org + fsg * tm.Fs * tm.fstep;
                for (int kb = 0; kb < nkb; ++kb) {
                    const long long t0 = prof ? clock64() : 0;
                    mbar_wait<32>(empty_bar(ps), pphase ^ 1u);
                    if (prof) w_empty += clock64() - t0;
                    const uint32_t stage = tiles + (uint32_t)ps * S::STAGE_BYTES;
                    const int k0 = s_koff[4 * kb], k1 = s_koff[4 * kb + 1], k2 = s_koff[4 * kb + 2];
                    if (elect_one()) {
                        if (PAIR) {
                            const uint32_t lead_full = mapa_rank(full_bar(ps), 0);
                            if (crank == 0) mbar_arrive_expect_tx(full_bar(ps), tx);
                            tma_load_4d_pair(stage, &tm.a, lead_full, k0, cf + k1, ct + k2, cb);
                            tma_load_2d_pair(stage + A_STAGE_BYTES, &tm.w, lead_full, kb * BKE, n0 + (int)crank * wrows);
                        } else {
                            mbar_arrive_expect_tx(full_bar(ps), tx);
                            tma_load_4d(stage, &tm.a, full_bar(ps), k0, cf + k1, ct + k2, cb);
                            tma_load_2d(stage + A_STAGE_BYTES, &tm.w, full_bar(ps), kb * BKE, n0);
                        }
                    }
                    __syncwarp();
                    if (++ps == STAGES) {
                        ps = 0;
                        pphase ^= 1u;
                    }
                }
            }
            if (prof && lane == 0) {
                atomicAdd(&g_gemm_prof[3], (unsigned long long)w_empty);
                atomicAdd(&g_gemm_prof[4], (unsigned long long)(clock64() - t_begin));
            }
        }
    } else if (warp_u < 4) {
        // ============================ producers ============================
        // thread (g = tid/8, j = tid%8) serves chunk j of rows g, g+16, g+32, ... of both operand tiles
        const int j = tid & 7;
        const int g = tid >> 3;
        const uint32_t dst_gj = (uint32_t)((g >> 3) * 1024 + (g & 7) * 128 + ((j ^ (g & 7)) << 4));
        constexpr int B_ITERS = BN / 16;
        uint32_t ps = 0, pphase = 0;  // stage ring position / phase (the ring runs on across tiles)
        // split form: this thread's chunks of stage s, once landed, become tf32 heads in place and tf32 tails in the
        // stage's second plane; then the stage is handed to the tensor core through the async proxy
        int split_ps = -1;  // stage whose loads are in flight and not split yet
        auto split_stage = [&](int s) {
            unsigned char* base = tiles_ptr + s * S::STAGE_BYTES + dst_gj;
#pragma unroll
            for (int i = 0; i < BM / 16; ++i) split16(base + i * 2048, base + S::PLANE_BYTES + i * 2048);
#pragma unroll
            for (int i = 0; i < B_ITERS; ++i)
                split16(base + A_STAGE_BYTES + i * 2048, base + S::PLANE_BYTES + A_STAGE_BYTES + i * 2048);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_arrive(full_bar(s));
        };
        const int q16 = 16 / p.Fo, r16 = 16 % p.Fo;
        for (int tile = tfirst; tile < ntiles; tile += tstep) {
            const int m0 = (tile / ntn) * BM;
            const int n0 = (tile % ntn) * BN;
            const AT* arow[BM / 16];
            uint32_t avalid = 0;
            {
                // rows m0 + g + 16 i: one division for the first row, then (q16 frames, r16 bins) steps
                int m = m0 + g;
                int bl = m / rowsPerStream;
                int rr = m - bl * rowsPerStream;
                int t = rr / p.Fo;
                int f = rr - t * p.Fo;
#pragma unroll
                for (int i = 0; i < BM / 16; ++i) {
                    arow[i] = Abase;
                    if (m < p.M) {
                        arow[i] = Abase + (p.b0 + bl) * p.sB + t * p.sT + f * p.sF;
                        avalid |= 1u << i;
                    }
                    m += 16;
                    f += r16;
                    t += q16;
                    if (f >= p.Fo) {
                        f -= p.Fo;
                        ++t;
                    }
                    while (t >= p.Tn) {
                        t -= p.Tn;
                        ++bl;
                    }
                }
            }
            uint32_t asz[BM / 16];
#pragma unroll
            for (int i = 0; i < BM / 16; ++i) asz[i] = ((avalid >> i) & 1u) ? 16u : 0u;  // 0: zero-fill the row
            const AT* wptr = Wbase + (long long)(n0 + g) * p.K + UE * j;
            const long long wstep = 16LL * p.K;
            const int* kptr = s_koff + j;
            for (int kb = 0; kb < nkb; ++kb) {
                mbar_wait<32>(empty_bar(ps), pphase ^ 1u);
                const uint32_t stage = tiles + (uint32_t)ps * S::STAGE_BYTES + dst_gj;
                const int ko = kptr[kb * 8];
#pragma unroll
                for (int i = 0; i < BM / 16; ++i) cp_async16(stage + (uint32_t)i * 2048u, arow[i] + ko, asz[i]);
                const AT* wp = wptr;
#pragma unroll
                for (int i = 0; i < B_ITERS; ++i) {
                    cp_async16(stage + A_STAGE_BYTES + (uint32_t)i * 2048u, wp, 16u);
                    wp += wstep;
                }
                wptr += BKE;
                if (SPLIT) {
                    // one k-block behind: the previous stage's chunks have landed while this one's loads are in flight
                    cp_async_commit();
                    if (split_ps >= 0) {
                        cp_async_wait<1>();
                        split_stage(split_ps);
                    }
                    split_ps = (int)ps;
                } else {
                    cp_async_mbar_arrive_noinc(full_bar(ps));
                }
                if (++ps == STAGES) {
                    ps = 0;
                    pphase ^= 1u;
                }
            }
        }
        if (SPLIT && split_ps >= 0) {
            cp_async_wait<0>();
            split_stage(split_ps);
        }
    } else if (warp_u == 4) {
        // ============================ MMA issuer ============================
        const uint32_t tmem_base_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        // instruction descriptor: D=f32 (1<<4), A/B format @7/@10 (tf32 = 2, f16 = 0), K-major both, N>>3 @17, M>>4 @24
        constexpr uint32_t fmt = sizeof(AT) == 4 ? 2u : 0u;
        constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) |
                                   ((uint32_t)(BM >> 4) << 24);
        constexpr uint32_t idesc_pair = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
        if (!PAIR || crank == 0) {  // pair: only the leader issues (for both CTAs); the warp loops, one lane issues
            uint32_t ms = 0, mphase = 0, it = 0;
            const bool prof = kProf && TMA && tm.profile != 0;
            long long w_full = 0, w_tempty = 0;
            const long long t_begin = kProf ? clock64() : 0;
            for (int tile = tfirst; tile < ntiles; tile += tstep, ++it) {
                const int g = it % NACC;
                const long long t0 = prof ? clock64() : 0;
                mbar_wait<0>(tempty_bar(g), ((it / NACC) & 1) ^ 1);  // the epilogue has drained this accumulator
                if (prof) w_tempty += clock64() - t0;
                tc_fence_after();
                const uint32_t tacc = tmem_base_u + (uint32_t)(g * BN);
                uint32_t acc = 0;
                for (int kb = 0; kb < nkb; ++kb) {
                    const long long t1 = prof ? clock64() : 0;
                    mbar_wait<0>(full_bar(ms), mphase);
                    if (prof) w_full += clock64() - t1;
                    // cp.async wrote the stage through the generic proxy; TMA stages are already async-proxy writes, and
                    // the fence would make this thread wait for its own MMAs in flight (one k-block at a time)
                    if (!TMA || SE_GEMM_TMA_FENCE) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    tc_fence_after();
                    const uint64_t adesc = make_desc(tiles + ms * (uint32_t)S::STAGE_BYTES);
                    const uint64_t bdesc = adesc + (uint64_t)(A_STAGE_BYTES >> 4);
                    constexpr uint64_t tail = (uint64_t)(S::PLANE_BYTES >> 4);  // split: heads -> tails plane
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            // one MMA consumes 32 bytes of K (8 tf32 / 16 fp16): +2 in the (addr >> 4) field of the atom
                            const uint32_t a1 = kk ? 1u : acc;
                            const uint64_t ad = adesc + (uint64_t)(2 * kk), bd = bdesc + (uint64_t)(2 * kk);
                            if (PAIR) {
                                tc_mma_f16_pair(tacc, ad, bd, idesc_pair, a1);
                            } else if (SPLIT) {  // small terms first: lo.hi + hi.lo, then hi.hi
                                tc_mma<AT>(tacc, ad + tail, bd, idesc, a1);
                                tc_mma<AT>(tacc, ad, bd + tail, idesc, 1u);
                                tc_mma<AT>(tacc, ad, bd, idesc, 1u);
                            } else {
                                tc_mma<AT>(tacc, ad, bd, idesc, a1);
                            }
                        }
                        if (PAIR) tc_commit_pair(empty_bar(ms), 3);  // the stage is free in BOTH CTAs
                        else tc_commit(empty_bar(ms));
                    }
                    __syncwarp();
                    acc = 1;
                    if (++ms == STAGES) {
                        ms = 0;
                        mphase ^= 1u;
                    }
                }
                if (elect_one()) {
                    if (PAIR) tc_commit_pair(tfull_bar(g), 3);  // each CTA's epilogue reads its own 128 TMEM lanes
                    else tc_commit(tfull_bar(g));
                }
                __syncwarp();
            }
            if (prof && lane == 0) {
                atomicAdd(&g_gemm_prof[0], (unsigned long long)w_full);
                atomicAdd(&g_gemm_prof[1], (unsigned long long)w_tempty);
                atomicAdd(&g_gemm_prof[2], (unsigned long long)(clock64() - t_begin));
                atomicAdd(&g_gemm_prof[7], (unsigned long long)it);
            }
        }
        __syncwarp();
    } else {
        // ============================ epilogue groups ============================
        const int ew = warp - kFirstEpiWarp;  // 0 .. 4*NACC-1
        const int g = ew >> 2;                // group = accumulator
        const int q = warp & 3;               // TMEM lane quarter this warp may access (warp id % 4)
        float* stg = reinterpret_cast<float*>(tiles_ptr + S::OFF_STG) + ew * 32 * SPW;
        float* sbias = reinterpret_cast<float*>(tiles_ptr + S::OFF_BIAS) + ew * BN;
        float* srow = stg + lane * SPW;
        const bool vec4 = p.vec4 != 0;
        // GRU tiles (BN = 96): every group works on every tile of this CTA (8 of its 32 hidden units each); all other
        // epilogues: group g owns the tiles g, g + NACC, ... and accumulator g
        const bool gru = BN == 96 && p.epi == EPI_GRU;
        uint32_t it = gru ? 0 : g;
        const uint32_t it_step = gru ? 1 : NACC;
        const uint32_t lead_tempty0 = PAIR ? mapa_rank(tempty_bar(0), 0) : 0u;  // pair: the leader's "accumulator drained"
        const long long t_epi_begin = kProf ? clock64() : 0;
        for (int tile = tfirst + it * tstep; tile < ntiles; tile += it_step * tstep, it += it_step) {
            const int acc = gru ? (int)(it % NACC) : g;
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
            const int tdiv = TMA ? div_mh(tile, tm.magic_ntn) : tile / ntn;
            const int m0 = (TMA ? tdiv * CS + (int)crank : tdiv) * BM;  // (used by the row = sequence epilogues: LSTM)
            const int n0 = (tile - tdiv * ntn) * BN;
            const int m = m0 + q * 32 + lane;
            int b = -1;
            long long ooff = -1;
            int nlim = p.N;  // columns this row owns (merged-parity transposed conv: half of them on the last bin)
            if (TMA) {  // rectangular tile: row r = (stream bi, frame ti, bin f) of tile (bgrp, tgrp)
                const int tile_m = tdiv * CS + (int)crank;
                const int tq = div_mh(tile_m, tm.magic_fsegs), fsg = tile_m - tq * tm.fsegs;
                const int bgrp = div_mh(tq, tm.magic_tgroups), tgrp = tq - bgrp * tm.tgroups;
                const int r = q * 32 + lane, rpf = tm.bt * tm.Fs;
                const int bi = r / rpf, rr = r - bi * rpf;
                const int ti = rr / tm.Fs, f = fsg * tm.Fs + (rr - ti * tm.Fs);
                const int bl = bgrp * tm.bb + bi, t = tgrp * tm.bt + ti;
                if (r < tm.rows && bl < nstreams && t < p.Tn) {
                    b = p.b0 + bl;
                    ooff = b * p.oB + t * p.oT + f * p.oF;
                    if (p.odd_tail && f == p.Fo - 1) nlim = p.N >> 1;
                }
            } else if (m < p.M) {
                const int bl = m / rowsPerStream;
                const int rr = m - bl * rowsPerStream;
                const int t = rr / p.Fo;
                const int f = rr - t * p.Fo;
                b = p.b0 + bl;
                ooff = b * p.oB + t * p.oT + f * p.oF;
                if (p.odd_tail && f == p.Fo - 1) nlim = p.N >> 1;
            }
            const bool row_ok = b >= 0;
            // this tile's bias row, warp-private (zero beyond Npad)
            for (int i = lane; i < BN; i += 32) sbias[i] = (n0 + i) < p.Npad ? __ldg(p.bias + n0 + i) : 0.f;
            __syncwarp();
            // one warp per group polls the mbarrier, the other three block on a hardware named barrier (no issue slots)
            float s_acc = 0.f, ss_acc = 0.f;
            auto wait_acc = [&]() {
                // one warp per group polls the mbarrier, the other three block on a hardware named barrier
                if ((ew & 3) == 0) {
                    const bool prof = kProf && TMA && tm.profile != 0 && lane == 0;
                    const long long t0 = prof ? clock64() : 0;
                    mbar_wait<64>(tfull_bar(acc), (it / NACC) & 1);
                    if (prof) atomicAdd(&g_gemm_prof[5], (unsigned long long)(clock64() - t0));
                }
                asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
                tc_fence_after();
            };

            if (BN == 96 && p.epi == EPI_GRU) {
                // tile columns: [r | z | n] of hidden units j0 .. j0+32; this group: units u0 .. u0+8
                constexpr int U = BN / 3;
                const int j0 = (tile % ntn) * U;
                const int u0 = 8 * g;
                const int ul = lane & 7;
                const int ju = j0 + u0 + ul;
                // the cell's other inputs do not depend on the MMA: fetch them while it runs
                float pr[8], pz[8], pn[8], ph[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int mm = m0 + q * 32 + i * 4 + (lane >> 3);
                    pr[i] = pz[i] = pn[i] = ph[i] = 0.f;
                    if (mm < p.M) {
                        const long long bb = p.b0 + mm;  // Tn = Fo = 1: row = stream
                        const float* gi = p.gi + bb * p.giB;
                        pr[i] = gi[ju];
                        pz[i] = gi[p.H + ju];
                        pn[i] = gi[2 * p.H + ju];
                        ph[i] = p.hprev[bb * p.hB + ju];
                    }
                }
                const float br = sbias[u0 + ul], bz = sbias[U + u0 + ul], bn = sbias[2 * U + u0 + ul];
                wait_acc();
                uint32_t v[24];
                tmem_ld8_nowait(tlane + u0, v);
                tmem_ld8_nowait(tlane + U + u0, v + 8);
                tmem_ld8_nowait(tlane + 2 * U + u0, v + 16);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(tempty_bar(acc));
#pragma unroll
                for (int i = 0; i < 24; i += 4)
                    *reinterpret_cast<uint4*>(srow + i) = make_uint4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = i * 4 + (lane >> 3);
                    const int mm = m0 + q * 32 + r;
                    if (mm < p.M) {
                        const float* sr = stg + r * SPW;
                        const float rg = epi_sigmoid<SPLIT>(pr[i] + sr[ul] + br);
                        const float zg = epi_sigmoid<SPLIT>(pz[i] + sr[8 + ul] + bz);
                        const float ng = epi_tanh<SPLIT>(pn[i] + rg * (sr[16 + ul] + bn));
                        const float hn = (1.0f - zg) * ng + zg * ph[i];
                        p.out[(p.b0 + mm) * p.oB + ju] = hn;
                        // fp16 copy = operand of the next step / the next layer's projection
                        if (p.out_h2) reinterpret_cast<__half*>(p.out_h2)[(p.b0 + mm) * p.o2B + ju] = __float2half_rn(hn);
                    }
                }
                __syncwarp();
            } else if ((BN == 128 || BN == 256) && p.epi == EPI_LSTM) {
                // tile columns: [i | f | g | o] of hidden units j0 .. j0+U (nn.LSTM gate order); 8 units per pass.
                // c_prev = hprev (row stride hB), h' -> out (oB), c' -> out2 (o2B); Tn = Fo = 1: row = sequence.
                // Thread = row (its TMEM lane): the four gate pre-activations of 8 units come straight out of TMEM, the cell
                // state is two 16-byte loads / stores of the thread's own row, h' one 16-byte store (fp16) -- no transposition
                // through shared memory, no per-cell address arithmetic (the first version spent 170 of its 443 instructions
                // per pass on that and made the LSTM step GEMMs epilogue-bound: tools/fsn_roles.py).
                constexpr int U = BN / 4;
                const int j0 = n0 / 4;  // = (tile % ntn) * U
                const bool ok = m < p.M;
                const long long row = p.b0 + (ok ? m : 0);
                const float* cin = p.hprev + row * p.hB + j0;
                float* cout = p.out2 + row * p.o2B + j0;
                __half* hout_h = reinterpret_cast<__half*>(p.out) + row * p.oB + j0;
                float* hout_f = p.out + row * p.oB + j0;
                const bool vec = ((p.hB | p.o2B) & 3) == 0 && (p.out_half ? (p.oB & 7) == 0 : (p.oB & 3) == 0) &&
                                 ((reinterpret_cast<uintptr_t>(p.hprev) | reinterpret_cast<uintptr_t>(p.out2) |
                                   reinterpret_cast<uintptr_t>(p.out)) & 15) == 0;
                // cell state of the FullSubNet models: UNIT-major [H][c_rows] (c_rows > 0), so that the 32 rows of a warp are
                // one 128-byte line per unit instead of 32 lines per 16-byte vector (the epilogue is bound by LSU wavefronts)
                const long long crs = p.c_rows;
                const float* cin_t = p.hprev + (long long)j0 * crs + row;
                float* cout_t = p.out2 + (long long)j0 * crs + row;
                auto load_c = [&](int u0, float* pc) {  // c_{t-1}: independent of the MMAs, fetched one pass ahead
                    if (crs) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) pc[k] = ok ? cin_t[(long long)(u0 + k) * crs] : 0.f;
                    } else if (vec) {
                        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        const float4 a = ok ? *reinterpret_cast<const float4*>(cin + u0) : z4;
                        const float4 c = ok ? *reinterpret_cast<const float4*>(cin + u0 + 4) : z4;
                        pc[0] = a.x, pc[1] = a.y, pc[2] = a.z, pc[3] = a.w, pc[4] = c.x, pc[5] = c.y, pc[6] = c.z, pc[7] = c.w;
                    } else {
#pragma unroll
                        for (int k = 0; k < 8; ++k) pc[k] = ok ? cin[u0 + k] : 0.f;
                    }
                };
                float pc[8], pcn[8];
                load_c(0, pc);
                wait_acc();
                // gate pre-activations of pass u0 + 8 are in flight (TMEM -> registers) while pass u0 is computed
                uint32_t vb[2][32];
                auto load_gates = [&](int u0, uint32_t* v) {
                    tmem_ld8_nowait(tlane + u0, v);
                    tmem_ld8_nowait(tlane + U + u0, v + 8);
                    tmem_ld8_nowait(tlane + 2 * U + u0, v + 16);
                    tmem_ld8_nowait(tlane + 3 * U + u0, v + 24);
                };
                load_gates(0, vb[0]);
#pragma unroll 2
                for (int u0 = 0; u0 < U; u0 += 8) {
                    uint32_t* v = vb[(u0 >> 3) & 1];
                    tmem_ld_wait();
                    if (u0 + 8 < U) {
                        load_c(u0 + 8, pcn);
                        load_gates(u0 + 8, vb[((u0 >> 3) + 1) & 1]);
                    } else {  // the whole accumulator is in registers: hand it back to the MMA warp
                        tc_fence_before();
                        if (PAIR) mbar_arrive_cluster(lead_tempty0 + 8u * (uint32_t)acc);
                        else mbar_arrive(tempty_bar(acc));
                    }
                    float cn[8], hv[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float ig = epi_sigmoid<SPLIT>(__uint_as_float(v[k]) + sbias[u0 + k]);
                        const float fg = epi_sigmoid<SPLIT>(__uint_as_float(v[8 + k]) + sbias[U + u0 + k]);
                        const float gg = epi_tanh<SPLIT>(__uint_as_float(v[16 + k]) + sbias[2 * U + u0 + k]);
                        const float og = epi_sigmoid<SPLIT>(__uint_as_float(v[24 + k]) + sbias[3 * U + u0 + k]);
                        cn[k] = fmaf(fg, pc[k], ig * gg);
                        hv[k] = og * epi_tanh<SPLIT>(cn[k]);
                    }
                    if (ok && crs) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) cout_t[(long long)(u0 + k) * crs] = cn[k];
                    }
                    if (ok) {
                        if (vec) {
                            if (!crs) {
                                *reinterpret_cast<float4*>(cout + u0) = make_float4(cn[0], cn[1], cn[2], cn[3]);
                                *reinterpret_cast<float4*>(cout + u0 + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
                            }
                            if (p.out_half) {
                                const __half2 h0 = __floats2half2_rn(hv[0], hv[1]), h1 = __floats2half2_rn(hv[2], hv[3]),
                                              h2 = __floats2half2_rn(hv[4], hv[5]), h3 = __floats2half2_rn(hv[6], hv[7]);
                                uint4 u;
                                u.x = *reinterpret_cast<const uint32_t*>(&h0);
                                u.y = *reinterpret_cast<const uint32_t*>(&h1);
                                u.z = *reinterpret_cast<const uint32_t*>(&h2);
                                u.w = *reinterpret_cast<const uint32_t*>(&h3);
                                *reinterpret_cast<uint4*>(hout_h + u0) = u;
                            } else {
                                *reinterpret_cast<float4*>(hout_f + u0) = make_float4(hv[0], hv[1], hv[2], hv[3]);
                                *reinterpret_cast<float4*>(hout_f + u0 + 4) = make_float4(hv[4], hv[5], hv[6], hv[7]);
                            }
                        } else {
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                if (!crs) cout[u0 + k] = cn[k];
                                if (p.out_half) hout_h[u0 + k] = __float2half_rn(hv[k]);
                                else hout_f[u0 + k] = hv[k];
                            }
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 8; ++k) pc[k] = pcn[k];
                }
            } else if (B2B && p.epi == EPI_ELU_GATE && (BN > 16 || b2b)) {
                // conv + ELU, then the gated 1x1 pair of CRN_ELU.py:240 as a SECOND GEMM on the tensor core: this row of
                // the ELU tile goes as fp16 into the group's A-operand tile (logical 16-byte chunks 0 .. BN/8-1 of row r),
                // BN/16 MMAs M128 x N(2 BN) x K16 against the resident gate weights, gate on the 2 BN result columns
                const int r = q * 32 + lane;
                unsigned char* et = tiles_ptr + S::OFF_ETILE + g * (BM * BKB) + (r >> 3) * 1024 + (r & 7) * 128;
                wait_acc();
#pragma unroll
                for (int c0 = 0; c0 < BN; c0 += 16) {
                    uint32_t vr[16];
                    tmem_ld16_nowait(tlane + c0, vr);
                    tmem_ld_wait();
                    if (c0 + 16 >= BN) {  // conv accumulator fully read: hand it back to the MMA warp
                        tc_fence_before();
                        mbar_arrive(tempty_bar(acc));
                    }
                    float e[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) e[i] = fast_elu(__uint_as_float(vr[i]) + sbias[c0 + i]);
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const __half2 h0 = __floats2half2_rn(e[8 * j], e[8 * j + 1]), h1 = __floats2half2_rn(e[8 * j + 2], e[8 * j + 3]),
                                      h2 = __floats2half2_rn(e[8 * j + 4], e[8 * j + 5]), h3 = __floats2half2_rn(e[8 * j + 6], e[8 * j + 7]);
                        uint4 pk;
                        pk.x = *reinterpret_cast<const uint32_t*>(&h0);
                        pk.y = *reinterpret_cast<const uint32_t*>(&h1);
                        pk.z = *reinterpret_cast<const uint32_t*>(&h2);
                        pk.w = *reinterpret_cast<const uint32_t*>(&h3);
                        *reinterpret_cast<uint4*>(et + (((c0 / 8 + j) ^ (r & 7)) << 4)) = pk;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> MMA (async proxy)
                asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
                const uint32_t gate_bar = bar0 + 8u * (2 * STAGES + 2 * NACC + g);
                const uint32_t tgate = tmem_base + (uint32_t)(NACC * BN + g * 2 * BN);
                if ((ew & 3) == 0 && elect_one()) {
                    tc_fence_after();
                    constexpr uint32_t idesc2 = (1u << 4) | ((uint32_t)((2 * BN) >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
                    const uint64_t ad = make_desc(tiles + S::OFF_ETILE + (uint32_t)g * (BM * BKB));
                    const uint64_t bd = make_desc(tiles + S::OFF_W2T);
#pragma unroll
                    for (int kk = 0; kk < BN / 16; ++kk)
                        tc_mma<__half>(tgate, ad + (uint64_t)(2 * kk), bd + (uint64_t)(2 * kk), idesc2, kk ? 1u : 0u);
                    tc_commit(gate_bar);
                }
                if ((ew & 3) == 0) mbar_wait<32>(gate_bar, (it / NACC) & 1);
                asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
                tc_fence_after();
                const uint32_t tg = tgate + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
                for (int c0 = 0; c0 < 2 * BN; c0 += 32) {  // 32 gate columns = 16 output channels per pass
                    uint32_t gv[32];
                    tmem_ld16_nowait(tg + c0, gv);
                    tmem_ld16_nowait(tg + c0 + 16, gv + 16);
                    tmem_ld_wait();
                    const int ch0 = c0 / 2;
                    float y[16];
#pragma unroll
                    for (int c = 0; c < 16; ++c)
                        y[c] = ch0 + c < p.C2 ? (__uint_as_float(gv[2 * c]) + s_b2[c0 + 2 * c]) *
                                                    fast_sigmoid(__uint_as_float(gv[2 * c + 1]) + s_b2[c0 + 2 * c + 1])
                                              : 0.f;
                    if (row_ok) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            s_acc += y[i];
                            ss_acc += y[i] * y[i];
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 16; i += 4)
                        *reinterpret_cast<float4*>(srow + i) = make_float4(y[i], y[i + 1], y[i + 2], y[i + 3]);
                    __syncwarp();
                    float* outp = out_half ? reinterpret_cast<float*>(reinterpret_cast<__half*>(p.out) + ch0) : p.out + ch0;
                    store_chunk<16>(stg, 0, outp, ooff, min(16, p.C2 - ch0), vec4, lane, out_half);
                    __syncwarp();
                }
                tc_fence_before();
                stats_commit(p.stats, p.stats_stride ? p.stats_stride : 2, b, s_acc, ss_acc);
            } else if (BN == 16 && p.epi == EPI_ELU_GATE) {
                // tf32 mode: conv + ELU, then the gated 1x1 pair in registers (C2 <= 16 channels), + statistics
                uint32_t vr[16];
                float e[16], y[16];
                wait_acc();
                tmem_ld16_nowait(tlane, vr);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(tempty_bar(acc));
#pragma unroll
                for (int i = 0; i < 16; ++i) e[i] = epi_elu<SPLIT>(__uint_as_float(vr[i]) + sbias[i]);
                if (p.C2 <= 8) small_gate<8, SPLIT>(s_w2, e, p.C2, y);
                else small_gate<16, SPLIT>(s_w2, e, p.C2, y);
                if (row_ok) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        s_acc += y[i];
                        ss_acc += y[i] * y[i];
                    }
                }
#pragma unroll
                for (int i = 0; i < 16; i += 4)
                    *reinterpret_cast<float4*>(srow + i) = make_float4(y[i], y[i + 1], y[i + 2], y[i + 3]);
                __syncwarp();
                store_chunk<16>(stg, 0, p.out, ooff, p.C2, vec4, lane, out_half);
                __syncwarp();
                stats_commit(p.stats, p.stats_stride ? p.stats_stride : 2, b, s_acc, ss_acc);
            } else {
                const bool paired = (p.epi == EPI_GATE_STATS || p.epi == EPI_SKIP);
                const bool want_stats = (p.epi == EPI_ELU_STATS || p.epi == EPI_GATE_STATS || p.epi == EPI_SKIP ||
                                         p.epi == EPI_RELU_STATS);
                constexpr int CH = BN < 32 ? 16 : 32;  // accumulator columns per pass
                wait_acc();
#pragma unroll 1
                for (int c0 = 0; c0 < BN; c0 += CH) {
                    uint32_t vr[CH];
                    float v[CH];
#pragma unroll
                    for (int i = 0; i < CH; i += 16) tmem_ld16_nowait(tlane + c0 + i, vr + i);
                    tmem_ld_wait();
                    if (c0 + CH >= BN) {  // accumulator fully read: hand it back to the MMA warp
                        tc_fence_before();
                        if (PAIR) mbar_arrive_cluster(lead_tempty0 + 8u * (uint32_t)acc);  // the leader issues the next MMAs
                        else mbar_arrive(tempty_bar(acc));
                    }
                    const int n = n0 + c0;
                    if (n >= p.N) continue;  // (CTA-uniform) nothing but padding in this pass
                    // bias is zero beyond N and weight rows beyond N are zero: padded columns come out as 0
#pragma unroll
                    for (int i = 0; i < CH; ++i) v[i] = __uint_as_float(vr[i]) + sbias[c0 + i];
                    if (!paired) {
                        if (p.epi == EPI_RELU_STATS) {
#pragma unroll
                            for (int i = 0; i < CH; ++i) v[i] = fmaxf(v[i], 0.f);
                        } else if (p.epi != EPI_BIAS) {
#pragma unroll
                            for (int i = 0; i < CH; ++i) v[i] = epi_elu<SPLIT>(v[i]);
                        }
#pragma unroll
                        for (int i = 0; i < CH; i += 4)
                            *reinterpret_cast<float4*>(srow + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                        if (want_stats && row_ok) {
                            if (n + CH <= nlim) {
#pragma unroll
                                for (int i = 0; i < CH; ++i) {
                                    s_acc += v[i];
                                    ss_acc += v[i] * v[i];
                                }
                            } else {  // padded columns are 0 anyway; this only matters for the odd_tail rows
#pragma unroll
                                for (int i = 0; i < CH; ++i)
                                    if (n + i < nlim) {
                                        s_acc += v[i];
                                        ss_acc += v[i] * v[i];
                                    }
                            }
                        }
                        __syncwarp();
                        float* outp = out_half ? reinterpret_cast<float*>(reinterpret_cast<__half*>(p.out) + n) : p.out + n;
                        if (p.odd_tail) store_chunk<CH, true>(stg, 0, outp, ooff, min(CH, nlim - n), vec4, lane, out_half);
                        else store_chunk<CH>(stg, 0, outp, ooff, min(CH, p.N - n), vec4, lane, out_half);
                    } else {
                        constexpr int CO = CH / 2;  // output channels per pass
                        float w[CO];
                        if (p.epi == EPI_GATE_STATS) {
#pragma unroll
                            for (int i = 0; i < CO; ++i) w[i] = v[2 * i] * epi_sigmoid<SPLIT>(v[2 * i + 1]);
                        } else {
#pragma unroll
                            for (int i = 0; i < CO; ++i) w[i] = v[2 * i];
#pragma unroll
                            for (int i = 0; i < CO; i += 4)
                                *reinterpret_cast<float4*>(srow + CO + i) =
                                    make_float4(epi_elu<SPLIT>(v[2 * i + 1]), epi_elu<SPLIT>(v[2 * i + 3]),
                                                epi_elu<SPLIT>(v[2 * i + 5]), epi_elu<SPLIT>(v[2 * i + 7]));
                        }
#pragma unroll
                        for (int i = 0; i < CO; i += 4)
                            *reinterpret_cast<float4*>(srow + i) = make_float4(w[i], w[i + 1], w[i + 2], w[i + 3]);
                        if (row_ok) {
#pragma unroll
                            for (int i = 0; i < CO; ++i) {
                                s_acc += w[i];
                                ss_acc += w[i] * w[i];
                            }
                        }
                        __syncwarp();
                        const int cnt = min(CO, (p.N - n) >> 1);
                        const int co0 = n >> 1;
                        float* o1 = out_half ? reinterpret_cast<float*>(reinterpret_cast<__half*>(p.out) + co0) : p.out + co0;
                        store_chunk<CO>(stg, 0, o1, ooff, cnt, vec4, lane, out_half);
                        // out2 shares the row decomposition of out (gemm_tf32_supported checks the strides are equal)
                        if (p.epi == EPI_SKIP) {
                            float* o2 = out_half ? reinterpret_cast<float*>(reinterpret_cast<__half*>(p.out2) + co0)
                                                 : p.out2 + co0;
                            store_chunk<CO>(stg, CO, o2, ooff, cnt, vec4, lane, out_half);
                        }
                    }
                    __syncwarp();
                }
                if (want_stats) stats_commit(p.stats, p.stats_stride ? p.stats_stride : 2, b, s_acc, ss_acc);
            }
        }
        if (kProf && TMA && tm.profile != 0 && (ew & 3) == 0 && lane == 0)
            atomicAdd(&g_gemm_prof[6], (unsigned long long)(clock64() - t_epi_begin));
        tc_fence_before();
    }
    __syncthreads();
    if (PAIR) cluster_sync_all();  // neither CTA leaves (or frees TMEM) while the pair's MMAs / barriers may still touch it
    if (warp == 4) {
        tc_fence_after();
        if (PAIR)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(S::TMEM_COLS)
                         : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(S::TMEM_COLS)
                         : "memory");
    }
}

template <int BN, typename AT, bool B2B = (BN == 16), int TMA = 0>
__global__ void __launch_bounds__(Cfg<BN, B2B, TMA>::THREADS, 1)
    gemm_tc_kernel(const GemmParams p, const __grid_constant__ GemmTma tm) {
    gemm_tc_body<BN, AT, B2B, TMA, false>(p, tm);
}
// 3xTF32 form: gathered fp32 operands split into tf32 heads and tails, three MMAs per K = 8 step, exact-mode epilogues
template <int BN, bool B2B = (BN == 16)>
__global__ void __launch_bounds__(Cfg<BN, B2B, 0, true>::THREADS, 1)
    gemm_tc3x_kernel(const GemmParams p, const __grid_constant__ GemmTma tm) {
    gemm_tc_body<BN, float, B2B, 0, true>(p, tm);
}

template <int BN, typename AT, bool B2B = (BN == 16), bool SPLIT = false>
int launch_tc(const GemmParams& p, cudaStream_t st) {
    using S = Cfg<BN, B2B, 0, SPLIT>;
    int g_num_sms = 0;
    if (num_sms_current_device(&g_num_sms)) return 1;
    const int ntiles = ((p.M + BM - 1) / BM) * ((p.epi == EPI_GRU ? p.N : p.Npad) / BN);
    const int grid = ntiles < g_num_sms ? ntiles : g_num_sms;  // persistent: one CTA per SM
    static const GemmTma no_tma{};
    if constexpr (SPLIT) {
        SE_DYN_SMEM((gemm_tc3x_kernel<BN, B2B>), S::BYTES);
        gemm_tc3x_kernel<BN, B2B><<<grid, S::THREADS, S::BYTES, st>>>(p, no_tma);
    } else {
        SE_DYN_SMEM((gemm_tc_kernel<BN, AT, B2B, 0>), S::BYTES);
        gemm_tc_kernel<BN, AT, B2B, 0><<<grid, S::THREADS, S::BYTES, st>>>(p, no_tma);
    }
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

template <int BN>
int launch_tc_tma(const GemmParams& p, const GemmTma& tm_in, cudaStream_t st) {
    int g_num_sms = 0;
    if (num_sms_current_device(&g_num_sms)) return 1;
    GemmTma tm = tm_in;  // + the multiply-high reciprocals of this launch's three tile divisors
    const int nstreams = p.M / (p.Tn * p.Fo);
    const int ntiles_m = ((nstreams + tm.bb - 1) / tm.bb) * tm.tgroups * tm.fsegs;
    auto magic = [](int d) { return d <= 1 ? 0u : (uint32_t)(((1ull << 32) + (unsigned)d - 1) / (unsigned)d); };
    tm.magic_ntn = magic(p.Npad / BN);
    tm.magic_fsegs = magic(tm.fsegs);
    tm.magic_tgroups = magic(tm.tgroups);
    SE_REQUIRE((long long)(ntiles_m + 1) * (p.Npad / BN) < (1ll << 26) && p.Npad / BN <= 64 && tm.fsegs <= 64 && tm.tgroups <= 64,
               "gemm_tc: tile index range of the multiply-high division");
    if (!tm.pair) {
        using S = Cfg<BN, false, 1>;
        SE_DYN_SMEM((gemm_tc_kernel<BN, __half, false, 1>), S::BYTES);
        const int ntiles = ntiles_m * (p.Npad / BN);
        const int grid = ntiles < g_num_sms ? ntiles : g_num_sms;
        gemm_tc_kernel<BN, __half, false, 1><<<grid, S::THREADS, S::BYTES, st>>>(p, tm);
        SE_CUDA_OK(cudaGetLastError());
        return 0;
    }
    // CTA pairs: clusters of two CTAs (same TPC), one cluster per super-tile at a time
    using S = Cfg<BN, false, 2>;
    SE_DYN_SMEM((gemm_tc_kernel<BN, __half, false, 2>), S::BYTES);
    const int nsuper = ((ntiles_m + 1) / 2) * (p.Npad / BN);
    int nclusters = g_num_sms / 2;
    if (nsuper < nclusters) nclusters = nsuper;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * nclusters);
    cfg.blockDim = dim3(S::THREADS);
    cfg.dynamicSmemBytes = S::BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SE_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, __half, false, 2>, p, tm));
    return 0;
}

// split form: fp32 operands; tiles of at most 128 columns (a 256-column GEMM runs as twice as many 128-column tiles,
// an LSTM on 32-unit tiles)
int launch_split(const GemmParams& p, cudaStream_t st) {
    SE_REQUIRE(!p.a_half, "gemm_tc: the 3xTF32 form reads fp32 operands");
    SE_REQUIRE(p.epi != EPI_LSTM || p.lstm_units != 64, "gemm_tc: the 3xTF32 form runs LSTM steps on 32-unit tiles");
    if (p.epi == EPI_GRU) return launch_tc<96, float, false, true>(p, st);
    if (p.epi == EPI_LSTM) return launch_tc<128, float, false, true>(p, st);
    switch (gemm_tf32_tile_n(p.N)) {
        case 16: return launch_tc<16, float, true, true>(p, st);
        case 32: return launch_tc<32, float, false, true>(p, st);
        case 64: return launch_tc<64, float, false, true>(p, st);
        default: return launch_tc<128, float, false, true>(p, st);
    }
}

template <typename AT>
int launch_elem(const GemmParams& p, cudaStream_t st) {
    if (p.epi == EPI_GRU) return launch_tc<96, AT>(p, st);
    if (p.epi == EPI_LSTM) return p.lstm_units == 64 ? launch_tc<256, AT>(p, st) : launch_tc<128, AT>(p, st);
    if (p.epi == EPI_ELU_GATE && sizeof(AT) == 2 && p.Npad == 32) return launch_tc<32, AT, true>(p, st);
    if (p.epi == EPI_ELU_GATE && sizeof(AT) == 2 && p.Npad == 64) return launch_tc<64, AT, true>(p, st);
    switch (gemm_tf32_tile_n(p.N)) {
        case 16: return launch_tc<16, AT>(p, st);
        case 32: return launch_tc<32, AT>(p, st);
        case 64: return launch_tc<64, AT>(p, st);
        case 128: return launch_tc<128, AT>(p, st);
        default: return launch_tc<256, AT>(p, st);
    }
}

}  // namespace

bool gemm_tf32_supported(const GemmParams& p) {
    const int bke = p.a_half ? 64 : 32, ue = p.a_half ? 8 : 4;  // elements per k-block / per 16-byte gather unit
    if (p.K % bke != 0 || p.K < bke || p.K / ue > 512) return false;  // whole k-blocks (host pads with zero weights)
    if (p.epi == EPI_GRU) return p.H % 32 == 0 && p.Tn == 1 && p.Fo == 1 && p.N == 3 * p.H;
    if (p.epi == EPI_LSTM)
        return p.H % (p.lstm_units == 64 ? 64 : 32) == 0 && (p.lstm_units == 0 || p.lstm_units == 32 || p.lstm_units == 64) &&
               p.Tn == 1 && p.Fo == 1 && p.N == 4 * p.H && p.Npad == p.N;
    if (p.Npad % gemm_tf32_tile_n(p.N) != 0) return false;
    if (p.epi == EPI_ELU_GATE)  // register version: N <= 16; back-to-back tensor-core version (fp16 operands): N <= 64
        return (p.Npad == 16 || (p.a_half && (p.Npad == 32 || p.Npad == 64))) && p.C2 >= 1 && p.C2 <= p.Npad && p.W2 &&
               p.bias2;
    if (p.epi == EPI_SKIP && (p.o2B != p.oB || p.o2T != p.oT || p.o2F != p.oF)) return false;
    if (p.vec4 && ((p.oF % 4) || (p.oT % 4) || (p.oB % 4))) return false;
    return p.N >= 1;
}

bool gemm_tma_supported(const GemmParams& p) {
    if (!p.a_half || !gemm_tf32_supported(p)) return false;
    if (p.epi == EPI_GRU || p.epi == EPI_ELU_GATE) return false;  // their own tile walks
    if (p.epi == EPI_LSTM) return true;  // row = sequence (Tn = Fo = 1): a 128-row tile is 128 consecutive sequences
    return gemm_tf32_tile_n(p.N) >= 32 && p.Tn * p.Fo > 0 && p.Fo <= BM;
}

// Output-tile width of the TMA path.  The short-K gated 1x1 pairs are bound by their epilogue (two sigmoid-gated columns per
// output, statistics, stores): 128-column tiles run on four accumulators = 16 epilogue warps instead of the 8 of a
// 256-column tile, which is worth more than reading the (short) A rows twice.
int gemm_tma_tile_n(const GemmParams& p) {
    if (p.epi == EPI_LSTM) return p.lstm_units == 64 ? 256 : 128;  // [i | f | g | o] of 64 / 32 hidden units per tile
    const int bn = gemm_tf32_tile_n(p.N);
    if (bn == 256 && (p.epi == EPI_GATE_STATS || p.epi == EPI_SKIP) && p.K <= 256) return 128;
    return bn;
}

int launch_gemm_tma(const GemmParams& p, const GemmTma& tm, cudaStream_t st) {
    SE_REQUIRE(gemm_tma_supported(p), "gemm_tc: shape not supported by the TMA path");
    if (p.M <= 0) return 0;
    switch (gemm_tma_tile_n(p)) {
        case 32: return launch_tc_tma<32>(p, tm, st);
        case 64: return launch_tc_tma<64>(p, tm, st);
        case 128: return launch_tc_tma<128>(p, tm, st);
        default: return launch_tc_tma<256>(p, tm, st);
    }
}

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {  // the driver entry point is fetched at run time: the library does not link libcuda
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}
}  // namespace

int make_gemm_tma(GemmTma* out, const void* a_base, int C, int Fp, int Tp, long long sT, long long sB, int nB, int Fo,
                  int fstep, int Tn, const void* w_base, int K, int Npad, int BN) {
    static_assert(sizeof(TmaDesc) == sizeof(CUtensorMap), "TmaDesc must hold a CUtensorMap");
    EncodeTiledFn enc = encode_tiled_fn();
    SE_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
    SE_REQUIRE(C % 64 == 0 && BN <= 256 && K % 64 == 0 && Fo >= 1 && Tn >= 1, "make_gemm_tma: shape");
    // Tile shape: Fs bins (a divisor of Fo) x bt frames (a divisor of Tn: no ragged frame groups) x bb streams, as many
    // of the 128 rows as possible; among (nearly) equal fills the one with the longest contiguous run (bins, then frames)
    int Fs = 0, bt = 0, bb = 0, best = 0;
    for (int fs = Fo; fs >= 1; --fs) {
        if (Fo % fs != 0 || fs > BM) continue;
        for (int t = Tn; t >= 1; --t) {
            if (Tn % t != 0 || fs * t > BM) continue;
            int b = BM / (fs * t);
            if (b > 16 && fs * t > 1) b = 16;  // (row = stream GEMMs take all 128 rows from the stream dimension)
            const int rows = fs * t * b;
            if (rows > best + best / 20) {  // a candidate later in this order must fill > 5 % more rows to win
                best = rows;
                Fs = fs;
                bt = t;
                bb = b;
            }
        }
    }
    SE_REQUIRE(best > 0, "make_gemm_tma: no tile shape");
    {  // activations [nB][Tp][Fp][C] fp16: box = 64 channels x Fo bins (every fstep-th) x bt frames x bb streams
        const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)Fp, (cuuint64_t)Tp, (cuuint64_t)nB};
        const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)sT * 2, (cuuint64_t)sB * 2};
        const cuuint32_t box[4] = {64, (cuuint32_t)((Fs - 1) * fstep + 1), (cuuint32_t)bt, (cuuint32_t)bb};
        const cuuint32_t estr[4] = {1, (cuuint32_t)fstep, 1, 1};
        const CUresult r = enc(reinterpret_cast<CUtensorMap*>(&out->a), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4,
                               const_cast<void*>(a_base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        SE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (activations) failed with " + std::to_string((int)r));
    }
    // CTA pair mode (cta_group::2; SE_B200_TMA_PAIR=0 keeps one CTA per tile): each CTA of the pair holds half the weight
    // tile, so a 256-row M tile fetches the weights once.  With the tensor pipe fed at its own pace (tools/gemm_roles.py:
    // the MMA warp otherwise waits for operand stages ~45 % of the time) the operand stream from L2 is what bounds the
    // long-K GEMMs, and the pair cuts it by a quarter (BN 128) to a third (BN 256).  Measured at 1024 streams, pair vs
    // single: 768-column GRU projections 110 -> 94 us and 51 -> 48 us, 3x3 convolutions (K >= 576) 89 -> 85, 97 -> 93,
    // 91 -> 86 us; the short-K GEMMs (1x1 gates / skips, fc: K <= 256) are epilogue-bound and lose 4 us to the cluster
    // launch, so they stay single.  SE_B200_TMA_PAIR=2 forces the pair everywhere.
    int pair = BN == 256 || K >= 576;
    if (const char* e = getenv("SE_B200_TMA_PAIR")) pair = atoi(e) == 2 ? 1 : (atoi(e) != 0 && pair);
    if (BN / 2 < 16) pair = 0;
    out->pair = pair;
    out->profile = getenv("SE_B200_GEMM_PROFILE") ? atoi(getenv("SE_B200_GEMM_PROFILE")) : 0;
    {  // weights [Npad][K] fp16, K-major: box = 64 x BN (pair: x BN / 2, the slice of one CTA)
        const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Npad};
        const cuuint64_t strides[1] = {(cuuint64_t)K * 2};
        const cuuint32_t box[2] = {64, (cuuint32_t)(pair ? BN / 2 : BN)};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = enc(reinterpret_cast<CUtensorMap*>(&out->w), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                               const_cast<void*>(w_base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        SE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (weights) failed with " + std::to_string((int)r));
    }
    out->bt = bt;
    out->bb = bb;
    out->Fs = Fs;
    out->fsegs = Fo / Fs;
    out->fstep = fstep;
    out->tgroups = Tn / bt;
    out->rows = bb * bt * Fs;
    out->a_bytes = out->rows * BKB;
    return 0;
}

int make_tma_3d_f16(TmaDesc* out, const void* base, int d0, int d1, int d2, long long s1, long long s2, int b0, int b1,
                    int b2) {
    EncodeTiledFn enc = encode_tiled_fn();
    SE_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
    SE_REQUIRE(b0 * 2 == 128, "make_tma_3d_f16: the box must span one 128-byte swizzle row");
    const cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
    const cuuint64_t strides[2] = {(cuuint64_t)s1 * 2, (cuuint64_t)s2 * 2};
    const cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, (cuuint32_t)b2};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base),
                           dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (3-D) failed with " + std::to_string((int)r));
    return 0;
}

int make_tma_4d_f16(TmaDesc* out, const void* base, const long long dims[4], const long long strides[3], const int box[4],
                    int swizzle_bytes) {
    EncodeTiledFn enc = encode_tiled_fn();
    SE_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
    SE_REQUIRE((swizzle_bytes == 64 || swizzle_bytes == 128) && box[0] * 2 == swizzle_bytes,
               "make_tma_4d_f16: the box must span one swizzle row");
    const cuuint64_t d[4] = {(cuuint64_t)dims[0], (cuuint64_t)dims[1], (cuuint64_t)dims[2], (cuuint64_t)dims[3]};
    const cuuint64_t st[3] = {(cuuint64_t)strides[0], (cuuint64_t)strides[1], (cuuint64_t)strides[2]};
    const cuuint32_t bx[4] = {(cuuint32_t)box[0], (cuuint32_t)box[1], (cuuint32_t)box[2], (cuuint32_t)box[3]};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = enc(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base),
                           d, st, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (4-D) failed with " + std::to_string((int)r));
    return 0;
}

int gemm_profile_read(unsigned long long* out8, int reset) {
    SE_CUDA_OK(cudaDeviceSynchronize());
    if (out8) SE_CUDA_OK(cudaMemcpyFromSymbol(out8, g_gemm_prof, 8 * sizeof(unsigned long long)));
    if (reset) {
        const unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        SE_CUDA_OK(cudaMemcpyToSymbol(g_gemm_prof, z, sizeof(z)));
    }
    return 0;
}

int gemm_tf32_tile_n(int N) {
    if (N <= 16) return 16;
    if (N <= 32) return 32;
    if (N <= 64) return 64;
    if (N <= 128 || N % 256 != 0) return 128;
    return 256;
}

int launch_gemm_tf32(const GemmParams& p, cudaStream_t st, bool split) {
    SE_REQUIRE(gemm_tf32_supported(p), "gemm_tc: unsupported shape");
    if (p.M <= 0) return 0;
    if (split) return launch_split(p, st);
    return p.a_half ? launch_elem<__half>(p, st) : launch_elem<float>(p, st);
}

}  // namespace se
