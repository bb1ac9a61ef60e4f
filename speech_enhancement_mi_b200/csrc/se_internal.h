// Internal declarations shared by the .cu translation units of libse_b200.so (not part of the C-ABI).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <nvtx3/nvToolsExt.h>  // header-only (the tools library is dlopen'ed when a profiler is attached)

#include <functional>
#include <map>
#include <string>
#include <vector>

namespace se {

// NVTX range over a C-ABI call (nsys / ncu --nvtx time lines: "se.chunk_step", "se.train_forward", ...).  Costs a
// few nanoseconds when no tool is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};


constexpr int kFramesPerChunk = 21;  // T = 1 + K/hop for K=3200, hop=160 (reference: torch.stft center=True)

// GlobalLayerNorm mean and inverse denominator of one stream from its accumulated sum and sum of squares (double):
// teacher (x-mean)/(sqrt(var+1e-8)+1e-8) (CRN_ELU.py:51), student (x-mean)/(sqrt(var)+1e-8) (distillation_crn.py:51)
__host__ __device__ __forceinline__ void gln_mean_inv(double s, double ss, double count, int student, float& mean,
                                                      float& inv) {
    const double mu = s / count;
    double var = ss / count - mu * mu;
    if (var < 0.0) var = 0.0;
    const float varf = (float)var;
    const float den = student ? (sqrtf(varf) + 1e-8f) : (sqrtf(varf + 1e-8f) + 1e-8f);
    mean = (float)mu;
    inv = 1.0f / den;
}

// ---------------------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------------------
void set_error(const std::string& msg);
#define SE_CUDA_OK(expr)                                                                          \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            se::set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" +      \
                          __FILE__ + ":" + std::to_string(__LINE__) + ")");                       \
            return 1;                                                                             \
        }                                                                                         \
    } while (0)
#define SE_REQUIRE(cond, msg)                       \
    do {                                            \
        if (!(cond)) {                              \
            se::set_error(std::string(msg));        \
            return 2;                               \
        }                                           \
    } while (0)

// Per-device launch configuration (the C-ABI takes a device index, so one process may drive several GPUs):
// ensure_dyn_smem opts `func` into `bytes` of dynamic shared memory on the CURRENT device, once per (device, kernel,
// size); num_sms_current_device caches the SM count per device.  Both are thread-safe (crn.cu).
int ensure_dyn_smem(const void* func, int bytes);
int num_sms_current_device(int* out);
#define SE_DYN_SMEM(kernel, bytes)                                                     \
    do {                                                                               \
        if (se::ensure_dyn_smem(reinterpret_cast<const void*>(kernel), (int)(bytes))) return 1; \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------
// context plumbing shared by the CRN and FullSubNet contexts (arena.cu)
// ---------------------------------------------------------------------------------------------------------------
// zero-filled device buffer of `bytes`, recorded in `allocs` (freed when the owning context is destroyed)
int dev_alloc_bytes(std::vector<void*>& allocs, void** out, size_t bytes);
template <typename Owner, typename Tp>
int dev_alloc(Owner* c, Tp** out, size_t count) {
    return dev_alloc_bytes(c->allocs, reinterpret_cast<void**>(out), count * sizeof(Tp));
}
// the checks of se_*_create before a context is built: 3 = no CUDA device, 2 = bad index or not an sm_100 device,
// 1 = CUDA error; makes `device` current.  `fn` prefixes the error messages.
int check_create_device(int device, const char* fn);
// replays enq(stream) as a CUDA graph captured once per B into `graphs`.  The capture runs on *own (created on first
// use), so that the caller's stream is never put into capture mode.
int replay_graph(std::map<int, cudaGraphExec_t>& graphs, cudaStream_t* own, int B,
                 const std::function<int(cudaStream_t)>& enq, cudaStream_t st);

struct ParamInfo {  // one tensor of the reference model's state_dict
    std::string name;
    std::vector<int> shape;
    int64_t numel() const {
        int64_t n = 1;
        for (int s : shape) n *= s;
        return n;
    }
};
using HostParams = std::map<std::string, std::vector<float>>;
using PackFn = std::function<void(const HostParams&, float*)>;  // fills a host mirror of the packed-weight arena

// The packed weights of a context.  Building the program reserves regions of the fp32 weight arena (multiples of 4
// floats, so every region is 16-byte aligned) and of the koff table (gather offsets of 16-byte units), and registers
// for each region a packer that fills it from the reference parameters.  Each op registers a bind that sets its
// weight / bias / koff pointers (and builds whatever descriptor depends on them) once allocate() has created the device
// arenas.  With `half`, an fp16 mirror of the whole weight arena (same indexing) holds the fp16 weight operands.
struct WeightArena {
    std::vector<ParamInfo> params;  // registry in the order of the reference state_dict
    bool half = false;
    size_t floats = 0;
    std::vector<int> khost;
    std::vector<PackFn> packers;
    std::vector<std::function<int()>> binds;
    float* w = nullptr;          // device arenas (allocate)
    __half* wh = nullptr;        // fp16 mirror (half only)
    int* k = nullptr;
    bool bound = false;          // weights have been uploaded

    size_t reserve_w(size_t n) {
        const size_t off = floats;
        floats += (n + 3) / 4 * 4;
        return off;
    }
    int reserve_k(const std::vector<int>& v) {  // padded with offset-0 units to whole k-blocks of 8 units (weights there: 0)
        const int off = (int)khost.size();
        khost.insert(khost.end(), v.begin(), v.end());
        while ((khost.size() - off) % 8) khost.push_back(0);
        return off;
    }
    std::vector<float> pack(const HostParams& hp) const;  // runs every packer on a zeroed host arena
    // device arenas, koff upload, then every bind
    int allocate(std::vector<void*>& allocs);
    // gathers the `n` tensors of the registry from `ptrs` (host or device), packs them and uploads the arena (and its
    // fp16 mirror) once no work on `st` or the device still reads the old weights; `fn` prefixes the error messages
    int upload(const float* const* ptrs, int n, cudaStream_t st, const char* fn);
};

// ---------------------------------------------------------------------------------------------------------------
// gathered GEMM:  C[m][n] = sum_k A(m,k) * W[n][k],  m = (b*Tn + t)*Fo + f
//   A(m,k) = A[b*sB + t*sT + f*sF + koff[k/4] + k%4]          (implicit im2col over channels-last activations)
// Used for every dense contraction of the path: causal convs (CRN_ELU.py:239), 1x1 gate pairs (:240), transposed
// convs (:294), skip 1x1s (:305-306), GRU input / recurrent projections (:173) and the output Linear (:175).
// ---------------------------------------------------------------------------------------------------------------
enum Epilogue : int {
    EPI_BIAS = 0,        // out[n] = acc + bias[n]
    EPI_ELU = 1,         // out[n] = elu(acc + bias[n])
    EPI_ELU_STATS = 2,   // as EPI_ELU, and accumulate per-stream sum / sum-of-squares of out
    EPI_GATE_STATS = 3,  // columns interleaved (trans_c, gated_c): out[c] = (a0+b0)*sigmoid(a1+b1); stats of out
    EPI_SKIP = 4,        // columns interleaved (mask_c, resid_c): out[c] = a0+b0 (stats); out2[c] = elu(a1+b1)
    EPI_GRU = 5,         // TF32 path only: columns per 32-unit group [r|z|n]; fused GRU cell update
    EPI_LSTM = 7,        // TF32 path only: columns per 32-unit group [i|f|g|o]; fused LSTM cell (c in hprev, c' in out2)
    EPI_RELU_STATS = 8,  // out[n] = relu(acc + bias[n]); stats accumulate the sum (and sum of squares) of out
    EPI_ELU_GATE = 6,    // TF32 path only, N <= 16: e = elu(acc + bias), then the gated 1x1 pair of CRN_ELU.py:240 in
                         // registers: out[c] = (W2[2c].e + b2[2c]) * sigmoid(W2[2c+1].e + b2[2c+1]); stats of out
};

struct GemmParams {
    const void* A;         // fp32 (exact / tf32 path) or fp16 (a_half) activations
    int a_half;            // tensor-core path: operands A and W are fp16 (kind::f16), else fp32 read as tf32
    long long sB, sT, sF;  // element strides of the row decomposition
    int Tn, Fo, M;
    int b0;  // first stream of this launch: row m belongs to stream b0 + m / (Tn*Fo)  (tf32 path)
    const int* koff;  // element offset of every 16-byte unit (4 floats / 8 halves) of a row
    int K;            // padded to whole k-blocks (32 floats / 64 halves), weights zero there
    const void* W;    // [Npad][K] packed weights (same element type as A), rows >= N are zero
    int N;            // logical columns
    int Npad;         // rows available in W / bias (multiple of 16)
    const float* bias;
    int epi;
    float* out;    // with out_half: a __half* (operand of a following GEMM), strides in halves
    int out_half;
    long long oB, oT, oF;
    void* out_h2;  // EPI_GRU: optional fp16 copy of h' (row stride o2B halves)
    float* out2;
    long long o2B, o2T, o2F;
    double* stats;  // [B][2] (sum, sum of squares)
    int stats_stride;  // doubles per stream in `stats` (0 = 2)
    // EPI_GRU extras: gi = input projection (b_ih included) [B][Tn_gi][3H]; h_prev/h_out rows [B][.][H]
    const float* gi;
    long long giB;
    const float* hprev;
    long long hB;
    int H;
    // EPI_ELU_GATE extras: W2 [2*C2][16] (rows interleaved trans/gated, zero beyond C2 columns), bias2 [2*C2]
    const float* W2;
    const float* bias2;
    int C2;
    // tf32 path: rows may be written with 16-byte stores up to the next multiple of 4 columns (the destination pitch
    // is padded and aligned); 0 = element-wise stores of exactly the valid columns
    int vec4;
    // merged-parity transposed conv: rows with f == Fo-1 own only the first N/2 columns (nothing stored / counted beyond)
    int odd_tail;
    long long c_rows;  // EPI_LSTM: > 0 = the cell state (hprev / out2) is unit-major [H][c_rows] instead of [rows][H]
    // EPI_LSTM: hidden units per output tile (32 -> 128-column tiles, 64 -> 256-column tiles; 0 = 32).  Wider tiles
    // halve the re-reads of the [x_t | h_{t-1}] operand across the N tiles; the weight rows are packed to match.
    int lstm_units;
};

// TMA operand delivery for the tcgen05 GEMM (gemm_tc.cu; fp16 operands whose k-blocks are 64 contiguous channels).
// One elected thread issues two cp.async.bulk.tensor loads per k-block -- the activation tile and the weight tile, both
// landing in the canonical K-major SWIZZLE_128B layout the UMMA descriptors read -- instead of 128 threads gathering
// 16-byte units with cp.async.  Tiles are RECTANGLES of the activation tensor [B][T][F][C]: `bb` streams x `bt` frames x
// `Fs` bins of one of the `fsegs` equal segments of the Fo output bins (rows ordered stream, frame, bin; at most 128),
// so that one 4-D box (C: 64, F: Fs taken every `fstep`-th bin, T: bt, B: bb) is the whole A tile of a k-block; the
// per-k-block (channel, bin, frame) origin is a coordinate.
struct alignas(64) TmaDesc {
    unsigned long long opaque[16];  // CUtensorMap
};
struct GemmTma {
    TmaDesc a, w;
    int bt, bb;         // frames / streams per tile
    int Fs, fsegs;      // bins per tile and tiles per bin axis (Fs * fsegs = Fo)
    int fstep;          // input bins per output bin
    int profile;        // 1: the warp roles account their wait cycles in g_gemm_prof (diagnostic)
    uint32_t magic_ntn, magic_fsegs, magic_tgroups;  // ceil(2^32 / d) of the tile divisors (filled by the launcher)
    int pair;           // 1: CTA-pair kernel (cta_group::2, M256 MMAs over two SMs); the weight box is half a tile
    int rows;           // bb * bt * Fs rows of the 128-row tile are real
    int tgroups;        // ceil(Tn / bt) tiles per stream group
    int a_bytes;        // bytes one activation box delivers (rows * 128)
    int t_org, f_org;   // tensor coordinates of (frame 0, bin 0) of the row grid
    const int4* kcoord; // per k-block: (channel, bin, frame) offsets of the box origin
};
// builds the two tensor maps; A is the tensor [nB][Tp][Fp][C] (fp16) at `a_base` with element strides (sB, sT, C)
int make_gemm_tma(GemmTma* out, const void* a_base, int C, int Fp, int Tp, long long sT, long long sB, int nB, int Fo,
                  int fstep, int Tn, const void* w_base, int K, int Npad, int BN);
int launch_gemm_tma(const GemmParams& p, const GemmTma& tm, cudaStream_t st);
bool gemm_tma_supported(const GemmParams& p);
int gemm_profile_read(unsigned long long* out8, int reset);  // diagnostic cycle counters of the TMA GEMM roles

int launch_gemm_fp32(const GemmParams& p, cudaStream_t st);
// tcgen05 path (gemm_tc.cu); split: the 3xTF32 form (fp32 operands as tf32 head + tail, fp32-accurate products and
// exact-mode epilogues: SE_PRECISION_3XTF32)
int launch_gemm_tf32(const GemmParams& p, cudaStream_t st, bool split);
bool gemm_tf32_supported(const GemmParams& p);
int gemm_tf32_tile_n(int N);  // output-tile width (BN) the tcgen05 kernel uses for N logical columns
int gemm_tma_tile_n(const GemmParams& p);  // ... and the TMA path for this GEMM (may split 256-column tiles)

// ---------------------------------------------------------------------------------------------------------------
// GlobalLayerNorm application (CRN_ELU.py:37-56), fused with what follows it in the graph
// ---------------------------------------------------------------------------------------------------------------
struct NormApplyParams {
    int mode;  // 0: plain, 1: + residual (preconv, CRN_ELU.py:376), 2: gated skip blend (CRN_ELU.py:297-306)
    int B, T, F, C;         // logical extent of the output
    int b0;                 // first stream of this launch
    int student;            // distillation_crn.py:51 denominator
    int in_half;            // y, rm, rr are stored as fp16 (SE_PRECISION_FP16)
    const float* y;         // raw (pre-norm) tensor, [B][T][Fy][C] compact; rows f >= Fy read as post-norm 0 (mode 2)
    int Fy;
    const double* stats;    // [B][2] of y
    double count;           // number of real elements per stream in the statistics
    const float* w;         // per-channel [C] (or per-feature [F*C] when per_feature)
    const float* b;
    int per_feature;
    // mode 1: residual source (block input), mode 2 unused
    const float* res;
    long long rB, rT, rF;
    // mode 2: rm = raw residual mask [B][T][F][C] compact, rr = elu(residual) compact, stats/affine of rm
    const float* rm;
    const float* rr;
    const double* stats_r;
    double count_r;
    const float* wr;
    const float* br;
    // destination (channels-last, strided); out_half: a __half* (fp16 operand storage), strides in halves
    float* out;
    int out_half;
    long long oB, oT, oF;
};
int launch_norm_apply(const NormApplyParams& p, cudaStream_t st);

// ---------------------------------------------------------------------------------------------------------------
// pre-convolution block (CRN_ELU.py:337-339,375-376), one fused kernel per layer (preconv.cu).  Activations of this
// chain are channel-planar per stream: [5][25 frames: 4 carried + 21 new][FPP bins: 2d zero | 201 | 2d zero | pad]
// ---------------------------------------------------------------------------------------------------------------
#define PRECONV_FPP(D) ((204 + 4 * (D) + 3) / 4 * 4)
constexpr int PRECONV_TP = kFramesPerChunk + 4;
// packed weights: conv [(kt*5+ci)*28 + kf*5 + co], then bias, conv_trans, conv_gated, their biases, norm affine
constexpr int PRECONV_W_BIAS = 700, PRECONV_W_WT = 708, PRECONV_W_WG = 736, PRECONV_W_BT = 764, PRECONV_W_BG = 772,
              PRECONV_W_NW = 780, PRECONV_W_NB = 788, PRECONV_W_FLOATS = 800;
struct PreconvParams {
    float* in;           // planar input of this layer (frames 0..3 are rewritten with the carried state)
    long long in_sB;
    int d;               // frequency dilation 1 / 2 / 4
    const float* w;      // packed weights
    float* out;          // out(b, c, t, f) = out[b*oB + c*oC + t*oT + f*oF]  (interior of the next layer's input)
    long long oB, oC, oT, oF;
    int out_vec8;        // destination is channels-last with 8 channels: two 16-byte stores per position
    int out_half;        // ... stored as fp16 (one 16-byte store per position); only with out_vec8
    int student;
    int b0, B;
};
int launch_preconv(const PreconvParams& p, cudaStream_t st);

// the same block on the tensor cores (preconv_tc.cu; fp16 operand mode).  Activations of this chain are channels-last
// fp16 per stream: [25 frames: 4 carried + 21 new][PRECONV_TC_POS positions][8 halves], bin f of a layer with
// dilation d at position f + 2d, everything else zero (the conv's frequency padding and the tile overrun).
constexpr int PRECONV_TC_POS = 272;
struct PreconvTcParams {
    __half* in;          // this layer's input buffer (frames 0..3 are rewritten with the carried state)
    long long in_sB;     // halves per stream
    int d;               // frequency dilation 1 / 2 / 4
    const float* w;      // packed fp32 weights (same block as PreconvParams::w)
    __half* out;         // out(b, t, f) = 16-byte unit at out + b*oB + t*oT + f*oF (halves): interior of the next input
    long long oB, oT, oF;
    int student;
    int b0, B;
};
int launch_preconv_tc(const PreconvTcParams& p, cudaStream_t st);

// the three pre-convolution blocks in one launch and the small-channel encoder blocks (front_mma.cu; fp16 operand mode,
// warp-level mma.sync with the stream's activations resident in shared memory)
struct Preconv3Params {
    const __half* feat;   // this chunk's features [B][21 frames][224 positions][8 halves], bin f at position 8 + f
    long long feat_sB;    // halves per stream
    __half* state;        // carried frames [B][3 layers][4 frames][224][8 halves] (read, then replaced)
    long long state_sB;
    const float* w[3];    // packed fp32 parameter blocks (PRECONV_W_* offsets above)
    __half* out;          // out(b, t, f) = 16-byte unit at out + b*oB + t*oT + f*oF (halves)
    long long oB, oT, oF;
    int student;
    int b0, B;
};
int launch_preconv3(const Preconv3Params& p, cudaStream_t st);
constexpr int PRECONV3_POS = 224, PRECONV3_BORDER = 8;

struct EncMmaParams {
    const __half* in;     // zero-bordered input [B][Tp][Fp][Cin] (frame 0 = first carried frame, bin 0 = first pad bin)
    long long in_sB;
    int Tp, Fp, dt;       // Tp = 2 dt + 21 frames, Fp = F_in + 4 bins, time dilation dt
    int Fo;               // output bins
    const float* w;       // conv weights fp32 [>= Cout][Kp], column (kt * 5 + kf) * Cin + ci
    int Kp;
    const float* bias;
    const float* w2;      // gate weights fp32 [2 Cout][w2_pitch], rows interleaved (conv_trans c, conv_gated c)
    int w2_pitch;
    const float* bias2;   // [2 Cout], interleaved like the rows
    const float *nw, *nb; // GlobalLayerNorm affine [Cout]
    __half* out;          // out(b, t, f, :) at out + b*oB + t*oT + f*oF (halves), Cout contiguous
    long long oB, oT, oF;
    int student;
    int b0, B;
    int off_y, off_wf;    // shared-memory offsets (filled by the launcher)
    uint32_t magic_Jp, magic_Fo, magic_Fp;  // ceil(2^32 / d) of the three run-time divisors (filled by the launcher)
    int plane;            // enc_tc: 16-byte units per (parity, octet) plane (filled by the launcher)
    const __half *w1c, *w2c;  // enc_tc: conv / gate weights as fp16 UMMA operands in shared-memory order (crn.cu packs them)
};
bool enc_mma_supported(int Cin, int Cout, int Tp, int Fp, int Fo);
// the same block as an implicit GEMM on tcgen05 over the resident input (enc_tc.cu): 16 -> 32 and 32 -> 64 channels.
// mode is the context's SE_B200_ENC_TC: 0 never, 1 (default) 32 -> 64 only, 2 also 16 -> 32
bool enc_tc_supported(int mode, int Cin, int Cout, int Tp, int Fp, int Fo);
int launch_enc_tc(const EncMmaParams& p, int Cin, int Cout, cudaStream_t st);
int launch_enc_mma(const EncMmaParams& p, int Cin, int Cout, cudaStream_t st);

// one transposed-conv decoder block with few channels in one launch (back_mma.cu; fp16 operand mode): ConvTranspose2d
// (both output parities) + ELU + GlobalLayerNorm + the gated skip (1x1 mask / residual pair on the skip tensor,
// GlobalLayerNorm of the mask, sigmoid blend) of CRN_ELU.py:290-307
struct DecMmaParams {
    const __half* in;      // deconv input [B][Tp = 21 + 2 d][Fp = Fin + 2][Cin]: one zero bin each side, 2 d zero frames behind
    long long in_sB;
    int Tp, Fp, d, Fin;
    const float* w;        // deconv weights fp32 [2 Cout][Kp]: row parity * Cout + co, column (kt * 3 + j) * Cin + ci
    int Kp;
    const float* bias;     // [2 Cout]
    const __half* skip;    // skip tensor (b, t, f, :) at skip + b*sk_sB + t*sk_sT + f*sk_sF, Cout channels
    long long sk_sB, sk_sT, sk_sF;
    int Fs;                // bins of the skip tensor = bins of the block output (>= 2 Fin - 1)
    const float* w2;       // skip pair fp32 [2 Cout][K2p], rows interleaved (residualmask c, residual c)
    int K2p;
    const float* bias2;
    const float *nw, *nb, *nwr, *nbr;  // norm / residualnorm affine [Cout]
    __half* out;           // out(b, t, f, :) at out + b*oB + t*oT + f*oF
    long long oB, oT, oF;
    int student;
    int b0, B;
    int off_y, off_wf;                      // shared-memory offsets (filled by the launcher)
    uint32_t magic_Fp, magic_Fs, magic_in;  // ceil(2^32 / d) of the run-time divisors (filled by the launcher)
};
bool dec_mma_supported(int Cin, int Cout, int Tp, int Fp, int Fin, int Fs);
int launch_dec_mma(const DecMmaParams& p, int Cin, int Cout, cudaStream_t st);

// GRU cell pointwise update for the fp32 path (PyTorch nn.GRU gate order r,z,n; CRN_ELU.py:127-133)
int launch_gru_pointwise(const float* gi, long long giB, const float* gh, const float* hprev, long long hB,
                         float* hout, int B, int H, cudaStream_t st);

// state roll: copy `count` floats from src_off to dst_off inside each stream's slab of up to 16 buffers
struct RollEntry {
    float* base;
    long long sB;
    long long src_off, dst_off;
    int count;  // multiple of 4
};
struct RollTable {
    RollEntry e[24];
    int n;
    int first_block[25];  // filled by the launcher: blocks [first_block[i], first_block[i+1]) serve entry i
};
int launch_roll(const RollTable& tab, int first, int B, cudaStream_t st);
// x[i] = amp * u_i, u_i a hash of i in [-1, 1) (synthetic chunk content for the per-kernel timers)
int launch_fill_noise(float* x, long long n, float amp, cudaStream_t st);
int launch_zero(const RollTable& tab, int first, int B, cudaStream_t st);  // zero [dst_off, dst_off+count)

// ---------------------------------------------------------------------------------------------------------------
// STFT / features / mask / iSTFT / overlap-add
// ---------------------------------------------------------------------------------------------------------------
struct IoDesc {  // written by a 1-thread kernel before each step so that a captured graph can stay static
    const float* in;  // sample n of the chunk = in[b*in_stream_stride + m*in_mic_stride + in_offset + n] when that index
    long long in_stream_stride, in_mic_stride;  // lies in [0, in_len), else 0 (the zero padding of utility.py:327-336)
    long long in_offset, in_len;
    float* out;  // K/2 samples per stream; only the first n_valid are written (gap trimming, CRN_ELU.py:507-508)
    long long out_stream_stride;
    int n_valid;
};

struct StftParams {
    const IoDesc* io;  // chunk source
    int B, M;          // streams, microphones (3)
    int student;       // phase formula of distillation_crn.py:340
    // feat_h8 != nullptr: one 16-byte unit (5 features as fp16 + 3 zeros) per (frame, bin) at feat_h8 + b*fB + t*fT + f*fF
    // (halves) instead of the fp32 planes below (tensor-core pre-convolutions)
    __half* feat_h8;
    float* feat;       // preconv-0 input buffer interior: feat[b*fB + c*fC + t*fT + f*fF], c < 5
    long long fB, fC, fT, fF;
    float* noisy;  // mic-0 spectrum [B][T][F][2]
    // optional full spectrum in the reference layout [R][M][F][T][2] (se_stft_trans); feat/noisy may be null
    float* spec_ref;
    // training layout: stream s = n*nb + i reads utterance i at in_offset + n*hop_chunk (0: every stream is its own row)
    int nb;
    long long hop_chunk;
};
int launch_stft_features(const StftParams& p, cudaStream_t st);
// features from a spectrum in the reference layout [B][M][F][T][2] (for TemporalCRN.forward, CRN_ELU.py:369-373)
int launch_features_from_spec(const float* spec, int B, int M, int student, float* feat, long long fB, long long fC,
                              long long fT, long long fF, float* noisy, cudaStream_t st, __half* feat_h8 = nullptr);

struct MaskIstftParams {
    const IoDesc* io;     // out pointer for the fused streaming path (may be null when out_chunk is set)
    int B;
    int student;
    const float* y;       // raw last-deconv output [B][T][F][2]
    const double* stats;  // its statistics
    double count;
    const float* w;  // norm affine, 2 channels
    const float* b;
    const float* noisy;  // mic-0 spectrum [B][T][F][2]
    float* carry;        // [B][K/2] overlap-add carry (null: no streaming OLA)
    float* out_chunk;    // optional [B][K] full per-chunk iSTFT output
    float* spec_ref;     // optional enhanced spectrum in the reference layout [B][F][T][2] (forward()); skips iSTFT
    const float* spec_in;  // optional: take the enhanced spectrum [B][F][T][2] from here instead (se_istft_trans)
    int fast;  // tensor-core precisions (tf32 / fp16): decompress_cIRM by two lg2.approx instead of an IEEE division + logf
    // with spec_in: spec_in is d loss / d (STFT of a chunk) and out_chunk receives d loss / d chunk, the adjoint of the
    // framing + window + real DFT (per frame sum_k Re(D_k e^{+2 pi i k n / N}) times the window, overlap-added, centre pad
    // dropped, no envelope division)
    int adjoint;
};
int launch_mask_istft(const MaskIstftParams& p, cudaStream_t st);
int init_fft_tables();  // uploads twiddles / window / envelope to constant memory of the current device

int launch_set_io(IoDesc* dst, const IoDesc& v, cudaStream_t st);
int launch_segmentation(const float* x, int B, int C, long long L, int K, int gap, int N, float* out, cudaStream_t st);
int launch_over_add(const float* chunks, int C, int N, int K, int gap, float* out, cudaStream_t st);

// ---------------------------------------------------------------------------------------------------------------
// training step (train.py:195-204): backward kernels (train_kernels.cu).  All fp32 on CUDA cores; gradients of the
// packed weights are accumulated in a twin of the weight arena and scattered back to the reference layout.
// ---------------------------------------------------------------------------------------------------------------
struct StridedRows {  // row m = (b*Tn + t)*Fo + f of a [B][Tn][Fo] grid lives at base + b*sB + t*sT + f*sF
    long long sB, sT, sF;
};
// dW[n][k] += sum_m G(m,n) * A(m,k), dbias[n] += sum_m G(m,n)   (A gathered exactly like the forward GEMM `p`)
// G(m,n) = G[b*g.sB + t*g.sT + f*g.sF + n], n < N (odd_tail as in the forward).  dW has the packed layout [Npad][K].
// mode: which arithmetic carries the contraction (train_kernels.cu)
enum { BWD_CUDA_CORES = 0,  // fp32 FMA
       BWD_3XTF32 = 1,      // mma.sync tf32 with head / tail operands (fp32-accurate)
       BWD_TF32 = 2 };      // mma.sync tf32, single pass
int launch_wgrad(const GemmParams& p, const float* G, StridedRows g, float* dW, float* dbias, cudaStream_t st,
                 int mode = BWD_3XTF32);
// dA(m,k) = sum_n G(m,n) * W[n][k], scatter-added at dA + (same offsets as the forward gather); dA is a twin of the
// forward operand buffer (zero-initialised by the caller; contributions of overlapping taps accumulate)
int launch_dgrad(const GemmParams& p, const float* G, StridedRows g, float* dA, cudaStream_t st, int mode = BWD_3XTF32);

struct GlnBwdParams {
    int B, T, F, C;       // y is compact [B][T][F][C]; statistics count = `count` real elements
    int student, per_feature, elu;  // elu: y = elu(z) and the result is d loss / d z
    const float* y;
    const double* stats;
    double count;
    const float* w;       // affine weight [C] (or [F*C] per feature)
    const float* g;       // d loss / d normalised output, element (b,t,f,c) at g[b*gB + t*gT + f*gF + c]
    long long gB, gT, gF;
    float* dw;            // accumulated (atomics), same indexing as w
    float* db;
    double* red;          // [B][2] scratch: sum g*w, sum g*w*(y-mean)
    float* dy;            // element (b,t,f,c) at dy[((b*T+t)*F+f)*oC + c*ostep + ooff]
    int oC, ostep, ooff;
};
int launch_gln_bwd(const GlnBwdParams& p, cudaStream_t st);

struct BlendBwdParams {  // gated skip blend of CRN_ELU.py:297-306, backward
    int B, T, Fs, Fy, C, student;
    const float* g;  // d loss / d block output [B][T][Fs][C] strided
    long long gB, gT, gF;
    const float *y, *rm, *rr;  // saved: raw deconv+elu [B][T][Fy][C], raw mask conv, elu(residual conv) [B][T][Fs][C]
    const double *stats, *stats_r;
    double count, count_r;
    const float *w, *b, *wr, *br;
    float* g_o;   // [B][T][Fy][C]  d loss / d GLN(y)
    float* g_r;   // [B][T][Fs][C]  d loss / d GLN_r(rm)
    float* G2;    // [B*T*Fs][2C]: column 2c+1 = d loss / d (pre-ELU residual conv); column 2c left for the GLN_r backward
};
int launch_blend_bwd(const BlendBwdParams& p, cudaStream_t st);
// uv [rows][2C] (u_c, v_c interleaved, bias included), dy [rows][C] -> uv := (dy*sig(v), dy*u*sig(v)*(1-sig(v)))
int launch_gate_bwd(float* uv, const float* dy, long long rows, int C, cudaStream_t st);
// de [n] *= (e > 0 ? 1 : e + 1)
int launch_elu_bwd(float* de, const float* e, long long n, cudaStream_t st);
// dst(b,t,f,c) += src(b,t,f,c) over [B][T][F][C] with independent strides (residual path of the pre-convolutions)
int launch_add_strided(float* dst, StridedRows d, const float* src, StridedRows s, int B, int T, int F, int C,
                       cudaStream_t st);
// dst(b,t,f,c) = [add ? dst(b,t,f,c) : 0] + src(b,t,f,c) over [B][T][F][C], every axis with its own stride on both sides
// (feature taps of the distillation loss: channels-last activations <-> the reference's [B][C][F][T] tensors)
struct Strides4 {
    long long sB, sT, sF, sC;
};
int launch_permute4(float* dst, Strides4 d, const float* src, Strides4 s, int B, int T, int F, int C, int add,
                    cudaStream_t st);
// GRU cell backward for one step (PyTorch gate order r,z,n): dh = dH + dhrec; writes dgi, dgh (3H each) and dhrec := dh*z
int launch_gru_bwd_pw(const float* gi, long long giB, const float* gh, long long ghB, const float* hprev, long long hB,
                      const float* dH, long long dHB, float* dhrec, float* dgi, float* dgh, long long dgB, int B, int H,
                      cudaStream_t st);
// small-channel layers on CUDA cores (small_layers.cu; fp16 operand mode)
struct DeconvLastParams {
    const __half* in;      // last decoder input buffer (padded row 0, frame 0), element strides below
    long long sB, sT, sF;
    int Fin, d;            // input bins, time dilation
    const float* w;        // fp32 packed [4][Kp]: row n = parity * 2 + co, column (kt * 3 + j) * Cin + ci
    int Kp;
    const float* bias;
    float* y;              // [B][T][2 Fin - 1][2] fp32 (raw elu output; normalised inside the mask kernel)
    double* stats;
    int B;
};
struct SkipSmallParams {
    const __half* in;      // skip tensor = interior of an encoder input buffer
    long long sB, sT, sF;
    int Fs;
    const float* w;        // fp32 packed [2C][Kp], rows interleaved (mask_c, residual_c)
    int Kp;
    const float* bias;
    __half *rm, *rr;       // [B][T][Fs][C]
    double* stats;
    int B;
};
bool deconv_last_supported(int Cin);
bool skip_small_supported(int C);
int launch_deconv_last(const DeconvLastParams& p, int Cin, cudaStream_t st);
int launch_skip_small(const SkipSmallParams& p, int C, cudaStream_t st);

// persistent tensor-core GRU recurrence of the streaming path (gru_tc_persist.cu; fp16 operand mode)
struct GruTcParams {
    const __half* Whh;   // packed as for EPI_GRU: row n = gate (n % 96) / 32 of unit 32 (n / 96) + n % 32; pitch Kp halves
    int Kp;
    const float* bhh;    // same row order
    const float* gi;     // input projections incl. b_ih, PyTorch gate order: gi[b*giB + t*3H + {0,H,2H} + j]
    long long giB;
    __half* hseq;        // [B][T+1][H] fp16: slot t = operand of step t, slot t+1 = its result
    long long hB;
    float* h32;          // [B][H] fp32 master state, updated in place
    int* counters;       // [ceil(B/128)] release/acquire counters of the m-tile groups (zeroed by the launcher)
    int H, T, B;
};
bool gru_tc_persist_supported(int H);
int launch_gru_tc_persist(const GruTcParams& p, cudaStream_t st);

// two-layer wavefront recurrence (gru_wave.cu): both layers in one launch, layer 1 one step behind layer 0 and fed by
// h0_t directly (no batched input projection of layer 1)
struct GruWaveParams {
    TmaDesc h0map, h1map;  // [maxB][T+1][H] fp16 state histories, box 64 x 1 x 128 (make_gru_wave_maps)
    const __half *Whh0, *Wih1, *Whh1;  // packed as for EPI_GRU (see GruTcParams), pitch Kp halves
    int Kp;
    const float *bhh0, *bih1, *bhh1;   // same row order
    const float* gi0;      // layer-0 input projections incl. b_ih, PyTorch gate order
    long long giB;
    __half *hseq0, *hseq1; // slot t = operand of step t, slot t+1 = its result
    long long hB;
    float *h32_0, *h32_1;  // [B][H] fp32 master states, updated in place
    int* counters;         // [2][cstride] release/acquire counters per (layer, m-tile) (zeroed by the launcher)
    int cstride;
    int H, T, B;
    int layers;            // 2: wavefront over both layers; 1: one layer (the *0 fields) -- H too large for two slices
    int b0, mtiles;        // set by the launcher: first stream / m-tiles of this launch
};
bool gru_wave_supported(int H, int layers);
int make_gru_wave_maps(GruWaveParams* p, int maxB);
int launch_gru_wave(const GruWaveParams& p, cudaStream_t st);
int gru_profile_read(unsigned long long* out16, int reset);  // diagnostic cycle counters of the roles (-DSE_GRU_PROFILE=1)
// 3-D tiled tensor map over fp16 data: dims (d0 fastest), strides of d1 / d2 in elements, box, SWIZZLE_128B
int make_tma_3d_f16(TmaDesc* out, const void* base, int d0, int d1, int d2, long long s1, long long s2, int b0, int b1,
                    int b2);
// 4-D tiled tensor map over fp16 data: dims (d0 fastest), byte strides of d1 .. d3, box; swizzle_bytes 64 or 128 (the
// box's d0 extent in bytes)
int make_tma_4d_f16(TmaDesc* out, const void* base, const long long dims[4], const long long strides[3], const int box[4],
                    int swizzle_bytes);

// gated skip path of the 32- / 64-channel decoder levels as one tcgen05 launch (skip_blend_tc.cu; fp16 inference):
// out = m elu(residual(skip)) + (1 - m) GLN(y), m = sigmoid(GLN(residualmask(skip)))
struct SkipBlendParams {
    TmaDesc skip;            // the padded skip buffer, one box = one stream's interior (make_skip_blend_maps)
    TmaDesc ymap;            // y, one box = one stream
    int t_org, f_org;        // tensor coordinates of the interior's (frame 0, bin 0)
    int Fs;                  // skip bins = output bins
    const __half* w;         // the skip pair's packed fp16 weights [2C][Kp], rows interleaved (residualmask c, residual c)
    int Kp;
    const float* bias;       // [2C], same interleaving
    const __half* y;         // [B][T][Fy][C] elu(deconv) of the level
    int Fy;
    const double* stats;     // [B][2] sum / sum of squares of y
    const float *nw, *nb;    // norm affine [C]
    const float *nwr, *nbr;  // residualnorm affine [C]
    __half* out;             // block output, element strides below
    long long oB, oT, oF;
    int student, B;
};
bool skip_blend_supported(int C, int Fs, int Fy);
int make_skip_blend_maps(SkipBlendParams* p, const void* skip_base, int C, int Fp, int Tp, long long sT, long long sB,
                         int nB);  // p->Fs, p->Fy, p->y set
int launch_skip_blend(const SkipBlendParams& p, int C, cudaStream_t st);

// persistent small-batch GRU recurrence (gru_seq.cu): one cooperative launch per layer for all chunks and steps
struct GruSeqParams {
    const float* Whh;  // packed [3H][Kp], rows r | z | n (PyTorch order), b_hh separately
    int Kp;
    const float* bhh;
    const float* gi;   // input projections incl. b_ih: gi[s*giB + t*3H + n]
    long long giB;
    float* hseq;       // hseq[s*hB + t*H + j], t in [0, T]: slot 0 = state entering the chunk
    long long hB;
    int H, T, nb, N;   // streams s = n*nb + i (chunk n of utterance i); chunk n starts from the last state of chunk n-1
    int n0;            // first chunk of this launch (chunks n0 .. n0 + N - 1; n0 > 0 continues from chunk n0 - 1)
};
struct GruSeqBwdParams {
    const float* Whh;
    int Kp;
    const float *gi, *gh;  // [B][T][3H] input / recurrent projections (biases included)
    long long gB;
    const float* hseq;     // [B][T+1][H]
    const float* dH;       // [B][T+1][H] d loss / d h_t from the layer above (slot t+1 for step t)
    long long hB;
    float *dgi, *dgh;      // out [B][T][3H]
    float* dhrec;          // scratch [2][B][H]
    int H, T, B;
};
bool gru_seq_supported(int H);
int launch_gru_seq_fwd(const GruSeqParams& p, cudaStream_t st);
int launch_gru_seq_bwd(const GruSeqBwdParams& p, cudaStream_t st);
// generic row copy between two strided slabs: dst[b*dB + i] = src[b*sB + i] (or 0 when src == nullptr), i < count
int launch_copy_rows(float* dst, long long dB, const float* src, long long sB, int count, int nb, cudaStream_t st);

// chunk-major training layout: stream s = n*b + i is chunk n of utterance i
// pred[i][j] = (chunk_{q/P-1}[..] + chunk_{q/P}[..]) * scale at q = j + P + front (utility.py:393-403), j < L
// (scale 1: the adjoint of the chunk segmentation, d mixture gathered from the one or two chunks that read each sample)
int launch_over_add_cm(const float* chunks, int nb, int N, int K, int front, long long L, float* pred, cudaStream_t st,
                       float scale = 0.5f);
// adjoint + envelope: dchunk[s][n] = 0.5 * dpred[i][n0*P + n - P - front] / env[n]  (zero outside [0,L))
int launch_over_add_cm_bwd(const float* dpred, int nb, int N, int K, int front, long long L, float* dchunks,
                           cudaStream_t st);
struct MaskBwdParams {
    int B, student;
    const float* dspec;   // STFT of dchunk/env, reference layout [B][1][F][T][2]
    const float* y;       // raw last deconv output [B][T][F][2]
    const double* stats;
    double count;
    const float *w, *b;
    const float* noisy;   // [B][T][F][2]
    float* g;             // out: d loss / d GLN(y) [B][T][F][2]
    float* dnoisy;        // optional out: d loss / d noisy [B][T][F][2] through the mask multiply (CRN_ELU.py:401-405)
};
int launch_mask_bwd(const MaskBwdParams& p, cudaStream_t st);
struct FeatBwdParams {  // adjoint of the input features (CRN_ELU.py:369-373, distillation_crn.py:340)
    int B, student;
    const float* dfeat;   // d loss / d features, channel c of (b, t, f) at dfeat[b*fB + c*fC + t*fT + f*fF], c < 5
    long long fB, fC, fT, fF;
    const float* dnoisy;  // d loss / d mic-0 spectrum from the mask multiply [B][T][F][2]
    const float* spec;    // the 3-mic spectrum of the chunk [B][3][F][T][2]
    float* dspec;         // out: d loss / d spectrum [B][3][F][T][2]
};
int launch_features_bwd(const FeatBwdParams& p, cudaStream_t st);
// arena <-> flat parameter vector (map[pos] = 1 + flat index, 0 = padding)
int launch_arena_gather(float* arena, const int* map, const float* theta, long long n, cudaStream_t st);
int launch_arena_scatter_add(const float* garena, const int* map, float* grad, long long n, cudaStream_t st);

// ---------------------------------------------------------------------------------------------------------------
// per-stream state export / import (state_io.cu)
// ---------------------------------------------------------------------------------------------------------------
// One entry of a context's carried state.  The state of row r is `count` runs of `run` bytes, the u-th at
// base + r * row_stride + u * unit_stride (count = 1: one contiguous run; count > 1 with a unit_stride that grows with
// max_streams: the "unit-major" form of the FullSubNet cell states [layer][H][maxB (* F)]).  In a record the entry
// occupies `run * count` bytes at rec_off, padded to a multiple of 16 with zeros.
struct StateEntry {
    char* base;
    long long row_stride, unit_stride;
    int run, count;
    int rec_off;
    int vec;  // bytes per access: 16 where base, strides and run allow it, else 4
};
constexpr int kMaxStateEntries = 24;
struct StateTable {
    StateEntry e[kMaxStateEntries];
    int n = 0;
    int first_block[kMaxStateEntries + 1];  // filled by the launcher: blocks [first_block[i], first_block[i+1]) serve entry i
    int record_bytes = 0;                   // multiple of 16
    std::string desc;                       // what fixes the record's bytes; hashed into the layout (host only)
};
// appends an entry (run, row_stride, unit_stride in bytes; multiples of 4) and describes it as `name` with elements of
// `esz` bytes in t.desc
int state_table_add(StateTable& t, const std::string& name, int esz, void* base, long long row_stride, long long run,
                    int count = 1, long long unit_stride = 0);
// FNV-1a 64 of t.desc: equal layouts <=> byte-compatible records
uint64_t state_layout_hash(const StateTable& t);
// host checks of a row list: rows[i] in [0, max_streams), and distinct if `unique`
int state_rows_check(const int32_t* rows, int n, int max_streams, bool unique, const char* what);
// record i <-> entries of row rows[i]; records are t.record_bytes apart at rec
int launch_state_pack(const StateTable& t, const int32_t* rows, int n, void* rec, cudaStream_t st);
int launch_state_unpack(const StateTable& t, const int32_t* rows, int n, const void* rec, cudaStream_t st);

}  // namespace se
