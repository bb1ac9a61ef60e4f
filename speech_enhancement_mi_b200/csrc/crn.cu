// Context, weight re-layout, chunk-step program and the C-ABI of the CRN_ELU streaming path (include/se_b200.h).
//
// Data layout in HBM (per stream, fp32, channels-last): every tensor that feeds a convolution lives in a physically
// zero-bordered buffer [Tp][Fp][C] so that the implicit-GEMM gather (GemmParams::koff) never needs a bounds check:
//   * causal convs (CRN_ELU.py:230-247): `pad` leading frames hold the carried state (= last `pad` frames of the
//     previous chunk's block input), F is bordered by the conv's frequency padding;
//   * transposed convs (CRN_ELU.py:290-307): 2*d trailing zero frames (the `[..., -T:]` crop turns the time taps into
//     look-ahead inside the chunk) and one zero row on each side of F (stride-2 phase split, taps {0,2,4} / {1,3}).
// The carried state of a stream is therefore the leading frames of its conv-input buffers, slot 0 of the two GRU
// hidden sequences and the K/2 overlap-add carry; "roll" moves the trailing frames to the front after each chunk.
// se_crn_state_export / _import gather and scatter exactly that state of chosen rows (state_tab, state_io.cu).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/se_b200.h"
#include "se_internal.h"

namespace se {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }

// ---- per-device launch configuration (se_internal.h) ----------------------------------------------------------------
namespace {
std::mutex g_cfg_mutex;
std::map<std::pair<int, const void*>, int> g_dyn_smem;  // (device, kernel) -> largest size opted in so far
std::map<int, int> g_sm_count;
}  // namespace
int ensure_dyn_smem(const void* func, int bytes) {
    int dev = 0;
    SE_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_cfg_mutex);
    int& have = g_dyn_smem[{dev, func}];
    if (have < bytes) {
        SE_CUDA_OK(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        have = bytes;
    }
    return 0;
}
int num_sms_current_device(int* out) {
    int dev = 0;
    SE_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_cfg_mutex);
    auto it = g_sm_count.find(dev);
    if (it == g_sm_count.end()) {
        int n = 0;
        SE_CUDA_OK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        it = g_sm_count.emplace(dev, n).first;
    }
    *out = it->second;
    return 0;
}

namespace {

constexpr int T = kFramesPerChunk;
constexpr int NBIN = 201;
constexpr int KCHUNK = 3200;
constexpr int PHOP = KCHUNK / 2;

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct Act {  // zero-bordered channels-last activation buffer [maxB][Tp][Fp][C]
    float* base = nullptr;
    int C = 0, F = 0;
    int padT0 = 0, padT1 = 0, padF0 = 0, padF1 = 0;
    int Tp = 0, Fp = 0;
    long long sB = 0, sT = 0, sF = 0;  // strides in ELEMENTS
    int esz = 4;                       // element size: 4 (fp32) or 2 (fp16 operand storage, SE_PRECISION_FP16)
    float* dbase = nullptr;            // training: gradient twin with the same layout (fp32)
    float* dinterior() const { return dbase + padT0 * sT + padF0 * sF; }
    float* at(long long elems) const { return reinterpret_cast<float*>(reinterpret_cast<char*>(base) + elems * esz); }
    float* interior() const { return at(padT0 * sT + padF0 * sF); }
    long long per_stream() const { return sB; }
};

enum OpKind { OP_GEMM, OP_NORM, OP_GRU_PW, OP_PRECONV, OP_GRU_SEQ, OP_DECONV_LAST, OP_SKIP_SMALL, OP_GRU_TC, OP_PRECONV_TC,
              OP_PRECONV3, OP_ENC_MMA, OP_DEC_MMA, OP_GRU_WAVE, OP_ENC_TC, OP_SKIP_BLEND };
enum Stage { ST_STFT = 0, ST_PRECONV, ST_ENCODER, ST_GRU, ST_DECODER, ST_MASK, ST_ROLL, ST_COUNT };
const char* kStageNames[ST_COUNT] = {"stft", "preconv", "encoder", "gru", "decoder", "mask_istft", "roll"};

struct Op {
    OpKind kind;
    int stage;
    std::string label;      // kernel name for reports (se_crn_kernel_info)
    double alg_flops = 0;   // algorithmic FLOPs (2*MACs of the reference op) per stream and chunk
    double alg_bytes = 0;   // algorithmic HBM bytes per stream and chunk: every operand read once, every result written once
    // fp16 operand mode: alg_bytes counts 4 bytes per element, se_crn_kernel_info scales it by this factor for the tensors
    // that really are 2 bytes wide (0.5; 0.75 for the last deconv's fp32 output; 1 for the pre-convolution kernels and
    // the GRU projections / recurrences, which keep fp32 streams)
    double f16_bytes = 1;
    GemmParams g;
    int rows_per_stream = 0;
    NormApplyParams n;
    PreconvParams pc;
    DeconvLastParams dl;
    SkipSmallParams sk;
    GruTcParams gt;
    GruWaveParams gw;
    PreconvTcParams pt;
    Preconv3Params p3;
    EncMmaParams em;
    DecMmaParams dm;
    SkipBlendParams sb;
    int em_cin = 0, em_cout = 0;  // channel counts of the mma.sync block kernels (encoder / decoder)
    int small_c = 0;  // channel count of the two small-layer kernels
    bool tma_ok = false;  // TMA operand delivery (gemm_tc.cu) with `tma`
    GemmTma tma{};
    // GRU pointwise
    const float* gi = nullptr;
    long long giB = 0;
    const float* gh = nullptr;
    const float* hprev = nullptr;
    long long hB = 0;
    float* hout = nullptr;
    int H = 0;
    // training forward (chunk-major batch): state_entry >= 0 -> the carried frames of this op's input come from the
    // previous chunk and are copied in right before the op; chunk_serial -> the op runs chunk by chunk (GRU recurrence)
    int state_entry = -1;
    int chunk_serial = 0;
    int gru_layer = 0;
};

// ---- training: what the backward needs to know about each block (indices into se_ctx::ops) ---------------------
struct ConvRec {
    int op_conv = -1, op_gate = -1, op_norm = -1;
    const Act* in = nullptr;
    float *e = nullptr, *y = nullptr;  // saved elu(conv) and gate output (pre-norm)
    int Cp_out = 0, Fo = 0;
    bool residual = false, need_dgrad = true;
    float* gout = nullptr;  // where d loss / d block output accumulates
    StridedRows gs{};
};
struct DeconvRec {
    int op_deconv = -1, op_skip = -1, op_norm = -1;
    const Act* in = nullptr;
    const Act* skip = nullptr;
    float *y = nullptr, *rm = nullptr, *rr = nullptr;
    int Cop = 0, Fy = 0, Fs = 0;
    float* gout = nullptr;
    StridedRows gs{};
};
struct GruRec {
    int op_in[2] = {-1, -1}, op_hh[2] = {-1, -1}, op_fc = -1, op_norm = -1;
};

struct PreBuf {  // channel-planar preconv input [maxB][5][25][Fpp] (se_internal.h: PRECONV_FPP)
    float* base = nullptr;
    int d = 1, Fpp = 0;
    long long sB = 0, sC = 0;
    float* interior() const { return base + 4 * Fpp + 2 * d; }  // frame 4 (first new frame), bin 0
};

}  // namespace
}  // namespace se

using namespace se;

struct se_ctx {
    se_crn_config cfg;
    int device = 0;
    int maxB = 0;
    int L = 0;        // levels
    int C0 = 0;       // 2M-1 real input channels
    int student = 0;
    std::vector<int> encF;  // F after each encoder level
    int Fg = 0, Cg = 0, feat = 0, H = 0;

    WeightArena wa;  // packed weights, their koff tables and the parameter registry
    std::vector<void*> allocs;

    // activations
    std::vector<PreBuf> pre_in;  // 3 preconv inputs
    std::vector<Act> enc_in;  // L encoder inputs
    std::vector<Act> dec_in;  // L decoder inputs
    float *xg = nullptr, *gi = nullptr, *gh = nullptr, *hseq[2] = {nullptr, nullptr}, *fcraw = nullptr;
    float *tmp_e = nullptr, *tmp_y = nullptr, *tmp_rm = nullptr, *tmp_rr = nullptr;
    float *noisy = nullptr, *ylast = nullptr, *carry = nullptr;
    double* stats = nullptr;
    int n_stats = 0;
    int stats_last = -1;  // slot of the last deconv's statistics
    const float *w_last = nullptr, *b_last = nullptr;

    std::vector<Op> ops;
    RollTable roll{};
    RollTable zero_tab{};
    int64_t roll_floats = 0;   // floats moved per stream by the roll kernel
    StateTable state_tab;       // what a stream carries between steps (se_crn_state_export / _import; state_io.cu)
    uint64_t state_layout = 0;  // hash of the record layout

    IoDesc* io_dev = nullptr;
    bool use_graph = true;
    bool tf32 = false;  // tensor-core path (tf32 or fp16 operands)
    bool half = false;  // operands of the tensor-core GEMMs are stored as fp16 (SE_PRECISION_FP16)
    bool split = false;  // tensor-core GEMMs in the 3xTF32 form, exact-mode epilogues (SE_PRECISION_3XTF32)
    int esz = 4;        // element size of the GEMM-operand activations
    int ue = 4;         // elements per 16-byte gather unit
    int kblock = 32;    // elements per k-block
    float* h32[2] = {nullptr, nullptr};  // fp16 mode: fp32 master copy of the GRU state [maxB][H] per layer
    float* E(float* base, long long elems) const {  // element offset into an operand buffer
        return reinterpret_cast<float*>(reinterpret_cast<char*>(base) + elems * esz);
    }
    int gru_wave = 1;          // SE_B200_GRU_WAVE=0: one persistent kernel per layer (+ the layer-1 projection GEMM) instead
                               // of the two-layer wavefront kernel (gru_wave.cu); 2: also where H is too large for the
                               // wavefront, use the one-layer form of gru_wave.cu instead of gru_tc_persist.cu
    bool gru_persist = true;   // SE_B200_GRU_PERSIST=0: one GEMM launch per recurrent step instead of the persistent kernel
    int* gru_counters = nullptr;
    // fp16 mode: pre-convolutions on the tensor cores (preconv_tc.cu: implicit conv through no-swizzle UMMA descriptors
    // over the SMEM-resident channels-last input, frequency taps as a shift-and-add in the epilogue); 0.164 ms per layer
    // against 0.231 ms for the fp32 CUDA-core kernel.  SE_B200_PRECONV_TC=0 keeps the CUDA-core kernel.
    bool preconv_tc = true;
    __half* pre_h[3] = {nullptr, nullptr, nullptr};  // tensor-core pre-convolution inputs [maxB][25][272][8] halves
    // fp16 mode: the three pre-convolutions as ONE launch and the small-channel encoder blocks as one launch each, warp-level
    // mma.sync with the stream resident in shared memory (front_mma.cu).  SE_B200_FRONT_MMA=0 / SE_B200_ENC_MMA=0 keep the
    // round-1 kernels (preconv_tc.cu per layer; back-to-back tcgen05 GEMM + separate GlobalLayerNorm pass).
    bool front_mma = true, enc_mma = true;
    int enc_tc = 1;  // SE_B200_ENC_TC=0: the 16 -> 32 / 32 -> 64 encoder levels on their round-2a kernels (mma.sync / b2b GEMM);
                     // 1: 32 -> 64 on the implicit-GEMM kernel (enc_tc.cu); 2: 16 -> 32 there too
    int bwd_mode = BWD_3XTF32;  // arithmetic of the backward contractions (train_kernels.cu), SE_B200_BWD_MMA
    bool dec_mma = true;  // SE_B200_DEC_MMA=0: small-channel decoder blocks as deconv GEMM + skip-pair kernel + blend kernel
    bool use_tma = true;  // SE_B200_TMA=0: every tcgen05 GEMM keeps the cp.async gather producers
    __half* feat_h = nullptr;     // features of the chunk [maxB][21][224][8] halves (borders stay zero)
    __half* pre_state = nullptr;  // carried frames of the three pre-convolutions [maxB][3][4][224][8] halves
    bool b2b_gate = true;      // SE_B200_B2B=0: 32- / 64-channel gates as separate GEMMs
    bool small_layers = true;  // SE_B200_SMALL_LAYERS=0: keep the two small-channel layers on the GEMM path (A/B switch)
    unsigned tc_mask = 0xffffffffu;  // SE_B200_TC_MASK: bit per Stage that may use the tensor-core GEMM (debug)
    std::map<int, cudaGraphExec_t> graphs;  // keyed by B
    cudaStream_t own_stream = nullptr;
    // training forward: second branch for the layer-1 GRU (input projection + recurrence per chunk group) beside layer 0
    cudaStream_t pipe_stream = nullptr;
    cudaEvent_t pipe_ev[17] = {};
    int gru_pipe = 1;  // SE_B200_GRU_PIPE=0: the two GRU layers one after the other
    int bwd_overlap = 1;  // SE_B200_BWD_OVERLAP=0: weight gradient, then data gradient, on one stream

    // ---- training (se_crn_config.training): chunk-major batch, activations of every layer kept, gradient twins --------
    bool train = false;
    bool alloc_failed = false;
    std::vector<Act> pre_act;  // the three pre-convolution inputs as zero-bordered channels-last buffers (GEMM path)
    float* gi_l[2] = {nullptr, nullptr};  // per-layer GRU input projections (kept for the backward)
    std::vector<ConvRec> conv_recs;       // preconv 0..2, encoder 0..L-1
    std::vector<DeconvRec> deconv_recs;   // decoder 0..L-1
    GruRec gru_rec;
    float* garena = nullptr;  // gradient twin of the weight arena
    int* wmap = nullptr;      // weight-arena position -> 1 + index into the flat parameter vector (0: padding)
    std::vector<int64_t> param_off;
    int64_t n_theta = 0;
    float *dxg = nullptr, *dH[2] = {nullptr, nullptr}, *dhrec = nullptr, *dgi = nullptr, *dgh = nullptr, *gh_all = nullptr;
    float* sc[4] = {nullptr, nullptr, nullptr, nullptr};  // scratch, 2 * tmp_floats * maxB each
    double* red = nullptr;                                 // [maxB][2]
    float *chunks = nullptr, *dchunks = nullptr, *dspec = nullptr;
    float* dnoisy = nullptr;  // d loss / d mic-0 spectrum through the mask multiply (input gradient only)
    bool t_wgrad = true;      // this backward computes parameter gradients (false: d mixture of a frozen model only)
    std::vector<std::pair<void*, size_t>> twins;  // zeroed at the start of every backward
    std::vector<float*> carry_store;              // per state entry: [maxB][count] state kept between flag=True pieces
    int t_nb = 0, t_N = 0, t_front = 0;
    long long t_L = 0;
    bool t_have_fwd = false;
    size_t tmp_floats = 0;

    // staging for the host variant
    float *h_in = nullptr, *h_out = nullptr;
    size_t h_in_floats = 0, h_out_floats = 0;
};

namespace {

int make_act(se_ctx* c, Act& a, int C, int F, int Tn, int padT0, int padT1, int padF0, int padF1) {
    a.C = C;
    a.F = F;
    a.padT0 = padT0;
    a.padT1 = padT1;
    a.padF0 = padF0;
    a.padF1 = padF1;
    a.Tp = padT0 + Tn + padT1;
    a.Fp = padF0 + F + padF1;
    a.sF = C;
    a.sT = (long long)a.Fp * C;
    a.sB = a.sT * a.Tp;
    a.esz = c->esz;
    return dev_alloc(c, reinterpret_cast<char**>(&a.base), (size_t)a.sB * c->maxB * a.esz);
}

// ---- parameter registry (order of TemporalCRN.state_dict() without the `net.0` aliases; CRN_ELU.py:335-365) -------
void register_params(se_ctx* c) {
    auto add = [&](const std::string& n, std::vector<int> s) { c->wa.params.push_back({n, std::move(s)}); };
    const se_crn_config& g = c->cfg;
    auto conv_block = [&](const std::string& p, int ci, int co, int kf, int kt) {
        add(p + ".conv.weight", {co, ci, kf, kt});
        add(p + ".conv.bias", {co});
        add(p + ".conv_trans.weight", {co, co, 1, 1});
        add(p + ".conv_trans.bias", {co});
        add(p + ".conv_gated.weight", {co, co, 1, 1});
        add(p + ".conv_gated.bias", {co});
        add(p + ".norm.weight", {1, co, 1, 1});
        add(p + ".norm.bias", {1, co, 1, 1});
    };
    for (int i = 0; i < 3; ++i) conv_block("preconvlist." + std::to_string(i), c->C0, c->C0, 5, 5);
    for (int i = 0; i < c->L; ++i)
        conv_block("convlist." + std::to_string(i), i == 0 ? c->C0 : g.num_channels[i - 1], g.num_channels[i], 5,
                   g.kernel_size);
    for (int j = 0; j < c->L; ++j) {
        const int ci = g.num_channels[c->L - 1 - j];
        const int co = j < c->L - 1 ? g.num_channels[c->L - 2 - j] : 2;
        const std::string p = "deconvlist." + std::to_string(j);
        add(p + ".conv.weight", {ci, co, 5, g.kernel_size});
        add(p + ".conv.bias", {co});
        add(p + ".residualmask.weight", {co, co, 1, 1});
        add(p + ".residualmask.bias", {co});
        add(p + ".residualnorm.weight", {1, co, 1, 1});
        add(p + ".residualnorm.bias", {1, co, 1, 1});
        add(p + ".residual.weight", {co, co, 1, 1});
        add(p + ".residual.bias", {co});
        add(p + ".norm.weight", {1, co, 1, 1});
        add(p + ".norm.bias", {1, co, 1, 1});
    }
    for (int l = 0; l < g.num_layers; ++l) {
        const std::string s = std::to_string(l);
        add("gru.sequence_model.weight_ih_l" + s, {3 * c->H, l == 0 ? c->feat : c->H});
        add("gru.sequence_model.weight_hh_l" + s, {3 * c->H, c->H});
        add("gru.sequence_model.bias_ih_l" + s, {3 * c->H});
        add("gru.sequence_model.bias_hh_l" + s, {3 * c->H});
    }
    add("gru.fc_output_layer.weight", {c->feat, c->H});
    add("gru.fc_output_layer.bias", {c->feat});
    add("gru.norm.weight", {1, 1, 1, c->feat});
    add("gru.norm.bias", {1, 1, 1, c->feat});
}

// A packed GEMM weight: W[Npad][K] followed by bias[Npad]
struct PackedW {
    size_t w_off, b_off;
    int Npad, K;
};
// Rows are padded to the output-tile width the tensor-core kernel will pick for N (gemm_tf32_tile_n) and the row
// pitch to whole 32-float k-blocks, all zero-filled, so that the kernels need no bounds checks on the weight operand.
PackedW reserve_packed(se_ctx* c, int N, int K) {
    PackedW pw;
    pw.Npad = round_up(N, gemm_tf32_tile_n(N));
    pw.K = round_up(K, c->kblock);
    pw.w_off = c->wa.reserve_w((size_t)pw.Npad * pw.K);
    pw.b_off = c->wa.reserve_w(pw.Npad);
    return pw;
}

void fill_gemm_common(se_ctx* c, GemmParams& g, const PackedW& pw, int N) {
    g.K = pw.K;
    g.N = N;
    g.Npad = pw.Npad;
    g.a_half = c->half ? 1 : 0;
}

constexpr size_t NONE = (size_t)-1;

// geometry of the tensor a GEMM's A operand is gathered from, [B][Tp][Fp][C] at `base`, with the row grid starting at
// (frame t_org, bin f_org) and advancing fstep bins per output bin (TMA operand delivery).  C = 0: not described.
struct TmaSrc {
    const void* base = nullptr;
    int C = 0, Fp = 0, Tp = 0;
    long long sT = 0, sB = 0;
    int fstep = 1, t_org = 0, f_org = 0;
};

// points a GEMM op at its packed weights, bias, koff table and (EPI_ELU_GATE) fused gate weights
int bind_gemm(se_ctx* c, Op& op, const PackedW& pw, int k_off, size_t w2_off, size_t b2_off, const TmaSrc& ts) {
    const WeightArena& wa = c->wa;
    op.g.W = (c->half && op.g.a_half) ? static_cast<const void*>(wa.wh + pw.w_off)
                                      : static_cast<const void*>(wa.w + pw.w_off);
    op.g.bias = wa.w + pw.b_off;
    op.g.koff = wa.k + k_off;
    if (w2_off != NONE) {
        op.g.W2 = wa.w + w2_off;
        op.g.bias2 = wa.w + b2_off;
    }
    // TMA delivery where every k-block of the gather is 64 contiguous channels of one (frame, bin) tap
    if (c->use_tma && ts.C > 0 && ts.C % 64 == 0 && op.g.a_half) {
        GemmParams probe = op.g;
        probe.M = op.rows_per_stream;
        const int nkb = op.g.K / 64;
        std::vector<int> kc(4 * nkb, 0);
        bool ok = gemm_tma_supported(probe) && op.g.Fo * op.g.Tn == op.rows_per_stream;
        for (int kb = 0; kb < nkb && ok; ++kb) {
            const int e = wa.khost[k_off + 8 * kb];
            for (int j = 1; j < 8; ++j) ok = ok && wa.khost[k_off + 8 * kb + j] == e + 8 * j;
            kc[4 * kb + 2] = (int)(e / ts.sT);
            const int rem = (int)(e % ts.sT);
            kc[4 * kb + 1] = rem / ts.C;
            kc[4 * kb] = rem % ts.C;
            ok = ok && kc[4 * kb] % 64 == 0;
        }
        // weights beyond the real K are zero, but their k-blocks must still address valid channels: the padding
        // units of the koff table point at offset 0 (frame 0, bin 0, channel 0), which the loop above maps there
        if (ok) {
            int* kdev = nullptr;
            if (dev_alloc(c, &kdev, kc.size())) return 1;
            SE_CUDA_OK(cudaMemcpy(kdev, kc.data(), kc.size() * sizeof(int), cudaMemcpyHostToDevice));
            if (make_gemm_tma(&op.tma, ts.base, ts.C, ts.Fp, ts.Tp, ts.sT, ts.sB, c->maxB, op.g.Fo, ts.fstep, op.g.Tn,
                              op.g.W, op.g.K, op.g.Npad, gemm_tma_tile_n(op.g)))
                return 1;
            op.tma.t_org = ts.t_org;
            op.tma.f_org = ts.f_org;
            op.tma.kcoord = reinterpret_cast<const int4*>(kdev);
            op.tma_ok = true;
        }
    }
    return 0;
}

struct Builder {
    se_ctx* c;
    std::string m_label;  // meta of the next pushed op
    double m_flops = 0, m_bytes = 0, m_f16 = 0.5;
    void meta(const std::string& label, double flops, double bytes, double f16_bytes = 0.5) {
        m_label = label;
        m_flops = flops;
        m_bytes = bytes;
        m_f16 = f16_bytes;
    }
    // appends `op` with the pending meta(); `bind` points it at its packed weights once the arena exists.  Returns its
    // index in se_ctx::ops.
    int push(Op op, std::function<int(Op&)> bind = nullptr) {
        op.label = m_label;
        op.alg_flops = m_flops;
        op.alg_bytes = m_bytes;
        op.f16_bytes = m_f16;
        meta("", 0, 0);
        c->ops.push_back(op);
        const int i = (int)c->ops.size() - 1;
        if (bind) {
            se_ctx* cc = c;
            c->wa.binds.push_back([cc, i, bind] { return bind(cc->ops[i]); });
        }
        return i;
    }

    // identity koff for a dense K-contiguous operand
    int koff_dense(int K) {
        const int U = c->ue;
        std::vector<int> v(K / U);
        for (int u = 0; u < K / U; ++u) v[u] = U * u;
        return c->wa.reserve_k(v);
    }

    // ts: the tensor the A operand is gathered from, for TMA delivery
    int push_gemm(int stage, GemmParams g, int rows_per_stream, const PackedW& pw, int k_off, TmaSrc ts = {},
                  size_t w2_off = NONE, size_t b2_off = NONE, OpKind kind = OP_GEMM) {
        Op op{};
        op.kind = kind;
        op.stage = stage;
        op.g = g;
        op.rows_per_stream = rows_per_stream;
        se_ctx* cc = c;
        return push(op, [=](Op& o) { return bind_gemm(cc, o, pw, k_off, w2_off, b2_off, ts); });
    }
    bool tc_stage(int stage) const { return c->tf32 && ((c->tc_mask >> stage) & 1u); }
    // inference: the per-layer temporaries share four buffers; training: every layer keeps its own (saved for backward)
    float* tmp_buf(float* shared, size_t floats_per_stream) {
        if (!c->train) return shared;
        float* p = nullptr;
        if (dev_alloc(c, &p, floats_per_stream * c->maxB)) c->alloc_failed = true;
        return p;
    }
    int push_norm(int stage, NormApplyParams n, size_t w_off, size_t b_off, size_t wr_off = NONE, size_t br_off = NONE) {
        Op op{};
        op.kind = OP_NORM;
        op.stage = stage;
        op.n = n;
        op.n.out_half = c->half ? 1 : 0;  // every normalised tensor is the operand of a following GEMM
        op.n.in_half = c->half ? 1 : 0;   // ... and the pre-norm tensors are stored as fp16 too
        se_ctx* cc = c;
        return push(op, [=](Op& o) {
            o.n.w = cc->wa.w + w_off;
            o.n.b = cc->wa.w + b_off;
            if (wr_off != NONE) {
                o.n.wr = cc->wa.w + wr_off;
                o.n.br = cc->wa.w + br_off;
            }
            return 0;
        });
    }
    int push_gru_pw(const float* gi, long long giB, const float* gh, const float* hprev, long long hB, float* hout, int H) {
        Op op{};
        op.kind = OP_GRU_PW;
        op.stage = ST_GRU;
        op.gi = gi;
        op.giB = giB;
        op.gh = gh;
        op.hprev = hprev;
        op.hB = hB;
        op.hout = hout;
        op.H = H;
        return push(op);
    }

    // per-channel affine [Cp] (zero beyond the real channels) -> arena
    size_t pack_affine(const std::string& key, int Creal, int Cp) {
        const size_t off = c->wa.reserve_w(Cp);
        c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
            const std::vector<float>& v = hp.at(key);
            for (int i = 0; i < Cp; ++i) arena[off + i] = i < Creal ? v[i] : 0.f;
        });
        return off;
    }

    // one pre-convolution block in the PRECONV_W_* layout (se_internal.h) -> arena
    size_t pack_preconv_block(const std::string& name) {
        const size_t w_off = c->wa.reserve_w(PRECONV_W_FLOATS);
        c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
            const std::vector<float>& w = hp.at(name + ".conv.weight");  // [Co][Ci][KF][KT]
            float* a = arena + w_off;
            for (int kt = 0; kt < 5; ++kt)
                for (int ci = 0; ci < 5; ++ci)
                    for (int kf = 0; kf < 5; ++kf)
                        for (int co = 0; co < 5; ++co)
                            a[(kt * 5 + ci) * 28 + kf * 5 + co] = w[((co * 5 + ci) * 5 + kf) * 5 + kt];
            for (int co = 0; co < 5; ++co) {
                a[PRECONV_W_BIAS + co] = hp.at(name + ".conv.bias")[co];
                for (int k = 0; k < 5; ++k) {
                    a[PRECONV_W_WT + co * 5 + k] = hp.at(name + ".conv_trans.weight")[co * 5 + k];
                    a[PRECONV_W_WG + co * 5 + k] = hp.at(name + ".conv_gated.weight")[co * 5 + k];
                }
                a[PRECONV_W_BT + co] = hp.at(name + ".conv_trans.bias")[co];
                a[PRECONV_W_BG + co] = hp.at(name + ".conv_gated.bias")[co];
                a[PRECONV_W_NW + co] = hp.at(name + ".norm.weight")[co];
                a[PRECONV_W_NB + co] = hp.at(name + ".norm.bias")[co];
            }
        });
        return w_off;
    }

    // ---- causal gated conv block (CRN_ELU.py:230-247) ---------------------------------------------------------
    // in: padded input; dst/dstB..: where the normalised output goes; residual: add the block input (preconv)
    void conv_block(int stage, const std::string& name, const Act& in, int Cin_real, int Cout_real, int KF, int KT,
                    int strideF, int dilF, int dilT, int Fo, float* dst, long long dB, long long dT, long long dF,
                    bool residual, int stats_slot, int state_entry = -1, float* dgrad_dst = nullptr) {
        const int Cp_in = in.C;
        const int Cp_out = round_up(Cout_real, 4);
        const int rows = T * Fo;
        // gate fused into the conv GEMM: in registers for <= 16 channels, as a back-to-back tensor-core GEMM (fp16 operands)
        // for 32 / 64 channels (SE_B200_B2B=0 keeps those two levels on separate kernels)
        // small-channel encoder levels (fp16 mode): conv + ELU + gate + GlobalLayerNorm as ONE launch (front_mma.cu)
        const bool enc_shape = stage == ST_ENCODER && !residual && KF == 5 && KT == 3 && strideF == 2 && dilF == 1 &&
                               Cp_out == Cout_real && in.padF0 == 2 && in.padT0 == 2 * dilT && c->half && !c->train;
        // ... as an implicit GEMM on tcgen05 over the resident input where the channel counts allow it (enc_tc.cu)
        const bool use_tc = enc_shape && enc_tc_supported(c->enc_tc, Cp_in, Cout_real, in.Tp, in.Fp, Fo);
        const bool use_mma = use_tc || (c->enc_mma && enc_shape && enc_mma_supported(Cp_in, Cout_real, in.Tp, in.Fp, Fo));
        const bool fuse_gate = use_mma || (tc_stage(stage) && !c->train &&
                               (Cp_out <= 16 || (c->half && c->b2b_gate && (Cout_real == 32 || Cout_real == 64))));
        const int w2_pitch = gemm_tf32_tile_n(Cout_real);
        double* stats = c->stats + (size_t)stats_slot * 2 * c->maxB;
        float* const tmp_e = tmp_buf(c->tmp_e, (size_t)rows * Cp_out);
        float* const tmp_y = tmp_buf(c->tmp_y, (size_t)rows * Cp_out);
        ConvRec rec;
        rec.in = &in;
        rec.e = tmp_e;
        rec.y = tmp_y;
        rec.Cp_out = Cp_out;
        rec.Fo = Fo;
        rec.residual = residual;
        rec.gout = dgrad_dst;
        rec.gs = StridedRows{dB, dT, dF};
        // (1) conv + ELU -> tmp_e [B][T][Fo][Cp_out]   (fuse_gate: + gated 1x1 pair + statistics -> tmp_y, skipping 2)
        {
            const int K = KT * KF * Cp_in;
            const int U = c->ue;
            std::vector<int> koff(K / U);
            for (int kt = 0; kt < KT; ++kt)
                for (int kf = 0; kf < KF; ++kf)
                    for (int cu = 0; cu < Cp_in / U; ++cu)
                        koff[((kt * KF + kf) * Cp_in) / U + cu] =
                            (int)(kt * dilT * in.sT + kf * dilF * in.sF + U * cu);
            const int k_off = c->wa.reserve_k(koff);
            PackedW pw = reserve_packed(c, Cout_real, K);
            c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                const std::vector<float>& w = hp.at(name + ".conv.weight");  // [Co][Ci][KF][KT]
                const std::vector<float>& b = hp.at(name + ".conv.bias");
                for (int n = 0; n < Cout_real; ++n) {
                    for (int kt = 0; kt < KT; ++kt)
                        for (int kf = 0; kf < KF; ++kf)
                            for (int ci = 0; ci < Cin_real; ++ci)
                                arena[pw.w_off + (size_t)n * pw.K + (kt * KF + kf) * Cp_in + ci] =
                                    w[((n * Cin_real + ci) * KF + kf) * KT + kt];
                    arena[pw.b_off + n] = b[n];
                }
            });
            size_t w2_off = NONE, b2_off = NONE;
            if (fuse_gate) {
                w2_off = c->wa.reserve_w((size_t)2 * Cout_real * w2_pitch);
                b2_off = c->wa.reserve_w((size_t)2 * Cout_real);
                c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                    const std::vector<float>& wt = hp.at(name + ".conv_trans.weight");
                    const std::vector<float>& bt = hp.at(name + ".conv_trans.bias");
                    const std::vector<float>& wg = hp.at(name + ".conv_gated.weight");
                    const std::vector<float>& bg = hp.at(name + ".conv_gated.bias");
                    for (int co = 0; co < Cout_real; ++co) {
                        for (int ci = 0; ci < Cout_real; ++ci) {
                            arena[w2_off + (size_t)(2 * co) * w2_pitch + ci] = wt[co * Cout_real + ci];
                            arena[w2_off + (size_t)(2 * co + 1) * w2_pitch + ci] = wg[co * Cout_real + ci];
                        }
                        arena[b2_off + 2 * co] = bt[co];
                        arena[b2_off + 2 * co + 1] = bg[co];
                    }
                });
            }
            GemmParams g{};
            g.A = in.base;
            g.sB = in.sB;
            g.sT = in.sT;
            g.sF = (long long)strideF * in.sF;
            g.Tn = T;
            g.Fo = Fo;
            fill_gemm_common(c, g, pw, Cout_real);
            g.epi = fuse_gate ? EPI_ELU_GATE : EPI_ELU;
            g.out = fuse_gate ? tmp_y : tmp_e;
            g.oB = (long long)rows * Cp_out;
            g.oT = (long long)Fo * Cp_out;
            g.oF = Cp_out;
            g.vec4 = 1;
            if (fuse_gate) {
                g.C2 = Cout_real;
                g.stats = stats;
            }
            g.out_half = c->half ? 1 : 0;  // tmp_e (operand of the gate GEMM) / tmp_y (pre-norm tensor) are fp16 then
            {
                const double in_b = 4.0 * Cin_real * in.Tp * in.F, conv_fl = 2.0 * rows * Cout_real * (KT * KF * Cin_real);
                if (fuse_gate)
                    meta(name + ".conv+elu+gate", conv_fl + 4.0 * rows * Cout_real * Cout_real, in_b + 4.0 * rows * Cout_real);
                else
                    meta(name + ".conv+elu", conv_fl, in_b + 4.0 * rows * Cout_real);
            }
            if (use_mma) {
                const size_t nw_off = pack_affine(name + ".norm.weight", Cout_real, Cp_out);
                const size_t nb_off = pack_affine(name + ".norm.bias", Cout_real, Cp_out);
                size_t w1c_off = NONE, w2c_off = NONE;
                if (use_tc) {  // the two B operands of enc_tc.cu, element for element in its shared-memory order
                    const int CI = Cp_in, CO = Cout_real, HP = CI / 16;
                    const size_t n1 = (size_t)15 * HP * 2 * CO * 8, n2 = (size_t)(CO / 16) * 2 * (2 * CO) * 8;
                    w1c_off = (c->wa.reserve_w(n1 + 8) + 7) / 8 * 8;  // 16-byte aligned in the fp16 copy of the arena (cp.async)
                    w2c_off = (c->wa.reserve_w(n2 + 8) + 7) / 8 * 8;
                    c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                        const std::vector<float>& w = hp.at(name + ".conv.weight");  // [Co][Ci][KF][KT]
                        const std::vector<float>& wt = hp.at(name + ".conv_trans.weight");
                        const std::vector<float>& wg = hp.at(name + ".conv_gated.weight");
                        for (size_t i = 0; i < n1; ++i) {
                            const int cc = (int)(i & 7), n = (int)((i >> 3) % CO), j = (int)(((i >> 3) / CO) & 1);
                            const int ks = (int)((i >> 3) / (2 * CO)), tap = ks / HP, hp_ = ks % HP;
                            const int ci = (2 * hp_ + j) * 8 + cc, kt = tap / 5, kf = tap % 5;
                            arena[w1c_off + i] = ci < Cin_real ? w[((size_t)(n * Cin_real + ci) * KF + kf) * KT + kt] : 0.f;
                        }
                        for (size_t i = 0; i < n2; ++i) {
                            const int cc = (int)(i & 7), r2 = (int)((i >> 3) % (2 * CO)), j = (int)(((i >> 3) / (2 * CO)) & 1);
                            const int ks2 = (int)((i >> 3) / (4 * CO)), kind = r2 / CO, ch = r2 % CO, k = ks2 * 16 + j * 8 + cc;
                            arena[w2c_off + i] = kind ? 0.5f * wg[(size_t)ch * CO + k] : wt[(size_t)ch * CO + k];
                        }
                    });
                }
                Op op{};
                op.kind = use_tc ? OP_ENC_TC : OP_ENC_MMA;
                op.stage = stage;
                op.em = EncMmaParams{};
                op.em.in = reinterpret_cast<const __half*>(in.base);
                op.em.in_sB = in.sB;
                op.em.Tp = in.Tp;
                op.em.Fp = in.Fp;
                op.em.dt = dilT;
                op.em.Fo = Fo;
                op.em.Kp = pw.K;
                op.em.w2_pitch = w2_pitch;
                op.em.out = reinterpret_cast<__half*>(dst);
                op.em.oB = dB;
                op.em.oT = dT;
                op.em.oF = dF;
                op.em.student = c->student;
                op.em_cin = Cp_in;
                op.em_cout = Cout_real;
                meta(name + ".conv+elu+gate+gln",
                     2.0 * rows * Cout_real * (KT * KF * Cin_real) + 4.0 * rows * Cout_real * Cout_real,
                     4.0 * Cin_real * in.Tp * in.F + 4.0 * rows * Cout_real);
                se_ctx* cc = c;
                push(op, [=](Op& o) {
                    const WeightArena& wa = cc->wa;
                    if (use_tc) {
                        o.em.w1c = wa.wh + w1c_off;
                        o.em.w2c = wa.wh + w2c_off;
                    }
                    o.em.w = wa.w + pw.w_off;
                    o.em.bias = wa.w + pw.b_off;
                    o.em.w2 = wa.w + w2_off;
                    o.em.bias2 = wa.w + b2_off;
                    o.em.nw = wa.w + nw_off;
                    o.em.nb = wa.w + nb_off;
                    return 0;
                });
                return;
            }
            rec.op_conv = push_gemm(stage, g, rows, pw, k_off, TmaSrc{in.base, in.C, in.Fp, in.Tp, in.sT, in.sB, strideF},
                                    w2_off, b2_off);
            c->ops.back().state_entry = state_entry;
        }
        // (2) gated 1x1 pair + statistics -> tmp_y [B][T][Fo][Cp_out]
        if (!fuse_gate) {
            const int K = Cp_out;
            const int k_off = koff_dense(K);
            PackedW pw = reserve_packed(c, 2 * Cout_real, K);
            c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                const std::vector<float>& wt = hp.at(name + ".conv_trans.weight");
                const std::vector<float>& bt = hp.at(name + ".conv_trans.bias");
                const std::vector<float>& wg = hp.at(name + ".conv_gated.weight");
                const std::vector<float>& bg = hp.at(name + ".conv_gated.bias");
                for (int co = 0; co < Cout_real; ++co) {
                    for (int ci = 0; ci < Cout_real; ++ci) {
                        arena[pw.w_off + (size_t)(2 * co) * pw.K + ci] = wt[co * Cout_real + ci];
                        arena[pw.w_off + (size_t)(2 * co + 1) * pw.K + ci] = wg[co * Cout_real + ci];
                    }
                    arena[pw.b_off + 2 * co] = bt[co];
                    arena[pw.b_off + 2 * co + 1] = bg[co];
                }
            });
            GemmParams g{};
            g.A = tmp_e;
            g.sB = (long long)rows * Cp_out;
            g.sT = (long long)Fo * Cp_out;
            g.sF = Cp_out;
            g.Tn = T;
            g.Fo = Fo;
            fill_gemm_common(c, g, pw, 2 * Cout_real);
            g.epi = EPI_GATE_STATS;
            g.out = tmp_y;
            g.oB = g.sB;
            g.oT = g.sT;
            g.oF = g.sF;
            g.vec4 = 1;
            g.stats = stats;
            g.out_half = c->half ? 1 : 0;
            meta(name + ".gate1x1", 4.0 * rows * Cout_real * Cout_real, 8.0 * rows * Cout_real);
            rec.op_gate = push_gemm(stage, g, rows, pw, k_off,
                                    TmaSrc{tmp_e, Cp_out, Fo, T, (long long)Fo * Cp_out, (long long)rows * Cp_out});
        }
        // (3) GlobalLayerNorm (+ residual) -> destination
        {
            NormApplyParams n{};
            n.mode = residual ? 1 : 0;
            n.T = T;
            n.F = Fo;
            n.C = Cp_out;
            n.student = c->student;
            n.y = tmp_y;
            n.Fy = Fo;
            n.stats = c->stats + (size_t)stats_slot * 2 * c->maxB;
            n.count = (double)Cout_real * Fo * T;
            n.per_feature = 0;
            if (residual) {
                n.res = in.interior();
                n.rB = in.sB;
                n.rT = in.sT;
                n.rF = in.sF;
            }
            n.out = dst;
            n.oB = dB;
            n.oT = dT;
            n.oF = dF;
            const size_t w_off = pack_affine(name + ".norm.weight", Cout_real, Cp_out);
            const size_t b_off = pack_affine(name + ".norm.bias", Cout_real, Cp_out);
            meta(name + ".gln" + (residual ? "+residual" : ""), 0, (residual ? 12.0 : 8.0) * rows * Cout_real);
            rec.op_norm = push_norm(stage, n, w_off, b_off);
        }
        if (c->train) c->conv_recs.push_back(rec);
    }

    // ---- transposed conv block (CRN_ELU.py:290-307) ---------------------------------------------------------
    // in: [T + 2d][Fin + 2][Cin]; skip: padded encoder-input buffer whose interior is the skip tensor (or null).
    // The weights of every form are packed first (deconv, skip pair, the four affines); then the form is chosen and
    // only its ops are pushed.
    void deconv_block(const std::string& name, const Act& in, int Cin, int Cout_real, int KT, int d, const Act* skip,
                      float* dst, long long dB, long long dT, long long dF, int stats_slot, int stats_slot_r,
                      float* dgrad_dst = nullptr) {
        const int Fin = in.F;
        const int Fy = 2 * Fin - 1;
        const int Fs = skip ? skip->F : Fy;
        const int rows = T * Fs;
        const int Cop = Cout_real < 4 ? Cout_real : round_up(Cout_real, 4);  // last layer keeps 2 (float2 consumer)
        float* y = skip ? tmp_buf(c->tmp_y, (size_t)T * Fy * Cop) : c->ylast;
        float* const tmp_rm = skip ? tmp_buf(c->tmp_rm, (size_t)rows * Cop) : nullptr;
        float* const tmp_rr = skip ? tmp_buf(c->tmp_rr, (size_t)rows * Cop) : nullptr;
        double* const stats = c->stats + (size_t)stats_slot * 2 * c->maxB;
        double* const stats_r = skip ? c->stats + (size_t)stats_slot_r * 2 * c->maxB : nullptr;
        DeconvRec rec;
        rec.in = &in;
        rec.skip = skip;
        rec.y = y;
        rec.rm = tmp_rm;
        rec.rr = tmp_rr;
        rec.Cop = Cop;
        rec.Fy = Fy;
        rec.Fs = Fs;
        rec.gout = dgrad_dst;
        rec.gs = StridedRows{dB, dT, dF};
        // Both output parities in one GEMM.  Output bin phi = 2f' (even) uses taps kf = 0,2,4 and phi = 2f'+1 (odd)
        // taps kf = 1,3, all on the padded input rows f'+2-j (j = kf/2): the odd half re-uses the rows gathered for
        // the even half.  Columns: [even channels | odd channels] = 2*Cout contiguous floats of y at bin 2f'.  The
        // odd half of the last row (phi = 2*Fin-1 = Fy) does not exist: GemmParams::odd_tail masks it.
        const int nkf = 3;
        const int K = KT * nkf * Cin;
        const int U = c->ue;
        std::vector<int> koff(K / U);
        for (int kt = 0; kt < KT; ++kt)
            for (int j = 0; j < nkf; ++j)
                for (int cu = 0; cu < Cin / U; ++cu) {
                    const long long frame = (long long)(KT - 1 - kt) * d;
                    koff[((kt * nkf + j) * Cin) / U + cu] = (int)(frame * in.sT + (2 - j) * in.sF + U * cu);
                }
        const int k_off = c->wa.reserve_k(koff);
        const PackedW pw = reserve_packed(c, 2 * Cout_real, K);
        c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
            const int KF = 5;
            const std::vector<float>& w = hp.at(name + ".conv.weight");  // [Ci][Co][KF][KT]
            const std::vector<float>& b = hp.at(name + ".conv.bias");
            for (int parity = 0; parity < 2; ++parity)
                for (int co = 0; co < Cout_real; ++co) {
                    const int n = parity * Cout_real + co;
                    for (int kt = 0; kt < KT; ++kt)
                        for (int j = 0; j < nkf; ++j) {
                            const int kf = 2 * j + parity;
                            if (kf >= KF) continue;  // odd rows have no third tap: weights stay zero
                            for (int ci = 0; ci < Cin; ++ci)
                                arena[pw.w_off + (size_t)n * pw.K + (kt * nkf + j) * Cin + ci] =
                                    w[((ci * Cout_real + co) * KF + kf) * KT + kt];
                        }
                    arena[pw.b_off + n] = b[co];
                }
        });
        // ConvTranspose2d counted over the T kept frames: even bins 3 taps, odd bins 2 taps
        const double deconv_flops = 2.0 * T * (3.0 * Fin + 2.0 * (Fin - 1)) * KT * Cin * Cout_real;
        const double skip_flops = 4.0 * rows * Cout_real * Cout_real;
        // residual mask / residual 1x1 pair on the skip tensor, then the affines of both GlobalLayerNorms
        int k2_off = -1;
        PackedW pw2{};
        size_t nw_off = NONE, nb_off = NONE, nwr_off = NONE, nbr_off = NONE;
        if (skip) {
            k2_off = koff_dense(skip->C);
            pw2 = reserve_packed(c, 2 * Cout_real, skip->C);
            c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                const std::vector<float>& wm = hp.at(name + ".residualmask.weight");
                const std::vector<float>& bm = hp.at(name + ".residualmask.bias");
                const std::vector<float>& wr = hp.at(name + ".residual.weight");
                const std::vector<float>& br = hp.at(name + ".residual.bias");
                for (int co = 0; co < Cout_real; ++co) {
                    for (int ci = 0; ci < Cout_real; ++ci) {
                        arena[pw2.w_off + (size_t)(2 * co) * pw2.K + ci] = wm[co * Cout_real + ci];
                        arena[pw2.w_off + (size_t)(2 * co + 1) * pw2.K + ci] = wr[co * Cout_real + ci];
                    }
                    arena[pw2.b_off + 2 * co] = bm[co];
                    arena[pw2.b_off + 2 * co + 1] = br[co];
                }
            });
            nw_off = pack_affine(name + ".norm.weight", Cout_real, Cop);
            nb_off = pack_affine(name + ".norm.bias", Cout_real, Cop);
            nwr_off = pack_affine(name + ".residualnorm.weight", Cout_real, Cop);
            nbr_off = pack_affine(name + ".residualnorm.bias", Cout_real, Cop);
        }
        se_ctx* cc = c;
        const bool fused_skip = skip && skip->C == Cout_real && Cop == Cout_real;
        // 32- / 64-channel levels (fp16 inference): the skip pair and the blend as ONE launch (skip_blend_tc.cu) after the
        // transposed-conv GEMM
        const bool blend = fused_skip && c->half && !c->train && skip_blend_supported(Cout_real, Fs, Fy);
        if (fused_skip && !blend && c->dec_mma && dec_mma_supported(Cin, Cout_real, in.Tp, in.Fp, Fin, Fs)) {
            // small-channel levels (fp16 mode): the whole block as ONE launch (back_mma.cu)
            Op op{};
            op.kind = OP_DEC_MMA;
            op.stage = ST_DECODER;
            op.dm = DecMmaParams{};
            op.dm.in = reinterpret_cast<const __half*>(in.base);
            op.dm.in_sB = in.sB;
            op.dm.Tp = in.Tp;
            op.dm.Fp = in.Fp;
            op.dm.d = d;
            op.dm.Fin = Fin;
            op.dm.Kp = pw.K;
            op.dm.skip = reinterpret_cast<const __half*>(skip->interior());
            op.dm.sk_sB = skip->sB;
            op.dm.sk_sT = skip->sT;
            op.dm.sk_sF = skip->sF;
            op.dm.Fs = Fs;
            op.dm.K2p = pw2.K;
            op.dm.out = reinterpret_cast<__half*>(dst);
            op.dm.oB = dB;
            op.dm.oT = dT;
            op.dm.oF = dF;
            op.dm.student = c->student;
            op.em_cin = Cin;
            op.em_cout = Cout_real;
            // input and skip tensor in, block output out
            meta(name + ".deconv+skip+blend", deconv_flops + skip_flops, 4.0 * Cin * T * Fin + 4.0 * 2 * T * Fs * Cout_real);
            push(op, [=](Op& o) {
                const float* w = cc->wa.w;
                o.dm.w = w + pw.w_off;
                o.dm.bias = w + pw.b_off;
                o.dm.w2 = w + pw2.w_off;
                o.dm.bias2 = w + pw2.b_off;
                o.dm.nw = w + nw_off;
                o.dm.nb = w + nb_off;
                o.dm.nwr = w + nwr_off;
                o.dm.nbr = w + nbr_off;
                return 0;
            });
            return;
        }
        meta(name + ".deconv+elu", deconv_flops, 4.0 * Cin * T * Fin + 4.0 * T * Fy * Cout_real);
        if (c->half && !c->train && !skip && Cout_real == 2 && KT == 3 && deconv_last_supported(Cin) && c->small_layers) {
            Op op{};  // the last level on the direct kernel (small_layers.cu): fp16 input, fp32 output
            op.kind = OP_DECONV_LAST;
            op.stage = ST_DECODER;
            op.small_c = Cin;
            op.dl = DeconvLastParams{};
            op.dl.in = reinterpret_cast<const __half*>(in.base);
            op.dl.sB = in.sB;
            op.dl.sT = in.sT;
            op.dl.sF = in.sF;
            op.dl.Fin = Fin;
            op.dl.d = d;
            op.dl.Kp = pw.K;
            op.dl.y = y;
            op.dl.stats = stats;
            m_f16 = 0.75;
            push(op, [=](Op& o) {
                o.dl.w = cc->wa.w + pw.w_off;
                o.dl.bias = cc->wa.w + pw.b_off;
                return 0;
            });
        } else {
            GemmParams g{};
            g.A = in.base;  // padded row 0, frame 0
            g.sB = in.sB;
            g.sT = in.sT;
            g.sF = in.sF;
            g.Tn = T;
            g.Fo = Fin;
            fill_gemm_common(c, g, pw, 2 * Cout_real);
            g.epi = EPI_ELU_STATS;
            g.out = y;
            g.oB = (long long)T * Fy * Cop;
            g.oT = (long long)Fy * Cop;
            g.oF = 2 * Cop;
            g.odd_tail = 1;
            g.out_half = (c->half && skip) ? 1 : 0;  // the last layer's output feeds the mask kernel in fp32
            g.stats = stats;
            g.vec4 = Cop % 4 == 0;
            rec.op_deconv = push_gemm(ST_DECODER, g, T * Fin, pw, k_off, TmaSrc{in.base, in.C, in.Fp, in.Tp, in.sT, in.sB});
        }
        if (!skip) {
            if (c->train) c->deconv_recs.push_back(rec);
            return;
        }
        const TmaSrc skip_src{skip->base, skip->C, skip->Fp, skip->Tp, skip->sT, skip->sB, 1, skip->padT0, skip->padF0};
        if (blend) {
            Op op{};
            op.kind = OP_SKIP_BLEND;
            op.stage = ST_DECODER;
            op.sb = SkipBlendParams{};
            op.sb.t_org = skip->padT0;
            op.sb.f_org = skip->padF0;
            op.sb.Fs = Fs;
            op.sb.Kp = pw2.K;
            op.sb.y = reinterpret_cast<const __half*>(y);
            op.sb.Fy = Fy;
            op.sb.stats = stats;
            op.sb.out = reinterpret_cast<__half*>(dst);
            op.sb.oB = dB;
            op.sb.oT = dT;
            op.sb.oF = dF;
            op.sb.student = c->student;
            op.em_cout = Cout_real;
            // y and skip tensor in, block output out
            meta(name + ".skip+gln+blend", skip_flops, 4.0 * T * Fy * Cout_real + 4.0 * 2 * T * Fs * Cout_real);
            push(op, [=](Op& o) {
                const float* w = cc->wa.w;
                o.sb.w = cc->wa.wh + pw2.w_off;
                o.sb.bias = w + pw2.b_off;
                o.sb.nw = w + nw_off;
                o.sb.nb = w + nb_off;
                o.sb.nwr = w + nwr_off;
                o.sb.nbr = w + nbr_off;
                return make_skip_blend_maps(&o.sb, skip_src.base, skip_src.C, skip_src.Fp, skip_src.Tp, skip_src.sT,
                                            skip_src.sB, cc->maxB);
            });
            return;
        }
        meta(name + ".skip1x1", skip_flops, 12.0 * rows * Cout_real);
        if (c->half && !c->train && skip->C == Cout_real && skip_small_supported(Cout_real) && c->small_layers) {
            Op op{};  // the skip pair on the small-channel kernel (small_layers.cu)
            op.kind = OP_SKIP_SMALL;
            op.stage = ST_DECODER;
            op.small_c = Cout_real;
            op.sk = SkipSmallParams{};
            op.sk.in = reinterpret_cast<const __half*>(skip->interior());
            op.sk.sB = skip->sB;
            op.sk.sT = skip->sT;
            op.sk.sF = skip->sF;
            op.sk.Fs = Fs;
            op.sk.Kp = pw2.K;
            op.sk.rm = reinterpret_cast<__half*>(tmp_rm);
            op.sk.rr = reinterpret_cast<__half*>(tmp_rr);
            op.sk.stats = stats_r;
            push(op, [=](Op& o) {
                o.sk.w = cc->wa.w + pw2.w_off;
                o.sk.bias = cc->wa.w + pw2.b_off;
                return 0;
            });
        } else {
            GemmParams g{};
            g.A = skip->interior();
            g.sB = skip->sB;
            g.sT = skip->sT;
            g.sF = skip->sF;
            g.Tn = T;
            g.Fo = Fs;
            fill_gemm_common(c, g, pw2, 2 * Cout_real);
            g.epi = EPI_SKIP;
            g.out = tmp_rm;
            g.oB = (long long)rows * Cop;
            g.oT = (long long)Fs * Cop;
            g.oF = Cop;
            g.out2 = tmp_rr;
            g.o2B = g.oB;
            g.o2T = g.oT;
            g.o2F = g.oF;
            g.stats = stats_r;
            g.vec4 = 1;
            g.out_half = c->half ? 1 : 0;
            rec.op_skip = push_gemm(ST_DECODER, g, rows, pw2, k2_off, skip_src);
        }
        {
            NormApplyParams n{};
            n.mode = 2;
            n.T = T;
            n.F = Fs;
            n.C = Cop;
            n.student = c->student;
            n.y = y;
            n.Fy = Fy;
            n.stats = stats;
            n.count = (double)Cout_real * Fy * T;
            n.rm = tmp_rm;
            n.rr = tmp_rr;
            n.stats_r = stats_r;
            n.count_r = (double)Cout_real * Fs * T;
            n.out = dst;
            n.oB = dB;
            n.oT = dT;
            n.oF = dF;
            meta(name + ".gln+skipblend", 0, 4.0 * T * Cout_real * (Fy + 3.0 * Fs));
            rec.op_norm = push_norm(ST_DECODER, n, nw_off, nb_off, nwr_off, nbr_off);
        }
        if (c->train) c->deconv_recs.push_back(rec);
    }
};

int build_ctx(se_ctx* c) {
    const se_crn_config& g = c->cfg;
    SE_REQUIRE(g.num_inputs == 3, "num_inputs must be 3 (features of CRN_ELU.py:369-373 are built for 3 microphones)");
    SE_REQUIRE(g.num_freqs == NBIN && g.n_fft == 400 && g.win_length == 400 && g.hop_length == 160,
               "STFT kernel is built for n_fft=win=400, hop=160, 201 bins (config.yaml:214-217)");
    SE_REQUIRE(g.segment_length == KCHUNK, "segment_length must be 3200 (config.yaml:209)");
    SE_REQUIRE(g.num_levels >= 2 && g.num_levels <= 4, "num_levels must be 2..4 (state pad 2*2^i must stay < 21 frames)");
    SE_REQUIRE(g.kernel_size == 3, "kernel_size must be 3 (config.yaml:211)");
    SE_REQUIRE(g.num_layers == 2, "num_layers must be 2 (config.yaml:210)");
    SE_REQUIRE(g.hidden % 16 == 0 && g.hidden > 0, "hidden must be a positive multiple of 16");
    SE_REQUIRE(g.max_streams > 0, "max_streams must be positive");
    SE_REQUIRE(g.precision == SE_PRECISION_FP32 || g.precision == SE_PRECISION_TF32 || g.precision == SE_PRECISION_FP16 ||
                   g.precision == SE_PRECISION_3XTF32,
               "unknown precision");
    SE_REQUIRE(g.variant == SE_VARIANT_CRN_ELU || g.variant == SE_VARIANT_DISTILLED, "unknown variant");
    c->maxB = g.max_streams;
    c->L = g.num_levels;
    c->C0 = 2 * g.num_inputs - 1;
    c->student = g.variant == SE_VARIANT_DISTILLED;
    c->H = g.hidden;
    c->tf32 = g.precision != SE_PRECISION_FP32;
    c->half = g.precision == SE_PRECISION_FP16;
    c->split = g.precision == SE_PRECISION_3XTF32;
    c->train = g.training != 0;
    SE_REQUIRE(!(c->train && c->half), "training keeps fp32 activations: use precision fp32, 3xtf32 or tf32");
    c->esz = c->half ? 2 : 4;
    c->ue = 16 / c->esz;
    c->kblock = 128 / c->esz;
    if (const char* e = getenv("SE_B200_TC_MASK")) c->tc_mask = (unsigned)strtoul(e, nullptr, 0);
    if (const char* e = getenv("SE_B200_SMALL_LAYERS")) c->small_layers = atoi(e) != 0;
    if (const char* e = getenv("SE_B200_GRU_PERSIST")) c->gru_persist = atoi(e) != 0;
    if (const char* e = getenv("SE_B200_GRU_WAVE")) c->gru_wave = atoi(e);
    if (const char* e = getenv("SE_B200_B2B")) c->b2b_gate = atoi(e) != 0;
    if (const char* e = getenv("SE_B200_PRECONV_TC")) c->preconv_tc = atoi(e) != 0;
    c->preconv_tc = c->preconv_tc && c->half && !c->train;
    if (const char* e = getenv("SE_B200_TMA")) c->use_tma = atoi(e) != 0;
    c->use_tma = c->use_tma && c->half && !c->train;
    if (const char* e = getenv("SE_B200_FRONT_MMA")) c->front_mma = atoi(e) != 0;
    if (const char* e = getenv("SE_B200_ENC_MMA")) c->enc_mma = atoi(e) != 0;
    if (const char* e = getenv("SE_B200_ENC_TC")) c->enc_tc = atoi(e);
    SE_REQUIRE(c->enc_tc >= 0 && c->enc_tc <= 2, "SE_B200_ENC_TC must be 0, 1 or 2");
    c->front_mma = c->front_mma && c->preconv_tc;  // replaces the per-layer tensor-core kernels
    c->enc_mma = c->enc_mma && c->half && !c->train;
    if (const char* e = getenv("SE_B200_DEC_MMA")) c->dec_mma = atoi(e) != 0;
    c->dec_mma = c->dec_mma && c->half && !c->train;
    // backward contractions of the training step: fp32-accurate 3xTF32 beside the exact and the 3xTF32 forward, one
    // tf32 pass beside the tf32 forward; SE_B200_BWD_MMA=0 keeps them on the CUDA cores (1 / 2 force a tensor-core form)
    c->bwd_mode = c->tf32 && !c->split ? BWD_TF32 : BWD_3XTF32;
    if (const char* e = getenv("SE_B200_BWD_MMA")) c->bwd_mode = atoi(e);
    SE_REQUIRE(c->bwd_mode >= 0 && c->bwd_mode <= 2, "SE_B200_BWD_MMA must be 0, 1 or 2");
    if (const char* e = getenv("SE_B200_GRU_PIPE")) c->gru_pipe = atoi(e);
    if (const char* e = getenv("SE_B200_BWD_OVERLAP")) c->bwd_overlap = atoi(e);
    if (c->train && (c->gru_pipe || c->bwd_overlap)) {  // created here, not at first use: the first use may sit inside a stream capture
        SE_CUDA_OK(cudaStreamCreateWithFlags(&c->pipe_stream, cudaStreamNonBlocking));
        for (cudaEvent_t& e : c->pipe_ev) SE_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    for (int i = 0; i < c->L; ++i) {
        SE_REQUIRE(g.num_channels[i] % 4 == 0 && g.num_channels[i] > 0, "num_channels must be multiples of 4");
        SE_REQUIRE(!c->half || g.num_channels[i] % 8 == 0, "fp16 mode: num_channels must be multiples of 8");
    }
    SE_REQUIRE(!c->half || g.hidden % 32 == 0, "fp16 mode: hidden must be a multiple of 32");
    int F = NBIN;
    for (int i = 0; i < c->L; ++i) {
        F = (F - 1) / 2 + 1;
        c->encF.push_back(F);
    }
    c->Fg = F;
    c->Cg = g.num_channels[c->L - 1];
    c->feat = c->Fg * c->Cg;
    SE_REQUIRE(c->Fg == NBIN / (1 << c->L) + 1, "frequency pyramid does not match CRN_ELU.py:364");
    register_params(c);

    const int maxB = c->maxB;
    const int C0p = 8;
    const int H = c->H;
    // ---- activations ------------------------------------------------------------------------------------------
    const long long pre_h_sB = (long long)PRECONV_TP * PRECONV_TC_POS * 8;  // halves per stream
    const long long feat_sB = (long long)T * PRECONV3_POS * 8, pre_state_sB = 3LL * 4 * PRECONV3_POS * 8;  // halves
    if (c->front_mma) {
        if (dev_alloc(c, &c->feat_h, (size_t)feat_sB * maxB)) return 1;
        if (dev_alloc(c, &c->pre_state, (size_t)pre_state_sB * maxB)) return 1;
    } else if (c->preconv_tc) {
        for (int i = 0; i < 3; ++i)
            if (dev_alloc(c, &c->pre_h[i], (size_t)pre_h_sB * maxB)) return 1;
    }
    c->pre_in.resize((c->train || c->preconv_tc) ? 0 : 3);
    for (int i = 0; i < (int)c->pre_in.size(); ++i) {
        PreBuf& pb = c->pre_in[i];
        pb.d = 1 << i;
        pb.Fpp = PRECONV_FPP(pb.d);
        pb.sC = (long long)PRECONV_TP * pb.Fpp;
        pb.sB = 5 * pb.sC;
        if (dev_alloc(c, &pb.base, (size_t)pb.sB * maxB)) return 1;
    }
    auto make_twin = [&](Act& a) -> int {
        if (!c->train) return 0;
        if (dev_alloc(c, &a.dbase, (size_t)a.sB * maxB)) return 1;
        c->twins.push_back({a.dbase, (size_t)a.sB * maxB * sizeof(float)});
        return 0;
    };
    if (c->train) {  // training: the pre-convolutions run on the generic GEMM path so that one backward serves all convs
        c->pre_act.resize(3);
        for (int i = 0; i < 3; ++i) {
            const int d = 1 << i;
            if (make_act(c, c->pre_act[i], C0p, NBIN, T, 4, 0, 2 * d, 2 * d)) return 1;
            if (make_twin(c->pre_act[i])) return 1;
        }
    }
    c->enc_in.resize(c->L);
    for (int i = 0; i < c->L; ++i) {
        const int Cin = i == 0 ? C0p : g.num_channels[i - 1];
        const int Fin = i == 0 ? NBIN : c->encF[i - 1];
        if (make_act(c, c->enc_in[i], Cin, Fin, T, 2 * (1 << i), 0, 2, 2)) return 1;
        if (make_twin(c->enc_in[i])) return 1;
    }
    c->dec_in.resize(c->L);
    for (int j = 0; j < c->L; ++j) {
        const int Cin = g.num_channels[c->L - 1 - j];
        const int Fin = j == 0 ? c->Fg : c->encF[c->L - 1 - j];
        const int d = 1 << j;
        if (make_act(c, c->dec_in[j], Cin, Fin, T, 0, 2 * d, 1, 1)) return 1;
        if (make_twin(c->dec_in[j])) return 1;
    }
    size_t tmp = 0;
    auto upd = [&](size_t v) { tmp = v > tmp ? v : tmp; };
    upd((size_t)T * NBIN * C0p);
    for (int i = 0; i < c->L; ++i) upd((size_t)T * c->encF[i] * g.num_channels[i]);
    for (int j = 0; j + 1 < c->L; ++j) {
        const int Fin = c->dec_in[j].F;
        const int Co = g.num_channels[c->L - 2 - j];
        upd((size_t)T * (2 * Fin) * Co);
    }
    if (dev_alloc(c, reinterpret_cast<char**>(&c->tmp_e), tmp * maxB * c->esz)) return 1;
    if (dev_alloc(c, reinterpret_cast<char**>(&c->tmp_y), tmp * maxB * c->esz)) return 1;
    if (dev_alloc(c, reinterpret_cast<char**>(&c->tmp_rm), tmp * maxB * c->esz)) return 1;
    if (dev_alloc(c, reinterpret_cast<char**>(&c->tmp_rr), tmp * maxB * c->esz)) return 1;
    if (dev_alloc(c, reinterpret_cast<char**>(&c->xg), (size_t)T * c->feat * maxB * c->esz)) return 1;
    if (dev_alloc(c, reinterpret_cast<char**>(&c->fcraw), (size_t)T * c->feat * maxB * c->esz)) return 1;
    c->tmp_floats = tmp;
    if (dev_alloc(c, &c->gi, (size_t)T * 3 * H * maxB)) return 1;
    c->gi_l[0] = c->gi_l[1] = c->gi;
    if (c->train) {
        if (dev_alloc(c, &c->gi_l[1], (size_t)T * 3 * H * maxB)) return 1;
        if (dev_alloc(c, &c->gh_all, (size_t)T * 3 * H * maxB)) return 1;
        if (dev_alloc(c, &c->dgi, (size_t)T * 3 * H * maxB)) return 1;
        if (dev_alloc(c, &c->dgh, (size_t)T * 3 * H * maxB)) return 1;
        if (dev_alloc(c, &c->dhrec, (size_t)2 * H * maxB)) return 1;
        if (dev_alloc(c, &c->dxg, (size_t)T * c->feat * maxB)) return 1;
        c->twins.push_back({c->dxg, (size_t)T * c->feat * maxB * sizeof(float)});
        for (int l = 0; l < 2; ++l) {
            if (dev_alloc(c, &c->dH[l], (size_t)(T + 1) * H * maxB)) return 1;
            c->twins.push_back({c->dH[l], (size_t)(T + 1) * H * maxB * sizeof(float)});
        }
        for (int i = 0; i < 4; ++i)
            if (dev_alloc(c, &c->sc[i], 2 * tmp * maxB)) return 1;
        if (dev_alloc(c, &c->red, (size_t)2 * maxB)) return 1;
        if (dev_alloc(c, &c->chunks, (size_t)KCHUNK * maxB)) return 1;
        if (dev_alloc(c, &c->dchunks, (size_t)KCHUNK * maxB)) return 1;
        if (dev_alloc(c, &c->dspec, (size_t)T * NBIN * 2 * maxB)) return 1;
        if (dev_alloc(c, &c->dnoisy, (size_t)T * NBIN * 2 * maxB)) return 1;
    }
    if (dev_alloc(c, &c->gh, (size_t)3 * H * maxB)) return 1;
    for (int l = 0; l < 2; ++l)
        if (dev_alloc(c, reinterpret_cast<char**>(&c->hseq[l]), (size_t)(T + 1) * H * maxB * c->esz)) return 1;
    if (c->half)
        for (int l = 0; l < 2; ++l)
            if (dev_alloc(c, &c->h32[l], (size_t)H * maxB)) return 1;
    if (dev_alloc(c, &c->noisy, (size_t)T * NBIN * 2 * maxB)) return 1;
    if (dev_alloc(c, &c->ylast, (size_t)T * NBIN * 2 * maxB)) return 1;
    if (dev_alloc(c, &c->carry, (size_t)PHOP * maxB)) return 1;
    c->n_stats = 3 + c->L + 1 + 2 * c->L;
    if (dev_alloc(c, &c->stats, (size_t)c->n_stats * 2 * maxB)) return 1;
    if (dev_alloc(c, &c->io_dev, 1)) return 1;
    if (dev_alloc(c, &c->gru_counters, (size_t)2 * ((maxB + 127) / 128))) return 1;

    // ---- program ----------------------------------------------------------------------------------------------
    Builder b{c};
    int slot = 0;
    for (int i = 0; i < 3 && c->train; ++i) {  // training: generic conv blocks with the residual add (CRN_ELU.py:376)
        const Act& in = c->pre_act[i];
        const Act& nx = i < 2 ? c->pre_act[i + 1] : c->enc_in[0];
        b.conv_block(ST_PRECONV, "preconvlist." + std::to_string(i), in, c->C0, c->C0, 5, 5, 1, 1 << i, 1, NBIN,
                     nx.interior(), nx.sB, nx.sT, nx.sF, true, slot++, i, nx.dinterior());
        c->conv_recs.back().need_dgrad = i > 0;
    }
    if (c->front_mma) {  // fp16 mode: the three pre-convolution blocks in one launch (front_mma.cu)
        size_t w_off[3];
        for (int i = 0; i < 3; ++i) w_off[i] = b.pack_preconv_block("preconvlist." + std::to_string(i));
        const Act& nx = c->enc_in[0];
        Op op{};
        op.kind = OP_PRECONV3;
        op.stage = ST_PRECONV;
        op.p3 = Preconv3Params{};
        op.p3.feat = c->feat_h;
        op.p3.feat_sB = feat_sB;
        op.p3.state = c->pre_state;
        op.p3.state_sB = pre_state_sB;
        op.p3.out = reinterpret_cast<__half*>(nx.interior());
        op.p3.oB = nx.sB;
        op.p3.oT = nx.sT;
        op.p3.oF = nx.sF;
        op.p3.student = c->student;
        // features in, block output out, 4 carried frames per layer read and written (fp32 sizes, as for every other op)
        b.meta("preconvlist.0-2.fused", 3 * 2.0 * T * NBIN * 5 * (125 + 10), 4.0 * 5 * NBIN * (T + T + 3 * 2 * 4));
        b.push(op, [=](Op& o) {
            for (int l = 0; l < 3; ++l) o.p3.w[l] = c->wa.w + w_off[l];
            return 0;
        });
        slot += 3;
    }
    for (int i = 0; i < 3 && c->preconv_tc && !c->front_mma; ++i) {  // fp16 mode: pre-convolutions on the tensor cores (preconv_tc.cu)
        const std::string name = "preconvlist." + std::to_string(i);
        const size_t w_off = b.pack_preconv_block(name);
        Op op{};
        op.kind = OP_PRECONV_TC;
        op.stage = ST_PRECONV;
        op.pt.in = c->pre_h[i];
        op.pt.in_sB = pre_h_sB;
        op.pt.d = 1 << i;
        op.pt.student = c->student;
        if (i < 2) {
            op.pt.out = c->pre_h[i + 1] + (4LL * PRECONV_TC_POS + 2 * (2 << i)) * 8;  // frame 4, bin 0 of the next layer
            op.pt.oB = pre_h_sB;
            op.pt.oT = (long long)PRECONV_TC_POS * 8;
            op.pt.oF = 8;
        } else {
            const Act& nx = c->enc_in[0];
            op.pt.out = reinterpret_cast<__half*>(nx.interior());
            op.pt.oB = nx.sB;
            op.pt.oT = nx.sT;
            op.pt.oF = nx.sF;
        }
        b.meta(name + ".fused", 2.0 * T * NBIN * 5 * (125 + 10), 2.0 * 8 * NBIN * (PRECONV_TP + T), 1);
        b.push(op, [=](Op& o) {
            o.pt.w = c->wa.w + w_off;
            return 0;
        });
        slot++;
    }
    for (int i = 0; i < 3 && !c->train && !c->preconv_tc; ++i) {  // pre-convolutions: one fused kernel per layer (preconv.cu), exact fp32
        const PreBuf& in = c->pre_in[i];
        const std::string name = "preconvlist." + std::to_string(i);
        const size_t w_off = b.pack_preconv_block(name);
        Op op{};
        op.kind = OP_PRECONV;
        op.stage = ST_PRECONV;
        op.pc.in = in.base;
        op.pc.in_sB = in.sB;
        op.pc.d = in.d;
        op.pc.student = c->student;
        if (i < 2) {
            const PreBuf& nx = c->pre_in[i + 1];
            op.pc.out = nx.interior();
            op.pc.oB = nx.sB;
            op.pc.oC = nx.sC;
            op.pc.oT = nx.Fpp;
            op.pc.oF = 1;
        } else {
            const Act& nx = c->enc_in[0];
            op.pc.out = nx.interior();
            op.pc.oB = nx.sB;
            op.pc.oC = 1;
            op.pc.oT = nx.sT;
            op.pc.oF = nx.sF;
            op.pc.out_vec8 = 1;
            op.pc.out_half = c->half ? 1 : 0;
        }
        b.meta(name + ".fused", 2.0 * T * NBIN * 5 * (125 + 10), 4.0 * 5 * NBIN * (PRECONV_TP + T), 1);
        b.push(op, [=](Op& o) {
            o.pc.w = c->wa.w + w_off;
            return 0;
        });
        slot++;
    }
    for (int i = 0; i < c->L; ++i) {
        const Act& in = c->enc_in[i];
        const int Cin_real = i == 0 ? c->C0 : g.num_channels[i - 1];
        float *dst, *gdst = nullptr;
        long long dB, dT, dF;
        if (i + 1 < c->L) {
            const Act& nx = c->enc_in[i + 1];
            dst = nx.interior();
            if (c->train) gdst = nx.dinterior();
            dB = nx.sB;
            dT = nx.sT;
            dF = nx.sF;
        } else {
            dst = c->xg;
            gdst = c->dxg;
            dB = (long long)T * c->feat;
            dT = c->feat;
            dF = c->Cg;
        }
        b.conv_block(ST_ENCODER, "convlist." + std::to_string(i), in, Cin_real, g.num_channels[i], 5, 3, 2, 1, 1 << i,
                     c->encF[i], dst, dB, dT, dF, false, slot++, c->train ? 3 + i : -1, gdst);
    }
    // ---- GRU + Linear + ELU + GLN(last) (CRN_ELU.py:160-186) --------------------------------------------------
    // feature index: reference c*Fg + f  ->  ours f*Cg + c (channels-last)
    const int Fg = c->Fg, Cg = c->Cg, feat = c->feat;
    auto perm = [=](int ours) { return (ours % Cg) * Fg + ours / Cg; };
    const int gru_slot = slot++;
    // fp16 inference: both recurrences and the layer-1 projection as ONE wavefront launch (gru_wave.cu)
    const bool wave = !c->train && c->half && c->gru_persist && c->gru_wave && gru_tc_persist_supported(H) &&
                      gru_wave_supported(H, 2);
    PackedW wave_pw[3];  // W_hh0, W_ih1 (gate-tile order), W_hh1
    for (int l = 0; l < 2; ++l) {
        const int Kin = l == 0 ? feat : H;
        const std::string s = std::to_string(l);
        if (wave && l == 1) {  // W_ih1 in the gate-tile order of the fused cell; no batched projection
            PackedW pw = reserve_packed(c, 3 * H, H);
            wave_pw[1] = pw;
            c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                const std::vector<float>& w = hp.at("gru.sequence_model.weight_ih_l1");
                const std::vector<float>& bi = hp.at("gru.sequence_model.bias_ih_l1");
                for (int n = 0; n < 3 * H; ++n) {
                    const int src = ((n % 96) / 32) * H + (n / 96) * 32 + n % 32;
                    for (int k = 0; k < H; ++k) arena[pw.w_off + (size_t)n * pw.K + k] = w[(size_t)src * H + k];
                    arena[pw.b_off + n] = bi[src];
                }
            });
        } else {  // input projection for all T frames at once
            const int k_off = b.koff_dense(Kin);
            PackedW pw = reserve_packed(c, 3 * H, Kin);
            c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
                const std::vector<float>& w = hp.at("gru.sequence_model.weight_ih_l" + s);
                const std::vector<float>& bi = hp.at("gru.sequence_model.bias_ih_l" + s);
                for (int n = 0; n < 3 * H; ++n) {
                    for (int k = 0; k < Kin; ++k)
                        arena[pw.w_off + (size_t)n * pw.K + k] = w[(size_t)n * Kin + (l == 0 ? perm(k) : k)];
                    arena[pw.b_off + n] = bi[n];
                }
            });
            GemmParams gp{};
            if (l == 0) {
                gp.A = c->xg;
                gp.sB = (long long)T * feat;
                gp.sT = feat;
            } else {
                gp.A = c->E(c->hseq[0], H);
                gp.sB = (long long)(T + 1) * H;
                gp.sT = H;
            }
            gp.sF = 0;
            gp.Tn = T;
            gp.Fo = 1;
            fill_gemm_common(c, gp, pw, 3 * H);
            gp.epi = EPI_BIAS;
            gp.out = c->gi_l[l];
            gp.oB = (long long)T * 3 * H;
            gp.oT = 3 * H;
            gp.oF = 0;
            gp.vec4 = 1;
            b.meta("gru.l" + s + ".input_proj", 2.0 * T * 3 * H * Kin, 4.0 * T * (Kin + 3 * H), 1);
            c->gru_rec.op_in[l] = b.push_gemm(ST_GRU, gp, T, pw, k_off,
                                              l == 0 ? TmaSrc{c->xg, feat, 1, T, feat, (long long)T * feat}
                                                     : TmaSrc{c->hseq[0], H, 1, T + 1, H, (long long)(T + 1) * H, 1, 1, 0});
        }
        const int k_off = b.koff_dense(H);
        PackedW pw = reserve_packed(c, 3 * H, H);
        const bool fused = !c->train && (c->half || (c->tf32 && ((c->tc_mask >> ST_GRU) & 1u) && H % 32 == 0));
        c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
            const std::vector<float>& w = hp.at("gru.sequence_model.weight_hh_l" + s);
            const std::vector<float>& bh = hp.at("gru.sequence_model.bias_hh_l" + s);
            for (int n = 0; n < 3 * H; ++n) {
                // fused tensor-core cell: tile y holds [r | z | n] of hidden units 32y .. 32y+31 (gemm_tc.cu EPI_GRU)
                const int src = fused ? ((n % 96) / 32) * H + (n / 96) * 32 + n % 32 : n;
                for (int k = 0; k < H; ++k) arena[pw.w_off + (size_t)n * pw.K + k] = w[(size_t)src * H + k];
                arena[pw.b_off + n] = bh[src];
            }
        });
        const bool persist = fused && c->half && c->gru_persist && gru_tc_persist_supported(H);
        if (wave) {
            wave_pw[2 * l] = pw;
            if (l == 1) {
                Op op{};
                op.kind = OP_GRU_WAVE;
                op.stage = ST_GRU;
                op.rows_per_stream = 1;
                op.gw = GruWaveParams{};
                op.gw.Kp = pw.K;
                op.gw.gi0 = c->gi_l[0];
                op.gw.giB = (long long)T * 3 * H;
                op.gw.hseq0 = reinterpret_cast<__half*>(c->hseq[0]);
                op.gw.hseq1 = reinterpret_cast<__half*>(c->hseq[1]);
                op.gw.hB = (long long)(T + 1) * H;
                op.gw.h32_0 = c->h32[0];
                op.gw.h32_1 = c->h32[1];
                op.gw.H = H;
                op.gw.T = T;
                op.gw.layers = 2;
                // W_hh0, W_ih1, W_hh1; gi0 (fp32) read; h0 history written, read by both layers; h1 written + read (fp16)
                b.meta("gru.l0+l1.recurrence(wavefront)", 2.0 * T * 3 * H * H * 3, 22.0 * T * H, 1);
                b.push(op, [=](Op& o) {
                    const WeightArena& wa = c->wa;
                    o.gw.Whh0 = wa.wh + wave_pw[0].w_off;
                    o.gw.bhh0 = wa.w + wave_pw[0].b_off;
                    o.gw.Wih1 = wa.wh + wave_pw[1].w_off;
                    o.gw.bih1 = wa.w + wave_pw[1].b_off;
                    o.gw.Whh1 = wa.wh + wave_pw[2].w_off;
                    o.gw.bhh1 = wa.w + wave_pw[2].b_off;
                    o.gw.cstride = (c->maxB + 127) / 128;
                    o.gw.counters = c->gru_counters;
                    return make_gru_wave_maps(&o.gw, c->maxB);
                });
            }
            continue;
        }
        if (persist) {  // the whole recurrence of the layer: one persistent tensor-core kernel (gru_tc_persist.cu)
            Op op{};
            op.stage = ST_GRU;
            op.rows_per_stream = 1;
            op.gru_layer = l;
            b.meta("gru.l" + s + ".recurrence", 2.0 * T * 3 * H * H, 4.0 * T * (3 * H + 2 * H), 1);
            if (c->gru_wave == 2 && gru_wave_supported(H, 1)) {  // H too large for the wavefront: its one-layer form (measured
                                                               // 151 us vs 146 us per layer at H = 512: opt-in)
                op.kind = OP_GRU_WAVE;
                op.gw = GruWaveParams{};
                op.gw.Kp = pw.K;
                op.gw.gi0 = c->gi_l[l];
                op.gw.giB = (long long)T * 3 * H;
                op.gw.hseq0 = reinterpret_cast<__half*>(c->hseq[l]);
                op.gw.hB = (long long)(T + 1) * H;
                op.gw.h32_0 = c->h32[l];
                op.gw.H = H;
                op.gw.T = T;
                op.gw.layers = 1;
                b.push(op, [=](Op& o) {
                    o.gw.Whh0 = c->wa.wh + pw.w_off;
                    o.gw.bhh0 = c->wa.w + pw.b_off;
                    o.gw.cstride = (c->maxB + 127) / 128;
                    o.gw.counters = c->gru_counters + (size_t)l * o.gw.cstride;
                    return make_gru_wave_maps(&o.gw, c->maxB);
                });
                continue;
            }
            op.kind = OP_GRU_TC;
            op.gt = GruTcParams{};
            op.gt.Kp = pw.K;
            op.gt.gi = c->gi_l[l];
            op.gt.giB = (long long)T * 3 * H;
            op.gt.hseq = reinterpret_cast<__half*>(c->hseq[l]);
            op.gt.hB = (long long)(T + 1) * H;
            op.gt.h32 = c->h32[l];
            op.gt.H = H;
            op.gt.T = T;
            b.push(op, [=](Op& o) {
                o.gt.Whh = c->wa.wh + pw.w_off;
                o.gt.bhh = c->wa.w + pw.b_off;
                o.gt.counters = c->gru_counters + (size_t)l * ((c->maxB + 127) / 128);
                return 0;
            });
        }
        for (int t = 0; t < T && fused && !persist; ++t) {
            GemmParams gp{};
            gp.A = c->E(c->hseq[l], (long long)t * H);
            gp.sB = (long long)(T + 1) * H;
            gp.Tn = 1;
            gp.Fo = 1;
            fill_gemm_common(c, gp, pw, 3 * H);
            gp.epi = EPI_GRU;
            gp.gi = c->gi_l[l] + (long long)t * 3 * H;
            gp.giB = (long long)T * 3 * H;
            if (c->half) {  // fp32 master state updated in place + fp16 history = operand of the following GEMMs
                gp.hprev = c->h32[l];
                gp.hB = H;
                gp.out = c->h32[l];
                gp.oB = H;
                gp.out_h2 = c->E(c->hseq[l], (long long)(t + 1) * H);
                gp.o2B = (long long)(T + 1) * H;
            } else {
                gp.out = c->hseq[l] + (long long)(t + 1) * H;
                gp.oB = (long long)(T + 1) * H;
                gp.hprev = c->hseq[l] + (long long)t * H;
                gp.hB = (long long)(T + 1) * H;
            }
            gp.H = H;
            b.meta("gru.l" + s + ".step" + std::to_string(t), 2.0 * 3 * H * H, 4.0 * (3 * H + 2 * H), 1);
            b.push_gemm(ST_GRU, gp, 1, pw, k_off);
        }
        const bool seq = c->train && gru_seq_supported(H);
        if (seq) {  // training: the whole recurrence of the layer is one persistent kernel (gru_seq.cu)
            GemmParams gp{};  // describes W_hh for the backward's batched recompute / weight gradient
            gp.A = c->hseq[l];
            gp.sB = (long long)(T + 1) * H;
            gp.Tn = 1;
            gp.Fo = 1;
            fill_gemm_common(c, gp, pw, 3 * H);
            gp.epi = EPI_BIAS;
            gp.out = c->gh;
            gp.oB = 3 * H;
            b.meta("gru.l" + s + ".recurrence", 2.0 * T * 3 * H * H, 4.0 * T * (3 * H + 2 * H));
            c->gru_rec.op_hh[l] = b.push_gemm(ST_GRU, gp, 1, pw, k_off, {}, NONE, NONE, OP_GRU_SEQ);
            c->ops.back().gru_layer = l;
        }
        for (int t = 0; t < T && !fused && !seq; ++t) {
            GemmParams gp{};
            gp.A = c->hseq[l] + (long long)t * H;
            gp.sB = (long long)(T + 1) * H;
            gp.sT = 0;
            gp.sF = 0;
            gp.Tn = 1;
            gp.Fo = 1;
            fill_gemm_common(c, gp, pw, 3 * H);
            gp.epi = EPI_BIAS;
            gp.out = c->gh;
            gp.oB = 3 * H;
            gp.oT = 0;
            gp.oF = 0;
            b.meta("gru.l" + s + ".step" + std::to_string(t) + ".hh", 2.0 * 3 * H * H, 4.0 * (H + 3 * H), 1);
            const int i = b.push_gemm(ST_GRU, gp, 1, pw, k_off);
            if (t == 0) c->gru_rec.op_hh[l] = i;
            c->ops.back().chunk_serial = 1;
            c->ops.back().gru_layer = l;
            b.meta("gru.l" + s + ".step" + std::to_string(t) + ".cell", 0, 4.0 * (6 * H + 2 * H), 1);
            b.push_gru_pw(c->gi_l[l] + (long long)t * 3 * H, (long long)T * 3 * H, c->gh, c->hseq[l] + (long long)t * H,
                          (long long)(T + 1) * H, c->hseq[l] + (long long)(t + 1) * H, H);
            c->ops.back().chunk_serial = 1;
            c->ops.back().gru_layer = l;
        }
    }
    {  // fc + ELU + stats, then per-feature GLN into the first decoder input
        const int k_off = b.koff_dense(H);
        PackedW pw = reserve_packed(c, feat, H);
        c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
            const std::vector<float>& w = hp.at("gru.fc_output_layer.weight");
            const std::vector<float>& bb = hp.at("gru.fc_output_layer.bias");
            for (int n = 0; n < feat; ++n) {
                const int r = perm(n);
                for (int k = 0; k < H; ++k) arena[pw.w_off + (size_t)n * pw.K + k] = w[(size_t)r * H + k];
                arena[pw.b_off + n] = bb[r];
            }
        });
        GemmParams gp{};
        gp.A = c->E(c->hseq[1], H);
        gp.sB = (long long)(T + 1) * H;
        gp.sT = H;
        gp.sF = 0;
        gp.Tn = T;
        gp.Fo = 1;
        fill_gemm_common(c, gp, pw, feat);
        gp.epi = EPI_ELU_STATS;
        gp.out = c->fcraw;
        gp.oB = (long long)T * feat;
        gp.oT = feat;
        gp.oF = 0;
        gp.stats = c->stats + (size_t)gru_slot * 2 * maxB;
        gp.vec4 = 1;
        gp.out_half = c->half ? 1 : 0;
        b.meta("gru.fc+elu", 2.0 * T * feat * H, 4.0 * T * (H + feat));
        c->gru_rec.op_fc =
            b.push_gemm(ST_GRU, gp, T, pw, k_off, TmaSrc{c->hseq[1], H, 1, T + 1, H, (long long)(T + 1) * H, 1, 1, 0});

        const Act& nx = c->dec_in[0];
        NormApplyParams n{};
        n.mode = 0;
        n.T = T;
        n.F = Fg;
        n.C = Cg;
        n.student = c->student;
        n.y = c->fcraw;
        n.Fy = Fg;
        n.stats = gp.stats;
        n.count = (double)feat * T;
        n.per_feature = 1;
        n.out = nx.interior();
        n.oB = nx.sB;
        n.oT = nx.sT;
        n.oF = nx.sF;
        const size_t w_off = c->wa.reserve_w(feat), b_off = c->wa.reserve_w(feat);
        c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
            const std::vector<float>& w = hp.at("gru.norm.weight");
            const std::vector<float>& bb = hp.at("gru.norm.bias");
            for (int n2 = 0; n2 < feat; ++n2) {
                arena[w_off + n2] = w[perm(n2)];
                arena[b_off + n2] = bb[perm(n2)];
            }
        });
        b.meta("gru.gln", 0, 8.0 * T * feat);
        c->gru_rec.op_norm = b.push_norm(ST_GRU, n, w_off, b_off);
    }
    // ---- decoder ----------------------------------------------------------------------------------------------
    size_t wl_off = NONE, bl_off = NONE;
    for (int j = 0; j < c->L; ++j) {
        const Act& in = c->dec_in[j];
        const int Cin = g.num_channels[c->L - 1 - j];
        const std::string name = "deconvlist." + std::to_string(j);
        if (j + 1 < c->L) {
            const int Co = g.num_channels[c->L - 2 - j];
            const Act* skip = &c->enc_in[c->L - 1 - j];  // interior = output of encoder level L-2-j
            const Act& nx = c->dec_in[j + 1];
            const int s0 = slot++, s1 = slot++;
            b.deconv_block(name, in, Cin, Co, 3, 1 << j, skip, nx.interior(), nx.sB, nx.sT, nx.sF, s0, s1,
                           c->train ? nx.dinterior() : nullptr);
        } else {
            c->stats_last = slot++;
            b.deconv_block(name, in, Cin, 2, 3, 1 << j, nullptr, nullptr, 0, 0, 0, c->stats_last, -1);
            wl_off = b.pack_affine(name + ".norm.weight", 2, 4);
            bl_off = b.pack_affine(name + ".norm.bias", 2, 4);
        }
    }
    SE_REQUIRE(slot <= c->n_stats, "internal: statistics slots");
    SE_REQUIRE(!c->alloc_failed, "out of device memory while allocating the per-layer training buffers");

    // ---- arenas -------------------------------------------------------------------------------------------------
    c->wa.half = c->half;
    if (c->wa.allocate(c->allocs)) return 1;
    c->w_last = c->wa.w + wl_off;
    c->b_last = c->wa.w + bl_off;
    if (c->train) {
        // position map of the packed arena: run the packers on index-coded parameters (value = 1 + flat index; every
        // packer only copies values, and 6.2 M indices are exact in fp32)
        if (dev_alloc(c, &c->garena, c->wa.floats)) return 1;
        if (dev_alloc(c, &c->wmap, c->wa.floats)) return 1;
        HostParams hp;
        int64_t off = 0;
        for (const ParamInfo& pi : c->wa.params) {
            c->param_off.push_back(off);
            std::vector<float> v((size_t)pi.numel());
            for (size_t i = 0; i < v.size(); ++i) v[i] = (float)(off + (int64_t)i + 1);
            hp.emplace(pi.name, std::move(v));
            off += pi.numel();
        }
        c->n_theta = off;
        SE_REQUIRE(off < (1 << 24), "internal: parameter count exceeds the exact-integer range of the index coding");
        const std::vector<float> arena = c->wa.pack(hp);
        std::vector<int> map(arena.size());
        for (size_t i = 0; i < arena.size(); ++i) map[i] = (int)arena[i];
        SE_CUDA_OK(cudaMemcpy(c->wmap, map.data(), map.size() * sizeof(int), cudaMemcpyHostToDevice));
    }

    // ---- state tables -------------------------------------------------------------------------------------------
    auto add_state = [&](float* base, long long sB, long long src, int count) {
        RollEntry e{base, sB, src, 0, count};
        c->roll.e[c->roll.n++] = e;
        c->zero_tab.e[c->zero_tab.n++] = e;
        c->roll_floats += count;
    };
    if (c->train)
        for (const Act& a : c->pre_act) add_state(a.base, a.sB, (long long)T * a.sT, (int)(a.padT0 * a.sT));
    if (c->front_mma) {  // rolled by the kernel itself; the borders of the feature buffer are never written
        RollEntry e{reinterpret_cast<float*>(c->pre_state), pre_state_sB / 2, 0, 0, (int)(pre_state_sB / 2)};
        c->zero_tab.e[c->zero_tab.n++] = e;
    }
    for (int i = 0; i < 3 && c->preconv_tc && !c->front_mma; ++i) {  // rolled by the kernel itself; a reset clears the whole slab
        RollEntry e{reinterpret_cast<float*>(c->pre_h[i]), pre_h_sB / 2, 0, 0, (int)(pre_h_sB / 2)};
        c->zero_tab.e[c->zero_tab.n++] = e;
    }
    for (const PreBuf& pb : c->pre_in) {  // rolled by the preconv kernel itself; a reset clears the whole slab
        RollEntry e{pb.base, pb.sB, 0, 0, (int)pb.sB};
        c->zero_tab.e[c->zero_tab.n++] = e;
    }
    const int fpe = 4 / c->esz;  // operand elements per float: the roll / zero kernels move 4-byte units
    for (const Act& a : c->enc_in)
        add_state(a.base, a.sB / fpe, (long long)T * a.sT / fpe, (int)(a.padT0 * a.sT / fpe));
    for (int l = 0; l < 2; ++l) add_state(c->hseq[l], (long long)(T + 1) * H / fpe, (long long)T * H / fpe, H / fpe);
    if (c->half)
        for (int l = 0; l < 2; ++l) {
            RollEntry e{c->h32[l], H, 0, 0, H};
            c->zero_tab.e[c->zero_tab.n++] = e;
        }
    {
        RollEntry e{c->carry, PHOP, 0, 0, PHOP};
        c->zero_tab.e[c->zero_tab.n++] = e;
    }
    if (c->train) {
        SE_REQUIRE(c->roll.n == 3 + c->L + 2, "internal: training state table");
        for (int e = 0; e < c->roll.n; ++e) {
            float* p = nullptr;
            if (dev_alloc(c, &p, (size_t)c->roll.e[e].count * maxB)) return 1;
            c->carry_store.push_back(p);
        }
    }
    // export / import: exactly what the next step reads, where it sits between steps.  The front kernels roll their own
    // inputs when they load them (frames 21..24 -> 0..3), launch_roll moves the other entries at the end of the step, so
    // between steps every carried frame is a LEADING frame and slot 0 of hseq is h_T.
    if (!c->train) {
        StateTable& t = c->state_tab;
        t.desc = "crn variant=" + std::to_string(g.variant) + " precision=" + std::to_string(g.precision) +
                 " inputs=" + std::to_string(g.num_inputs) + " freqs=" + std::to_string(g.num_freqs) + " channels=";
        for (int i = 0; i < c->L; ++i) t.desc += std::to_string(g.num_channels[i]) + ",";
        t.desc += " hidden=" + std::to_string(g.hidden) + " layers=" + std::to_string(g.num_layers) + " kernel=" +
                  std::to_string(g.kernel_size) + " segment=" + std::to_string(g.segment_length) + " front=" +
                  (c->front_mma ? "mma" : c->preconv_tc ? "tc" : "planar") + " half=" + std::to_string(c->half);
        if (c->front_mma) {  // [3 layers][4 frames][224 positions][8 halves]: all of it is carried
            if (state_table_add(t, "pre_state", 2, c->pre_state, pre_state_sB * 2, pre_state_sB * 2)) return 1;
        }
        for (int i = 0; i < 3 && c->preconv_tc && !c->front_mma; ++i)  // frames 0..3 of [25][272][8] halves
            if (state_table_add(t, "pre_h" + std::to_string(i), 2, c->pre_h[i], pre_h_sB * 2,
                                4LL * PRECONV_TC_POS * 8 * 2))
                return 1;
        for (int i = 0; i < (int)c->pre_in.size(); ++i) {  // frames 0..3 of each of the 5 channel planes [25][Fpp]
            const PreBuf& pb = c->pre_in[i];
            if (state_table_add(t, "pre_in" + std::to_string(i), 4, pb.base, pb.sB * 4, 4LL * pb.Fpp * 4, 5, pb.sC * 4))
                return 1;
        }
        for (int i = 0; i < 2 * c->L; ++i) {  // the decoder inputs have no leading frames (padT0 = 0): look-ahead only
            const Act& a = i < c->L ? c->enc_in[i] : c->dec_in[i - c->L];
            if (a.padT0 > 0 && state_table_add(t, (i < c->L ? "enc_in" : "dec_in") + std::to_string(i % c->L), c->esz,
                                               a.base, a.sB * c->esz, a.padT0 * a.sT * c->esz))
                return 1;
        }
        for (int l = 0; l < 2; ++l)
            if (state_table_add(t, "hseq" + std::to_string(l), c->esz, c->hseq[l], (long long)(T + 1) * H * c->esz,
                                (long long)H * c->esz))
                return 1;
        for (int l = 0; l < 2 && c->half; ++l)  // the fp32 master copy the fp16 recurrence continues from
            if (state_table_add(t, "h32_" + std::to_string(l), 4, c->h32[l], (long long)H * 4, (long long)H * 4)) return 1;
        if (state_table_add(t, "carry", 4, c->carry, PHOP * 4, PHOP * 4)) return 1;
        c->state_layout = state_layout_hash(t);
    }
    if (init_fft_tables()) return 1;
    return 0;
}

int run_gemm_impl(const se_ctx* c, const GemmParams& g, int stage, const std::string& label, cudaStream_t st);
// SE_B200_SYNC=1 (debug): synchronise after every GEMM launch and report the op that faulted
int run_gemm(const se_ctx* c, const GemmParams& g, int stage, const std::string& label, cudaStream_t st) {
    static const bool sync = getenv("SE_B200_SYNC") != nullptr;
    if (run_gemm_impl(c, g, stage, label, st)) return 1;
    if (sync) {
        const cudaError_t e = cudaStreamSynchronize(st);
        SE_REQUIRE(e == cudaSuccess, "GEMM '" + label + "' (M=" + std::to_string(g.M) + " N=" + std::to_string(g.N) +
                                         " K=" + std::to_string(g.K) + " epi=" + std::to_string(g.epi) +
                                         ") failed: " + cudaGetErrorString(e));
    }
    return 0;
}
int run_gemm_impl(const se_ctx* c, const GemmParams& g, int stage, const std::string& label, cudaStream_t st) {
    if (g.epi == EPI_GRU || g.epi == EPI_ELU_GATE) return launch_gemm_tf32(g, st, c->split);
    if (c->tf32 && (c->half || ((c->tc_mask >> stage) & 1u)) && gemm_tf32_supported(g))
        return launch_gemm_tf32(g, st, c->split);
    SE_REQUIRE(!c->half, "internal: fp16 operands need the tensor-core GEMM (" + label + ")");
    return launch_gemm_fp32(g, st);
}

// s0: first stream of the launch (training forward runs the recurrent ops chunk by chunk on a slice of the batch)
int launch_op(const se_ctx* c, const Op& op, int B, cudaStream_t st, int s0 = 0) {
    switch (op.kind) {
        case OP_GEMM: {
            GemmParams g = op.g;
            g.M = B * op.rows_per_stream;
            if (s0) {
                SE_REQUIRE(!g.a_half && !g.out_half, "internal: stream-offset launches are fp32 only");
                g.A = reinterpret_cast<const float*>(g.A) + (long long)s0 * g.sB;
                g.out += (long long)s0 * g.oB;
                if (g.out2) g.out2 += (long long)s0 * g.o2B;
                if (g.gi) g.gi += (long long)s0 * g.giB;
                if (g.hprev) g.hprev += (long long)s0 * g.hB;
                g.b0 = s0;
                // per-chunk recurrent GEMMs have a handful of rows: CUDA-core kernel (the tensor-core kernel's scalar
                // store path needs 16-byte aligned rows, which a 1-row slice of the shared gh buffer does not guarantee)
                return launch_gemm_fp32(g, st);
            }
            if (op.chunk_serial) return launch_gemm_fp32(g, st);
            if (op.tma_ok) return launch_gemm_tma(g, op.tma, st);
            return run_gemm(c, g, op.stage, op.label, st);
        }
        case OP_NORM: {
            NormApplyParams n = op.n;
            n.B = B;
            return launch_norm_apply(n, st);
        }
        case OP_PRECONV: {
            PreconvParams pc = op.pc;
            pc.b0 = 0;
            pc.B = B;
            return launch_preconv(pc, st);
        }
        case OP_PRECONV_TC: {
            PreconvTcParams pt = op.pt;
            pt.b0 = 0;
            pt.B = B;
            return launch_preconv_tc(pt, st);
        }
        case OP_PRECONV3: {
            Preconv3Params p3 = op.p3;
            p3.b0 = 0;
            p3.B = B;
            return launch_preconv3(p3, st);
        }
        case OP_ENC_MMA: {
            EncMmaParams em = op.em;
            em.b0 = 0;
            em.B = B;
            return launch_enc_mma(em, op.em_cin, op.em_cout, st);
        }
        case OP_ENC_TC: {
            EncMmaParams em = op.em;
            em.b0 = 0;
            em.B = B;
            return launch_enc_tc(em, op.em_cin, op.em_cout, st);
        }
        case OP_DEC_MMA: {
            DecMmaParams dm = op.dm;
            dm.b0 = 0;
            dm.B = B;
            return launch_dec_mma(dm, op.em_cin, op.em_cout, st);
        }
        case OP_SKIP_BLEND: {
            SkipBlendParams sb = op.sb;
            sb.B = B;
            return launch_skip_blend(sb, op.em_cout, st);
        }
        case OP_GRU_WAVE: {
            GruWaveParams gw = op.gw;
            gw.B = B;
            gw.b0 = 0;
            return launch_gru_wave(gw, st);
        }
        case OP_GRU_TC: {
            GruTcParams gt = op.gt;
            gt.B = B;
            return launch_gru_tc_persist(gt, st);
        }
        case OP_DECONV_LAST: {
            DeconvLastParams dl = op.dl;
            dl.B = B;
            return launch_deconv_last(dl, op.small_c, st);
        }
        case OP_SKIP_SMALL: {
            SkipSmallParams sk = op.sk;
            sk.B = B;
            return launch_skip_small(sk, op.small_c, st);
        }
        case OP_GRU_SEQ:
            SE_REQUIRE(false, "internal: the persistent GRU op only runs inside the training forward");
        case OP_GRU_PW:
            return launch_gru_pointwise(op.gi + (long long)s0 * op.giB, op.giB, op.gh + (long long)s0 * 3 * op.H,
                                        op.hprev + (long long)s0 * op.hB, op.hB, op.hout + (long long)s0 * op.hB, B, op.H,
                                        st);
    }
    return 0;
}

// stage_filter < 0: everything
int enqueue_net(se_ctx* c, int B, cudaStream_t st, int stage_filter) {
    for (const Op& op : c->ops) {
        if (stage_filter >= 0 && op.stage != stage_filter) continue;
        if (launch_op(c, op, B, st)) return 1;
    }
    return 0;
}

int enqueue_stream_step(se_ctx* c, int B, cudaStream_t st, int stage_filter = -1) {
    auto want = [&](int s) { return stage_filter < 0 || stage_filter == s; };
    if (want(ST_STFT)) {
        SE_CUDA_OK(cudaMemsetAsync(c->stats, 0, (size_t)c->n_stats * 2 * c->maxB * sizeof(double), st));
        StftParams sp{};
        sp.io = c->io_dev;
        sp.B = B;
        sp.M = 3;
        sp.student = c->student;
        if (c->front_mma) {
            sp.feat_h8 = c->feat_h + PRECONV3_BORDER * 8;  // frame 0, bin 0
            sp.fB = (long long)T * PRECONV3_POS * 8;
            sp.fT = (long long)PRECONV3_POS * 8;
            sp.fF = 8;
        } else if (c->preconv_tc) {
            sp.feat_h8 = c->pre_h[0] + (4LL * PRECONV_TC_POS + 2) * 8;  // frame 4, bin 0 (dilation 1: position 2)
            sp.fB = (long long)PRECONV_TP * PRECONV_TC_POS * 8;
            sp.fT = (long long)PRECONV_TC_POS * 8;
            sp.fF = 8;
        } else {
            const PreBuf& a = c->pre_in[0];
            sp.feat = a.interior();
            sp.fB = a.sB;
            sp.fC = a.sC;
            sp.fT = a.Fpp;
            sp.fF = 1;
        }
        sp.noisy = c->noisy;
        if (launch_stft_features(sp, st)) return 1;
    }
    if (enqueue_net(c, B, st, stage_filter)) return 1;
    if (want(ST_MASK)) {
        MaskIstftParams mp{};
        mp.io = c->io_dev;
        mp.B = B;
        mp.student = c->student;
        mp.y = c->ylast;
        mp.stats = c->stats + (size_t)c->stats_last * 2 * c->maxB;
        mp.count = 2.0 * NBIN * T;
        mp.w = c->w_last;
        mp.b = c->b_last;
        mp.noisy = c->noisy;
        mp.carry = c->carry;
        mp.fast = (c->half || c->tf32) && !c->split ? 1 : 0;  // 3xtf32 keeps the exact cIRM decompression
        if (launch_mask_istft(mp, st)) return 1;
    }
    if (want(ST_ROLL)) {
        if (launch_roll(c->roll, 0, B, st)) return 1;
    }
    return 0;
}

// kernels of one chunk step, in launch order: 0 = STFT + features, 1..n = network ops, n+1 = mask + iSTFT + OLA, n+2 = roll
int num_kernels(const se_ctx* c) { return (int)c->ops.size() + 3; }

int enqueue_kernel(se_ctx* c, int idx, int B, cudaStream_t st) {
    const int n = (int)c->ops.size();
    if (idx == 0) return enqueue_stream_step(c, B, st, ST_STFT);
    if (idx <= n) return launch_op(c, c->ops[idx - 1], B, st);
    if (idx == n + 1) return enqueue_stream_step(c, B, st, ST_MASK);
    return enqueue_stream_step(c, B, st, ST_ROLL);
}

int count_launches(const se_ctx* c) {
    // memset + stft + ops + mask + roll
    return 1 + 1 + (int)c->ops.size() + 1 + 1;
}

int run_stream_step(se_ctx* c, const IoDesc& io, int B, cudaStream_t st) {
    if (launch_set_io(c->io_dev, io, st)) return 1;
    if (!c->use_graph) return enqueue_stream_step(c, B, st);
    return replay_graph(c->graphs, &c->own_stream, B, [=](cudaStream_t s) { return enqueue_stream_step(c, B, s); }, st);
}

int check_ready(se_ctx* c, int B, bool want_train = false) {
    SE_REQUIRE(c != nullptr, "null context");
    SE_REQUIRE(c->train == want_train, want_train ? "this entry point needs a context created with training = 1"
                                                  : "training context: use the se_crn_train_* entry points");
    SE_REQUIRE(c->wa.bound, "se_crn_bind_weights has not been called");
    SE_REQUIRE(B >= 0 && B <= c->maxB, "B exceeds max_streams of the context");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return 0;
}


// ======================================================================================================================
// training micro-step (train.py:195-198).  Batch layout: stream s = n * nb + i is chunk n of utterance i ("chunk-major").
// The convolutional layers and all batched GEMMs run once over all N * nb chunk-streams: the carried frames of chunk n
// are the trailing frames of chunk n-1's block input (CRN_ELU.py:243), copied in front of the op that consumes them.
// Only the GRU recurrence is serial over chunks (its hidden state crosses chunk boundaries, CRN_ELU.py:173,185).
// ======================================================================================================================
int train_forward(se_ctx* c, const float* mixture, int nb, long long L, int flag, float* pred, cudaStream_t st) {
    const int front = flag ? 0 : PHOP;  // CRN_ELU.py:474-476
    int gap = 0, N = 0;
    se_chunk_grid(L + front, KCHUNK, &gap, &N);
    const int Bp = N * nb;
    SE_REQUIRE(Bp <= c->maxB, "se_crn_train_forward: chunks * utterances = " + std::to_string(Bp) +
                                  " exceeds max_streams = " + std::to_string(c->maxB) + " of the training context");
    SE_REQUIRE(!flag || (c->t_have_fwd && c->t_nb == nb), "se_crn_train_forward: flag=1 needs a previous piece of the same batch");
    c->t_nb = nb;
    c->t_N = N;
    c->t_L = L;
    c->t_front = front;
    SE_CUDA_OK(cudaMemsetAsync(c->stats, 0, (size_t)c->n_stats * 2 * c->maxB * sizeof(double), st));
    // chunk 0: zero state (CRN_ELU.py:480-481) or the state carried from the previous piece (flag=True)
    for (int e = 0; e < c->roll.n; ++e) {
        const RollEntry& r = c->roll.e[e];
        if (launch_copy_rows(r.base + r.dst_off, r.sB, flag ? c->carry_store[e] : nullptr, r.count, r.count, nb, st)) return 1;
    }
    IoDesc io{mixture, 3 * L, L, -(long long)PHOP - front, L, nullptr, 0, 0};
    if (launch_set_io(c->io_dev, io, st)) return 1;
    {
        StftParams sp{};
        sp.io = c->io_dev;
        sp.B = Bp;
        sp.M = 3;
        sp.student = c->student;
        const Act& a = c->pre_act[0];
        sp.feat = a.interior();
        sp.fB = a.sB;
        sp.fC = 1;
        sp.fT = a.sT;
        sp.fF = a.sF;
        sp.noisy = c->noisy;
        sp.nb = nb;
        sp.hop_chunk = PHOP;
        if (launch_stft_features(sp, st)) return 1;
    }
    auto shift_state = [&](int e) -> int {  // chunk n (n >= 1) <- trailing frames of chunk n-1
        const RollEntry& r = c->roll.e[e];
        return launch_copy_rows(r.base + (long long)nb * r.sB + r.dst_off, r.sB, r.base + r.src_off, r.sB, r.count,
                                Bp - nb, st);
    };
    for (size_t i = 0; i < c->ops.size();) {
        const Op& op = c->ops[i];
        if (op.chunk_serial) {
            size_t j = i;
            while (j < c->ops.size() && c->ops[j].chunk_serial && c->ops[j].gru_layer == op.gru_layer) ++j;
            const RollEntry& r = c->roll.e[3 + c->L + op.gru_layer];
            for (int n = 0; n < N; ++n) {
                if (n > 0 && launch_copy_rows(r.base + (long long)n * nb * r.sB + r.dst_off, r.sB,
                                              r.base + (long long)(n - 1) * nb * r.sB + r.src_off, r.sB, r.count, nb, st))
                    return 1;
                for (size_t k = i; k < j; ++k)
                    if (launch_op(c, c->ops[k], nb, st, n * nb)) return 1;
            }
            i = j;
            continue;
        }
        // Two GRU layers as a pipeline over chunk groups: layer 0 walks group g + 1 while the second branch runs the
        // layer-1 input projection and recurrence of group g (each sequence kernel occupies one cluster = 16 SMs, the
        // serial chain is what costs).  Streams are chunk-major, so a chunk group is a contiguous range of GEMM rows.
        if (op.kind == OP_GRU_SEQ && op.gru_layer == 0 && c->gru_pipe && c->pipe_stream && N >= 4 && i + 2 < c->ops.size() &&
            c->ops[i + 1].kind == OP_GEMM && !c->ops[i + 1].chunk_serial && c->ops[i + 1].state_entry < 0 &&
            !c->ops[i + 1].g.a_half && !c->ops[i + 1].g.out_half && c->ops[i + 2].kind == OP_GRU_SEQ &&
            c->ops[i + 2].gru_layer == 1) {
            const Op& proj = c->ops[i + 1];
            const Op& op1 = c->ops[i + 2];
            const int groups = N >= 16 ? 8 : N >= 8 ? 4 : 2;
            auto seq_params = [&](const Op& o, int n0, int n1) {
                GruSeqParams gp{};
                gp.Whh = reinterpret_cast<const float*>(o.g.W);
                gp.Kp = o.g.K;
                gp.bhh = o.g.bias;
                gp.gi = c->gi_l[o.gru_layer];
                gp.giB = (long long)T * 3 * c->H;
                gp.hseq = c->hseq[o.gru_layer];
                gp.hB = (long long)(T + 1) * c->H;
                gp.H = c->H;
                gp.T = T;
                gp.nb = nb;
                gp.N = n1 - n0;
                gp.n0 = n0;
                return gp;
            };
            for (int gidx = 0; gidx < groups; ++gidx) {
                const int n0 = (int)((long long)N * gidx / groups), n1 = (int)((long long)N * (gidx + 1) / groups);
                if (launch_gru_seq_fwd(seq_params(op, n0, n1), st)) return 1;
                SE_CUDA_OK(cudaEventRecord(c->pipe_ev[gidx], st));
                SE_CUDA_OK(cudaStreamWaitEvent(c->pipe_stream, c->pipe_ev[gidx], 0));
                GemmParams g = proj.g;  // rows of the chunk group (whole streams: the tensor-core path keeps its alignment)
                const int s0 = n0 * nb;
                g.M = (n1 - n0) * nb * proj.rows_per_stream;
                // the tensor-core kernel addresses rows as stream b0 + m / rows_per_stream itself; the CUDA-core kernel
                // starts at the pointers it is given
                const bool tc = c->tf32 && ((c->tc_mask >> proj.stage) & 1u) && gemm_tf32_supported(g);
                if (tc) {
                    g.b0 = s0;
                    if (launch_gemm_tf32(g, c->pipe_stream, c->split)) return 1;
                } else {
                    g.A = reinterpret_cast<const float*>(g.A) + (long long)s0 * g.sB;
                    g.out += (long long)s0 * g.oB;
                    if (g.out2) g.out2 += (long long)s0 * g.o2B;
                    if (launch_gemm_fp32(g, c->pipe_stream)) return 1;
                }
                if (launch_gru_seq_fwd(seq_params(op1, n0, n1), c->pipe_stream)) return 1;
            }
            SE_CUDA_OK(cudaEventRecord(c->pipe_ev[16], c->pipe_stream));
            SE_CUDA_OK(cudaStreamWaitEvent(st, c->pipe_ev[16], 0));
            i += 3;
            continue;
        }
        if (op.kind == OP_GRU_SEQ) {
            GruSeqParams gp{};
            gp.Whh = reinterpret_cast<const float*>(op.g.W);
            gp.Kp = op.g.K;
            gp.bhh = op.g.bias;
            gp.gi = c->gi_l[op.gru_layer];
            gp.giB = (long long)T * 3 * c->H;
            gp.hseq = c->hseq[op.gru_layer];
            gp.hB = (long long)(T + 1) * c->H;
            gp.H = c->H;
            gp.T = T;
            gp.nb = nb;
            gp.N = N;
            if (launch_gru_seq_fwd(gp, st)) return 1;
            ++i;
            continue;
        }
        if (op.state_entry >= 0 && N > 1 && shift_state(op.state_entry)) return 1;
        if (launch_op(c, op, Bp, st)) return 1;
        ++i;
    }
    {
        MaskIstftParams mp{};
        mp.B = Bp;
        mp.student = c->student;
        mp.y = c->ylast;
        mp.stats = c->stats + (size_t)c->stats_last * 2 * c->maxB;
        mp.count = 2.0 * NBIN * T;
        mp.w = c->w_last;
        mp.b = c->b_last;
        mp.noisy = c->noisy;
        mp.out_chunk = c->chunks;
        if (launch_mask_istft(mp, st)) return 1;
    }
    if (launch_over_add_cm(c->chunks, nb, N, KCHUNK, front, L, pred, st)) return 1;
    // state carried to a following flag=True piece: trailing frames / last hidden state of the last chunk
    for (int e = 0; e < c->roll.n; ++e) {
        const RollEntry& r = c->roll.e[e];
        if (launch_copy_rows(c->carry_store[e], r.count, r.base + (long long)(N - 1) * nb * r.sB + r.src_off, r.sB, r.count,
                             nb, st))
            return 1;
    }
    c->t_have_fwd = true;
    return 0;
}

// ---- distillation feature taps (distillation_crn.py:343-377) -------------------------------------------------------
// The reference returns the PRE-activation outputs of the last encoder conv (TemporalConv2d: `feature = self.net(inp)`,
// distillation_crn.py:198), of the GRU's Linear (`feature = o`, :140) and of the L-1 gated-skip transposed convs
// (`feature = out`, :253).  The forward keeps only the activated tensors, so a tap is recomputed on demand by re-running
// the layer's own GEMM over its saved input with the bias-only epilogue: same operands, same arithmetic, no extra
// stores in the training step that does not ask for taps.  The same five points accept an injected gradient in
// train_backward (the distillation loss's d loss / d tap).
struct Tap {
    const Op* op = nullptr;
    int C = 0, Cp = 0, F = 0;
    bool fc = false;
};
int tap_of(const se_ctx* c, int k, Tap& t) {
    SE_REQUIRE(c->train, "feature taps need a context created with training = 1");
    SE_REQUIRE(k >= 0 && k <= c->L, "feature tap index out of range (0 .. num_levels)");
    if (k == 0) {
        const ConvRec& r = c->conv_recs.back();
        t.op = &c->ops[r.op_conv];
        t.C = t.op->g.N;
        t.Cp = r.Cp_out;
        t.F = r.Fo;
    } else if (k == 1) {
        t.op = &c->ops[c->gru_rec.op_fc];
        t.C = t.Cp = c->Cg;
        t.F = c->Fg;
        t.fc = true;
    } else {
        const DeconvRec& r = c->deconv_recs[k - 2];
        t.op = &c->ops[r.op_deconv];
        t.C = t.op->g.N / 2;
        t.Cp = r.Cop;
        t.F = r.Fy;
    }
    return 0;
}
Strides4 tap_ours(const Tap& t) {  // channels-last [Bp][T][F][Cp]
    return Strides4{(long long)T * t.F * t.Cp, (long long)t.F * t.Cp, t.Cp, 1};
}
Strides4 tap_theirs(const Tap& t) {
    // [Bp][C][F][T]; the GRU tap is the Linear's [Bp][T][C*F] memory merely RE-SHAPED to (Bp, C, F, T)
    // (distillation_crn.py:364 `ft.reshape(B, C, F, T)`), i.e. element (t, c, f) sits at t*C*F + c*F + f
    if (t.fc) return Strides4{(long long)T * t.C * t.F, (long long)t.C * t.F, 1, t.F};
    return Strides4{(long long)t.C * t.F * T, 1, T, (long long)t.F * T};
}
int train_tap(se_ctx* c, int k, float* out, cudaStream_t st) {
    SE_REQUIRE(c->t_have_fwd, "se_crn_train_tap: no forward pass to read");
    Tap t;
    if (tap_of(c, k, t)) return 1;
    const int Bp = c->t_N * c->t_nb;
    GemmParams g = t.op->g;
    g.M = Bp * t.op->rows_per_stream;
    g.epi = EPI_BIAS;
    g.stats = nullptr;
    g.out = c->sc[1];
    g.out_half = 0;
    if (run_gemm(c, g, t.op->stage, "tap." + t.op->label, st)) return 1;
    return launch_permute4(out, tap_theirs(t), c->sc[1], tap_ours(t), Bp, T, t.F, t.C, 0, st);
}
// s[...] += dtaps[k] (reference layout) where s is d loss / d pre-activation in our layout
int inject_tap(const se_ctx* c, const float* const* dtaps, int k, float* s, int Bp, cudaStream_t st) {
    if (dtaps == nullptr || dtaps[k] == nullptr) return 0;
    Tap t;
    if (tap_of(c, k, t)) return 1;
    return launch_permute4(s, tap_ours(t), dtaps[k], tap_theirs(t), Bp, T, t.F, t.C, 1, st);
}

float* garena_of(const se_ctx* c, const void* w) {
    return c->garena + (reinterpret_cast<const float*>(w) - c->wa.w);
}

// weight + data gradient of one forward GEMM op.  G: d loss / d (pre-activation output), rows addressed by `gs`.
int dense_bwd(se_ctx* c, const Op& op, int B, const float* G, StridedRows gs, float* dA, cudaStream_t st) {
    GemmParams g = op.g;
    g.M = B * op.rows_per_stream;
    if (!c->t_wgrad) return dA != nullptr ? launch_dgrad(g, G, gs, dA, st, c->bwd_mode) : 0;
    // weight and data gradient read the same G and write disjoint buffers: side by side on two branches, joined before
    // anything downstream may overwrite G (at one piece per rank most of these launches leave SMs idle)
    if (dA != nullptr && c->pipe_stream && c->bwd_overlap) {
        SE_CUDA_OK(cudaEventRecord(c->pipe_ev[14], st));
        SE_CUDA_OK(cudaStreamWaitEvent(c->pipe_stream, c->pipe_ev[14], 0));
        if (launch_wgrad(g, G, gs, garena_of(c, g.W), garena_of(c, g.bias), c->pipe_stream, c->bwd_mode)) return 1;
        if (launch_dgrad(g, G, gs, dA, st, c->bwd_mode)) return 1;
        SE_CUDA_OK(cudaEventRecord(c->pipe_ev[15], c->pipe_stream));
        SE_CUDA_OK(cudaStreamWaitEvent(st, c->pipe_ev[15], 0));
        return 0;
    }
    if (launch_wgrad(g, G, gs, garena_of(c, g.W), garena_of(c, g.bias), st, c->bwd_mode)) return 1;
    if (dA != nullptr && launch_dgrad(g, G, gs, dA, st, c->bwd_mode)) return 1;
    return 0;
}

int gln_bwd(se_ctx* c, const NormApplyParams& n, int B, int F, const float* y, const double* stats, double count,
            const float* w, const float* g, StridedRows gs, float* dy, int oC, int ostep, int ooff, int elu,
            cudaStream_t st) {
    GlnBwdParams p{};
    p.B = B;
    p.T = T;
    p.F = F;
    p.C = n.C;
    p.student = c->student;
    p.per_feature = n.per_feature;
    p.elu = elu;
    p.y = y;
    p.stats = stats;
    p.count = count;
    p.w = w;
    p.g = g;
    p.gB = gs.sB;
    p.gT = gs.sT;
    p.gF = gs.sF;
    p.dw = garena_of(c, w);
    p.db = garena_of(c, w == n.w ? n.b : n.br);
    p.red = c->red;
    p.dy = dy;
    p.oC = oC;
    p.ostep = ostep;
    p.ooff = ooff;
    return launch_gln_bwd(p, st);
}

// grad_flat == nullptr: no parameter gradient (weight-gradient GEMMs and the arena scatter skipped).  dmixture != nullptr:
// also d loss / d mixture [nb][3][t_L]; `mixture` is the signal the forward read (its 3-mic spectrum is recomputed).
int train_backward(se_ctx* c, const float* dpred, const float* const* dtaps, float* grad_flat, const float* mixture,
                   float* dmixture, cudaStream_t st) {
    SE_REQUIRE(c->t_have_fwd, "se_crn_train_backward: no forward pass to differentiate");
    const int nb = c->t_nb, N = c->t_N, Bp = N * nb, H = c->H, L = c->L, feat = c->feat;
    c->t_wgrad = grad_flat != nullptr;
    SE_CUDA_OK(cudaMemsetAsync(c->garena, 0, c->wa.floats * sizeof(float), st));
    for (auto& tw : c->twins) SE_CUDA_OK(cudaMemsetAsync(tw.first, 0, tw.second, st));
    float *s0 = c->sc[0], *s1 = c->sc[1], *s2 = c->sc[2], *s3 = c->sc[3];

    // ---- over_add / iSTFT adjoint / mask -> gradient w.r.t. the normalised last deconv output ------------------------
    if (launch_over_add_cm_bwd(dpred, nb, N, KCHUNK, c->t_front, c->t_L, c->dchunks, st)) return 1;
    {
        IoDesc io{c->dchunks, (long long)KCHUNK, 0, 0, KCHUNK, nullptr, 0, 0};
        if (launch_set_io(c->io_dev, io, st)) return 1;
        StftParams sp{};
        sp.io = c->io_dev;
        sp.B = Bp;
        sp.M = 1;
        sp.spec_ref = c->dspec;
        if (launch_stft_features(sp, st)) return 1;
        MaskBwdParams mb{};
        mb.B = Bp;
        mb.student = c->student;
        mb.dspec = c->dspec;
        mb.y = c->ylast;
        mb.stats = c->stats + (size_t)c->stats_last * 2 * c->maxB;
        mb.count = 2.0 * NBIN * T;
        mb.w = c->w_last;
        mb.b = c->b_last;
        mb.noisy = c->noisy;
        mb.g = s0;  // [Bp][T][201][2]
        mb.dnoisy = dmixture != nullptr ? c->dnoisy : nullptr;
        if (launch_mask_bwd(mb, st)) return 1;
    }
    // ---- decoder, last block first --------------------------------------------------------------------------------
    for (int j = L - 1; j >= 0; --j) {
        const DeconvRec& r = c->deconv_recs[j];
        const Op& dop = c->ops[r.op_deconv];
        const int C = r.Cop;
        const StridedRows ys{(long long)T * r.Fy * C, (long long)r.Fy * C, 2LL * C};  // rows of the merged-parity GEMM in y
        if (r.skip == nullptr) {
            NormApplyParams n{};
            n.C = C;
            n.w = c->w_last;
            n.b = c->b_last;
            const StridedRows gs{(long long)T * r.Fy * C, (long long)r.Fy * C, C};
            if (gln_bwd(c, n, Bp, r.Fy, r.y, c->stats + (size_t)c->stats_last * 2 * c->maxB, 2.0 * NBIN * T, n.w, s0, gs, s1,
                        C, 1, 0, 1, st))
                return 1;
        } else {
            const Op& nop = c->ops[r.op_norm];
            const Op& sop = c->ops[r.op_skip];
            const NormApplyParams& n = nop.n;
            BlendBwdParams bp{};
            bp.B = Bp;
            bp.T = T;
            bp.Fs = r.Fs;
            bp.Fy = r.Fy;
            bp.C = C;
            bp.student = c->student;
            bp.g = r.gout;
            bp.gB = r.gs.sB;
            bp.gT = r.gs.sT;
            bp.gF = r.gs.sF;
            bp.y = r.y;
            bp.rm = r.rm;
            bp.rr = r.rr;
            bp.stats = n.stats;
            bp.stats_r = n.stats_r;
            bp.count = n.count;
            bp.count_r = n.count_r;
            bp.w = n.w;
            bp.b = n.b;
            bp.wr = n.wr;
            bp.br = n.br;
            bp.g_o = s0;  // [Bp][T][Fy][C]
            bp.g_r = s2;  // [Bp][T][Fs][C]
            bp.G2 = s3;   // [Bp*T*Fs][2C]
            if (launch_blend_bwd(bp, st)) return 1;
            // residual-mask norm backward -> even columns of G2, then the skip 1x1 pair (dgrad into the skip tensor)
            const StridedRows rs{(long long)T * r.Fs * C, (long long)r.Fs * C, C};
            if (gln_bwd(c, n, Bp, r.Fs, r.rm, n.stats_r, n.count_r, n.wr, s2, rs, s3, 2 * C, 2, 0, 0, st)) return 1;
            const StridedRows g2s{(long long)T * r.Fs * 2 * C, (long long)r.Fs * 2 * C, 2LL * C};
            if (dense_bwd(c, sop, Bp, s3, g2s, r.skip->dbase + (r.skip->interior() - r.skip->base), st)) return 1;
            // main norm backward fused with the ELU backward -> s1 = d loss / d deconv pre-activation
            const StridedRows os{(long long)T * r.Fy * C, (long long)r.Fy * C, C};
            if (gln_bwd(c, n, Bp, r.Fy, r.y, n.stats, n.count, n.w, s0, os, s1, C, 1, 0, 1, st)) return 1;
            if (inject_tap(c, dtaps, 2 + j, s1, Bp, st)) return 1;
        }
        if (dense_bwd(c, dop, Bp, s1, ys, r.in->dbase, st)) return 1;
    }
    // ---- GRU + Linear + ELU + GLN(last) -----------------------------------------------------------------------------
    {
        const GruRec& gr = c->gru_rec;
        const Op& nop = c->ops[gr.op_norm];
        const Op& fop = c->ops[gr.op_fc];
        const Act& d0 = c->dec_in[0];
        const StridedRows gs{d0.sB, d0.sT, d0.sF};
        if (gln_bwd(c, nop.n, Bp, c->Fg, c->fcraw, nop.n.stats, nop.n.count, nop.n.w, d0.dinterior(), gs, s1, c->Cg, 1, 0, 1,
                    st))
            return 1;
        if (inject_tap(c, dtaps, 1, s1, Bp, st)) return 1;
        const StridedRows fs{(long long)T * feat, feat, 0};
        if (dense_bwd(c, fop, Bp, s1, fs, c->dH[1] + H, st)) return 1;
        const StridedRows g3{(long long)T * 3 * H, 3LL * H, 0};
        for (int l = 1; l >= 0; --l) {
            const Op& hop = c->ops[gr.op_hh[l]];
            const Op& iop = c->ops[gr.op_in[l]];
            // recurrent projections of all T steps at once: gh[t] = W_hh h[t-1] + b_hh  (h[0..T-1] are saved in hseq)
            GemmParams gh = hop.g;
            gh.A = c->hseq[l];
            gh.sB = (long long)(T + 1) * H;
            gh.sT = H;
            gh.Tn = T;
            gh.M = Bp * T;
            gh.epi = EPI_BIAS;
            gh.out = c->gh_all;
            gh.oB = (long long)T * 3 * H;
            gh.oT = 3 * H;
            gh.vec4 = 1;
            if (run_gemm(c, gh, ST_GRU, "gru.bwd.hh", st)) return 1;
            if (gru_seq_supported(H)) {
                GruSeqBwdParams bp{};
                bp.Whh = reinterpret_cast<const float*>(hop.g.W);
                bp.Kp = hop.g.K;
                bp.gi = c->gi_l[l];
                bp.gh = c->gh_all;
                bp.gB = (long long)T * 3 * H;
                bp.hseq = c->hseq[l];
                bp.dH = c->dH[l];
                bp.hB = (long long)(T + 1) * H;
                bp.dgi = c->dgi;
                bp.dgh = c->dgh;
                bp.dhrec = c->dhrec;
                bp.H = H;
                bp.T = T;
                bp.B = Bp;
                if (launch_gru_seq_bwd(bp, st)) return 1;
            }
            SE_CUDA_OK(cudaMemsetAsync(c->dhrec, 0, (size_t)Bp * H * sizeof(float), st));
            GemmParams rec = hop.g;  // dhrec[b][:] += dgh_t . W_hh
            rec.A = c->dhrec;
            rec.sB = H;
            rec.sT = 0;
            rec.sF = 0;
            rec.Tn = 1;
            rec.M = Bp;
            for (int t = T - 1; t >= 0 && !gru_seq_supported(H); --t) {
                if (launch_gru_bwd_pw(c->gi_l[l] + (long long)t * 3 * H, (long long)T * 3 * H,
                                      c->gh_all + (long long)t * 3 * H, (long long)T * 3 * H,
                                      c->hseq[l] + (long long)t * H, (long long)(T + 1) * H,
                                      c->dH[l] + (long long)(t + 1) * H, (long long)(T + 1) * H, c->dhrec,
                                      c->dgi + (long long)t * 3 * H, c->dgh + (long long)t * 3 * H, (long long)T * 3 * H, Bp,
                                      H, st))
                    return 1;
                if (t > 0 && launch_dgrad(rec, c->dgh + (long long)t * 3 * H, StridedRows{(long long)T * 3 * H, 0, 0},
                                          c->dhrec, st, c->bwd_mode))
                    return 1;
            }
            gh.out = nullptr;
            if (c->t_wgrad && launch_wgrad(gh, c->dgh, g3, garena_of(c, gh.W), garena_of(c, gh.bias), st, c->bwd_mode)) return 1;
            if (dense_bwd(c, iop, Bp, c->dgi, g3, l == 1 ? c->dH[0] + H : c->dxg, st)) return 1;
        }
    }
    // ---- encoder and pre-convolutions, last block first ------------------------------------------------------------
    for (int i = (int)c->conv_recs.size() - 1; i >= 0; --i) {
        const ConvRec& r = c->conv_recs[i];
        const Op& cop = c->ops[r.op_conv];
        const Op& gop = c->ops[r.op_gate];
        const Op& nop = c->ops[r.op_norm];
        const int C = r.Cp_out;
        const long long rows = (long long)Bp * T * r.Fo;
        if (r.residual)  // out = GLN(..) + x: the block input receives the output gradient as well (CRN_ELU.py:376)
            if (launch_add_strided(r.in->dinterior(), StridedRows{r.in->sB, r.in->sT, r.in->sF}, r.gout, r.gs, Bp, T, r.Fo,
                                   r.in->C, st))
                return 1;
        if (gln_bwd(c, nop.n, Bp, r.Fo, r.y, nop.n.stats, nop.n.count, nop.n.w, r.gout, r.gs, s0, C, 1, 0, 0, st)) return 1;
        GemmParams uv = gop.g;  // recompute the two 1x1 pre-activations (u, v) from the saved elu(conv)
        uv.M = (int)rows;
        uv.epi = EPI_BIAS;
        uv.out = s1;
        uv.oB = (long long)T * r.Fo * 2 * C;
        uv.oT = (long long)r.Fo * 2 * C;
        uv.oF = 2 * C;
        uv.stats = nullptr;
        uv.vec4 = 1;
        if (run_gemm(c, uv, gop.stage, "gate.bwd.uv", st)) return 1;
        if (launch_gate_bwd(s1, s0, rows, C, st)) return 1;
        SE_CUDA_OK(cudaMemsetAsync(s2, 0, (size_t)rows * C * sizeof(float), st));
        const StridedRows g2{(long long)T * r.Fo * 2 * C, (long long)r.Fo * 2 * C, 2LL * C};
        if (dense_bwd(c, gop, Bp, s1, g2, s2, st)) return 1;
        if (launch_elu_bwd(s2, r.e, rows * C, st)) return 1;
        if (i == (int)c->conv_recs.size() - 1 && inject_tap(c, dtaps, 0, s2, Bp, st)) return 1;
        const StridedRows g1{(long long)T * r.Fo * C, (long long)r.Fo * C, C};
        // the first pre-convolution's data gradient lands in the twin of the features (beside its residual path)
        const bool dgrad = r.need_dgrad || dmixture != nullptr;
        if (dense_bwd(c, cop, Bp, s2, g1, dgrad ? r.in->dbase : nullptr, st)) return 1;
    }
    // ---- features -> spectrum -> chunk -> mixture (CRN_ELU.py:369-373,417-424, utility.py:312-370) -------------------
    // Only the interior frames of the feature twin count: the leading state frames are the previous chunk's features,
    // detached in the reference (CRN_ELU.py:243), so no gradient crosses chunk state.
    if (dmixture != nullptr) {
        IoDesc io{mixture, 3 * c->t_L, c->t_L, -(long long)PHOP - c->t_front, c->t_L, nullptr, 0, 0};
        if (launch_set_io(c->io_dev, io, st)) return 1;
        StftParams sp{};
        sp.io = c->io_dev;
        sp.B = Bp;
        sp.M = 3;
        sp.spec_ref = s0;  // the 3-mic spectrum the forward's features were computed from, [Bp][3][F][T][2]
        sp.nb = nb;
        sp.hop_chunk = PHOP;
        if (launch_stft_features(sp, st)) return 1;
        const Act& a = c->pre_act[0];
        FeatBwdParams fb{};
        fb.B = Bp;
        fb.student = c->student;
        fb.dfeat = a.dinterior();
        fb.fB = a.sB;
        fb.fC = 1;
        fb.fT = a.sT;
        fb.fF = a.sF;
        fb.dnoisy = c->dnoisy;
        fb.spec = s0;
        fb.dspec = s1;
        if (launch_features_bwd(fb, st)) return 1;
        MaskIstftParams mp{};  // per (stream, mic) row: the adjoint of framing + window + real DFT -> d chunk [Bp][3][K]
        mp.B = Bp * 3;
        mp.spec_in = s1;
        mp.out_chunk = s2;
        mp.adjoint = 1;
        if (launch_mask_istft(mp, st)) return 1;
        // chunk n of utterance i read mixture[i][m][n*P + j - P - front]: rows (n*nb + i)*3 + m gathered like the output
        // overlap-add (utterance-mic rows i*3 + m), weight 1, pads and gap dropped
        if (launch_over_add_cm(s2, 3 * nb, N, KCHUNK, c->t_front, c->t_L, dmixture, st, 1.f)) return 1;
    }
    if (grad_flat == nullptr) return 0;
    // ---- packed-arena gradients -> flat vector in the reference layout (registry order) --------------------------------
    SE_CUDA_OK(cudaMemsetAsync(grad_flat, 0, (size_t)c->n_theta * sizeof(float), st));
    return launch_arena_scatter_add(c->garena, c->wmap, grad_flat, (long long)c->wa.floats, st);
}

}  // namespace

// ======================================================================================================================
// C-ABI
// ======================================================================================================================
extern "C" {

const char* se_last_error(void) { return g_err.c_str(); }
const char* se_version(void) { return "se_b200 0.1 sm_100a"; }

int se_ctx_create(se_ctx** out, int device, const se_crn_config* cfg) {
    if (!out || !cfg) {
        set_error("se_ctx_create: null argument");
        return 2;
    }
    *out = nullptr;
    if (const int rc = check_create_device(device, "se_ctx_create")) return rc;
    se_ctx* c = new se_ctx();
    c->cfg = *cfg;
    c->device = device;
    if (build_ctx(c)) {
        se_ctx_destroy(c);
        return 1;
    }
    *out = c;
    return 0;
}

int se_ctx_destroy(se_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto& kv : c->graphs) cudaGraphExecDestroy(kv.second);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    if (c->pipe_stream) cudaStreamDestroy(c->pipe_stream);
    for (cudaEvent_t e : c->pipe_ev)
        if (e) cudaEventDestroy(e);
    for (void* p : c->allocs) cudaFree(p);
    if (c->h_in) cudaFree(c->h_in);
    if (c->h_out) cudaFree(c->h_out);
    delete c;
    return 0;
}

int se_crn_num_params(const se_ctx* c) { return c ? (int)c->wa.params.size() : 0; }
const char* se_crn_param_name(const se_ctx* c, int i) {
    return (c && i >= 0 && i < (int)c->wa.params.size()) ? c->wa.params[i].name.c_str() : nullptr;
}
int64_t se_crn_param_numel(const se_ctx* c, int i) {
    return (c && i >= 0 && i < (int)c->wa.params.size()) ? c->wa.params[i].numel() : -1;
}

int se_crn_bind_weights(se_ctx* c, const float* const* ptrs, int n, void* stream) {
    SE_REQUIRE(c != nullptr && ptrs != nullptr, "se_crn_bind_weights: null argument");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return c->wa.upload(ptrs, n, (cudaStream_t)stream, "se_crn_bind_weights");
}

int se_crn_state_reset(se_ctx* c, int first, int count, void* stream) {
    SE_REQUIRE(c != nullptr, "null context");
    SE_REQUIRE(first >= 0 && count >= 0 && first + count <= c->maxB, "se_crn_state_reset: stream range");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return launch_zero(c->zero_tab, first, count, (cudaStream_t)stream);
}

int64_t se_crn_state_bytes_per_stream(const se_ctx* c) {
    if (!c) return -1;
    return c->state_tab.record_bytes;
}

uint64_t se_crn_state_layout(const se_ctx* c) { return c ? c->state_layout : 0; }

int se_crn_state_export(se_ctx* c, const int32_t* rows_host, int n, void* dst_dev, void* stream) {
    NvtxRange nvtx_range("se.state_export");
    SE_REQUIRE(c != nullptr, "null context");
    SE_REQUIRE(!c->train, "se_crn_state_export: a training context carries no per-stream streaming state");
    if (state_rows_check(rows_host, n, c->maxB, false, "se_crn_state_export")) return 2;
    SE_REQUIRE(n == 0 || (dst_dev != nullptr && reinterpret_cast<uintptr_t>(dst_dev) % 16 == 0),
               "se_crn_state_export: dst must be a 16-byte aligned device buffer");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return launch_state_pack(c->state_tab, rows_host, n, dst_dev, (cudaStream_t)stream);
}

int se_crn_state_import(se_ctx* c, const int32_t* rows_host, int n, const void* src_dev, uint64_t layout, void* stream) {
    NvtxRange nvtx_range("se.state_import");
    SE_REQUIRE(c != nullptr, "null context");
    SE_REQUIRE(!c->train, "se_crn_state_import: a training context carries no per-stream streaming state");
    SE_REQUIRE(layout == c->state_layout,
               "se_crn_state_import: record layout mismatch (records from another model, configuration, precision or "
               "front path; this context:" + c->state_tab.desc + ")");
    if (state_rows_check(rows_host, n, c->maxB, true, "se_crn_state_import")) return 2;
    SE_REQUIRE(n == 0 || (src_dev != nullptr && reinterpret_cast<uintptr_t>(src_dev) % 16 == 0),
               "se_crn_state_import: src must be a 16-byte aligned device buffer");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return launch_state_unpack(c->state_tab, rows_host, n, src_dev, (cudaStream_t)stream);
}

int se_crn_process_chunk(se_ctx* c, const float* in, int64_t in_stream_stride, int64_t in_mic_stride, float* out,
                         int64_t out_stream_stride, int B, void* stream) {
    NvtxRange nvtx_range("se.chunk_step");
    if (check_ready(c, B)) return 1;
    SE_REQUIRE(in != nullptr && out != nullptr, "se_crn_process_chunk: null buffer");
    if (B == 0) return 0;
    IoDesc io{in, in_stream_stride, in_mic_stride, 0, KCHUNK, out, out_stream_stride, PHOP};
    return run_stream_step(c, io, B, (cudaStream_t)stream);
}

int se_chunk_grid(int64_t L, int K, int* gap, int* n_chunks) {
    SE_REQUIRE(L >= 0 && K > 0 && K % 2 == 0, "se_chunk_grid: bad arguments");
    const int P = K / 2;
    const int g = K - (int)((P + L % K) % K);  // utility.py:325
    if (gap) *gap = g;
    if (n_chunks) *n_chunks = (int)(2 * (L + g + P) / K);  // utility.py:357-368
    return 0;
}

int se_crn_realtime_process(se_ctx* c, const float* mixture, int B, int64_t L, int flag, float* out, void* stream) {
    NvtxRange nvtx_range("se.realtime_process");
    if (check_ready(c, B)) return 1;
    SE_REQUIRE(mixture != nullptr && out != nullptr, "se_crn_realtime_process: null buffer");
    SE_REQUIRE(L > 0, "se_crn_realtime_process: empty signal");
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int front = flag ? 0 : PHOP;  // CRN_ELU.py:474-476
    int gap = 0, N = 0;
    se_chunk_grid(L + front, KCHUNK, &gap, &N);
    if (!flag) {
        if (se_crn_state_reset(c, 0, B, stream)) return 1;  // CRN_ELU.py:480-481
    }
    // chunk n covers samples [n*P - P - front, ... + K) of the caller's signal; its step emits the overlap-added
    // samples [n*P - P - front, n*P - front) (utility.py:393-403), of which [0, L) are kept.
    for (int n = 0; n < N; ++n) {
        IoDesc io{};
        io.in = mixture;
        io.in_stream_stride = 3 * L;
        io.in_mic_stride = L;
        io.in_offset = (long long)n * PHOP - PHOP - front;
        io.in_len = L;
        const long long o0 = (long long)n * PHOP - PHOP - front;
        long long nv = 0;
        if (o0 >= 0) nv = (L - o0) < PHOP ? (L - o0) : PHOP;
        if (nv < 0) nv = 0;
        io.out = out + (o0 >= 0 ? o0 : 0);
        io.out_stream_stride = L;
        io.n_valid = (int)nv;
        if (run_stream_step(c, io, B, st)) return 1;
    }
    return 0;
}

int se_crn_realtime_process_host(se_ctx* c, const float* mixture, int B, int64_t L, int flag, float* out) {
    NvtxRange nvtx_range("se.realtime_process_host");
    if (check_ready(c, B)) return 1;
    const size_t nin = (size_t)B * 3 * L, nout = (size_t)B * L;
    if (c->h_in_floats < nin) {
        if (c->h_in) cudaFree(c->h_in);
        SE_CUDA_OK(cudaMalloc(&c->h_in, nin * sizeof(float)));
        c->h_in_floats = nin;
    }
    if (c->h_out_floats < nout) {
        if (c->h_out) cudaFree(c->h_out);
        SE_CUDA_OK(cudaMalloc(&c->h_out, nout * sizeof(float)));
        c->h_out_floats = nout;
    }
    SE_CUDA_OK(cudaMemcpy(c->h_in, mixture, nin * sizeof(float), cudaMemcpyHostToDevice));
    if (se_crn_realtime_process(c, c->h_in, B, L, flag, c->h_out, nullptr)) return 1;
    SE_CUDA_OK(cudaMemcpy(out, c->h_out, nout * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
}

// STFT / iSTFT do not depend on a model: with ctx == NULL they run on the current device with a per-device descriptor cell
static int fft_cell(IoDesc** cell) {
    static std::map<int, IoDesc*> cells;
    int dev = 0;
    SE_CUDA_OK(cudaGetDevice(&dev));
    auto it = cells.find(dev);
    if (it == cells.end()) {
        void* p = nullptr;
        SE_CUDA_OK(cudaMalloc(&p, sizeof(IoDesc)));
        if (init_fft_tables()) return 1;
        it = cells.emplace(dev, reinterpret_cast<IoDesc*>(p)).first;
    }
    *cell = it->second;
    return 0;
}

int se_stft_trans(se_ctx* c, const float* chunks, int R, float* spec, void* stream) {
    SE_REQUIRE(chunks != nullptr && spec != nullptr, "se_stft_trans: null argument");
    IoDesc* cell = nullptr;
    if (c) {
        SE_CUDA_OK(cudaSetDevice(c->device));
        cell = c->io_dev;
    } else if (fft_cell(&cell)) {
        return 1;
    }
    if (R == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    IoDesc io{chunks, 3LL * KCHUNK, KCHUNK, 0, KCHUNK, nullptr, 0, 0};
    if (launch_set_io(cell, io, st)) return 1;
    StftParams sp{};
    sp.io = cell;
    sp.B = R;
    sp.M = 3;
    sp.student = c ? c->student : 0;
    sp.spec_ref = spec;
    return launch_stft_features(sp, st);
}

int se_istft_trans(se_ctx* c, const float* spec, int R, float* out, void* stream) {
    SE_REQUIRE(spec != nullptr && out != nullptr, "se_istft_trans: null argument");
    if (c) {
        SE_CUDA_OK(cudaSetDevice(c->device));
    } else {
        IoDesc* cell = nullptr;
        if (fft_cell(&cell)) return 1;  // constant tables of this device
    }
    if (R == 0) return 0;
    MaskIstftParams mp{};
    mp.B = R;
    mp.spec_in = spec;
    mp.out_chunk = out;
    return launch_mask_istft(mp, (cudaStream_t)stream);
}

int se_crn_forward_chunk(se_ctx* c, const float* spec_in, float* spec_out, int B, void* stream) {
    NvtxRange nvtx_range("se.forward_chunk");
    if (check_ready(c, B)) return 1;
    SE_REQUIRE(spec_in != nullptr && spec_out != nullptr, "se_crn_forward_chunk: null buffer");
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_OK(cudaMemsetAsync(c->stats, 0, (size_t)c->n_stats * 2 * c->maxB * sizeof(double), st));
    if (c->front_mma) {
        if (launch_features_from_spec(spec_in, B, 3, c->student, nullptr, (long long)T * PRECONV3_POS * 8, 0,
                                      (long long)PRECONV3_POS * 8, 8, c->noisy, st, c->feat_h + PRECONV3_BORDER * 8))
            return 1;
    } else if (c->preconv_tc) {
        if (launch_features_from_spec(spec_in, B, 3, c->student, nullptr, (long long)PRECONV_TP * PRECONV_TC_POS * 8, 0,
                                      (long long)PRECONV_TC_POS * 8, 8, c->noisy, st,
                                      c->pre_h[0] + (4LL * PRECONV_TC_POS + 2) * 8))
            return 1;
    } else {
        const PreBuf& a = c->pre_in[0];
        if (launch_features_from_spec(spec_in, B, 3, c->student, a.interior(), a.sB, a.sC, a.Fpp, 1, c->noisy, st)) return 1;
    }
    if (enqueue_net(c, B, st, -1)) return 1;
    MaskIstftParams mp{};
    mp.B = B;
    mp.student = c->student;
    mp.y = c->ylast;
    mp.stats = c->stats + (size_t)c->stats_last * 2 * c->maxB;
    mp.count = 2.0 * NBIN * T;
    mp.w = c->w_last;
    mp.b = c->b_last;
    mp.noisy = c->noisy;
    mp.spec_ref = spec_out;
    if (launch_mask_istft(mp, st)) return 1;
    return launch_roll(c->roll, 0, B, st);
}

int se_segmentation(const float* x, int B, int C, int64_t L, int K, float* out, int* gap, int* n_chunks,
                    void* stream) {
    SE_REQUIRE(x != nullptr && out != nullptr, "se_segmentation: null buffer");
    int g = 0, N = 0;
    if (se_chunk_grid(L, K, &g, &N)) return 1;
    if (gap) *gap = g;
    if (n_chunks) *n_chunks = N;
    return launch_segmentation(x, B, C, L, K, g, N, out, (cudaStream_t)stream);
}

int se_over_add(const float* chunks, int C, int N, int K, int gap, float* out, void* stream) {
    SE_REQUIRE(chunks != nullptr && out != nullptr, "se_over_add: null buffer");
    SE_REQUIRE(N >= 2 && K > 0 && K % 2 == 0 && gap >= 0, "se_over_add: bad arguments");
    return launch_over_add(chunks, C, N, K, gap, out, (cudaStream_t)stream);
}

int se_debug_read(se_ctx* c, const char* name, int b, float* host_dst, int64_t max_floats, int* dims) {
    SE_REQUIRE(c != nullptr && name != nullptr && host_dst != nullptr && dims != nullptr, "se_debug_read: null argument");
    SE_REQUIRE(b >= 0 && b < c->maxB, "se_debug_read: stream index");
    SE_CUDA_OK(cudaSetDevice(c->device));
    SE_CUDA_OK(cudaDeviceSynchronize());
    const std::string n(name);
    const float* src = nullptr;
    int t = T, f = 1, ch = 1;
    int src_esz = 4;
    long long sT = 0, sF = 0;
    auto from_act = [&](const Act& a) {
        src_esz = a.esz;
        src = a.at(a.padT0 * a.sT + a.padF0 * a.sF + (long long)b * a.sB);
        f = a.F;
        ch = a.C;
        sT = a.sT;
        sF = a.sF;
    };
    auto compact = [&](const float* base, int F_, int C_, int T_ = T) {
        t = T_;
        f = F_;
        ch = C_;
        sF = C_;
        sT = (long long)F_ * C_;
        src = base + (long long)b * T_ * sT;
    };
    auto idx_of = [&](const char* prefix, int limit) -> int {
        const size_t len = strlen(prefix);
        if (n.compare(0, len, prefix) != 0 || n.size() != len + 1) return -1;
        const int i = n[len] - '0';
        return (i >= 0 && i < limit) ? i : -1;
    };
    int i;
    if ((i = idx_of("pre_in", 3)) >= 0 && c->front_mma) {  // only the features reach HBM: layers 1, 2 live in shared memory
        SE_REQUIRE(i == 0, "se_debug_read: pre_in1 / pre_in2 are not materialised by the fused pre-convolution kernel");
        dims[0] = T;
        dims[1] = NBIN;
        dims[2] = 5;
        SE_REQUIRE((int64_t)T * NBIN * 5 <= max_floats, "se_debug_read: destination too small");
        const size_t n = (size_t)T * PRECONV3_POS * 8;
        std::vector<__half> slab(n);
        SE_CUDA_OK(cudaMemcpy(slab.data(), c->feat_h + (size_t)b * n, n * sizeof(__half), cudaMemcpyDeviceToHost));
        for (int tt = 0; tt < T; ++tt)
            for (int ff = 0; ff < NBIN; ++ff)
                for (int cc = 0; cc < 5; ++cc)
                    host_dst[((size_t)tt * NBIN + ff) * 5 + cc] =
                        __half2float(slab[((size_t)tt * PRECONV3_POS + ff + PRECONV3_BORDER) * 8 + cc]);
        return 0;
    } else if ((i = idx_of("pre_in", 3)) >= 0 && c->preconv_tc) {  // channels-last fp16 units -> [T][F][5] on the host
        dims[0] = T;
        dims[1] = NBIN;
        dims[2] = 5;
        SE_REQUIRE((int64_t)T * NBIN * 5 <= max_floats, "se_debug_read: destination too small");
        const size_t n = (size_t)PRECONV_TP * PRECONV_TC_POS * 8;
        std::vector<__half> slab(n);
        SE_CUDA_OK(cudaMemcpy(slab.data(), c->pre_h[i] + (size_t)b * n, n * sizeof(__half), cudaMemcpyDeviceToHost));
        for (int tt = 0; tt < T; ++tt)
            for (int ff = 0; ff < NBIN; ++ff)
                for (int cc = 0; cc < 5; ++cc)
                    host_dst[((size_t)tt * NBIN + ff) * 5 + cc] =
                        __half2float(slab[((size_t)(tt + 4) * PRECONV_TC_POS + ff + 2 * (1 << i)) * 8 + cc]);
        return 0;
    } else if ((i = idx_of("pre_in", 3)) >= 0 && c->train) {
        from_act(c->pre_act[i]);
    } else if ((i = idx_of("pre_in", 3)) >= 0) {  // planar -> [T][F][5] on the host
        const PreBuf& pb = c->pre_in[i];
        dims[0] = T;
        dims[1] = NBIN;
        dims[2] = 5;
        SE_REQUIRE((int64_t)T * NBIN * 5 <= max_floats, "se_debug_read: destination too small");
        std::vector<float> slab((size_t)pb.sB);
        SE_CUDA_OK(cudaMemcpy(slab.data(), pb.base + (long long)b * pb.sB, slab.size() * sizeof(float),
                              cudaMemcpyDeviceToHost));
        for (int tt = 0; tt < T; ++tt)
            for (int ff = 0; ff < NBIN; ++ff)
                for (int cc = 0; cc < 5; ++cc)
                    host_dst[((size_t)tt * NBIN + ff) * 5 + cc] =
                        slab[(size_t)cc * pb.sC + (size_t)(tt + 4) * pb.Fpp + ff + 2 * pb.d];
        return 0;
    } else if ((i = idx_of("enc_in", c->L)) >= 0) from_act(c->enc_in[i]);
    else if ((i = idx_of("dec_in", c->L)) >= 0) from_act(c->dec_in[i]);
    else if ((i = idx_of("hseq", 2)) >= 0) {
        compact(c->hseq[i], 1, c->H, T + 1);
        src_esz = c->esz;
        src = c->E(c->hseq[i], (long long)b * (T + 1) * c->H);
    } else if (n == "xg") {
        compact(c->xg, c->Fg, c->Cg);
        src_esz = c->esz;
        src = c->E(c->xg, (long long)b * T * c->feat);
    }
    else if (n == "fcraw") {
        compact(c->fcraw, c->Fg, c->Cg);
        src_esz = c->esz;
        src = c->E(c->fcraw, (long long)b * T * c->feat);
    }
    else if (n == "ylast") compact(c->ylast, NBIN, 2);
    else if (n == "noisy") compact(c->noisy, NBIN, 2);
    else SE_REQUIRE(false, "se_debug_read: unknown tensor " + n);
    dims[0] = t;
    dims[1] = f;
    dims[2] = ch;
    SE_REQUIRE((int64_t)t * f * ch <= max_floats, "se_debug_read: destination too small");
    if (src_esz == 2) {  // fp16 operand buffer: convert on the host
        std::vector<__half> tmp((size_t)t * f * ch);
        SE_CUDA_OK(cudaMemcpy2D(tmp.data(), (size_t)f * ch * 2, src, (size_t)sT * 2, (size_t)f * ch * 2, t,
                                cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < tmp.size(); ++i) host_dst[i] = __half2float(tmp[i]);
        return 0;
    }
    SE_CUDA_OK(cudaMemcpy2D(host_dst, (size_t)f * ch * sizeof(float), src, (size_t)sT * sizeof(float),
                            (size_t)f * ch * sizeof(float), t, cudaMemcpyDeviceToHost));
    (void)sF;
    return 0;
}


int se_debug_gru_counters(uint64_t* out16, int reset) {
    return gru_profile_read(reinterpret_cast<unsigned long long*>(out16), reset);
}

int se_debug_gemm_counters(uint64_t* out8, int reset) {
    static_assert(sizeof(uint64_t) == sizeof(unsigned long long), "counter width");
    return gemm_profile_read(reinterpret_cast<unsigned long long*>(out8), reset);
}

int se_debug_mask_spectrum(se_ctx* c, const float* mask, const float* noisy, float* spec_out, int B) {
    SE_REQUIRE(c != nullptr && mask != nullptr && noisy != nullptr && spec_out != nullptr && B > 0,
               "se_debug_mask_spectrum: bad arguments");
    SE_CUDA_OK(cudaSetDevice(c->device));
    // identity GlobalLayerNorm in front of the mask: sum = 0, sum of squares = count  ->  mean 0, variance 1 (the
    // denominator sqrt(1 + 1e-8) + 1e-8 differs from 1 by 1.5e-8); affine weight 1, bias 0
    const double count = 2.0 * NBIN * T;
    std::vector<double> st(2 * (size_t)B);
    for (int b = 0; b < B; ++b) {
        st[2 * b] = 0.0;
        st[2 * b + 1] = count;
    }
    const float wb[4] = {1.f, 1.f, 0.f, 0.f};
    double* d_st = nullptr;
    float* d_wb = nullptr;
    SE_CUDA_OK(cudaMalloc(&d_st, st.size() * sizeof(double)));
    SE_CUDA_OK(cudaMalloc(&d_wb, sizeof(wb)));
    SE_CUDA_OK(cudaMemcpy(d_st, st.data(), st.size() * sizeof(double), cudaMemcpyHostToDevice));
    SE_CUDA_OK(cudaMemcpy(d_wb, wb, sizeof(wb), cudaMemcpyHostToDevice));
    MaskIstftParams mp{};
    mp.B = B;
    mp.student = c->student;
    mp.y = mask;
    mp.stats = d_st;
    mp.count = count;
    mp.w = d_wb;
    mp.b = d_wb + 2;
    mp.noisy = noisy;
    mp.spec_ref = spec_out;
    const int rc = launch_mask_istft(mp, nullptr);
    const cudaError_t e = cudaDeviceSynchronize();
    cudaFree(d_st);
    cudaFree(d_wb);
    if (rc) return rc;
    SE_CUDA_OK(e);
    return 0;
}

// ---- training ---------------------------------------------------------------------------------------------------
int64_t se_crn_num_theta(const se_ctx* c) { return c ? c->n_theta : -1; }
int64_t se_crn_param_offset(const se_ctx* c, int i) {
    return (c && c->train && i >= 0 && i < (int)c->param_off.size()) ? c->param_off[i] : -1;
}

int se_crn_bind_weights_flat(se_ctx* c, const float* theta, void* stream) {
    SE_REQUIRE(c != nullptr && theta != nullptr, "se_crn_bind_weights_flat: null argument");
    SE_REQUIRE(c->train, "se_crn_bind_weights_flat needs a context created with training = 1");
    SE_CUDA_OK(cudaSetDevice(c->device));
    if (launch_arena_gather(c->wa.w, c->wmap, theta, (long long)c->wa.floats, (cudaStream_t)stream)) return 1;
    c->wa.bound = true;
    return 0;
}

int se_crn_train_forward(se_ctx* c, const float* mixture, int B, int64_t L, int flag, float* pred, void* stream) {
    NvtxRange nvtx_range("se.train_forward");
    if (check_ready(c, 0, true)) return 1;
    SE_REQUIRE(mixture != nullptr && pred != nullptr, "se_crn_train_forward: null buffer");
    SE_REQUIRE(B > 0 && L > 0, "se_crn_train_forward: empty batch");
    return train_forward(c, mixture, B, L, flag, pred, (cudaStream_t)stream);
}

int se_crn_train_backward(se_ctx* c, const float* dpred, float* grad_flat, void* stream) {
    NvtxRange nvtx_range("se.train_backward");
    if (check_ready(c, 0, true)) return 1;
    SE_REQUIRE(dpred != nullptr && grad_flat != nullptr, "se_crn_train_backward: null buffer");
    return train_backward(c, dpred, nullptr, grad_flat, nullptr, nullptr, (cudaStream_t)stream);
}

int se_crn_train_num_taps(const se_ctx* c) { return (c && c->train) ? c->L + 1 : 0; }

int se_crn_train_tap_shape(const se_ctx* c, int tap, int* C_out, int* F_out, int* T_out) {
    SE_REQUIRE(c != nullptr && C_out && F_out && T_out, "se_crn_train_tap_shape: null argument");
    Tap t;
    if (tap_of(c, tap, t)) return 1;
    *C_out = t.C;
    *F_out = t.F;
    *T_out = T;
    return 0;
}

int se_crn_train_tap(se_ctx* c, int tap, float* out, void* stream) {
    NvtxRange nvtx_range("se.train_tap");
    if (check_ready(c, 0, true)) return 1;
    SE_REQUIRE(out != nullptr, "se_crn_train_tap: null buffer");
    return train_tap(c, tap, out, (cudaStream_t)stream);
}

int se_crn_train_backward_taps(se_ctx* c, const float* dpred, const float* const* dtaps, int n_taps, float* grad_flat,
                               void* stream) {
    NvtxRange nvtx_range("se.train_backward_taps");
    if (check_ready(c, 0, true)) return 1;
    SE_REQUIRE(dpred != nullptr && grad_flat != nullptr, "se_crn_train_backward_taps: null buffer");
    SE_REQUIRE(dtaps == nullptr || n_taps == c->L + 1, "se_crn_train_backward_taps: one gradient slot per feature tap");
    return train_backward(c, dpred, dtaps, grad_flat, nullptr, nullptr, (cudaStream_t)stream);
}

int se_crn_train_backward_input(se_ctx* c, const float* mixture, const float* dpred, const float* const* dtaps, int n_taps,
                                float* grad_flat, float* dmixture, void* stream) {
    NvtxRange nvtx_range("se.train_backward_input");
    if (check_ready(c, 0, true)) return 1;
    SE_REQUIRE(dpred != nullptr, "se_crn_train_backward_input: null dpred");
    SE_REQUIRE(grad_flat != nullptr || dmixture != nullptr, "se_crn_train_backward_input: nothing to compute");
    SE_REQUIRE(dmixture == nullptr || mixture != nullptr, "se_crn_train_backward_input: d mixture needs the mixture");
    SE_REQUIRE(dtaps == nullptr || n_taps == c->L + 1, "se_crn_train_backward_input: one gradient slot per feature tap");
    return train_backward(c, dpred, dtaps, grad_flat, mixture, dmixture, (cudaStream_t)stream);
}

int se_crn_launches_per_chunk(const se_ctx* c) { return c ? count_launches(c) : 0; }

int se_crn_set_graph(se_ctx* c, int enable) {
    SE_REQUIRE(c != nullptr, "null context");
    c->use_graph = enable != 0;
    return 0;
}

int se_crn_num_kernels(const se_ctx* c) { return c ? num_kernels(c) : 0; }

int se_crn_kernel_info(const se_ctx* c, int index, char* name, int name_cap, double* flops_per_stream,
                       double* bytes_per_stream, int* stage) {
    SE_REQUIRE(c != nullptr && index >= 0 && index < num_kernels(c), "se_crn_kernel_info: bad index");
    const int n = (int)c->ops.size();
    std::string label;
    double fl = 0, by = 0;
    int stg = 0;
    if (index == 0) {
        label = "stft+features";
        fl = 0;
        by = 4.0 * (3 * KCHUNK + 5 * NBIN * T + 2 * NBIN * T);  // SURVEY.md section 8(d)
        stg = ST_STFT;
    } else if (index <= n) {
        const Op& op = c->ops[index - 1];
        label = op.label;
        fl = op.alg_flops;
        by = op.alg_bytes;
        stg = op.stage;
        if (c->half) by *= op.f16_bytes;
    } else if (index == n + 1) {
        label = "mask+istft+ola";
        by = 4.0 * (2 * 2 * NBIN * T + PHOP + 2 * PHOP);
        stg = ST_MASK;
    } else {
        label = "state_roll";
        by = 2.0 * 4.0 * (double)c->roll_floats;
        stg = ST_ROLL;
    }
    if (name && name_cap > 0) {
        strncpy(name, label.c_str(), (size_t)name_cap - 1);
        name[name_cap - 1] = 0;
    }
    if (flops_per_stream) *flops_per_stream = fl;
    if (bytes_per_stream) *bytes_per_stream = by;
    if (stage) *stage = stg;
    return 0;
}

static int time_filter(se_ctx* c, int filter, int kernel, int B, int iters, float* ms);

int se_crn_time_kernel(se_ctx* c, int index, int B, int iters, float* ms) {
    if (check_ready(c, B)) return 1;
    SE_REQUIRE(ms != nullptr && iters > 0 && B > 0 && index >= 0 && index < num_kernels(c),
               "se_crn_time_kernel: bad arguments");
    return time_filter(c, -2, index, B, iters, ms);
}

int se_crn_time_stage(se_ctx* c, const char* stage, int B, int iters, float* ms) {
    if (check_ready(c, B)) return 1;
    SE_REQUIRE(stage != nullptr && ms != nullptr && iters > 0 && B > 0, "se_crn_time_stage: bad arguments");
    int filter = -2;
    if (strcmp(stage, "step") == 0) filter = -1;
    for (int s = 0; s < ST_COUNT; ++s)
        if (strcmp(stage, kStageNames[s]) == 0) filter = s;
    SE_REQUIRE(filter != -2, std::string("se_crn_time_stage: unknown stage ") + stage);
    return time_filter(c, filter, -1, B, iters, ms);
}

// filter >= -1: a stage (or the whole step); filter == -2: the single kernel `kernel`
static int time_filter(se_ctx* c, int filter, int kernel, int B, int iters, float* ms) {
    cudaStream_t st = nullptr;
    // a self-contained chunk source so that the stage can run without caller buffers: the carry/out of the previous
    // run are reused as scratch (timing only; state is garbage afterwards -> caller must reset)
    static thread_local float* scratch = nullptr;
    static thread_local size_t scratch_floats = 0;
    const size_t need = (size_t)B * (3 * KCHUNK + PHOP);
    if (scratch_floats < need) {
        if (scratch) cudaFree(scratch);
        SE_CUDA_OK(cudaMalloc(&scratch, need * sizeof(float)));
        SE_CUDA_OK(cudaMemset(scratch, 0, need * sizeof(float)));
        // noise-like chunk content (the arithmetic of the STFT / feature kernel is not data independent: atan2 branches)
        if (launch_fill_noise(scratch, (long long)B * 3 * KCHUNK, 0.3f, st)) return 1;
        scratch_floats = need;
    }
    IoDesc io{scratch, 3LL * KCHUNK, KCHUNK, 0, KCHUNK, scratch + (size_t)B * 3 * KCHUNK, PHOP, PHOP};
    if (launch_set_io(c->io_dev, io, st)) return 1;
    cudaEvent_t e0, e1;
    SE_CUDA_OK(cudaEventCreate(&e0));
    SE_CUDA_OK(cudaEventCreate(&e1));
    auto run = [&]() { return filter == -2 ? enqueue_kernel(c, kernel, B, st) : enqueue_stream_step(c, B, st, filter); };
    if (run()) return 1;  // warm-up
    SE_CUDA_OK(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; ++i)
        if (run()) return 1;
    SE_CUDA_OK(cudaEventRecord(e1, st));
    SE_CUDA_OK(cudaEventSynchronize(e1));
    float t = 0.f;
    SE_CUDA_OK(cudaEventElapsedTime(&t, e0, e1));
    *ms = t / iters;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return 0;
}

}  // extern "C"
