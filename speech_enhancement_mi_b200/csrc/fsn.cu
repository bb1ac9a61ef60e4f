// FullSubNet chunk step (fullsubnet.py:769-824) behind the C-ABI of include/se_b200.h (se_fsn_*).
//
//   magnitude of the 3 microphones -> CumLayerNorm (in-place, running mean, fullsubnet.py:177-205) -> full-band LSTM
//   (603 -> 512, 2 layers) + Linear(201) + ReLU -> unfold of the NORMALISED mic-0 magnitude (31 reflect-padded
//   neighbours, fullsubnet.py:299-331) ++ full-band output -> CumLayerNorm -> sub-band LSTM (32 -> 384, 2 layers) on
//   B*201 independent sequences + Linear(2) -> cIRM mask.
//
// Every LSTM step is ONE tcgen05 GEMM (gemm_tc.cu, EPI_LSTM): A = [x_t | h_{t-1}] gathered from a per-sequence record
// through the koff table, W = [W_ih | W_hh] with rows re-ordered to [i|f|g|o] per 32-unit tile, bias = b_ih + b_hh, and
// the cell update fused in the epilogue -- the input projection is never materialised.  Per-sequence record (fp32):
//   [ x: T x Kin_pad | h(layer 0): (T+1) x H | h(layer 1): (T+1) x H ]      slot 0 of an h history = carried state
// (se_fsn_state_export / _import gather and scatter the carried state of chosen rows: state_tab, state_io.cu)
// The reflect-padded neighbour gather is expanded once per chunk into the x part of the sub-band records (540 KB per
// stream and chunk, against 15.4 GFLOP of LSTM work per stream and chunk).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <string.h>

#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/se_b200.h"
#include "se_internal.h"

using namespace se;

namespace {

constexpr int T = kFramesPerChunk;
constexpr int KCHUNK = 3200;         // samples per chunk (config.yaml:172 segment_length)
constexpr int PHOP = KCHUNK / 2;     // samples a streaming step returns
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct FsnGemm {
    GemmParams g;
    int rows_per_stream;
    bool tma_ok = false;  // TMA descriptors (fp16 LSTM steps) in `tma`
    GemmTma tma{};
};

}  // namespace

struct se_fsn {
    se_fsn_config cfg;
    int device = 0, maxB = 0;
    int F = 0, M = 0, Hf = 0, Hs = 0, NB = 0;  // NB = 2*sb_neighbors + 1
    int Kf = 0;                                // padded full-band input size (603 -> 608)
    int Ks = 0;                                // sub-band input size (32)
    long long recF = 0, recS = 0;              // record strides (floats)
    long long f_h0 = 0, f_h1 = 0, s_h0 = 0, s_h1 = 0;  // offsets of the h histories inside a record
    WeightArena wa;  // packed weights, their koff tables and the parameter registry
    std::vector<void*> allocs;
    float *fbrec = nullptr, *sbrec = nullptr, *fbc = nullptr, *sbc = nullptr, *fbout = nullptr, *pline = nullptr;
    float *crm = nullptr;  // [B*F][T][2]
    double* sums = nullptr;      // [B][4]: sum |X|, weighted sum of the unfolded mic-0 magnitude, (sum, sumsq) of fb_out
    float* cstate = nullptr;     // [B][4]: running mean fb, running mean sb, inv fb, inv sb
    int* cstep = nullptr;        // [B][2]
    // SE_PRECISION_FP16: the sub-band records (x_t and the h histories, 98.7 % of the FLOPs read them) and the sub-band
    // weights are stored as fp16 (tcgen05 kind::f16, fp32 accumulate; cell state c and all statistics stay fp32)
    bool half = false;
    bool split = false;  // SE_PRECISION_3XTF32: every GEMM in the 3xTF32 form (fp32-accurate products, exact cells)
    bool wide_tiles = true;  // 256-column LSTM tiles where the hidden size allows (SE_B200_FSN_WIDE=0: 128-column tiles)
    bool use_tma = true;     // TMA operand delivery of the fp16 LSTM steps (SE_B200_FSN_TMA=0: cp.async gather)
    int sesz = 4;   // element size of the sub-band records
    int Ksp = 0;    // sub-band input size padded to whole k-blocks (32 floats / 64 halves)
    std::vector<FsnGemm> gemms;  // in launch order, interleaved with the elementwise kernels by enqueue()
    std::map<int, cudaGraphExec_t> graphs;
    cudaStream_t own_stream = nullptr;
    // scratch of se_fsn_realtime_process (grown on demand; see there for which buffer scales with what)
    float *rt_spec = nullptr, *rt_xin = nullptr, *rt_x0 = nullptr, *rt_crm = nullptr, *rt_s = nullptr, *rt_enh = nullptr,
          *rt_chunks = nullptr, *rt_pline = nullptr, *rt_fbout = nullptr;
    size_t rt_rows = 0, rt_rows_train = 0, rt_xin_rows = 0;
    IoDesc* rt_io = nullptr;
    // se_fsn_process_chunk: the overlap-add carry [maxB][K/2] is stream state (allocated with the context, zeroed by
    // se_fsn_reset_state); the step's scratch is allocated for maxB streams on the first call, and its graphs (one per
    // B, each setting its own cells) are kept apart from `graphs`, which holds the bare network
    float* carry = nullptr;
    StateTable state_tab;       // what a stream carries between steps (se_fsn_state_export / _import; state_io.cu)
    uint64_t state_layout = 0;  // hash of the record layout
    float *st_spec = nullptr, *st_xin = nullptr, *st_x0 = nullptr, *st_crm = nullptr, *st_enh = nullptr;
    IoDesc* st_io = nullptr;
    std::map<int, cudaGraphExec_t> step_graphs;
    const float* cur_x = nullptr;  // indirection cell for graph replay
    const float** x_cell = nullptr;
    float** out_cell = nullptr;
};

namespace {

// ---------------------------------------------------------------------------------------------------------------
// elementwise kernels
// ---------------------------------------------------------------------------------------------------------------
// |X| of one (stream, microphone): x [B][2M][F][T] (M real planes, then M imaginary planes; fullsubnet.py:782) ->
// record x part [t][c*F + f], plus the per-stream sum for CumLayerNorm.  grid (M, B)
__global__ void __launch_bounds__(256) fsn_mag_kernel(const float* const* xcell, int M, int F, float* rec, long long recB,
                                                      int Kf, double* sums) {
    extern __shared__ float sm[];  // [F*T]
    const float* x = *xcell;
    const int c = blockIdx.x, b = blockIdx.y;
    const float* re = x + (((long long)b * 2 * M + c) * F) * T;
    const float* im = x + (((long long)b * 2 * M + M + c) * F) * T;
    float part = 0.f;
    for (int i = threadIdx.x; i < F * T; i += blockDim.x) {
        const float r = re[i], q = im[i];
        const float m = sqrtf(r * r + q * q + 1e-8f);
        sm[i] = m;
        part += m;
    }
    __syncthreads();
    float* dst = rec + (long long)b * recB + c * F;
    for (int i = threadIdx.x; i < F * T; i += blockDim.x) {
        const int t = i / F, f = i - t * F;
        dst[(long long)t * Kf + f] = sm[f * T + t];
    }
    __shared__ double red[8];
    double d = part;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
        atomicAdd(sums + 4 * b, s);
    }
}

// CumLayerNorm state update (fullsubnet.py:184-201): mean over the whole per-stream tensor, running average with
// alpha = step/(step+1), step capped at 80; which: 0 = full-band norm, 1 = sub-band norm.  One thread per stream.
__global__ void fsn_cumnorm_kernel(const double* sums, float* cstate, int* cstep, int which, double count, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double total = which == 0 ? sums[4 * b] : sums[4 * b + 1] + sums[4 * b + 2];
    const float mean = (float)(total / count);
    int step = cstep[2 * b + which];
    float run = cstate[4 * b + which];
    if (step == 0) {
        run = mean;  // self.mean is None
    } else {
        const float alpha = (float)step / (float)(step + 1);
        run = alpha * run + (1.0f - alpha) * mean;
    }
    step = step + 1 < 80 ? step + 1 : 80;
    cstep[2 * b + which] = step;
    cstate[4 * b + which] = run;
    cstate[4 * b + 2 + which] = 1.0f / (run + 1e-8f);
}

// in-place division of the magnitudes (the sub-band branch sees the NORMALISED mic-0 plane: fullsubnet.py:788,796),
// reflect-padded mic-0 line P[t][0 .. F+2n) and the sum of the unfolded tensor's mic-0 part.  grid (T, B)
__global__ void __launch_bounds__(256) fsn_scale_fb_kernel(float* rec, long long recB, int Kf, int MF, int F, int nb,
                                                           const float* cstate, float* pline, int Pp, double* sums) {
    const int t = blockIdx.x, b = blockIdx.y;
    const float inv = cstate[4 * b + 2];
    float* row = rec + (long long)b * recB + (long long)t * Kf;
    for (int i = threadIdx.x; i < MF; i += blockDim.x) row[i] *= inv;
    __syncthreads();
    float* P = pline + ((long long)b * T + t) * Pp;
    const int W = 2 * nb + 1;
    float part = 0.f;
    for (int j = threadIdx.x; j < F + 2 * nb; j += blockDim.x) {
        int f = j - nb;  // reflect (no edge repeat), functional.pad(mode="reflect")
        if (f < 0) f = -f;
        if (f > F - 1) f = 2 * (F - 1) - f;
        const float v = row[f];
        P[j] = v;
        const int lo = j - (W - 1) > 0 ? j - (W - 1) : 0, hi = j < F - 1 ? j : F - 1;  // windows f' with f' <= j <= f'+W-1
        part += v * (float)(hi - lo + 1);
    }
    __shared__ double red[8];
    double d = part;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
        atomicAdd(sums + 4 * b + 1, s);
    }
}

// sub-band input of sequence (b, f) at frame t: [P[t][f .. f+W) | fb_out[t][f]] / running mean  (fullsubnet.py:800-814)
// grid (T, B), one thread per (f, k)
__global__ void __launch_bounds__(256) fsn_unfold_kernel(const float* pline, int Pp, const float* fbout, int Fp, int F,
                                                         int W, const float* cstate, float* sbrec, long long recS,
                                                         int Ks, int Ksp, int half) {
    const int t = blockIdx.x, b = blockIdx.y;
    const float inv = cstate[4 * b + 3];
    const float* P = pline + ((long long)b * T + t) * Pp;
    const float* fo = fbout + ((long long)b * T + t) * Fp;
    for (int i = threadIdx.x; i < F * Ks; i += blockDim.x) {
        const int f = i / Ks, k = i - f * Ks;
        float v = 0.f;
        if (k < W) v = P[f + k];
        else if (k == W) v = fo[f];
        const long long o = ((long long)b * F + f) * recS + (long long)t * Ksp + k;
        if (half) reinterpret_cast<__half*>(sbrec)[o] = __float2half_rn(v * inv);
        else sbrec[o] = v * inv;
    }
}

// carried state: h history slot T -> slot 0 for both layers.  grid (rows, ceil(H/256))
template <typename E>
__global__ void fsn_roll_kernel(E* rec, long long recB, long long h0, long long h1, int H) {
    const long long r = blockIdx.x;
    const int j = blockIdx.y * blockDim.x + threadIdx.x;
    if (j >= H) return;
    E* base = rec + r * recB;
    base[h0 + j] = base[h0 + (long long)T * H + j];
    base[h1 + j] = base[h1 + (long long)T * H + j];
}

// [B*F][T][2] -> [B][2][F][T]  (fullsubnet.py:817)
__global__ void fsn_out_kernel(const float* crm, float* const* outcell, int F, long long total) {
    float* out = *outcell;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % T);
        const int f = (int)((i / T) % F);
        const int c = (int)((i / ((long long)T * F)) % 2);
        const long long b = i / ((long long)2 * T * F);
        out[i] = crm[((b * F + f) * T + t) * 2 + c];
    }
}

__global__ void fsn_set_cells(const float** xcell, const float* x, float** outcell, float* out) {
    *xcell = x;
    *outcell = out;
}

__device__ __forceinline__ float decompress_cirm(float m) {  // utility.py:439-442
    const float limit = 9.9f;
    const float ge = (m >= limit) ? 1.f : 0.f;
    const float le = (m <= -limit) ? 1.f : 0.f;
    const float in = (fabsf(m) < limit) ? 1.f : 0.f;
    m = limit * ge - limit * le + m * in;
    return -10.f * logf((10.f - m) / (10.f + m));
}
// crm [R][2][F][T], x [R][2][F][T] (mic-0 real / imaginary) -> enhanced [R][F][T][2]   (fullsubnet.py:949-953)
__global__ void fsn_apply_mask_kernel(const float* crm, const float* x, float* out, int F, int Tn, long long total) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long ft = i % ((long long)F * Tn);
        const long long r = i / ((long long)F * Tn);
        const long long base = r * 2 * F * Tn + ft;
        const float mr = decompress_cirm(crm[base]), mi = decompress_cirm(crm[base + (long long)F * Tn]);
        const float xr = x[base], xi = x[base + (long long)F * Tn];
        out[2 * i] = mr * xr - mi * xi;
        out[2 * i + 1] = mi * xr + mr * xi;
    }
}

// BaseModel.unfold (fullsubnet.py:299-331): [B][C][F][T] -> [B][F][C][2n+1][T], reflect padding of F
__global__ void unfold_kernel(const float* in, float* out, int C, int F, int Tn, int n, long long total) {
    const int W = 2 * n + 1;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % Tn);
        long long r = i / Tn;
        const int k = (int)(r % W);
        r /= W;
        const int c = (int)(r % C);
        r /= C;
        const int f = (int)(r % F);
        const long long b = r / F;
        int g = f + k - n;
        if (g < 0) g = -g;
        if (g > F - 1) g = 2 * (F - 1) - g;
        out[i] = in[((b * C + c) * F + g) * Tn + t];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// program
// ---------------------------------------------------------------------------------------------------------------
void register_params(se_fsn* c) {
    auto add = [&](const std::string& n, std::vector<int> s) { c->wa.params.push_back({n, std::move(s)}); };
    auto seq = [&](const std::string& p, int in, int H, int out) {
        for (int l = 0; l < 2; ++l) {
            const std::string s = std::to_string(l);
            add(p + ".sequence_model.weight_ih_l" + s, {4 * H, l == 0 ? in : H});
            add(p + ".sequence_model.weight_hh_l" + s, {4 * H, H});
            add(p + ".sequence_model.bias_ih_l" + s, {4 * H});
            add(p + ".sequence_model.bias_hh_l" + s, {4 * H});
        }
        add(p + ".fc_output_layer.weight", {out, H});
        add(p + ".fc_output_layer.bias", {out});
    };
    seq("fb_model", c->F * c->M, c->Hf, c->F);
    seq("sb_model", c->Ks, c->Hs, 2);
}

// one LSTM layer: T step GEMMs.  rec/recB: record buffer; xoff(t), hoff(t): offsets of x_t / h_{t-1} inside a record
void build_lstm(se_fsn* c, const std::string& prefix, int layer, int Kin, int Kin_pad, int H, float* rec,
                long long recB, std::function<long long(int)> xoff, long long hhist, float* cbuf, int rows_per_stream,
                bool half = false) {
    const int U = half ? 8 : 4;    // elements per 16-byte gather unit
    const int esz = half ? 2 : 4;
    // hidden units per output tile (the 3xTF32 form has 128-column tiles: 32 units)
    const int U_tile = (H % 64 == 0 && c->wide_tiles && !c->split) ? 64 : 32;
    const int K = Kin_pad + H;
    const int N = 4 * H;
    const size_t w_off = c->wa.reserve_w((size_t)N * K), b_off = c->wa.reserve_w(N);
    const std::string s = std::to_string(layer);
    c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
        const std::vector<float>& wi = hp.at(prefix + ".sequence_model.weight_ih_l" + s);
        const std::vector<float>& wh = hp.at(prefix + ".sequence_model.weight_hh_l" + s);
        const std::vector<float>& bi = hp.at(prefix + ".sequence_model.bias_ih_l" + s);
        const std::vector<float>& bh = hp.at(prefix + ".sequence_model.bias_hh_l" + s);
        for (int n = 0; n < N; ++n) {
            // tile y holds [i | f | g | o] of hidden units U*y .. U*y+U-1 (gemm_tc.cu EPI_LSTM; nn.LSTM gate order i,f,g,o)
            const int src = ((n % (4 * U_tile)) / U_tile) * H + (n / (4 * U_tile)) * U_tile + n % U_tile;
            float* row = arena + w_off + (size_t)n * K;
            for (int k = 0; k < Kin; ++k) row[k] = wi[(size_t)src * Kin + k];
            for (int k = 0; k < H; ++k) row[Kin_pad + k] = wh[(size_t)src * H + k];
            arena[b_off + n] = bi[src] + bh[src];
        }
    });
    for (int t = 0; t < T; ++t) {
        std::vector<int> koff(K / U);
        for (int u = 0; u < Kin_pad / U; ++u) koff[u] = (int)(xoff(t) + U * u);
        for (int u = 0; u < H / U; ++u) koff[Kin_pad / U + u] = (int)(hhist + (long long)t * H + U * u);
        GemmParams g{};
        g.a_half = half ? 1 : 0;
        g.out_half = half ? 1 : 0;
        g.A = rec;
        g.sB = recB;
        g.Tn = 1;
        g.Fo = 1;
        g.K = K;
        g.N = N;
        g.Npad = N;
        g.epi = EPI_LSTM;
        g.lstm_units = U_tile;
        g.out = reinterpret_cast<float*>(reinterpret_cast<char*>(rec) + (hhist + (long long)(t + 1) * H) * esz);  // h_t
        g.oB = recB;
        g.hprev = cbuf;  // c_{t-1}, updated in place; unit-major [H][maxB * rows_per_stream] (gemm_tc.cu EPI_LSTM)
        g.hB = H;
        g.out2 = cbuf;
        g.o2B = H;
        g.c_rows = (long long)c->maxB * rows_per_stream;
        g.H = H;
        const int k_off = c->wa.reserve_k(koff);
        const size_t i = c->gemms.size();
        c->gemms.push_back({g, rows_per_stream});
        c->wa.binds.push_back([=] {
            FsnGemm& e = c->gemms[i];
            e.g.W = half ? static_cast<const void*>(c->wa.wh + w_off) : static_cast<const void*>(c->wa.w + w_off);
            e.g.bias = c->wa.w + b_off;
            e.g.koff = c->wa.k + k_off;
            // fp16 LSTM steps of the sub-band model: TMA operand delivery + CTA pairs (gemm_tc.cu).  A row of the GEMM is
            // one (stream, bin) sequence record; every 64-wide k-block of [x_t | h_{t-1}] is contiguous inside the record,
            // so the A tile of a k-block is ONE 2-D box (64 halves at the block's offset x 128 consecutive records).
            if (!(c->use_tma && half && e.g.sB % 64 == 0)) return 0;
            GemmParams probe = e.g;
            probe.M = rows_per_stream;
            if (!gemm_tma_supported(probe)) return 0;
            const int nkb = K / 64;
            std::vector<int> kc(4 * nkb, 0);
            bool ok = true;
            for (int kb = 0; kb < nkb && ok; ++kb) {
                const int u = c->wa.khost[k_off + 8 * kb];
                for (int j = 1; j < 8; ++j) ok = ok && c->wa.khost[k_off + 8 * kb + j] == u + 8 * j;
                ok = ok && u % 8 == 0;
                kc[4 * kb] = u;
            }
            if (!ok) return 0;
            int* kdev = nullptr;
            if (dev_alloc(c, &kdev, kc.size())) return 1;
            SE_CUDA_OK(cudaMemcpy(kdev, kc.data(), kc.size() * sizeof(int), cudaMemcpyHostToDevice));
            const int nrows = c->maxB * rows_per_stream;
            if (make_gemm_tma(&e.tma, e.g.A, (int)e.g.sB, 1, 1, e.g.sB, e.g.sB, nrows, 1, 1, 1, e.g.W, e.g.K, e.g.Npad,
                              gemm_tma_tile_n(e.g)))
                return 1;
            e.tma.t_org = 0;
            e.tma.f_org = 0;
            e.tma.kcoord = reinterpret_cast<const int4*>(kdev);
            e.tma_ok = true;
            return 0;
        });
    }
}

void build_fc(se_fsn* c, const std::string& prefix, int H, int N, float* rec, long long recB, long long h1hist, int epi,
              float* out, long long oB, long long oT, int vec4, double* stats, int rows_per_stream_T, bool half = false) {
    const int U = half ? 8 : 4;
    const int esz = half ? 2 : 4;
    const int Npad = round_up(N, gemm_tf32_tile_n(N));
    const size_t w_off = c->wa.reserve_w((size_t)Npad * H), b_off = c->wa.reserve_w(Npad);
    c->wa.packers.push_back([=](const HostParams& hp, float* arena) {
        const std::vector<float>& w = hp.at(prefix + ".fc_output_layer.weight");
        const std::vector<float>& b = hp.at(prefix + ".fc_output_layer.bias");
        for (int n = 0; n < N; ++n) {
            for (int k = 0; k < H; ++k) arena[w_off + (size_t)n * H + k] = w[(size_t)n * H + k];
            arena[b_off + n] = b[n];
        }
    });
    std::vector<int> koff(H / U);
    for (int u = 0; u < H / U; ++u) koff[u] = U * u;
    GemmParams g{};
    g.a_half = half ? 1 : 0;
    g.A = reinterpret_cast<char*>(rec) + (h1hist + H) * esz;  // h_1 .. h_T of the top layer
    g.sB = recB;
    g.sT = H;
    g.Tn = T;
    g.Fo = 1;
    g.K = H;
    g.N = N;
    g.Npad = Npad;
    g.epi = epi;
    g.out = out;
    g.oB = oB;
    g.oT = oT;
    g.vec4 = vec4;
    g.stats = stats;
    const int k_off = c->wa.reserve_k(koff);
    const size_t i = c->gemms.size();
    c->gemms.push_back({g, rows_per_stream_T});
    c->wa.binds.push_back([=] {
        GemmParams& e = c->gemms[i].g;
        e.W = half ? static_cast<const void*>(c->wa.wh + w_off) : static_cast<const void*>(c->wa.w + w_off);
        e.bias = c->wa.w + b_off;
        e.koff = c->wa.k + k_off;
        return 0;
    });
}

int build(se_fsn* c) {
    const se_fsn_config& g = c->cfg;
    SE_REQUIRE(g.num_freqs == 201, "FullSubNet: num_freqs must be 201 (config.yaml:154)");
    SE_REQUIRE(g.num_mics >= 1 && g.num_mics <= 4, "FullSubNet: num_mics must be 1..4");
    SE_REQUIRE(g.num_layers == 2, "FullSubNet: num_layers must be 2 (config.yaml:166)");
    SE_REQUIRE(g.fb_num_neighbors == 0, "FullSubNet: fb_num_neighbors must be 0 (config.yaml:157)");
    SE_REQUIRE(g.sb_num_neighbors >= 1 && g.sb_num_neighbors < g.num_freqs, "FullSubNet: bad sb_num_neighbors");
    SE_REQUIRE((2 * g.sb_num_neighbors + 2) % 4 == 0, "FullSubNet: sub-band input size must be a multiple of 4");
    SE_REQUIRE(g.fb_hidden % 32 == 0 && g.sb_hidden % 32 == 0 && g.fb_hidden > 0 && g.sb_hidden > 0,
               "FullSubNet: hidden sizes must be positive multiples of 32");
    SE_REQUIRE(g.max_streams > 0, "FullSubNet: max_streams must be positive");
    c->maxB = g.max_streams;
    c->F = g.num_freqs;
    c->M = g.num_mics;
    c->Hf = g.fb_hidden;
    c->Hs = g.sb_hidden;
    c->NB = 2 * g.sb_num_neighbors + 1;
    c->Ks = c->NB + 1;
    c->Kf = round_up(c->F * c->M, 32) ;  // whole k-blocks, so that [x | h] stays k-block aligned
    SE_REQUIRE(g.precision == SE_PRECISION_TF32 || g.precision == SE_PRECISION_FP16 || g.precision == SE_PRECISION_3XTF32,
               "FullSubNet: precision must be SE_PRECISION_TF32, SE_PRECISION_3XTF32 or SE_PRECISION_FP16");
    c->half = g.precision == SE_PRECISION_FP16;
    c->split = g.precision == SE_PRECISION_3XTF32;
    if (const char* e = getenv("SE_B200_FSN_WIDE")) c->wide_tiles = atoi(e) != 0;
    if (const char* e = getenv("SE_B200_FSN_TMA")) c->use_tma = atoi(e) != 0;
    c->sesz = c->half ? 2 : 4;
    SE_REQUIRE(round_up(c->Ks, 32) == c->Ks, "FullSubNet: sub-band input size must be a multiple of 32 (31 neighbours + 1)");
    c->Ksp = round_up(c->Ks, c->half ? 64 : 32);
    SE_REQUIRE(!c->half || g.sb_hidden % 64 == 0, "FullSubNet fp16: sb_hidden must be a multiple of 64");
    register_params(c);
    const int B = c->maxB, F = c->F, Hf = c->Hf, Hs = c->Hs;
    c->f_h0 = (long long)T * c->Kf;
    c->f_h1 = c->f_h0 + (long long)(T + 1) * Hf;
    c->recF = c->f_h1 + (long long)(T + 1) * Hf;
    c->s_h0 = (long long)T * c->Ksp;
    c->s_h1 = c->s_h0 + (long long)(T + 1) * Hs;
    c->recS = c->s_h1 + (long long)(T + 1) * Hs;
    const int Fp = round_up(F, 4), Pp = round_up(F + 2 * g.sb_num_neighbors, 4);
    if (dev_alloc(c, &c->fbrec, (size_t)c->recF * B)) return 1;
    if (dev_alloc(c, reinterpret_cast<char**>(&c->sbrec), (size_t)c->recS * B * F * c->sesz)) return 1;
    if (dev_alloc(c, &c->fbc, (size_t)2 * B * Hf)) return 1;
    if (dev_alloc(c, &c->sbc, (size_t)2 * B * F * Hs)) return 1;
    if (dev_alloc(c, &c->fbout, (size_t)B * T * Fp)) return 1;
    if (dev_alloc(c, &c->pline, (size_t)B * T * Pp)) return 1;
    if (dev_alloc(c, &c->crm, (size_t)B * F * T * 2)) return 1;
    if (dev_alloc(c, &c->sums, (size_t)4 * B)) return 1;
    if (dev_alloc(c, &c->cstate, (size_t)4 * B)) return 1;
    if (dev_alloc(c, &c->cstep, (size_t)2 * B)) return 1;
    if (dev_alloc(c, &c->carry, (size_t)B * PHOP)) return 1;
    if (dev_alloc(c, &c->x_cell, 1)) return 1;
    if (dev_alloc(c, &c->out_cell, 1)) return 1;
    {  // export / import (state_io.cu): h_T in slot 0 of both records (after fsn_roll_kernel), the cell states, both
       // CumLayerNorms and the step carry.  `sums` is not state: every step zeroes it before it accumulates.
        StateTable& t = c->state_tab;
        t.desc = "fsn freqs=" + std::to_string(F) + " mics=" + std::to_string(c->M) + " fb_hidden=" + std::to_string(Hf) +
                 " sb_hidden=" + std::to_string(Hs) + " layers=" + std::to_string(g.num_layers) + " sb_neighbors=" +
                 std::to_string(g.sb_num_neighbors) + " fb_neighbors=" + std::to_string(g.fb_num_neighbors) +
                 " precision=" + std::to_string(g.precision);
        const long long rF = c->recF * 4, rS = c->recS * c->sesz;
        if (state_table_add(t, "fb_h0", 4, c->fbrec + c->f_h0, rF, Hf * 4LL) ||
            state_table_add(t, "fb_h1", 4, c->fbrec + c->f_h1, rF, Hf * 4LL) ||
            state_table_add(t, "sb_h0", c->sesz, reinterpret_cast<char*>(c->sbrec) + c->s_h0 * c->sesz, F * rS,
                            (long long)Hs * c->sesz, F, rS) ||
            state_table_add(t, "sb_h1", c->sesz, reinterpret_cast<char*>(c->sbrec) + c->s_h1 * c->sesz, F * rS,
                            (long long)Hs * c->sesz, F, rS) ||
            // cell states, unit-major [layer][H][maxB (* F)]: one column (F columns) per stream in each of 2H unit rows
            state_table_add(t, "fb_c", 4, c->fbc, 4, 4, 2 * Hf, (long long)B * 4) ||
            state_table_add(t, "sb_c", 4, c->sbc, F * 4LL, F * 4LL, 2 * Hs, (long long)B * F * 4) ||
            state_table_add(t, "cstate", 4, c->cstate, 16, 16) || state_table_add(t, "cstep", 4, c->cstep, 8, 8) ||
            state_table_add(t, "carry", 4, c->carry, PHOP * 4LL, PHOP * 4LL))
            return 1;
        c->state_layout = state_layout_hash(t);
    }

    const long long recF = c->recF, recS = c->recS;
    const int Kf = c->Kf, Ks = c->Ks;
    const long long fh0 = c->f_h0, fh1 = c->f_h1, sh0 = c->s_h0, sh1 = c->s_h1;
    // gemm order: fb l0 (T), fb l1 (T), fb fc, sb l0 (T), sb l1 (T), sb fc
    build_lstm(c, "fb_model", 0, F * c->M, Kf, Hf, c->fbrec, recF, [=](int t) { return (long long)t * Kf; }, fh0, c->fbc, 1);
    build_lstm(c, "fb_model", 1, Hf, Hf, Hf, c->fbrec, recF, [=](int t) { return fh0 + (long long)(t + 1) * Hf; }, fh1,
               c->fbc + (size_t)B * Hf, 1);
    build_fc(c, "fb_model", Hf, F, c->fbrec, recF, fh1, EPI_RELU_STATS, c->fbout, (long long)T * Fp, Fp, 1, nullptr, T);
    const int Ksp = c->Ksp;
    build_lstm(c, "sb_model", 0, Ks, Ksp, Hs, c->sbrec, recS, [=](int t) { return (long long)t * Ksp; }, sh0, c->sbc, F,
               c->half);
    build_lstm(c, "sb_model", 1, Hs, Hs, Hs, c->sbrec, recS, [=](int t) { return sh0 + (long long)(t + 1) * Hs; }, sh1,
               c->sbc + (size_t)B * F * Hs, F, c->half);
    build_fc(c, "sb_model", Hs, 2, c->sbrec, recS, sh1, EPI_BIAS, c->crm, 2LL * T, 2, 0, nullptr, F * T, c->half);

    c->wa.half = c->half;
    if (c->wa.allocate(c->allocs)) return 1;
    return init_fft_tables();  // se_fsn_realtime_process frames and transforms on this device
}

int run_gemm(se_fsn* c, int i, int B, cudaStream_t st) {
    const FsnGemm& e = c->gemms[i];
    GemmParams g = e.g;
    g.M = B * e.rows_per_stream;
    if (e.tma_ok) return launch_gemm_tma(g, e.tma, st);
    return launch_gemm_tf32(g, st, c->split);
}

// The chunk step in four phases.  whole = 0: the streaming chunk step (fullsubnet.py:932-945), both CumLayerNorms advance
// once per chunk.  whole = 1 (train=True, :921-927: all chunks as ONE forward): the caller runs phase 0 over all chunks
// first (sum of |X| over the whole utterance), one full-band norm update, phase 1 over all chunks (full-band model, sums
// of the sub-band input), one sub-band norm update, phase 2 over all chunks.
int phase_mag(se_fsn* c, int B, cudaStream_t st) {  // |X| -> full-band record, sum of |X|
    fsn_mag_kernel<<<dim3(c->M, B), 256, (size_t)c->F * T * sizeof(float), st>>>(c->x_cell, c->M, c->F, c->fbrec, c->recF,
                                                                               c->Kf, c->sums);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}
int phase_norm(se_fsn* c, int which, double count, int B, cudaStream_t st) {
    fsn_cumnorm_kernel<<<(B + 127) / 128, 128, 0, st>>>(c->sums, c->cstate, c->cstep, which, count, B);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}
int phase_fullband(se_fsn* c, int B, cudaStream_t st) {  // scale, reflect-padded line, full-band LSTM + Linear + ReLU
    const int F = c->F, M = c->M;
    const int Pp = round_up(F + 2 * c->cfg.sb_num_neighbors, 4);
    fsn_scale_fb_kernel<<<dim3(T, B), 256, 0, st>>>(c->fbrec, c->recF, c->Kf, M * F, F, c->cfg.sb_num_neighbors,
                                                    c->cstate, c->pline, Pp, c->sums);
    int gi = 0;
    for (int i = 0; i < 2 * T; ++i)
        if (run_gemm(c, gi++, B, st)) return 1;
    {  // fb fc + ReLU; its statistics slot is sums[b][2..3]
        GemmParams g = c->gemms[gi].g;
        g.M = B * c->gemms[gi].rows_per_stream;
        g.stats = c->sums + 2;
        g.stats_stride = 4;  // sums holds 4 doubles per stream
        if (launch_gemm_tf32(g, st, c->split)) return 1;
    }
    fsn_roll_kernel<float><<<dim3(B, (c->Hf + 255) / 256), 256, 0, st>>>(c->fbrec, c->recF, c->f_h0, c->f_h1, c->Hf);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}
int phase_subband(se_fsn* c, int B, cudaStream_t st) {  // unfold, sub-band LSTM + Linear, compressed cIRM out
    const int F = c->F, Hs = c->Hs;
    const int Fp = round_up(F, 4), Pp = round_up(F + 2 * c->cfg.sb_num_neighbors, 4);
    fsn_unfold_kernel<<<dim3(T, B), 256, 0, st>>>(c->pline, Pp, c->fbout, Fp, F, c->NB, c->cstate, c->sbrec, c->recS,
                                                  c->Ks, c->Ksp, c->half ? 1 : 0);
    int gi = 2 * T + 1;
    for (int i = 0; i < 2 * T; ++i)
        if (run_gemm(c, gi++, B, st)) return 1;
    if (run_gemm(c, gi++, B, st)) return 1;
    const long long total = (long long)B * 2 * F * T;
    fsn_out_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(c->crm, c->out_cell, F, total);
    if (c->half)
        fsn_roll_kernel<__half><<<dim3(B * F, (Hs + 255) / 256), 256, 0, st>>>(reinterpret_cast<__half*>(c->sbrec), c->recS,
                                                                             c->s_h0, c->s_h1, Hs);
    else
        fsn_roll_kernel<float><<<dim3(B * F, (Hs + 255) / 256), 256, 0, st>>>(c->sbrec, c->recS, c->s_h0, c->s_h1, Hs);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int enqueue(se_fsn* c, int B, cudaStream_t st) {
    SE_CUDA_OK(cudaMemsetAsync(c->sums, 0, (size_t)4 * c->maxB * sizeof(double), st));
    if (phase_mag(c, B, st)) return 1;
    if (phase_norm(c, 0, (double)c->M * c->F * T, B, st)) return 1;
    if (phase_fullband(c, B, st)) return 1;
    if (phase_norm(c, 1, (double)c->F * c->Ks * T, B, st)) return 1;
    return phase_subband(c, B, st);
}

// spectrum [R][M][F][T][2] (se_stft layout) -> x [R][2M][F][T] (M real planes, then M imaginary planes; fullsubnet.py:
// 835-844) and, optionally, the mic-0 pair x0 [R][2][F][T] (:950)
__global__ void fsn_planes_kernel(const float* spec, int M, int F, float* x, float* x0, long long total) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long ft = i % ((long long)F * T);
        const long long rm = i / ((long long)F * T);
        const int m = (int)(rm % M);
        const long long r = rm / M;
        const float2 v = reinterpret_cast<const float2*>(spec)[i];
        if (x) {
            x[((r * 2 * M + m) * F) * T + ft] = v.x;
            x[((r * 2 * M + M + m) * F) * T + ft] = v.y;
        }
        if (x0 && m == 0) {
            x0[(r * 2 * F) * T + ft] = v.x;
            x0[((r * 2 + 1) * F) * T + ft] = v.y;
        }
    }
}

// The streaming step of se_fsn_process_chunk for streams [0, B): framing + STFT of the chunk the IoDesc cell st_io
// describes, network input and mic-0 pair, the chunk network on them, decompress_cIRM + complex mask (the arithmetic of
// se_fsn_realtime_process), iSTFT and the overlap-add with the carried half, written where st_io points.
int enqueue_step(se_fsn* c, int B, cudaStream_t st) {
    StftParams sp{};
    sp.io = c->st_io;
    sp.B = B;
    sp.M = c->M;
    sp.spec_ref = c->st_spec;
    if (launch_stft_features(sp, st)) return 1;
    const long long total = (long long)B * c->M * c->F * T;
    fsn_planes_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(c->st_spec, c->M, c->F, c->st_xin, c->st_x0, total);
    fsn_set_cells<<<1, 1, 0, st>>>(c->x_cell, c->st_xin, c->out_cell, c->st_crm);
    SE_CUDA_OK(cudaGetLastError());
    if (enqueue(c, B, st)) return 1;
    if (se_fsn_apply_mask(c->st_crm, c->st_x0, c->st_enh, B, c->F, T, st)) return 1;
    MaskIstftParams mp{};
    mp.io = c->st_io;
    mp.B = B;
    mp.spec_in = c->st_enh;
    mp.carry = c->carry;
    return launch_mask_istft(mp, st);
}

int run_chunk_graph(se_fsn* c, int B, cudaStream_t st) {
    return replay_graph(c->graphs, &c->own_stream, B, [=](cudaStream_t s) { return enqueue(c, B, s); }, st);
}

template <typename Tp>
int regrow(se_fsn* c, Tp** buf, size_t count) {  // scratch: freed and re-allocated larger (registered for destroy)
    if (*buf) {
        for (void*& q : c->allocs)
            if (q == *buf) q = nullptr;
        SE_CUDA_OK(cudaFree(*buf));
        *buf = nullptr;
    }
    return dev_alloc(c, buf, count);
}

}  // namespace

extern "C" {

int se_fsn_create(se_fsn** out, int device, const se_fsn_config* cfg) {
    if (!out || !cfg) {
        set_error("se_fsn_create: null argument");
        return 2;
    }
    *out = nullptr;
    if (const int rc = check_create_device(device, "se_fsn_create")) return rc;
    se_fsn* c = new se_fsn();
    c->cfg = *cfg;
    c->device = device;
    if (build(c)) {
        se_fsn_destroy(c);
        return 1;
    }
    *out = c;
    return 0;
}

int se_fsn_destroy(se_fsn* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto& kv : c->graphs) cudaGraphExecDestroy(kv.second);
    for (auto& kv : c->step_graphs) cudaGraphExecDestroy(kv.second);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    for (void* p : c->allocs) cudaFree(p);
    delete c;
    return 0;
}

int se_fsn_num_params(const se_fsn* c) { return c ? (int)c->wa.params.size() : 0; }
const char* se_fsn_param_name(const se_fsn* c, int i) {
    return (c && i >= 0 && i < (int)c->wa.params.size()) ? c->wa.params[i].name.c_str() : nullptr;
}
int64_t se_fsn_param_numel(const se_fsn* c, int i) {
    return (c && i >= 0 && i < (int)c->wa.params.size()) ? c->wa.params[i].numel() : -1;
}

int se_fsn_bind_weights(se_fsn* c, const float* const* ptrs, int n, void* stream) {
    SE_REQUIRE(c != nullptr && ptrs != nullptr, "se_fsn_bind_weights: null argument");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return c->wa.upload(ptrs, n, (cudaStream_t)stream, "se_fsn_bind_weights");
}

int se_fsn_reset_state(se_fsn* c, int first, int count, void* stream) {
    SE_REQUIRE(c != nullptr, "null context");
    SE_REQUIRE(first >= 0 && count >= 0 && first + count <= c->maxB, "se_fsn_reset_state: stream range");
    SE_CUDA_OK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t F = c->F;
    // zero LSTM states (fullsubnet.py:826-830) and reset both CumLayerNorms (:831-832)
    SE_CUDA_OK(cudaMemsetAsync(c->fbrec + c->recF * first, 0, (size_t)c->recF * count * sizeof(float), st));
    SE_CUDA_OK(cudaMemsetAsync(reinterpret_cast<char*>(c->sbrec) + (size_t)c->recS * first * F * c->sesz, 0,
                               (size_t)c->recS * count * F * c->sesz, st));
    for (int l = 0; l < 2; ++l) {
        // cell states are unit-major [layer][H][maxB (* F)]: the streams' columns of every unit row
        if (count > 0) {
            SE_CUDA_OK(cudaMemset2DAsync(c->fbc + (size_t)l * c->maxB * c->Hf + first, (size_t)c->maxB * sizeof(float), 0,
                                         (size_t)count * sizeof(float), (size_t)c->Hf, st));
            SE_CUDA_OK(cudaMemset2DAsync(c->sbc + (size_t)l * c->maxB * F * c->Hs + (size_t)first * F,
                                         (size_t)c->maxB * F * sizeof(float), 0, (size_t)count * F * sizeof(float),
                                         (size_t)c->Hs, st));
        }
    }
    SE_CUDA_OK(cudaMemsetAsync(c->cstate + 4 * (size_t)first, 0, 4 * (size_t)count * sizeof(float), st));
    SE_CUDA_OK(cudaMemsetAsync(c->cstep + 2 * (size_t)first, 0, 2 * (size_t)count * sizeof(int), st));
    // overlap-add carry of se_fsn_process_chunk
    SE_CUDA_OK(cudaMemsetAsync(c->carry + (size_t)PHOP * first, 0, (size_t)PHOP * count * sizeof(float), st));
    return 0;
}

int64_t se_fsn_state_bytes_per_stream(const se_fsn* c) { return c ? c->state_tab.record_bytes : -1; }

uint64_t se_fsn_state_layout(const se_fsn* c) { return c ? c->state_layout : 0; }

int se_fsn_state_export(se_fsn* c, const int32_t* rows_host, int n, void* dst_dev, void* stream) {
    NvtxRange nvtx_range("se.fsn_state_export");
    SE_REQUIRE(c != nullptr, "null context");
    if (state_rows_check(rows_host, n, c->maxB, false, "se_fsn_state_export")) return 2;
    SE_REQUIRE(n == 0 || (dst_dev != nullptr && reinterpret_cast<uintptr_t>(dst_dev) % 16 == 0),
               "se_fsn_state_export: dst must be a 16-byte aligned device buffer");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return launch_state_pack(c->state_tab, rows_host, n, dst_dev, (cudaStream_t)stream);
}

int se_fsn_state_import(se_fsn* c, const int32_t* rows_host, int n, const void* src_dev, uint64_t layout, void* stream) {
    NvtxRange nvtx_range("se.fsn_state_import");
    SE_REQUIRE(c != nullptr, "null context");
    SE_REQUIRE(layout == c->state_layout,
               "se_fsn_state_import: record layout mismatch (records from another model, configuration or precision; "
               "this context:" + c->state_tab.desc + ")");
    if (state_rows_check(rows_host, n, c->maxB, true, "se_fsn_state_import")) return 2;
    SE_REQUIRE(n == 0 || (src_dev != nullptr && reinterpret_cast<uintptr_t>(src_dev) % 16 == 0),
               "se_fsn_state_import: src must be a 16-byte aligned device buffer");
    SE_CUDA_OK(cudaSetDevice(c->device));
    return launch_state_unpack(c->state_tab, rows_host, n, src_dev, (cudaStream_t)stream);
}

int se_fsn_forward_chunk(se_fsn* c, const float* x, float* out, int B, void* stream) {
    NvtxRange nvtx_range("se.fsn_forward_chunk");
    SE_REQUIRE(c != nullptr && c->wa.bound, "se_fsn_forward_chunk: context without weights");
    SE_REQUIRE(x != nullptr && out != nullptr, "se_fsn_forward_chunk: null buffer");
    SE_REQUIRE(B >= 0 && B <= c->maxB, "se_fsn_forward_chunk: B exceeds max_streams");
    if (B == 0) return 0;
    SE_CUDA_OK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    fsn_set_cells<<<1, 1, 0, st>>>(c->x_cell, x, c->out_cell, out);
    return run_chunk_graph(c, B, st);
}

int se_fsn_process_chunk(se_fsn* c, const float* in, int64_t in_stream_stride, int64_t in_mic_stride, float* out,
                         int64_t out_stream_stride, int B, void* stream) {
    NvtxRange nvtx_range("se.fsn_chunk_step");
    SE_REQUIRE(c != nullptr && c->wa.bound, "se_fsn_process_chunk: context without weights");
    SE_REQUIRE(in != nullptr && out != nullptr, "se_fsn_process_chunk: null buffer");
    SE_REQUIRE(B >= 0 && B <= c->maxB, "se_fsn_process_chunk: B exceeds max_streams");
    SE_REQUIRE(c->M <= 3, "se_fsn_process_chunk: the framing kernel serves at most 3 microphones");
    if (B == 0) return 0;
    SE_CUDA_OK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (!c->st_io) {  // the step's scratch, for the context's capacity: a graph captured for one B keeps its pointers
        const size_t per = (size_t)c->F * T, R = c->maxB;
        if (dev_alloc(c, &c->st_spec, R * c->M * per * 2)) return 1;
        if (dev_alloc(c, &c->st_xin, R * 2 * c->M * per)) return 1;
        if (dev_alloc(c, &c->st_x0, R * 2 * per)) return 1;
        if (dev_alloc(c, &c->st_crm, R * 2 * per)) return 1;
        if (dev_alloc(c, &c->st_enh, R * 2 * per)) return 1;
        if (dev_alloc(c, &c->st_io, 1)) return 1;
    }
    IoDesc io{in, in_stream_stride, in_mic_stride, 0, KCHUNK, out, out_stream_stride, PHOP};
    if (launch_set_io(c->st_io, io, st)) return 1;
    return replay_graph(c->step_graphs, &c->own_stream, B, [=](cudaStream_t s) { return enqueue_step(c, B, s); }, st);
}

int se_fsn_realtime_process(se_fsn* c, const float* mixture, const float* source, int B, int64_t L, int flag, int train,
                            float* pred, float* crm_out, float* s_out, float* x0_out, void* stream) {
    NvtxRange nvtx_range("se.fsn_realtime_process");
    SE_REQUIRE(c != nullptr && c->wa.bound, "se_fsn_realtime_process: context without weights");
    SE_REQUIRE(mixture != nullptr && pred != nullptr && L > 0, "se_fsn_realtime_process: null buffer");
    SE_REQUIRE(B >= 1 && B <= c->maxB, "se_fsn_realtime_process: B exceeds max_streams");
    SE_REQUIRE(c->M <= 3, "se_fsn_realtime_process: the framing kernel serves at most 3 microphones");
    SE_CUDA_OK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int F = c->F, M = c->M, K = 3200, P = K / 2;
    const int front = flag ? 0 : P;  // fullsubnet.py:905-908
    int gap = 0, N = 0;
    if (se_chunk_grid(L + front, K, &gap, &N)) return 1;
    const size_t R = (size_t)N * B;
    const size_t per = (size_t)F * T;
    const int Fp = round_up(F, 4), Pp = round_up(F + 2 * c->cfg.sb_num_neighbors, 4);
    // Scratch, kept across calls.  The buffers of one chunk of every stream (the spectrum rt_spec, and with train=False
    // the network input rt_xin) scale with the streams B; they are sized for the context's capacity maxB, since a later
    // call may bring more streams in fewer chunks.  The buffers of every chunk of every stream (rt_x0, rt_crm, rt_s,
    // rt_enh, rt_chunks; with train=True also rt_xin, rt_pline and rt_fbout) scale with the rows R = N * B and grow with R.
    if (!c->rt_spec && dev_alloc(c, &c->rt_spec, (size_t)c->maxB * M * per * 2)) return 1;
    const size_t xin_rows = train ? R : (size_t)B;
    if (xin_rows > c->rt_xin_rows) {
        c->rt_xin_rows = xin_rows > (size_t)c->maxB ? xin_rows : (size_t)c->maxB;
        if (regrow(c, &c->rt_xin, c->rt_xin_rows * 2 * M * per)) return 1;
    }
    if (R > c->rt_rows) {
        if (regrow(c, &c->rt_x0, R * 2 * per)) return 1;
        if (regrow(c, &c->rt_crm, R * 2 * per)) return 1;
        if (regrow(c, &c->rt_s, R * 2 * per)) return 1;
        if (regrow(c, &c->rt_enh, R * 2 * per)) return 1;
        if (regrow(c, &c->rt_chunks, R * K)) return 1;
        if (!c->rt_io && dev_alloc(c, &c->rt_io, 1)) return 1;
        c->rt_rows = R;
    }
    if (train && R > c->rt_rows_train) {  // train=True keeps every chunk's full-band results
        if (regrow(c, &c->rt_pline, R * T * Pp)) return 1;
        if (regrow(c, &c->rt_fbout, R * T * Fp)) return 1;
        c->rt_rows_train = R;
    }
    if (!flag && se_fsn_reset_state(c, 0, B, stream)) return 1;  // :913-915
    float* crm_all = crm_out ? crm_out : c->rt_crm;
    float* x0_all = x0_out ? x0_out : c->rt_x0;
    // STFT of chunk n of every stream straight from the signal: the zero padding of utility.padding (P samples in front,
    // gap + P behind) and the front pad of :905-908 are the out-of-range reads of the framing kernel
    auto stft_chunk = [&](const float* sig, int n, float* xin, float* x0) -> int {
        IoDesc io{sig, (long long)M * L, L, -(long long)P - front + (long long)n * P, L, nullptr, 0, 0};
        if (launch_set_io(c->rt_io, io, st)) return 1;
        StftParams sp{};
        sp.io = c->rt_io;
        sp.B = B;
        sp.M = M;
        sp.spec_ref = c->rt_spec;
        if (launch_stft_features(sp, st)) return 1;
        const long long total = (long long)B * M * per;
        fsn_planes_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(c->rt_spec, M, F, xin, x0, total);
        SE_CUDA_OK(cudaGetLastError());
        return 0;
    };
    if (!train) {
        for (int n = 0; n < N; ++n) {  // strictly serial: LSTM states and running norms are carried (:932-945)
            if (stft_chunk(mixture, n, c->rt_xin, x0_all + (size_t)n * B * 2 * per)) return 1;
            fsn_set_cells<<<1, 1, 0, st>>>(c->x_cell, c->rt_xin, c->out_cell, crm_all + (size_t)n * B * 2 * per);
            if (run_chunk_graph(c, B, st)) return 1;
        }
    } else {
        const size_t xin_chunk = (size_t)B * 2 * M * per;
        SE_CUDA_OK(cudaMemsetAsync(c->sums, 0, (size_t)4 * c->maxB * sizeof(double), st));
        for (int n = 0; n < N; ++n) {
            if (stft_chunk(mixture, n, c->rt_xin + n * xin_chunk, x0_all + (size_t)n * B * 2 * per)) return 1;
            fsn_set_cells<<<1, 1, 0, st>>>(c->x_cell, c->rt_xin + n * xin_chunk, c->out_cell, crm_all);
            if (phase_mag(c, B, st)) return 1;
        }
        if (phase_norm(c, 0, (double)M * F * T * N, B, st)) return 1;  // ONE CumLayerNorm step over all N*T frames
        SE_CUDA_OK(cudaMemsetAsync(c->sums, 0, (size_t)4 * c->maxB * sizeof(double), st));
        for (int n = 0; n < N; ++n) {
            fsn_set_cells<<<1, 1, 0, st>>>(c->x_cell, c->rt_xin + n * xin_chunk, c->out_cell, crm_all);
            if (phase_mag(c, B, st)) return 1;  // re-creates the record of this chunk (its sum slot is not used again)
            if (phase_fullband(c, B, st)) return 1;
            SE_CUDA_OK(cudaMemcpyAsync(c->rt_pline + (size_t)n * B * T * Pp, c->pline, (size_t)B * T * Pp * sizeof(float),
                                       cudaMemcpyDeviceToDevice, st));
            SE_CUDA_OK(cudaMemcpyAsync(c->rt_fbout + (size_t)n * B * T * Fp, c->fbout, (size_t)B * T * Fp * sizeof(float),
                                       cudaMemcpyDeviceToDevice, st));
        }
        if (phase_norm(c, 1, (double)F * c->Ks * T * N, B, st)) return 1;
        for (int n = 0; n < N; ++n) {
            SE_CUDA_OK(cudaMemcpyAsync(c->pline, c->rt_pline + (size_t)n * B * T * Pp, (size_t)B * T * Pp * sizeof(float),
                                       cudaMemcpyDeviceToDevice, st));
            SE_CUDA_OK(cudaMemcpyAsync(c->fbout, c->rt_fbout + (size_t)n * B * T * Fp, (size_t)B * T * Fp * sizeof(float),
                                       cudaMemcpyDeviceToDevice, st));
            fsn_set_cells<<<1, 1, 0, st>>>(c->x_cell, c->rt_xin + n * xin_chunk, c->out_cell,
                                           crm_all + (size_t)n * B * 2 * per);
            if (phase_subband(c, B, st)) return 1;
        }
    }
    if (source != nullptr && s_out != nullptr)  // spectrum of the clean source, mic 0 (:880-886), returned to the caller
        for (int n = 0; n < N; ++n)
            if (stft_chunk(source, n, nullptr, s_out + (size_t)n * B * 2 * per)) return 1;
    // decompress_cIRM + complex mask (:949-953), per-chunk iSTFT and the 50 % chunk overlap-add (:955-957)
    if (se_fsn_apply_mask(crm_all, x0_all, c->rt_enh, (int)R, F, T, stream)) return 1;
    MaskIstftParams mp{};
    mp.B = (int)R;
    mp.spec_in = c->rt_enh;
    mp.out_chunk = c->rt_chunks;
    if (launch_mask_istft(mp, st)) return 1;
    return launch_over_add_cm(c->rt_chunks, B, N, K, front, L, pred, st);
}

int se_fsn_planes(const float* spec, int R, int M, int F, int Tn, float* x, float* x0, void* stream) {
    SE_REQUIRE(spec != nullptr && (x != nullptr || x0 != nullptr), "se_fsn_planes: null buffer");
    SE_REQUIRE(R >= 0 && M >= 1 && F >= 1 && Tn == T, "se_fsn_planes: bad shape (T must be 21)");
    const long long total = (long long)R * M * F * T;
    if (total == 0) return 0;
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 32) grid = 148 * 32;
    fsn_planes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(spec, M, F, x, x0, total);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int se_fsn_apply_mask(const float* crm, const float* x, float* out, int R, int F, int Tn, void* stream) {
    SE_REQUIRE(crm != nullptr && x != nullptr && out != nullptr, "se_fsn_apply_mask: null buffer");
    const long long total = (long long)R * F * Tn;
    if (total <= 0) return 0;
    long long grid = (total + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    fsn_apply_mask_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(crm, x, out, F, Tn, total);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

int se_unfold(const float* in, int B, int C, int F, int Tn, int num_neighbor, float* out, void* stream) {
    SE_REQUIRE(in != nullptr && out != nullptr, "se_unfold: null buffer");
    SE_REQUIRE(num_neighbor >= 0 && num_neighbor < F, "se_unfold: reflect padding needs num_neighbor < F");
    const long long total = (long long)B * F * C * (2 * num_neighbor + 1) * Tn;
    if (total <= 0) return 0;
    long long grid = (total + 255) / 256;
    if (grid > 148 * 32) grid = 148 * 32;
    unfold_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(in, out, C, F, Tn, num_neighbor, total);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
