// Engine + C-ABI (include/facodec_b200.h): checkpoint folding/packing, workspace, and the
// launch sequences of Encoder.forward (dac/model/dac.py:69-104), FAquantizer.forward_v2
// (modules/quantize.py:375-454) and Decoder.forward (dac/model/dac.py:131-165).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/facodec_b200.h"
#include "../../include/facodec_b200_debug.h"
#include "common.cuh"
#include "kernels.h"

using namespace fac;

namespace {

constexpr int HOP = 300;
constexpr int LATENT = 1024;
constexpr int N_FFT = 2048;
constexpr int WIN = 1200;
constexpr int N_BINS = 1025;
constexpr int SPEC_LD = 2052;   // 2*1025 rounded up to a multiple of 4
constexpr int SPEC_TC_LD = 2176; // ... and to 17 channel tiles of 128 for the tensor-core DFT
constexpr int N_MELS = 80;

struct HostTensor {
    std::vector<float> data;
    std::vector<int64_t> shape;
    size_t numel() const { size_t n = 1; for (auto s : shape) n *= (size_t)s; return n; }
};

struct ConvW {
    size_t w = 0, b = 0; int Cin = 0, Cout = 0, K = 1, ldw = 0;
    // tensor-core blob (conv_tc.cu): present when the layer is eligible
    bool tc = false; size_t tcw = 0; int vf = 1, Kr = 0, tcN = 0;   // tcN: channel tile the blob was laid out for
    bool promoted = false;   // blob built for conv_tcp_kernel (layers upstream of the VQ)
    bool has16 = false; size_t tcw16 = 0;   // 16-bit-operand blob: bf16 hi/lo (non-promoted layers) or fp16 hi / scaled lo (promoted)
    bool has_f16s = false; size_t tcw_f16s = 0;   // hi-only fp16 blob: the one-pass class of the k = 7 convs downstream of the VQ
    bool has_tt = false; size_t tcw_tt = 0; // transposed-formulation blob (conv_tt_kernel, promoted layers): [co tile of 128][chunk][tap][hi|lo']
};
struct SnakeW { size_t a = 0, ia = 0; int C = 0; };
struct LstmW { ConvW ih[2]; size_t whh[2] = {0, 0}; size_t whh16[2] = {0, 0}; bool has16 = false; int H = 0, U = 0, G = 0;
               size_t whh2[2][2] = {{0, 0}, {0, 0}}; bool has2[2] = {false, false}; };   // lstm2 packs: [layer][pass3]
struct ResW { SnakeW s1; ConvW c7; SnakeW s2; ConvW c1; int dil = 1; };
struct VqW { size_t w_in, b_in, cb, cbn, cbn2, w_out, b_out; };

struct EncW {
    ConvW conv0;
    struct Block { ResW res[3]; SnakeW snake; ConvW down; int stride; } blk[4];
    LstmW lstm; SnakeW snake; ConvW conv_out;
};
struct DecW {
    ConvW conv0; LstmW lstm;
    struct Block { SnakeW snake; ConvW up; int stride; int cout; ResW res[3]; } blk[4];
    SnakeW snake; ConvW conv_out;
    bool causal = true, has_lstm = true;   // the redecoder's decoder: causal = false, no SLSTM (config_redecoder.yml)
};
// modules/redecoder.py Redecoder(encoder_type = "wavenet"): embeddings + WN(512, k5, 16 layers, gin 1024) + conv_out
struct RedW {
    size_t emb_p = 0, emb_c[2] = {0, 0};
    ConvW cond, wn_in[16], wn_rs[16], conv_out;
    int hidden = 512, layers = 16;
};
struct QuantW {
    VqW vq[6];
    ConvW spec0, spec3, glu[2], cq, ck, cv, co, fc, timbre_linear;
    ConvW mel_lin, wn_in[8], wn_rs[8], mel_lin2;
    ConvW dft; size_t fb = 0;
    ConvW dft_tc;      // same basis as a K=1 GEMM over gathered frames: Cin = 1200, Cout padded to 2176 (17 x 128)
};
struct RvqSet { int nq; VqW vq[8]; };

}  // namespace

struct fac_handle {
    int device = 0;
    std::string err;
    std::map<std::string, HostTensor> host[FAC_NUM_MODULES];
    bool have[FAC_NUM_MODULES] = {false, false, false, false, false};
    bool finalized = false;
    std::vector<float> pack;        // host staging of the weight arena
    float* warena = nullptr; size_t wfloats = 0;
    EncW enc; DecW dec; QuantW qw;
    RedW red; DecW dec2;            // voice-conversion model: Redecoder + its non-causal, LSTM-free decoder
    std::vector<RvqSet> rvqs; std::vector<float*> rvq_arenas;
    struct Stream;                  // chunked (streaming) encoder / decoder state (fac_stream_*)
    std::vector<Stream*> streams;
    struct HeadSet;                 // modules/quantize.py:106-125 CNNLSTM instances (fac_head_*)
    std::vector<HeadSet*> heads;
    char* ws = nullptr; size_t ws_bytes = 0;
    int launches = 0;
    // tcgen05 3xTF32 path (fac_set_option "tensor_cores"): 0 = never, 1 = layers downstream of the VQ only
    // (decoder, timbre branch), 2 = every eligible layer (default; promoted accumulation upstream of the VQ)
    int use_tc = 2;
    int fuse_res = 1;               // fused ResidualUnit launches (fac_set_option "fuse_resunit"); 2 = only where the
                                    // fused tile still allows two CTAs per SM (C <= 128)
    int lstm_v2 = 1;                // fac_set_option "lstm_v2": resident-W fp16 recurrence kernel (lstm2.cu); 0 = round-1 kernel
    int dec_lstm_fp16 = 1;          // fac_set_option "decoder_lstm_fp16": downstream LSTMs run ONE fp16 pass (0 = bf16 hi/lo 3-pass)
    int enc_mufu = 0;               // fac_set_option "encoder_snake_mufu" (experiment)
    int attn_stream = 0;            // fac_set_option "attention_stream": 1 forces the recomputing attention kernel (test aid)
    int dec_c7_f16 = 1;             // fac_set_option "decoder_conv7_fp16": k = 7 convs downstream of the VQ take ONE fp16 pass (0 = bf16 hi/lo 3-pass)
    int enc_tt = 1;                 // fac_set_option "encoder_tt": promoted layers run the transposed kernel (conv_tt_kernel)
    int enc_f16 = 0;                // fac_set_option "encoder_f16x2": promoted layers use the fp16 hi + scaled-lo split
    int tc_occ2 = 256;              // fac_set_option "tc_occ2_maxn": conv_tc tiles with N <= this are planned for two CTAs per SM (0 = off)
    bool dec_bf16 = true;           // decoder-side layers use the bf16x3 split (fac_set_option "decoder_bf16")
    // second stream for the waveform-only half of the quantizer (fac_set_option "overlap_front")
    int overlap_front = 1; cudaStream_t side = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    float* aa_filter = nullptr;
    // dataset-side mel (meldataset.py:29-47: MelSpectrogram with its default sample_rate 16000): own constants, built lazily
    float* mel16_arena = nullptr; ConvW mel16_dft, mel16_dft_tc; size_t mel16_fb = 0;
    // losses.py:65-89 reconstruction_loss: per scale s = 64 << i the window-folded DFT basis [s][ld] (+ tensor-core blobs)
    // and the 64-band HTK filterbank [n_fft/2 + 1][64]; built on first use
    struct LossScale { ConvW dft; size_t fb = 0; int s = 0, nfft = 0, nb = 0, ld = 0; };
    float* loss_arena = nullptr; LossScale loss_scale[6];
    // dac/nn/loss.py MultiScaleSTFTLoss / MelSpectrogramLoss: one cached configuration (rebuilt when the arguments change)
    struct SpecScale { ConvW dft; size_t fb = 0; int w = 0, nb = 0, ld = 0, n_out = 0; bool mel = false; };
    float* spec_arena = nullptr; std::vector<SpecScale> spec_scales; std::vector<double> spec_key;
    // optional per-kernel-family timing (fac_profile_*): CUDA events around every launch
    bool profiling = false;
    struct ProfRec { std::string name; cudaEvent_t a, b; double flops, bytes; };
    std::vector<ProfRec> prof;
    struct ProfAgg { double ms = 0, flops = 0, bytes = 0; long launches = 0; };
    std::map<std::string, ProfAgg> prof_agg;
    // debug taps: named intermediates copied out during a forward (fac_debug_tap)
    std::map<std::string, std::pair<float*, size_t>> taps;
};

// Streaming state of one batch of utterances: the encoder and the decoder are causal (README.md:105-107), so a chunk's
// outputs depend on the past only through (a) a bounded window of earlier samples / frames of every FIR-like conv stack
// and (b) the LSTM states.  Histories are kept on the device; chunks are computed on [history | chunk] windows with the
// ordinary kernels and the history part of the output is dropped.
struct fac_handle::Stream {
    int B = 0;
    bool alive = false;
    long long enc_samples = 0, dec_frames = 0;
    float* x_hist = nullptr; int x_hist_len = 0;            // [B][kEncCtx] last samples
    float* ey_hist = nullptr; int ey_hist_len = 0;          // [B][2][1024] last encoder-LSTM output frames (conv_out, k = 3)
    float* z_hist = nullptr; int z_hist_len = 0;            // [B][6][1024] last latent frames (decoder conv0, k = 7)
    float* dy_hist = nullptr; int dy_hist_len = 0;          // [B][kDecCtx][1536] last decoder-LSTM output frames
    uint32_t* enc_h[2] = {nullptr, nullptr}; float* enc_c[2] = {nullptr, nullptr};
    uint32_t* dec_h[2] = {nullptr, nullptr}; float* dec_c[2] = {nullptr, nullptr};
    void* all[12] = {nullptr};
};

// One CNNLSTM predictor head (modules/quantize.py:106-125): 3 ResidualUnits (alias-free SnakeBeta, k7 conv dilation
// 1/2/3 with zero padding, alias-free SnakeBeta, 1x1 conv, +x), a final alias-free SnakeBeta, nheads Linear layers.
// Built through a private staging handle so that the conv packing code is shared; weights live in their own arena.
struct fac_handle::HeadSet {
    int indim = 0, outdim = 0, nheads = 0, global_pred = 0;
    struct Unit { size_t a1, b1, a2, b2; ConvW c7, c1; int dil; } unit[3];
    size_t af, bf;                  // final activation exp(alpha), exp(beta)
    ConvW lin[8];
    std::map<std::string, HostTensor> staged;
    float* arena = nullptr;
    bool ready = false;
};

namespace {

// ------------------------------------------------------------------------------------------
// packing helpers (host)
// ------------------------------------------------------------------------------------------
size_t pack_alloc(fac_handle* h, size_t n) {
    size_t off = (h->pack.size() + 63) / 64 * 64;
    h->pack.resize(off + n, 0.f);
    return off;
}

const HostTensor* find(fac_handle* h, int m, const std::string& k) {
    auto it = h->host[m].find(k);
    return it == h->host[m].end() ? nullptr : &it->second;
}

struct PackError { std::string msg; };
const HostTensor& need(fac_handle* h, int m, const std::string& k) {
    const HostTensor* t = find(h, m, k);
    if (!t) throw PackError{"missing tensor '" + k + "' in module " + std::to_string(m)};
    return *t;
}

// Folded conv weight in PyTorch layout [d0][d1][K] (weight-norm over dims != 0, encodec.py:42-51).
std::vector<float> folded_weight(fac_handle* h, int m, const std::string& prefix, std::vector<int64_t>& shape) {
    if (const HostTensor* w = find(h, m, prefix + ".weight")) {
        shape = w->shape;
        return w->data;
    }
    const HostTensor& v = need(h, m, prefix + ".weight_v");
    const HostTensor& g = need(h, m, prefix + ".weight_g");
    shape = v.shape;
    size_t d0 = (size_t)v.shape[0], inner = v.numel() / d0;
    if (g.numel() != d0) throw PackError{"weight_g shape mismatch at " + prefix};
    std::vector<float> w(v.numel());
    for (size_t i = 0; i < d0; ++i) {
        double s = 0.0;
        for (size_t j = 0; j < inner; ++j) { double x = v.data[i * inner + j]; s += x * x; }
        float scale = g.data[i] / (float)std::sqrt(s);
        for (size_t j = 0; j < inner; ++j) w[i * inner + j] = v.data[i * inner + j] * scale;
    }
    return w;
}

// Builds the tcgen05 weight blob for a packed conv (stride-1 in rows; `stride` > 1 means the
// kernel-2*stride down-conv viewed as a 2-tap conv over rows of `stride` samples).
void attach_tc(fac_handle* h, ConvW& c, int stride, bool promoted) {
    TcConvParams tp;
    tp.Cin = c.Cin; tp.Cout = c.Cout; tp.dil = 1; tp.promoted = promoted ? 1 : 0;
    if (stride == 1) { tp.vf = 1; tp.Kr = c.K; }
    else if (c.K == 2 * stride) { tp.vf = stride; tp.Kr = 2; }
    else return;
    if (!tc_conv_plan(tp)) return;
    c.vf = tp.vf; c.Kr = tp.Kr; c.promoted = promoted; c.tcN = tp.N;
    size_t n = tc_blob_floats(tp);
    c.tcw = pack_alloc(h, n);
    tc_pack_blob(tp, h->pack.data() + c.w, c.ldw, h->pack.data() + c.tcw);
    c.tc = true;
    if (promoted) {
        TcConvParams tt = tp;
        if (tt_conv_plan(tt)) {
            c.tcw_tt = pack_alloc(h, tt_blob_floats(tt));
            tt_pack_blob(tt, h->pack.data() + c.w, c.ldw, h->pack.data() + c.tcw_tt);
            c.has_tt = true;
        }
        TcConvParams t16 = tp;
        t16.f16x2 = 1;
        if (tc_conv_plan(t16) && t16.N == tp.N) {
            c.tcw16 = pack_alloc(h, tc_blob_floats(t16));
            tc_pack_blob(t16, h->pack.data() + c.w, c.ldw, h->pack.data() + c.tcw16);
            c.has16 = true;
        }
    } else {
        TcConvParams t16 = tp;
        t16.bf16 = 1;
        if (tc_conv_plan(t16) && t16.N == tp.N) {
            c.tcw16 = pack_alloc(h, tc_blob_floats(t16));
            tc_pack_blob(t16, h->pack.data() + c.w, c.ldw, h->pack.data() + c.tcw16);
            c.has16 = true;
        }
    }
}

// hi-only fp16 blob of a stride-1 layer downstream of the VQ (conv_tc_kernel's one-pass class; the dilated k = 7 convs of
// the ResidualUnits: 7/8 of a unit's MACs, 1.4e-5 RMS on the waveform, scripts/cpu_decoder_precision.py)
void attach_f16_single(fac_handle* h, ConvW& c) {
    if (!c.tc || c.promoted || !c.has16 || c.vf != 1) return;
    TcConvParams t1;
    t1.Cin = c.Cin; t1.Cout = c.Cout; t1.dil = 1; t1.vf = 1; t1.Kr = c.K; t1.bf16 = 1; t1.g1f16 = 1;
    if (!tc_conv_plan(t1) || t1.N != c.tcN) return;
    c.tcw_f16s = pack_alloc(h, tc_blob_floats(t1));
    tc_pack_blob(t1, h->pack.data() + c.w, c.ldw, h->pack.data() + c.tcw_f16s);
    c.has_f16s = true;
}

// nn.Conv1d [Cout][Cin][K] -> packed [K*Cin][ldw]
ConvW pack_conv(fac_handle* h, int m, const std::string& prefix, int stride = 1, bool promoted = false) {
    std::vector<int64_t> shp;
    std::vector<float> w = folded_weight(h, m, prefix, shp);
    if (shp.size() == 2) shp.push_back(1);
    if (shp.size() != 3) throw PackError{"conv weight rank at " + prefix};
    ConvW c;
    c.Cout = (int)shp[0]; c.Cin = (int)shp[1]; c.K = (int)shp[2];
    c.ldw = (c.Cout + 3) / 4 * 4;
    c.w = pack_alloc(h, (size_t)c.K * c.Cin * c.ldw);
    for (int co = 0; co < c.Cout; ++co)
        for (int ci = 0; ci < c.Cin; ++ci)
            for (int k = 0; k < c.K; ++k)
                h->pack[c.w + ((size_t)k * c.Cin + ci) * c.ldw + co] = w[((size_t)co * c.Cin + ci) * c.K + k];
    const HostTensor& b = need(h, m, prefix + ".bias");
    c.b = pack_alloc(h, c.Cout);
    for (int co = 0; co < c.Cout; ++co) h->pack[c.b + co] = b.data[co];
    attach_tc(h, c, stride, promoted);
    return c;
}

// nn.ConvTranspose1d [Cin][Cout][2s] stride s + right trim (encodec.py:248-270) -> K=2 conv with
// Cout*s phase-major output channels: tap0 (x[t-1]) = w[..][r+s], tap1 (x[t]) = w[..][r].
ConvW pack_convtr(fac_handle* h, int m, const std::string& prefix, int stride) {
    std::vector<int64_t> shp;
    std::vector<float> w = folded_weight(h, m, prefix, shp);
    if (shp.size() != 3 || shp[2] != 2 * stride) throw PackError{"convtr kernel != 2*stride at " + prefix};
    int Cin = (int)shp[0], Cout = (int)shp[1], K = (int)shp[2];
    ConvW c;
    c.Cin = Cin; c.Cout = Cout * stride; c.K = 2; c.ldw = (c.Cout + 3) / 4 * 4;
    c.w = pack_alloc(h, (size_t)2 * Cin * c.ldw);
    for (int ci = 0; ci < Cin; ++ci)
        for (int co = 0; co < Cout; ++co)
            for (int r = 0; r < stride; ++r) {
                h->pack[c.w + ((size_t)0 * Cin + ci) * c.ldw + r * Cout + co] = w[((size_t)ci * Cout + co) * K + r + stride];
                h->pack[c.w + ((size_t)1 * Cin + ci) * c.ldw + r * Cout + co] = w[((size_t)ci * Cout + co) * K + r];
            }
    const HostTensor& b = need(h, m, prefix + ".bias");
    c.b = pack_alloc(h, c.Cout);
    for (int r = 0; r < stride; ++r)
        for (int co = 0; co < Cout; ++co) h->pack[c.b + r * Cout + co] = b.data[co];
    attach_tc(h, c, 1, false);
    return c;
}

// Non-causal variant (encodec.py:264-269: trim padding_total - padding_total/2 on the left, padding_total/2 on the right):
// output sample n = t*s + r reads full[n + pl], pl = s - s/2, i.e. x[t-1]*w[a+s] (a < s) + x[t]*w[a] + x[t+1]*w[a-s] (a >= s)
// with a = r + pl: a 3-tap conv over (x[t-1], x[t], x[t+1]), zero padding 1 | 1, s*Cout phase-major channels.
ConvW pack_convtr_noncausal(fac_handle* h, int m, const std::string& prefix, int stride) {
    std::vector<int64_t> shp;
    std::vector<float> w = folded_weight(h, m, prefix, shp);
    if (shp.size() != 3 || shp[2] != 2 * stride) throw PackError{"convtr kernel != 2*stride at " + prefix};
    int Cin = (int)shp[0], Cout = (int)shp[1], K = (int)shp[2];
    const int pl = stride - stride / 2;
    ConvW c;
    c.Cin = Cin; c.Cout = Cout * stride; c.K = 3; c.ldw = (c.Cout + 3) / 4 * 4;
    c.w = pack_alloc(h, (size_t)3 * Cin * c.ldw);
    for (int ci = 0; ci < Cin; ++ci)
        for (int co = 0; co < Cout; ++co)
            for (int r = 0; r < stride; ++r) {
                const int a = r + pl;
                const float* wk = &w[((size_t)ci * Cout + co) * K];
                h->pack[c.w + ((size_t)0 * Cin + ci) * c.ldw + r * Cout + co] = a < stride ? wk[a + stride] : 0.f;
                h->pack[c.w + ((size_t)1 * Cin + ci) * c.ldw + r * Cout + co] = wk[a];
                h->pack[c.w + ((size_t)2 * Cin + ci) * c.ldw + r * Cout + co] = a >= stride ? wk[a - stride] : 0.f;
            }
    const HostTensor& b = need(h, m, prefix + ".bias");
    c.b = pack_alloc(h, c.Cout);
    for (int r = 0; r < stride; ++r)
        for (int co = 0; co < Cout; ++co) h->pack[c.b + r * Cout + co] = b.data[co];
    attach_tc(h, c, 1, false);
    return c;
}

SnakeW pack_snake(fac_handle* h, int m, const std::string& key) {
    const HostTensor& a = need(h, m, key);
    SnakeW s;
    s.C = (int)a.numel();
    s.a = pack_alloc(h, s.C);
    s.ia = pack_alloc(h, s.C);
    for (int i = 0; i < s.C; ++i) {
        h->pack[s.a + i] = a.data[i];
        h->pack[s.ia + i] = 1.0f / (a.data[i] + 1e-9f);   // (alpha + 1e-9).reciprocal(), fp32
    }
    return s;
}

ResW pack_res(fac_handle* h, int m, const std::string& prefix, int dil, bool promoted = false) {
    ResW r;
    r.dil = dil;
    r.s1 = pack_snake(h, m, prefix + ".block.0.alpha");
    r.c7 = pack_conv(h, m, prefix + ".block.1.conv.conv", 1, promoted);
    if (!promoted) attach_f16_single(h, r.c7);
    r.s2 = pack_snake(h, m, prefix + ".block.2.alpha");
    r.c1 = pack_conv(h, m, prefix + ".block.3.conv.conv", 1, promoted);
    return r;
}

LstmW pack_lstm(fac_handle* h, int m, const std::string& prefix, bool promoted = false) {
    LstmW L;
    const HostTensor& w0 = need(h, m, prefix + ".weight_hh_l0");
    L.H = (int)w0.shape[1];
    L.U = lstm_units_per_cta(L.H);
    if (L.U == 0) throw PackError{"unsupported LSTM width " + std::to_string(L.H)};
    L.G = L.H / L.U;
    const int H = L.H, U = L.U, R = 4 * U;
    for (int l = 0; l < 2; ++l) {
        std::string sfx = "_l" + std::to_string(l);
        const HostTensor& wih = need(h, m, prefix + ".weight_ih" + sfx);
        const HostTensor& whh = need(h, m, prefix + ".weight_hh" + sfx);
        const HostTensor& bih = need(h, m, prefix + ".bias_ih" + sfx);
        const HostTensor& bhh = need(h, m, prefix + ".bias_hh" + sfx);
        ConvW c;
        c.Cin = H; c.Cout = 4 * H; c.K = 1; c.ldw = 4 * H;
        c.w = pack_alloc(h, (size_t)H * c.ldw);
        for (int row = 0; row < 4 * H; ++row)
            for (int k = 0; k < H; ++k) h->pack[c.w + (size_t)k * c.ldw + row] = wih.data[(size_t)row * H + k];
        c.b = pack_alloc(h, 4 * H);
        for (int row = 0; row < 4 * H; ++row) h->pack[c.b + row] = bih.data[row] + bhh.data[row];
        attach_tc(h, c, 1, promoted);
        L.ih[l] = c;
        L.whh[l] = pack_alloc(h, (size_t)L.G * H * R);
        for (int cta = 0; cta < L.G; ++cta)
            for (int k = 0; k < H; ++k)
                for (int g = 0; g < 4; ++g)
                    for (int u = 0; u < U; ++u)
                        h->pack[L.whh[l] + ((size_t)cta * H + k) * R + g * U + u] =
                            whh.data[((size_t)g * H + cta * U + u) * H + k];
        for (int p3 = 0; p3 < 2; ++p3) {
            // second-generation kernel: promoted (upstream) layers use the 3-pass pack, the others the one-pass pack; the
            // 3-pass pack of a downstream layer backs fac_set_option("decoder_bf16", 0)
            if (p3 == 0 && promoted) continue;
            if ((H / 16) % 8 != 0 || lstm2_smem_bytes(H, U, p3) > 227 * 1024) continue;
            const size_t nw = lstm2_pack_words(H, U, p3);
            L.whh2[l][p3] = pack_alloc(h, nw);
            lstm2_pack(whh.data.data(), H, U, p3, reinterpret_cast<uint32_t*>(h->pack.data() + L.whh2[l][p3]));
            L.has2[p3] = true;
        }
        if (!promoted) {
            // bf16 hi/lo words for the recurrence downstream of the VQ: [cta][H/16][hi|lo][8 k-pairs][R]
            auto bf16_rn = [](float f) { uint32_t u; memcpy(&u, &f, 4); u += 0x7FFFu + ((u >> 16) & 1u); return (uint32_t)(u >> 16); };
            auto bf16_f = [](uint32_t b) { uint32_t u = b << 16; float f; memcpy(&f, &u, 4); return f; };
            L.whh16[l] = pack_alloc(h, (size_t)L.G * H * R);
            for (int cta = 0; cta < L.G; ++cta)
                for (int sub = 0; sub < H / 16; ++sub)
                    for (int k2 = 0; k2 < 8; ++k2)
                        for (int r = 0; r < R; ++r) {
                            const int g = r / U, u = r % U;
                            const float* wrow = &whh.data[((size_t)g * H + cta * U + u) * H + sub * 16 + 2 * k2];
                            uint32_t h0 = bf16_rn(wrow[0]), h1 = bf16_rn(wrow[1]);
                            uint32_t l0 = bf16_rn(wrow[0] - bf16_f(h0)), l1 = bf16_rn(wrow[1] - bf16_f(h1));
                            uint32_t hw = h0 | (h1 << 16), lw = l0 | (l1 << 16);
                            size_t base = L.whh16[l] + ((size_t)cta * (H / 16) + sub) * 16 * R;
                            memcpy(&h->pack[base + (size_t)k2 * R + r], &hw, 4);
                            memcpy(&h->pack[base + (size_t)(8 + k2) * R + r], &lw, 4);
                        }
            L.has16 = true;
        }
    }
    return L;
}

VqW pack_vq_raw(std::vector<float>& pack, const float* in_w, const float* in_b, const float* out_w,
                const float* out_b, const float* codebook, fac_handle* h = nullptr) {
    auto alloc = [&](size_t n) {
        size_t off = (pack.size() + 63) / 64 * 64;
        pack.resize(off + n, 0.f);
        return off;
    };
    VqW v;
    v.w_in = alloc(8 * 1024);
    for (int i = 0; i < 8 * 1024; ++i) pack[v.w_in + i] = in_w[i];
    v.b_in = alloc(8);
    for (int i = 0; i < 8; ++i) pack[v.b_in + i] = in_b[i];
    v.cb = alloc(1024 * 8);
    v.cbn = alloc(1024 * 8);
    v.cbn2 = alloc(1024);
    for (int j = 0; j < 1024; ++j) {
        float n2 = 0.f;
        for (int k = 0; k < 8; ++k) n2 = fmaf(codebook[j * 8 + k], codebook[j * 8 + k], n2);
        float nrm = fmaxf(sqrtf(n2), 1e-12f);
        float c2 = 0.f;
        for (int k = 0; k < 8; ++k) {
            float cn = codebook[j * 8 + k] / nrm;
            pack[v.cb + j * 8 + k] = codebook[j * 8 + k];
            pack[v.cbn + j * 8 + k] = cn;
            c2 = fmaf(cn, cn, c2);
        }
        pack[v.cbn2 + j] = c2;
    }
    v.w_out = alloc(8 * 1024);   // transposed [k][c]
    for (int c = 0; c < 1024; ++c)
        for (int k = 0; k < 8; ++k) pack[v.w_out + (size_t)k * 1024 + c] = out_w[c * 8 + k];
    v.b_out = alloc(1024);
    for (int c = 0; c < 1024; ++c) pack[v.b_out + c] = out_b[c];
    (void)h;
    return v;
}

VqW pack_vq(fac_handle* h, int m, const std::string& prefix) {
    std::vector<int64_t> s1, s2;
    std::vector<float> win = folded_weight(h, m, prefix + ".in_proj", s1);
    std::vector<float> wout = folded_weight(h, m, prefix + ".out_proj", s2);
    if (s1[0] != 8 || s1[1] != 1024 || s2[0] != 1024 || s2[1] != 8) throw PackError{"VQ shape at " + prefix};
    const HostTensor& bi = need(h, m, prefix + ".in_proj.bias");
    const HostTensor& bo = need(h, m, prefix + ".out_proj.bias");
    const HostTensor& cb = need(h, m, prefix + ".codebook.weight");
    if (cb.shape[0] != 1024 || cb.shape[1] != 8) throw PackError{"codebook shape at " + prefix};
    return pack_vq_raw(h->pack, win.data(), bi.data.data(), wout.data(), bo.data.data(), cb.data.data());
}

void pack_encoder(fac_handle* h) {
    EncW& e = h->enc;
    const int m = FAC_ENCODER;
    const int rates[4] = {2, 5, 5, 6};
    e.conv0 = pack_conv(h, m, "block.0.conv.conv");
    for (int i = 0; i < 4; ++i) {
        std::string p = "block." + std::to_string(i + 1);
        const int dils[3] = {1, 3, 9};
        for (int j = 0; j < 3; ++j) e.blk[i].res[j] = pack_res(h, m, p + ".block." + std::to_string(j), dils[j], true);
        e.blk[i].snake = pack_snake(h, m, p + ".block.3.alpha");
        e.blk[i].down = pack_conv(h, m, p + ".block.4.conv.conv", rates[i], true);
        e.blk[i].stride = rates[i];
        if (e.blk[i].down.K != 2 * rates[i]) throw PackError{"encoder stride/kernel mismatch"};
    }
    e.lstm = pack_lstm(h, m, "block.5.lstm", true);
    e.snake = pack_snake(h, m, "block.6.alpha");
    e.conv_out = pack_conv(h, m, "block.7.conv.conv", 1, true);
}

void pack_decoder_into(fac_handle* h, int m, DecW& d, bool lstm, bool causal) {
    const int rates[4] = {6, 5, 5, 2};
    d.causal = causal; d.has_lstm = lstm;
    d.conv0 = pack_conv(h, m, "model.0.conv.conv");
    int base = 1;
    if (lstm) { d.lstm = pack_lstm(h, m, "model.1.lstm"); base = 2; }
    for (int i = 0; i < 4; ++i) {
        std::string p = "model." + std::to_string(i + base);
        d.blk[i].snake = pack_snake(h, m, p + ".block.0.alpha");
        d.blk[i].up = causal ? pack_convtr(h, m, p + ".block.1.convtr.convtr", rates[i])
                             : pack_convtr_noncausal(h, m, p + ".block.1.convtr.convtr", rates[i]);
        d.blk[i].stride = rates[i];
        d.blk[i].cout = d.blk[i].up.Cout / rates[i];
        const int dils[3] = {1, 3, 9};
        for (int j = 0; j < 3; ++j) d.blk[i].res[j] = pack_res(h, m, p + ".block." + std::to_string(j + 2), dils[j]);
    }
    d.snake = pack_snake(h, m, "model." + std::to_string(4 + base) + ".alpha");
    d.conv_out = pack_conv(h, m, "model." + std::to_string(5 + base) + ".conv.conv");
}

void pack_decoder(fac_handle* h) { pack_decoder_into(h, FAC_DECODER, h->dec, true, true); }

// modules/redecoder.py:5-21 (encoder_type "wavenet"); key names of modules/wavenet.py:103-136 under "encoder."
void pack_redecoder(fac_handle* h) {
    RedW& r = h->red;
    const int m = FAC_REDECODER;
    auto emb = [&](const std::string& key) {
        const HostTensor& t = need(h, m, key);
        if (t.shape.size() != 2 || t.shape[0] != 1024 || t.shape[1] != r.hidden) throw PackError{"embedding shape at " + key};
        size_t off = pack_alloc(h, t.numel());
        for (size_t i = 0; i < t.numel(); ++i) h->pack[off + i] = t.data[i];
        return off;
    };
    r.emb_p = emb("prosody_embed.0.weight");
    r.emb_c[0] = emb("content_embed.0.weight");
    r.emb_c[1] = emb("content_embed.1.weight");
    r.cond = pack_conv(h, m, "encoder.cond_layer.conv.conv");
    for (int i = 0; i < r.layers; ++i) {
        r.wn_in[i] = pack_conv(h, m, "encoder.in_layers." + std::to_string(i) + ".conv.conv");
        r.wn_rs[i] = pack_conv(h, m, "encoder.res_skip_layers." + std::to_string(i) + ".conv.conv");
    }
    r.conv_out = pack_conv(h, m, "conv_out");
    if (r.cond.Cin != LATENT || r.cond.Cout != 2 * r.hidden * r.layers || r.wn_in[0].K != 5 || r.conv_out.Cout != LATENT)
        throw PackError{"redecoder geometry (expects WN(512, kernel 5, 16 layers, gin 1024))"};
}

// The mel front-end's constants: [1200][2*1025] windowed DFT basis (fp64 -> fp32), its tensor-core variant, the filterbank.
void pack_mel_frontend(fac_handle* h, ConvW& dft, ConvW& dft_tc, size_t& fb_off, const float* win, const float* fb) {
    dft.Cin = 1; dft.Cout = 2 * N_BINS; dft.K = WIN; dft.ldw = SPEC_LD;
    dft.w = pack_alloc(h, (size_t)WIN * SPEC_LD);
    dft.b = 0;
    const int left = (N_FFT - WIN) / 2;
    for (int n = 0; n < WIN; ++n)
        for (int k = 0; k < N_BINS; ++k) {
            // reduce the phase index mod N_FFT in integers so the fp64 angle stays small
            long long ph = ((long long)k * (n + left)) % N_FFT;
            double ang = 2.0 * M_PI * (double)ph / (double)N_FFT;
            h->pack[dft.w + (size_t)n * SPEC_LD + 2 * k] = (float)((double)win[n] * std::cos(ang));
            h->pack[dft.w + (size_t)n * SPEC_LD + 2 * k + 1] = (float)(-(double)win[n] * std::sin(ang));
        }
    // tensor-core variant: [1200][2176] with zero columns beyond 2*1025, zero bias
    dft_tc.Cin = WIN; dft_tc.Cout = SPEC_TC_LD; dft_tc.K = 1; dft_tc.ldw = SPEC_TC_LD;
    dft_tc.w = pack_alloc(h, (size_t)WIN * SPEC_TC_LD);
    for (int n = 0; n < WIN; ++n)
        for (int k = 0; k < 2 * N_BINS; ++k) h->pack[dft_tc.w + (size_t)n * SPEC_TC_LD + k] = h->pack[dft.w + (size_t)n * SPEC_LD + k];
    dft_tc.b = pack_alloc(h, SPEC_TC_LD);
    attach_tc(h, dft_tc, 1, true);
    fb_off = pack_alloc(h, (size_t)N_BINS * N_MELS);
    for (size_t i = 0; i < (size_t)N_BINS * N_MELS; ++i) h->pack[fb_off + i] = fb[i];
}

void pack_quantizer(fac_handle* h) {
    QuantW& q = h->qw;
    const int m = FAC_QUANTIZER;
    q.vq[0] = pack_vq(h, m, "prosody_quantizer.quantizers.0");
    q.vq[1] = pack_vq(h, m, "content_quantizer.quantizers.0");
    q.vq[2] = pack_vq(h, m, "content_quantizer.quantizers.1");
    for (int i = 0; i < 3; ++i) q.vq[3 + i] = pack_vq(h, m, "residual_quantizer.quantizers." + std::to_string(i));
    q.spec0 = pack_conv(h, m, "timbre_encoder.spectral.0", 1, true);
    q.spec3 = pack_conv(h, m, "timbre_encoder.spectral.3", 1, true);
    q.glu[0] = pack_conv(h, m, "timbre_encoder.temporal.0.conv1", 1, true);
    q.glu[1] = pack_conv(h, m, "timbre_encoder.temporal.1.conv1", 1, true);
    q.cq = pack_conv(h, m, "timbre_encoder.slf_attn.conv_q", 1, true);
    q.ck = pack_conv(h, m, "timbre_encoder.slf_attn.conv_k", 1, true);
    q.cv = pack_conv(h, m, "timbre_encoder.slf_attn.conv_v", 1, true);
    q.co = pack_conv(h, m, "timbre_encoder.slf_attn.conv_o", 1, true);
    q.fc = pack_conv(h, m, "timbre_encoder.fc", 1, true);
    q.timbre_linear = pack_conv(h, m, "timbre_linear", 1, true);
    q.mel_lin = pack_conv(h, m, "melspec_linear.conv.conv");
    for (int i = 0; i < 8; ++i) {
        q.wn_in[i] = pack_conv(h, m, "melspec_encoder.in_layers." + std::to_string(i) + ".conv.conv", 1, true);
        q.wn_rs[i] = pack_conv(h, m, "melspec_encoder.res_skip_layers." + std::to_string(i) + ".conv.conv", 1, true);
    }
    q.mel_lin2 = pack_conv(h, m, "melspec_linear2.conv.conv", 1, true);
    // STFT basis with the Hann window folded in: frame sample n+424 of the zero-padded window
    const HostTensor& win = need(h, m, "to_mel.spectrogram.window");
    const HostTensor& fb = need(h, m, "to_mel.mel_scale.fb");
    if ((int)win.numel() != WIN || fb.shape[0] != N_BINS || fb.shape[1] != N_MELS) throw PackError{"mel buffers shape"};
    pack_mel_frontend(h, q.dft, q.dft_tc, q.fb, win.data.data(), fb.data.data());
}

// ------------------------------------------------------------------------------------------
// forward context: bump allocator over the handle's workspace + launch helpers
// ------------------------------------------------------------------------------------------
struct Ctx {
    fac_handle* h;
    cudaStream_t st;
    bool dry;          // size pass: allocate only
    bool vq_critical = false;   // inside the encoder / prosody branch: feeds the bit-exact VQ argmin
    size_t off = 0;
    cudaError_t cerr = cudaSuccess;
    const char* where = "";

    template <typename T>
    T* alloc(size_t n) {
        size_t bytes = (n * sizeof(T) + 255) / 256 * 256;
        char* p = h->ws ? h->ws + off : nullptr;
        off += bytes;
        return reinterpret_cast<T*>(p);
    }
    const float* W(size_t o) const { return h->warena + o; }
    bool ok() const { return cerr == cudaSuccess; }
    void check(cudaError_t e, const char* w) {     // a kernel launch
        if (!dry) h->launches++;
        if (e != cudaSuccess && cerr == cudaSuccess) { cerr = e; where = w; }
    }
    void check_nk(cudaError_t e, const char* w) {  // memset / memcpy: not a kernel
        if (e != cudaSuccess && cerr == cudaSuccess) { cerr = e; where = w; }
    }
    void tap(const char* name, const float* src, size_t n) {
        if (dry || h->taps.empty()) return;
        auto it = h->taps.find(name);
        if (it == h->taps.end()) return;
        size_t m = n < it->second.second ? n : it->second.second;
        check_nk(cudaMemcpyAsync(it->second.first, src, m * sizeof(float), cudaMemcpyDeviceToDevice, st), "tap");
    }
    // profiling: begin()/end() bracket one launch with events on the launching stream
    void begin(const char* fam, double flops, double bytes, const char* detail = nullptr) {
        if (dry || !h->profiling) return;
        fac_handle::ProfRec r;
        r.name = fam; r.flops = flops; r.bytes = bytes;
        if (detail) { r.name += ":"; r.name += detail; }
        cudaEventCreate(&r.a); cudaEventCreate(&r.b);
        cudaEventRecord(r.a, st);
        h->prof.push_back(r);
    }
    void end() {
        if (dry || !h->profiling) return;
        cudaEventRecord(h->prof.back().b, st);
    }
};

struct ConvOpts {
    int dil = 1, stride = 1, pad_left = 0, pad_right = 0, reflect = 0;
    const SnakeW* in_snake = nullptr;
    const SnakeW* out_snake = nullptr;
    int act = ACT_NONE;
    const float* res = nullptr;
    const int* valid_len = nullptr;
    int transposed = 0;
    int ldx = 0;            // input row stride (0 = Cin)
    int ldy = 0;            // output row stride (0 = Cout)
    bool no_bias = false;
};

// SConv1d padding rule (encodec.py:212-228): causal => (k_eff - stride) on the left (reflect),
// plus "extra" on the right so the last window is full (encodec.py:71-78).
int conv_out_len(int T, int k_eff, int stride) {
    int padding_total = k_eff - stride;
    double n_frames = (double)(T - k_eff + padding_total) / stride + 1.0;
    int ideal = ((int)std::ceil(n_frames) - 1) * stride + (k_eff - padding_total);
    int extra = ideal - T;
    return (T + padding_total + extra - k_eff) / stride + 1;
}
int conv_extra_pad(int T, int k_eff, int stride) {
    int padding_total = k_eff - stride;
    double n_frames = (double)(T - k_eff + padding_total) / stride + 1.0;
    int ideal = ((int)std::ceil(n_frames) - 1) * stride + (k_eff - padding_total);
    return ideal - T;
}

void run_conv(Ctx& c, const ConvW& w, const float* x, float* y, int B, int Tin, int Tout, const ConvOpts& o,
              const char* name) {
    if (c.dry) return;
    if (c.h->use_tc >= (c.vq_critical ? 2 : 1) && w.tc && !o.transposed && !o.valid_len && (o.ldx == 0 || o.ldx == w.Cin) &&
        (o.ldy == 0 || o.ldy == w.Cout) && o.stride == w.vf && (w.vf == 1 || o.dil == 1) && !o.no_bias) {
        TcConvParams tp;
        tp.Cin = w.Cin; tp.Cout = w.Cout; tp.vf = w.vf; tp.Kr = w.Kr; tp.promoted = w.promoted ? 1 : 0;
        // A layer whose whole K loop is at most one promotion window (<= 48 chained MMAs: the 1x1 convs of the 64- and
        // 128-channel encoder stages) gains nothing from register promotion: same error class through conv_tc_kernel,
        // which runs two CTAs per SM and prefetches the residual.
        bool short_chain = false;
        if (w.promoted && (w.Cin * w.vf / 16) * w.Kr * 6 <= 48) {
            TcConvParams probe = tp;
            probe.promoted = 0; probe.occ2_maxn = c.h->tc_occ2;
            if (tc_conv_plan(probe) && probe.N == w.tcN) { tp.promoted = 0; short_chain = true; }
        }
        tp.dil = w.vf == 1 ? o.dil : 1;
        tp.bf16 = (c.h->dec_bf16 && w.has16 && !w.promoted && !c.vq_critical) ? 1 : 0;
        tp.g1f16 = (tp.bf16 && w.has_f16s && c.h->dec_c7_f16) ? 1 : 0;
        tp.f16x2 = (tp.promoted && c.h->enc_f16 && w.has16) ? 1 : 0;
        tp.occ2_maxn = c.h->tc_occ2;
        tp.Tout = Tout;
        const bool use_tt = tp.promoted && c.h->enc_tt && w.has_tt;
        tp.snake_mufu = c.h->enc_mufu;
        if (use_tt ? tt_conv_plan(tp) : tc_conv_plan(tp)) {
            tp.x = x; tp.y = y; tp.wblob = c.W(use_tt ? w.tcw_tt : (tp.g1f16 ? w.tcw_f16s : ((tp.bf16 || tp.f16x2) ? w.tcw16 : w.tcw))); tp.bias = c.W(w.b);
            if (o.in_snake) { tp.in_alpha = c.W(o.in_snake->a); tp.in_inv_alpha = c.W(o.in_snake->ia); }
            tp.out_act = o.act;
            if (o.out_snake) { tp.out_act = ACT_SNAKE; tp.out_alpha = c.W(o.out_snake->a); tp.out_inv_alpha = c.W(o.out_snake->ia); }
            tp.res = o.res;
            tp.B = B; tp.Tin = Tin; tp.ldx = w.Cin;
            tp.PLr = o.pad_left / w.vf;
            tp.pad_left_s = o.pad_left; tp.pad_right_s = o.pad_right; tp.reflect = o.reflect;
            tp.Tout = Tout; tp.ldy = w.Cout;
            tp.x_bstride = (size_t)Tin * w.Cin; tp.y_bstride = (size_t)Tout * w.Cout;
            double flops = 2.0 * B * Tout * (double)w.Cout * w.K * w.Cin;
            double bytes = 4.0 * ((double)B * Tin * w.Cin + (double)B * Tout * w.Cout * (o.res ? 2 : 1) + (double)w.K * w.Cin * w.Cout);
            char det[96];
            snprintf(det, sizeof det, "%s Cin%d Cout%d K%d d%d T%d", name, w.Cin, w.Cout, w.K, o.dil, Tout);
            c.begin(use_tt ? "conv_tt" : (tp.promoted ? "conv_tcp" : "conv_tc"), flops, bytes, det);
            (void)short_chain;
            c.check(use_tt ? launch_conv_tt(tp, c.st) : launch_conv_tc(tp, c.st), name);
            c.end();
            return;
        }
    }
    ConvParams p;
    p.x = x; p.y = y;
    p.w = c.W(w.w);
    p.bias = o.no_bias ? nullptr : c.W(w.b);
    if (o.in_snake) { p.in_alpha = c.W(o.in_snake->a); p.in_inv_alpha = c.W(o.in_snake->ia); }
    p.out_act = o.act;
    if (o.out_snake) { p.out_act = ACT_SNAKE; p.out_alpha = c.W(o.out_snake->a); p.out_inv_alpha = c.W(o.out_snake->ia); }
    p.res = o.res; p.valid_len = o.valid_len;
    p.B = B; p.Tin = Tin; p.Cin = w.Cin; p.Tout = Tout; p.Cout = w.Cout;
    p.K = w.K; p.dil = o.dil; p.stride = o.stride;
    p.pad_left = o.pad_left; p.pad_right = o.pad_right; p.pad_reflect = o.reflect;
    p.ldw = w.ldw; p.ldy = o.ldy ? o.ldy : w.Cout; p.ldx = o.ldx ? o.ldx : w.Cin;
    p.y_transposed = o.transposed;
    p.x_bstride = (size_t)Tin * p.ldx;
    p.y_bstride = (size_t)Tout * p.ldy;
    // algorithmic work of this launch: 2*MACs; bytes = input + output (+ residual) + weights once
    double flops = 2.0 * B * Tout * (double)w.Cout * w.K * w.Cin;
    double bytes = 4.0 * ((double)B * Tin * w.Cin + (double)B * Tout * w.Cout * (o.res ? 2 : 1) + (double)w.K * w.Cin * w.Cout);
    char det[96];
    snprintf(det, sizeof det, "%s Cin%d Cout%d K%d d%d T%d", name, w.Cin, w.Cout, w.K, o.dil, Tout);
    c.begin("conv", flops, bytes, det);
    c.check(launch_conv(p, c.st), name);
    c.end();
}

// SConv1d with reflect padding (encodec.py:212-228): causal = everything on the left, else padding_total - padding_total/2
// on the left and padding_total/2 (+ extra) on the right; returns output length
int sconv(Ctx& c, const ConvW& w, const float* x, float* y, int B, int T, int dil, int stride, ConvOpts o,
          const char* name, bool causal = true) {
    int k_eff = (w.K - 1) * dil + 1;
    o.dil = dil; o.stride = stride;
    const int total = k_eff - stride, extra = conv_extra_pad(T, k_eff, stride);
    o.pad_left = causal ? total : total - total / 2;
    o.pad_right = (causal ? 0 : total / 2) + extra;
    o.reflect = 1;
    int Tout = conv_out_len(T, k_eff, stride);
    run_conv(c, w, x, y, B, T, Tout, o, name);
    return Tout;
}

// Whole ResidualUnit in one tcgen05 launch (conv_tc_kernel<true>) when every channel fits one CTA tile.
bool residual_unit_fused(Ctx& c, const ResW& r, const float* x, float* y, int B, int T, bool causal) {
    if (c.h->use_tc < 1 || !c.h->fuse_res || c.vq_critical || !r.c7.tc || !r.c1.tc || r.c7.promoted || r.c1.promoted ||
        r.c7.Cin != r.c7.Cout || r.c1.K != 1 || r.c7.vf != 1)
        return false;
    TcConvParams tp;
    tp.Cin = r.c7.Cin; tp.Cout = r.c7.Cout; tp.vf = 1; tp.Kr = r.c7.K; tp.dil = r.dil; tp.fused = 1;
    tp.bf16 = (c.h->dec_bf16 && r.c7.has16 && r.c1.has16) ? 1 : 0;
    tp.g1f16 = (tp.bf16 && r.c7.has_f16s && c.h->dec_c7_f16) ? 1 : 0;
    tp.occ2_maxn = c.h->tc_occ2;
    tp.Tout = T;
    if (c.h->fuse_res == 2 && r.c7.Cout > 128) return false;
    if (!tc_conv_plan(tp)) return false;
    if (c.dry) return true;
    const int k_eff = (r.c7.K - 1) * r.dil + 1;
    tp.x = x; tp.y = y; tp.res = x;
    tp.wblob = c.W(tp.g1f16 ? r.c7.tcw_f16s : (tp.bf16 ? r.c7.tcw16 : r.c7.tcw)); tp.bias = c.W(r.c7.b);
    tp.wblob2 = c.W(tp.bf16 ? r.c1.tcw16 : r.c1.tcw); tp.bias2 = c.W(r.c1.b);
    tp.in_alpha = c.W(r.s1.a); tp.in_inv_alpha = c.W(r.s1.ia);
    tp.out_act = ACT_SNAKE; tp.out_alpha = c.W(r.s2.a); tp.out_inv_alpha = c.W(r.s2.ia);
    tp.B = B; tp.Tin = T; tp.ldx = r.c7.Cin;
    const int pl = causal ? k_eff - 1 : (k_eff - 1) - (k_eff - 1) / 2;
    tp.PLr = pl; tp.pad_left_s = pl; tp.pad_right_s = k_eff - 1 - pl; tp.reflect = 1;
    tp.Tout = T; tp.ldy = r.c7.Cout;
    tp.x_bstride = (size_t)T * r.c7.Cin; tp.y_bstride = (size_t)T * r.c7.Cout;
    double flops = 2.0 * B * T * (double)r.c7.Cout * r.c7.Cin * (r.c7.K + 1);
    double bytes = 4.0 * ((double)B * T * r.c7.Cin * 2 + (double)B * T * r.c7.Cout + (double)(r.c7.K + 1) * r.c7.Cin * r.c7.Cout);
    char det[96];
    snprintf(det, sizeof det, "res.fused C%d K%d d%d T%d", r.c7.Cin, r.c7.K, r.dil, T);
    c.begin("conv_tc", flops, bytes, det);
    c.check(launch_conv_tc(tp, c.st), "res.fused");
    c.end();
    return true;
}

// ResidualUnit (dac.py:25-42): y = x + conv1(snake2(conv7_d(snake1(x))))
void residual_unit(Ctx& c, const ResW& r, const float* x, float* tmp, float* y, int B, int T, bool causal = true) {
    if (residual_unit_fused(c, r, x, y, B, T, causal)) return;
    ConvOpts o1;
    o1.in_snake = &r.s1;
    o1.out_snake = &r.s2;
    sconv(c, r.c7, x, tmp, B, T, r.dil, 1, o1, "res.conv7", causal);
    ConvOpts o2;
    o2.res = x;
    sconv(c, r.c1, tmp, y, B, T, 1, 1, o2, "res.conv1", causal);
}

// Carried state of one 2-layer SLSTM (streaming): h in the kernel's published fp16 layout, c per CTA.
struct LstmState { uint32_t* h[2] = {nullptr, nullptr}; float* c[2] = {nullptr, nullptr}; };

// SLSTM (encodec.py:272-288) on channels-last x [B][T][H]; y = lstm2(lstm1(x)) + x.  st (streaming, B <= 32, resident-W
// kernel only): initial state read from / final state written to st.
void slstm(Ctx& c, const LstmW& L, const float* x, float* y, int B, int T, LstmState* st = nullptr) {
    const int H = L.H;
    float* xg = c.alloc<float>((size_t)B * T * 4 * H);
    float* h1 = c.alloc<float>((size_t)B * T * H);
    float* hT = c.alloc<float>((size_t)2 * H * 32);
    uint32_t* h16 = c.alloc<uint32_t>((size_t)2 * 2 * (H / 2) * 32);
    unsigned int* bar = c.alloc<unsigned int>(64);
    for (int l = 0; l < 2; ++l) {
        const float* in = l == 0 ? x : h1;
        ConvOpts o;
        run_conv(c, L.ih[l], in, xg, 1, B * T, B * T, o, "lstm.ih");
        if (c.dry) continue;
        // precision class: 3-pass fp32-faithful upstream of the VQ (and when "decoder_bf16" is off), one fp16 pass downstream
        const int pass3 = (c.vq_critical || !c.h->dec_bf16) ? 1 : 0;
        const bool v2 = c.h->lstm_v2 && L.has2[pass3] && (pass3 || c.h->dec_lstm_fp16);
        for (int b0 = 0; b0 < B; b0 += 32) {
            int nb = B - b0 < 32 ? B - b0 : 32;
            LstmParams p;
            p.xg = xg + (size_t)b0 * T * 4 * H;
            p.whh_p = c.W(L.whh[l]);
            if (c.h->dec_bf16 && L.has16 && !c.vq_critical) { p.bf16 = 1; p.whh_p16 = c.W(L.whh16[l]); }
            p.skip = l == 1 ? x + (size_t)b0 * T * H : nullptr;
            p.y = (l == 0 ? h1 : y) + (size_t)b0 * T * H;
            p.hT = hT; p.bar = bar;
            p.B = nb; p.T = T; p.H = H; p.U = L.U; p.G = L.G;
            c.begin("lstm_rec", 2.0 * nb * T * 4.0 * H * H, 4.0 * ((double)nb * T * 5 * H + 4.0 * H * H));
            if (st && (!v2 || B > 32)) { c.check(cudaErrorNotSupported, "lstm.stream (needs the resident-W kernel and B <= 32)"); c.end(); continue; }
            if (v2) {
                p.whh_p2 = reinterpret_cast<const uint32_t*>(c.W(L.whh2[l][pass3]));
                p.h16 = h16; p.pass3 = pass3;
                if (st) { p.state_h = st->h[l]; p.state_c = st->c[l]; }
                c.check(launch_lstm2_layer(p, c.st), "lstm.rec2");
            } else {
                c.check(launch_lstm_layer(p, c.st), "lstm.rec");
            }
            c.end();
        }
    }
}

size_t enc_stage_floats(int B, int T) {
    // largest activation of the encoder: [B][T][64] (== [B][T/2][128])
    return (size_t)B * ((size_t)T + 16) * 64;
}

// Encoder.forward (dac.py:69-104): x [B][T][1] -> z channels-last [B][Tz][1024] (or NCT when z_nct)
// Encoder front: conv0 + the four EncoderBlocks (a causal FIR stack) -> features [B][ceil(T/300)][1024] in workspace.
float* encoder_front(Ctx& c, const float* x, int B, int T, int* frames) {
    const EncW& e = c.h->enc;
    size_t stage = enc_stage_floats(B, T);
    float* buf[3] = {c.alloc<float>(stage), c.alloc<float>(stage), c.alloc<float>(stage)};
    int cur = 0;
    int t = sconv(c, e.conv0, x, buf[0], B, T, 1, 1, ConvOpts(), "enc.conv0");
    c.tap("enc_conv0", buf[0], (size_t)B * t * 64);
    static const char* blk_names[4] = {"enc_block1", "enc_block2", "enc_block3", "enc_block4"};
    for (int i = 0; i < 4; ++i) {
        for (int j = 0; j < 3; ++j) {
            int tmp = (cur + 1) % 3, nxt = (cur + 2) % 3;
            residual_unit(c, e.blk[i].res[j], buf[cur], buf[tmp], buf[nxt], B, t);
            cur = nxt;
        }
        ConvOpts o;
        o.in_snake = &e.blk[i].snake;
        int nxt = (cur + 1) % 3;
        t = sconv(c, e.blk[i].down, buf[cur], buf[nxt], B, t, 1, e.blk[i].stride, o, "enc.down");
        cur = nxt;
        c.tap(blk_names[i], buf[cur], (size_t)B * t * e.blk[i].down.Cout);
    }
    *frames = t;
    return buf[cur];
}

// Encoder.forward (dac.py:69-104): x [B][T][1] -> z channels-last [B][Tz][1024] (or NCT when z_nct)
int encoder_forward(Ctx& c, const float* x, int B, int T, float* z_out, bool z_nct) {
    const EncW& e = c.h->enc;
    c.vq_critical = true;
    int t = 0;
    float* feats = encoder_front(c, x, B, T, &t);
    float* ylstm = c.alloc<float>((size_t)B * t * LATENT);
    slstm(c, e.lstm, feats, ylstm, B, t);
    c.tap("enc_lstm", ylstm, (size_t)B * t * 1024);
    ConvOpts o;
    o.in_snake = &e.snake;
    if (z_nct) {
        // same kernel as the channels-last path (bit-identical z), then a [B][T][C] -> [B][C][T] transpose
        float* zcl = c.alloc<float>((size_t)B * t * LATENT);
        sconv(c, e.conv_out, ylstm, zcl, B, t, 1, 1, o, "enc.conv_out");
        if (!c.dry) c.check(launch_transpose(zcl, z_out, B, t, LATENT, c.st), "enc.z_T");
    } else {
        sconv(c, e.conv_out, ylstm, z_out, B, t, 1, 1, o, "enc.conv_out");
    }
    c.vq_critical = false;
    return t;
}

// Decoder.forward (dac.py:131-165): z channels-last [B][Tf][1024] -> y [B][300 Tf][1].  d = the codec's decoder (causal,
// SLSTM) or the redecoder's (non-causal, no SLSTM).
// The upsampling stack after the (optional) SLSTM: 4 DecoderBlocks, Snake, final conv, tanh.  in [B][Tf][1536] -> y [B][300 Tf].
// buf[0..2]: three stage buffers of decoder_stage_floats(B, Tf) each; `in` may be one of them (index in_idx) or external (-1).
size_t decoder_stage_floats(int B, int Tf) {
    size_t stage = (size_t)B * (size_t)Tf * 28800 + 1024;   // largest: [B][Tf*150][192] == [B][Tf*300][96]
    size_t first = (size_t)B * Tf * 1536;
    return first > stage ? first : stage;
}
void decoder_stack(Ctx& c, const DecW& d, const float* in, int in_idx, float* const* buf, int B, int Tf, float* y) {
    int t = Tf;
    const float* cur_p = in;
    int cur = in_idx;
    static const char* dblk_names[4] = {"dec_block1", "dec_block2", "dec_block3", "dec_block4"};
    for (int i = 0; i < 4; ++i) {
        // Snake -> SConvTranspose1d(k=2s, stride s) as a zero-padded conv with s*Cout phase-major channels:
        // causal = 2 taps (x[t-1], x[t]), non-causal = 3 taps (x[t-1], x[t], x[t+1])
        ConvOpts o;
        o.in_snake = &d.blk[i].snake;
        o.pad_left = 1; o.pad_right = d.causal ? 0 : 1; o.reflect = 0;
        int nxt = cur < 0 ? 0 : (cur + 1) % 3;
        run_conv(c, d.blk[i].up, cur_p, buf[nxt], B, t, t, o, "dec.up");
        cur = nxt; cur_p = buf[cur];
        t *= d.blk[i].stride;
        for (int j = 0; j < 3; ++j) {
            int tmp = (cur + 1) % 3, nx2 = (cur + 2) % 3;
            residual_unit(c, d.blk[i].res[j], buf[cur], buf[tmp], buf[nx2], B, t, d.causal);
            cur = nx2; cur_p = buf[cur];
        }
        c.tap(dblk_names[i], buf[cur], (size_t)B * t * d.blk[i].cout);
    }
    ConvOpts o;
    o.in_snake = &d.snake;
    o.act = ACT_TANH;
    sconv(c, d.conv_out, buf[cur], y, B, t, 1, 1, o, "dec.conv_out", d.causal);
}

void decoder_forward(Ctx& c, const DecW& d, const float* z, int B, int Tf, float* y) {
    const size_t stage = decoder_stage_floats(B, Tf);
    float* buf[3] = {c.alloc<float>(stage), c.alloc<float>(stage), c.alloc<float>(stage)};
    int cur = 0;
    int t = sconv(c, d.conv0, z, buf[0], B, Tf, 1, 1, ConvOpts(), "dec.conv0", d.causal);
    c.tap("dec_conv0", buf[0], (size_t)B * t * 1536);
    if (d.has_lstm) {
        slstm(c, d.lstm, buf[0], buf[1], B, t);
        cur = 1;
        c.tap("dec_lstm", buf[1], (size_t)B * t * 1536);
    }
    decoder_stack(c, d, buf[cur], cur, buf, B, t, y);
}

__global__ void embed_sum_kernel(const int64_t* __restrict__ codes_p, const int64_t* __restrict__ codes_c, int cc_stride,
                                 const float* __restrict__ ep, const float* __restrict__ ec0, const float* __restrict__ ec1,
                                 float* __restrict__ out, int T, int hidden, int use_p, int n_c) {
    // one CTA per (b, t): out[b][t][:] = [use_p] E_p[codes_p[b,0,t]] + sum_{i < n_c} E_c[i][codes_c[b,i,t]]  (redecoder.py:36-46)
    const int bt = blockIdx.x, b = bt / T, t = bt - b * T;
    const long long ip = use_p ? codes_p[(size_t)b * T + t] : -1;
    const long long i0 = n_c > 0 ? codes_c[(size_t)b * cc_stride + t] : -1;
    const long long i1 = n_c > 1 ? codes_c[(size_t)b * cc_stride + T + t] : -1;
    for (int c = threadIdx.x; c < hidden; c += blockDim.x) {
        float pe = 0.f, ce = 0.f;                 // the reference sums the prosody and the content embeddings apart
        if (ip >= 0) pe += ep[(size_t)ip * hidden + c];
        if (i0 >= 0) ce += ec0[(size_t)i0 * hidden + c];
        if (i1 >= 0) ce += ec1[(size_t)i1 * hidden + c];
        out[(size_t)bt * hidden + c] = pe + ce;
    }
}

// Redecoder.forward (modules/redecoder.py:35-48): codes -> embeddings -> WN conditioned on the timbre -> conv_out.
// codes_p [B][1][T], codes_c [B][ncc][T] int64 (device), timbre [B][1024]; returns channels-last z [B][T][1024] in workspace.
float* redecoder_forward(Ctx& c, const int64_t* codes_p, const int64_t* codes_c, int ncc, const float* timbre, int B, int T,
                         int use_p, int use_c, int n_c) {
    const RedW& r = c.h->red;
    const int Hd = r.hidden;
    float* x = c.alloc<float>((size_t)B * T * Hd);
    float* pin = c.alloc<float>((size_t)B * T * 2 * Hd);
    float* acts = c.alloc<float>((size_t)B * T * Hd);
    float* rs = c.alloc<float>((size_t)B * T * 2 * Hd);
    float* skip = c.alloc<float>((size_t)B * T * Hd);
    float* g = c.alloc<float>((size_t)B * 2 * Hd * r.layers);
    float* z = c.alloc<float>((size_t)B * T * LATENT);
    if (!c.dry) {
        embed_sum_kernel<<<B * T, 128, 0, c.st>>>(codes_p, codes_c, ncc * T, c.W(r.emb_p), c.W(r.emb_c[0]), c.W(r.emb_c[1]), x, T, Hd,
                                                  use_p, use_c ? n_c : 0);
        c.check(cudaGetLastError(), "red.embed");
    }
    run_conv(c, r.cond, timbre, g, 1, B, B, ConvOpts(), "red.cond");        // cond_layer on g [B,1024,1]: a Linear per utterance
    if (!c.dry) c.check_nk(cudaMemsetAsync(skip, 0, sizeof(float) * (size_t)B * T * Hd, c.st), "red.zero");
    for (int i = 0; i < r.layers; ++i) {
        sconv(c, r.wn_in[i], x, pin, B, T, 1, 1, ConvOpts(), "red.in", false);
        if (!c.dry) c.check(launch_wn_gate(pin, acts, (size_t)B * T, Hd, c.st, g + (size_t)i * 2 * Hd, (size_t)T, (size_t)2 * Hd * r.layers), "red.gate");
        sconv(c, r.wn_rs[i], acts, rs, B, T, 1, 1, ConvOpts(), "red.rs", false);
        if (!c.dry) c.check(launch_wn_update(rs, x, skip, (size_t)B * T, Hd, i == r.layers - 1, c.st), "red.upd");
    }
    run_conv(c, r.conv_out, skip, z, B, T, T, ConvOpts(), "red.conv_out");
    return z;
}

// mel [B][Tm][80] from wave [B][T] (Tm = T/300), preprocess modules/quantize.py:239-242
struct MelW { const ConvW* dft; const ConvW* dft_tc; size_t fb; };
float* mel_forward(Ctx& c, const float* wave, int B, int T, int Tm, const MelW* mw = nullptr) {
    MelW q;
    if (mw) q = *mw; else { q.dft = &c.h->qw.dft; q.dft_tc = &c.h->qw.dft_tc; q.fb = c.h->qw.fb; }
    if (c.h->use_tc >= 2 && q.dft_tc->tc) {
        // frames gather + K=1 GEMM on the promoted tcgen05 kernel (the mel feeds the prosody VQ: fp32-grade sums)
        float* frames = c.alloc<float>((size_t)B * Tm * WIN);
        float* spec = c.alloc<float>((size_t)B * Tm * SPEC_TC_LD);
        float* mel = c.alloc<float>((size_t)B * Tm * N_MELS);
        if (!c.dry) c.check(launch_stft_frames(wave, frames, B, T, Tm, HOP, WIN, N_FFT / 2 - (N_FFT - WIN) / 2, c.st), "mel.frames");
        run_conv(c, *q.dft_tc, frames, spec, 1, B * Tm, B * Tm, ConvOpts(), "mel.dft");
        if (!c.dry) c.check(launch_mel_from_spec(spec, SPEC_TC_LD, c.W(q.fb), mel, B, Tm, Tm, c.st), "mel.fb");
        c.tap("mel80", mel, (size_t)B * Tm * N_MELS);
        return mel;
    }
    float* spec = c.alloc<float>((size_t)B * Tm * SPEC_LD);
    float* mel = c.alloc<float>((size_t)B * Tm * N_MELS);
    ConvOpts o;
    o.stride = HOP;
    o.pad_left = N_FFT / 2 - (N_FFT - WIN) / 2;   // 1024 - 424 = 600
    o.pad_right = 600;
    o.reflect = 1;
    o.no_bias = true;
    o.ldy = SPEC_LD;
    run_conv(c, *q.dft, wave, spec, B, T, Tm, o, "mel.dft");
    if (!c.dry) c.check(launch_mel_from_spec(spec, SPEC_LD, c.W(q.fb), mel, B, Tm, Tm, c.st), "mel.fb");
    c.tap("mel80", mel, (size_t)B * Tm * N_MELS);
    return mel;
}

// StyleEncoder.forward (modules/style_encoder.py:63-81): mel80 [B][Tm][80] -> timbre [B][1024]
void style_encoder(Ctx& c, const float* mel, int B, int Tm, const int* vlen, float* timbre) {
    const QuantW& q = c.h->qw;
    float* a = c.alloc<float>((size_t)B * Tm * 512);
    float* x = c.alloc<float>((size_t)B * Tm * 512);
    float* y2 = c.alloc<float>((size_t)B * Tm * 1024);
    float* qb = c.alloc<float>((size_t)B * Tm * 512);
    float* kb = c.alloc<float>((size_t)B * Tm * 512);
    float* vb = c.alloc<float>((size_t)B * Tm * 512);
    float* ob = c.alloc<float>((size_t)B * Tm * 512);
    ConvOpts o;
    o.act = ACT_MISH;
    run_conv(c, q.spec0, mel, a, B, Tm, Tm, o, "se.spec0");
    o.valid_len = vlen;
    run_conv(c, q.spec3, a, x, B, Tm, Tm, o, "se.spec3");
    for (int i = 0; i < 2; ++i) {
        ConvOpts g;
        g.pad_left = 2; g.pad_right = 2; g.reflect = 0;
        run_conv(c, q.glu[i], x, y2, B, Tm, Tm, g, "se.glu");
        if (!c.dry) c.check(launch_glu_res(y2, x, B, Tm, 512, i == 1 ? vlen : nullptr, c.st), "se.glu_res");
    }
    ConvOpts p;
    run_conv(c, q.cq, x, qb, B, Tm, Tm, p, "se.q");
    run_conv(c, q.ck, x, kb, B, Tm, Tm, p, "se.k");
    run_conv(c, q.cv, x, vb, B, Tm, Tm, p, "se.v");
    if (!c.dry) c.check(launch_attention(qb, kb, vb, ob, B, Tm, 2, 256, vlen, c.st, c.h->attn_stream), "se.attn");
    ConvOpts r;
    r.res = x;
    run_conv(c, q.co, ob, a, B, Tm, Tm, r, "se.o");          // a = x + conv_o(attn)
    run_conv(c, q.fc, a, y2, B, Tm, Tm, ConvOpts(), "se.fc");
    if (!c.dry) c.check(launch_mean_pool(y2, timbre, B, Tm, 1024, vlen, c.st), "se.pool");
}

__global__ void lens_to_frames_kernel(const int64_t* lens, int* out, int B, int hop, int maxf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) {
        long long f = lens[i] / hop;
        out[i] = (int)(f < maxf ? f : maxf);
    }
}

struct QuantOut {
    float* outs_cl; float* zp_cl; float* zc_cl; float* zr_cl; int Tq;
};

// FAquantizer.forward_v2, the part that depends on the waveform only (modules/quantize.py:378-404): timbre (mel ->
// StyleEncoder -> timbre_linear) and the prosody features (mel[:, :20] -> melspec_linear -> WN -> melspec_linear2).  Nothing
// here reads the encoder's latents, so fac_codec_forward runs it on a second stream beside the encoder.
struct QuantFront { float* gb; float* f0; int Tm; };
QuantFront quantizer_front(Ctx& c, const float* wave, int B, int T, const float* full_waves, int T_full, const int64_t* wave_lens,
                           float* timbre) {
    const QuantW& q = c.h->qw;
    const int Tm = T / HOP;
    const bool was_critical = c.vq_critical;
    c.vq_critical = true;      // quantizer-side layers are tiny: all of them use the promoted kernel
    // --- timbre ---
    float* mel = mel_forward(c, wave, B, T, Tm);
    float* timbre_ws = c.alloc<float>((size_t)B * 1024);
    if (!timbre) timbre = timbre_ws;
    if (full_waves) {
        int Tmf = T_full / HOP;
        float* melf = mel_forward(c, full_waves, B, T_full, Tmf);
        int* vlen = c.alloc<int>(B);
        if (!c.dry) {
            lens_to_frames_kernel<<<(B + 127) / 128, 128, 0, c.st>>>(wave_lens, vlen, B, HOP, Tmf);
            c.check(cudaGetLastError(), "lens");
        }
        style_encoder(c, melf, B, Tmf, vlen, timbre);
    } else {
        style_encoder(c, mel, B, Tm, nullptr, timbre);
    }
    float* gb = c.alloc<float>((size_t)B * 2048);
    run_conv(c, q.timbre_linear, timbre, gb, 1, B, B, ConvOpts(), "timbre_linear");
    c.tap("gamma_beta", gb, (size_t)B * 2048);
    // --- prosody branch: mel[:, :20] -> melspec_linear -> WN -> melspec_linear2 ---
    float* px = c.alloc<float>((size_t)B * Tm * 256);
    float* pin = c.alloc<float>((size_t)B * Tm * 512);
    float* acts = c.alloc<float>((size_t)B * Tm * 256);
    float* rs = c.alloc<float>((size_t)B * Tm * 512);
    float* skip = c.alloc<float>((size_t)B * Tm * 256);
    float* f0 = c.alloc<float>((size_t)B * Tm * 1024);
    {
        ConvW lin = q.mel_lin;
        ConvOpts o;
        o.ldx = N_MELS;
        run_conv(c, lin, mel, px, B, Tm, Tm, o, "melspec_linear");
        if (!c.dry) c.check_nk(cudaMemsetAsync(skip, 0, sizeof(float) * (size_t)B * Tm * 256, c.st), "wn.zero");
        for (int i = 0; i < 8; ++i) {
            sconv(c, q.wn_in[i], px, pin, B, Tm, 1, 1, ConvOpts(), "wn.in");
            if (!c.dry) c.check(launch_wn_gate(pin, acts, (size_t)B * Tm, 256, c.st), "wn.gate");
            sconv(c, q.wn_rs[i], acts, rs, B, Tm, 1, 1, ConvOpts(), "wn.rs");
            if (!c.dry) c.check(launch_wn_update(rs, px, skip, (size_t)B * Tm, 256, i == 7, c.st), "wn.upd");
        }
        sconv(c, q.mel_lin2, skip, f0, B, Tm, 1, 1, ConvOpts(), "melspec_linear2");
        c.tap("f0_input", f0, (size_t)B * Tm * 1024);
    }
    c.vq_critical = was_critical;
    QuantFront fr;
    fr.gb = gb; fr.f0 = f0; fr.Tm = Tm;
    return fr;
}

// FAquantizer.forward_v2 on channels-last z; returns channels-last outputs in workspace
QuantOut quantizer_forward(Ctx& c, const float* z_cl, const float* wave, int B, int T, int Tz, int n_c,
                           const float* full_waves, int T_full, const int64_t* wave_lens, float* losses2,
                           float* timbre, int64_t* codes_p, int64_t* codes_c, int64_t* codes_r, bool want_parts,
                           const QuantFront* pre = nullptr) {
    const QuantW& q = c.h->qw;
    const int Tm = T / HOP;
    const int Tq = Tm < Tz ? Tm : Tz;
    c.vq_critical = true;
    QuantFront fr = pre ? *pre : quantizer_front(c, wave, B, T, full_waves, T_full, wave_lens, timbre);
    float* gb = fr.gb;
    float* f0 = fr.f0;
    // --- fused per-frame VQ + AdaLN ---
    QuantOut out;
    out.Tq = Tq;
    out.outs_cl = c.alloc<float>((size_t)B * Tq * 1024);
    out.zp_cl = want_parts ? c.alloc<float>((size_t)B * Tq * 1024) : nullptr;
    out.zc_cl = want_parts ? c.alloc<float>((size_t)B * Tq * 1024) : nullptr;
    out.zr_cl = want_parts ? c.alloc<float>((size_t)B * Tq * 1024) : nullptr;
    float* sqerr = c.alloc<float>((size_t)6 * B * Tq);
    int64_t* cp = c.alloc<int64_t>((size_t)B * Tq);
    int64_t* cc = c.alloc<int64_t>((size_t)B * 2 * Tq);
    int64_t* cr = c.alloc<int64_t>((size_t)B * 3 * Tq);
    float* loss_ws = c.alloc<float>(2);
    c.vq_critical = false;
    if (c.dry) return out;
    FaqParams fp;
    fp.f0 = f0; fp.z = z_cl;
    for (int i = 0; i < 6; ++i) {
        const VqW& v = q.vq[i];
        fp.vq[i] = VqWeights{c.W(v.w_in), c.W(v.b_in), c.W(v.cb), c.W(v.cbn), c.W(v.cbn2), c.W(v.w_out), c.W(v.b_out)};
    }
    fp.n_c = n_c;
    fp.gamma_beta = gb;
    fp.outs = out.outs_cl; fp.zp = out.zp_cl; fp.zc = out.zc_cl; fp.zr = out.zr_cl;
    fp.codes_p = codes_p ? codes_p : cp;
    fp.codes_c = codes_c ? codes_c : cc;
    fp.codes_r = codes_r ? codes_r : cr;
    fp.sqerr = sqerr;
    fp.B = B; fp.Tq = Tq; fp.Tz = Tz; fp.Tf0 = Tm;
    c.begin("fa_quantize", 2.0 * B * Tq * (3 + n_c + 1) * (8.0 * 1024 * 3), 4.0 * (double)B * Tq * 1024 * (3 + (want_parts ? 3 : 0)));
    c.check(launch_fa_quantize(fp, c.st), "fa_quantize");
    c.end();
    c.check(launch_vq_loss_reduce(sqerr, 6, B, Tq, losses2 ? losses2 : loss_ws, c.st), "vq_loss");
    return out;
}

// Runs the waveform-only half of the quantizer on the handle's side stream, forked after whatever the main stream has
// queued so far (the input copy) and joined by the caller with join_front() before fa_quantize.
bool fork_front(Ctx& c, QuantFront& fr, const float* wave, int B, int T, float* timbre) {
    fac_handle* h = c.h;
    if (!h->overlap_front || h->profiling) { return false; }
    if (c.dry) { fr = quantizer_front(c, wave, B, T, nullptr, 0, nullptr, timbre); return true; }
    if (!h->side) {
        if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            h->overlap_front = 0;
            return false;
        }
    }
    cudaStream_t main_st = c.st;
    c.check_nk(cudaEventRecord(h->ev_fork, main_st), "front.fork");
    c.check_nk(cudaStreamWaitEvent(h->side, h->ev_fork, 0), "front.fork_wait");
    c.st = h->side;
    fr = quantizer_front(c, wave, B, T, nullptr, 0, nullptr, timbre);
    c.check_nk(cudaEventRecord(h->ev_join, h->side), "front.join");
    c.st = main_st;
    return true;
}
void join_front(Ctx& c) {
    if (!c.dry) c.check_nk(cudaStreamWaitEvent(c.st, c.h->ev_join, 0), "front.join_wait");
}

// Decoding from codes: ResidualVectorQuantize.from_codes of each group (dac/nn/quantize.py:200-220) and the forward_v2
// tail (modules/quantize.py:435-449).  gamma, beta = timbre_linear(timbre) in the precision class quantizer_front uses,
// so the forward's own timbre gives the forward's gamma_beta bit for bit; then one dequantize_kernel.  Returns
// channels-last outs [B][T][1024] in workspace; zp_cl / zc_cl / zr_cl (channels-last, may be null) receive the groups.
float* dequantize_forward(Ctx& c, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, int n_c, const int64_t* codes_r,
                          int n_r_rows, int n_r, const float* timbre, int B, int T, float* zp_cl, float* zc_cl, float* zr_cl) {
    const QuantW& q = c.h->qw;
    float* gb = c.alloc<float>((size_t)B * 2048);
    float* outs = c.alloc<float>((size_t)B * T * LATENT);
    const bool was_critical = c.vq_critical;
    c.vq_critical = true;
    run_conv(c, q.timbre_linear, timbre, gb, 1, B, B, ConvOpts(), "timbre_linear");
    c.vq_critical = was_critical;
    c.tap("gamma_beta", gb, (size_t)B * 2048);
    if (c.dry) return outs;
    DequantParams dp;
    dp.codes_p = codes_p; dp.codes_c = codes_c; dp.codes_r = codes_r;
    dp.n_c_rows = n_c_rows; dp.n_c = n_c; dp.n_r_rows = n_r_rows; dp.n_r = n_r;
    for (int i = 0; i < 6; ++i) {
        const VqW& v = q.vq[i];
        dp.vq[i] = VqWeights{c.W(v.w_in), c.W(v.b_in), c.W(v.cb), c.W(v.cbn), c.W(v.cbn2), c.W(v.w_out), c.W(v.b_out)};
    }
    dp.gamma_beta = gb;
    dp.outs = outs; dp.zp = zp_cl; dp.zc = zc_cl; dp.zr = zr_cl;
    dp.B = B; dp.T = T;
    const double frames = (double)B * T;
    const int parts = (zp_cl ? 1 : 0) + (zc_cl ? 1 : 0) + (zr_cl ? 1 : 0);
    c.begin("dequantize", 2.0 * frames * (1 + n_c + n_r) * 8.0 * LATENT,   // 8 = codebook dim
            4.0 * frames * LATENT * (1 + parts) + 8.0 * frames * (1 + n_c + n_r));
    c.check(launch_dequantize(dp, c.st), "dequantize");
    c.end();
    return outs;
}

int ensure_ws(fac_handle* h, size_t bytes) {
    if (bytes <= h->ws_bytes) return FAC_OK;
    if (h->ws) { cudaDeviceSynchronize(); cudaFree(h->ws); h->ws = nullptr; h->ws_bytes = 0; }
    size_t want = bytes + (bytes >> 4) + (1 << 20);
    cudaError_t e = cudaMalloc(&h->ws, want);
    if (e != cudaSuccess) {
        h->err = std::string("workspace cudaMalloc failed: ") + cudaGetErrorString(e);
        cudaGetLastError();
        return FAC_ERR_CUDA;
    }
    h->ws_bytes = want;
    return FAC_OK;
}

int finish(fac_handle* h, Ctx& c) {
    if (c.cerr != cudaSuccess) {
        h->err = std::string("CUDA error at ") + c.where + ": " + cudaGetErrorString(c.cerr);
        return FAC_ERR_CUDA;
    }
    return FAC_OK;
}

// run `body` twice: size pass, then for real
template <typename F>
int two_pass(fac_handle* h, cudaStream_t st, F body) {
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return FAC_ERR_CUDA; }
    Ctx dry{h, st, true};
    body(dry);
    int rc = ensure_ws(h, dry.off);
    if (rc != FAC_OK) return rc;
    h->launches = 0;
    Ctx c{h, st, false};
    body(c);
    return finish(h, c);
}

}  // namespace

// ==========================================================================================
// C-ABI
// ==========================================================================================
extern "C" {

int fac_abi_version(void) { return 2; }

int fac_create(fac_handle** out, int device) {
    if (!out) return FAC_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) { cudaGetLastError(); return FAC_ERR_CUDA; }
    fac_handle* h = new fac_handle();
    h->device = device;
    *out = h;
    return FAC_OK;
}

int fac_destroy(fac_handle* h) {
    if (!h) return FAC_OK;
    cudaSetDevice(h->device);
    if (h->warena) cudaFree(h->warena);
    if (h->ws) cudaFree(h->ws);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->aa_filter) cudaFree(h->aa_filter);
    if (h->mel16_arena) cudaFree(h->mel16_arena);
    if (h->loss_arena) cudaFree(h->loss_arena);
    if (h->spec_arena) cudaFree(h->spec_arena);
    for (float* p : h->rvq_arenas) if (p) cudaFree(p);
    for (auto* hs : h->heads) { if (hs->arena) cudaFree(hs->arena); delete hs; }
    for (auto* ss : h->streams) { for (void* p : ss->all) if (p) cudaFree(p); delete ss; }
    delete h;
    return FAC_OK;
}

const char* fac_last_error(const fac_handle* h) { return h ? h->err.c_str() : "null handle"; }

int fac_load_tensor(fac_handle* h, int module, const char* key, const float* data_host, const int64_t* shape, int ndim) {
    if (!h || !key || !data_host || module < 0 || module >= FAC_NUM_MODULES || ndim < 0 || ndim > 4) return FAC_ERR_INVALID;
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; ++i) { if (shape[i] < 0) return FAC_ERR_INVALID; t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.data.assign(data_host, data_host + n);
    h->host[module][key] = std::move(t);
    h->have[module] = true;
    h->finalized = false;
    return FAC_OK;
}

int fac_finalize(fac_handle* h) {
    if (!h) return FAC_ERR_INVALID;
    h->pack.clear();
    h->pack.reserve(160u << 20);
    try {
        if (h->have[FAC_ENCODER]) pack_encoder(h);
        if (h->have[FAC_QUANTIZER]) pack_quantizer(h);
        if (h->have[FAC_DECODER]) pack_decoder(h);
        if (h->have[FAC_REDECODER]) pack_redecoder(h);
        if (h->have[FAC_REDECODER_DECODER]) pack_decoder_into(h, FAC_REDECODER_DECODER, h->dec2, false, false);
    } catch (const PackError& e) {
        h->err = e.msg;
        return FAC_ERR_STATE;
    }
    cudaError_t e = cudaSetDevice(h->device);
    if (e == cudaSuccess && h->warena) { cudaDeviceSynchronize(); cudaFree(h->warena); h->warena = nullptr; }
    size_t n = h->pack.size() + 64;
    if (e == cudaSuccess) e = cudaMalloc(&h->warena, n * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(h->warena, h->pack.data(), h->pack.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = std::string("weight upload: ") + cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    h->wfloats = n;
    h->pack.clear(); h->pack.shrink_to_fit();
    for (int m = 0; m < FAC_NUM_MODULES; ++m) h->host[m].clear();
    h->finalized = true;
    return FAC_OK;
}

int fac_encode_frames(int T) {
    const int rates[4] = {2, 5, 5, 6};
    int t = T;
    for (int i = 0; i < 4; ++i) t = conv_out_len(t, 2 * rates[i], rates[i]);
    return t;
}

static int check_ready(fac_handle* h, int m) {
    if (!h) return FAC_ERR_INVALID;
    if (!h->finalized || !h->have[m]) { h->err = "module weights not loaded/finalized"; return FAC_ERR_STATE; }
    return FAC_OK;
}

int fac_encode(fac_handle* h, const float* x, int B, int T, float* z, void* stream) {
    int rc = check_ready(h, FAC_ENCODER);
    if (rc) return rc;
    if (!x || !z || B <= 0 || T <= 0) { h->err = "fac_encode: bad arguments"; return FAC_ERR_INVALID; }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) { encoder_forward(c, x, B, T, z, true); });
}

int fac_decode(fac_handle* h, const float* z, int B, int Tf, float* y, void* stream) {
    int rc = check_ready(h, FAC_DECODER);
    if (rc) return rc;
    if (!z || !y || B <= 0 || Tf <= 0) { h->err = "fac_decode: bad arguments"; return FAC_ERR_INVALID; }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* zcl = c.alloc<float>((size_t)B * Tf * LATENT);
        if (!c.dry) c.check(launch_transpose(z, zcl, B, LATENT, Tf, c.st), "dec.z_transpose");
        decoder_forward(c, h->dec, zcl, B, Tf, y);
    });
}

int fac_quantize(fac_handle* h, const float* z, const float* wave, int B, int T, int Tz, int n_c,
                 const float* full_waves, int T_full, const int64_t* wave_lens, float* outs, float* zp, float* zc,
                 float* zr, float* losses2, float* timbre, int64_t* codes_p, int64_t* codes_c, int64_t* codes_r,
                 void* stream) {
    int rc = check_ready(h, FAC_QUANTIZER);
    if (rc) return rc;
    if (!z || !wave || !outs || B <= 0 || Tz <= 0 || n_c < 1 || n_c > 2) { h->err = "fac_quantize: bad arguments"; return FAC_ERR_INVALID; }
    if (T <= N_FFT / 2 || (full_waves && (T_full <= N_FFT / 2 || !wave_lens))) {
        h->err = "fac_quantize: wave shorter than the STFT reflect padding (1024), as torch.stft";
        return FAC_ERR_INVALID;
    }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* zcl = c.alloc<float>((size_t)B * Tz * LATENT);
        if (!c.dry) c.check(launch_transpose(z, zcl, B, LATENT, Tz, c.st), "q.z_transpose");
        QuantOut o = quantizer_forward(c, zcl, wave, B, T, Tz, n_c, full_waves, T_full, wave_lens, losses2, timbre,
                                       codes_p, codes_c, codes_r, zp || zc || zr);
        if (c.dry) return;
        c.check(launch_transpose(o.outs_cl, outs, B, o.Tq, LATENT, c.st), "q.outs_T");
        if (zp) c.check(launch_transpose(o.zp_cl, zp, B, o.Tq, LATENT, c.st), "q.zp_T");
        if (zc) c.check(launch_transpose(o.zc_cl, zc, B, o.Tq, LATENT, c.st), "q.zc_T");
        if (zr) c.check(launch_transpose(o.zr_cl, zr, B, o.Tq, LATENT, c.st), "q.zr_T");
    });
}

int fac_codec_forward(fac_handle* h, const float* x, int B, int T, int n_c, float* y, int64_t* codes_p,
                      int64_t* codes_c, int64_t* codes_r, float* timbre, void* stream) {
    for (int m = 0; m < 3; ++m) { int rc = check_ready(h, m); if (rc) return rc; }
    if (!x || !y || B <= 0 || T <= N_FFT / 2 || n_c < 1 || n_c > 2) { h->err = "fac_codec_forward: bad arguments"; return FAC_ERR_INVALID; }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        int Tz = fac_encode_frames(T);
        float* zcl = c.alloc<float>((size_t)B * Tz * LATENT);
        float* timbre_buf = timbre ? timbre : c.alloc<float>((size_t)B * 1024);
        QuantFront fr;
        const bool forked = fork_front(c, fr, x, B, T, timbre_buf);
        encoder_forward(c, x, B, T, zcl, false);
        if (forked) join_front(c);
        QuantOut o = quantizer_forward(c, zcl, x, B, T, Tz, n_c, nullptr, 0, nullptr, nullptr, timbre_buf, codes_p,
                                       codes_c, codes_r, false, forked ? &fr : nullptr);
        decoder_forward(c, h->dec, o.outs_cl, B, o.Tq, y);
    });
}

int fac_codec_forward_host(fac_handle* h, const float* x_host, int B, int T, int n_c, float* y_host,
                           int64_t* codes_p_host, int64_t* codes_c_host, int64_t* codes_r_host, void* stream) {
    for (int m = 0; m < 3; ++m) { int rc = check_ready(h, m); if (rc) return rc; }
    if (!x_host || !y_host || B <= 0 || T <= N_FFT / 2 || n_c < 1 || n_c > 2) { h->err = "fac_codec_forward_host: bad arguments"; return FAC_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    int Tq = 0;
    int rc = two_pass(h, st, [&](Ctx& c) {
        int Tz = fac_encode_frames(T);
        int Tm = T / HOP;
        Tq = Tm < Tz ? Tm : Tz;
        float* xd = c.alloc<float>((size_t)B * T);
        float* yd = c.alloc<float>((size_t)B * Tq * HOP);
        int64_t* cp = c.alloc<int64_t>((size_t)B * Tq);
        int64_t* cc = c.alloc<int64_t>((size_t)B * 2 * Tq);
        int64_t* cr = c.alloc<int64_t>((size_t)B * 3 * Tq);
        float* zcl = c.alloc<float>((size_t)B * Tz * LATENT);
        if (!c.dry) c.check_nk(cudaMemcpyAsync(xd, x_host, sizeof(float) * (size_t)B * T, cudaMemcpyHostToDevice, c.st), "h2d");
        float* timbre_buf = c.alloc<float>((size_t)B * 1024);
        QuantFront fr;
        const bool forked = fork_front(c, fr, xd, B, T, timbre_buf);
        encoder_forward(c, xd, B, T, zcl, false);
        if (forked) join_front(c);
        QuantOut o = quantizer_forward(c, zcl, xd, B, T, Tz, n_c, nullptr, 0, nullptr, nullptr, timbre_buf, cp, cc, cr, false,
                                       forked ? &fr : nullptr);
        decoder_forward(c, h->dec, o.outs_cl, B, o.Tq, yd);
        if (c.dry) return;
        c.check_nk(cudaMemcpyAsync(y_host, yd, sizeof(float) * (size_t)B * Tq * HOP, cudaMemcpyDeviceToHost, c.st), "d2h.y");
        if (codes_p_host) c.check_nk(cudaMemcpyAsync(codes_p_host, cp, sizeof(int64_t) * (size_t)B * Tq, cudaMemcpyDeviceToHost, c.st), "d2h.cp");
        if (codes_c_host) c.check_nk(cudaMemcpyAsync(codes_c_host, cc, sizeof(int64_t) * (size_t)B * n_c * Tq, cudaMemcpyDeviceToHost, c.st), "d2h.cc");
        if (codes_r_host) c.check_nk(cudaMemcpyAsync(codes_r_host, cr, sizeof(int64_t) * (size_t)B * 3 * Tq, cudaMemcpyDeviceToHost, c.st), "d2h.cr");
    });
    if (rc) return rc;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { h->err = std::string("stream sync: ") + cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_redecode(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, const float* timbre, int B, int T,
                 int use_p_code, int use_c_code, int n_c, float* z, void* stream) {
    int rc = check_ready(h, FAC_REDECODER);
    if (rc) return rc;
    if (!codes_p || !codes_c || !timbre || !z || B <= 0 || T <= 0 || n_c < 0 || n_c > 2 || n_c > n_c_rows) {
        h->err = "fac_redecode: bad arguments (n_c <= rows of codes_c <= 2)";
        return FAC_ERR_INVALID;
    }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* zcl = redecoder_forward(c, codes_p, codes_c, n_c_rows, timbre, B, T, use_p_code, use_c_code, n_c);
        if (!c.dry) c.check(launch_transpose(zcl, z, B, T, LATENT, c.st), "red.z_T");
    });
}

int fac_redecoder_decode(fac_handle* h, const float* z, int B, int Tf, float* y, void* stream) {
    int rc = check_ready(h, FAC_REDECODER_DECODER);
    if (rc) return rc;
    if (!z || !y || B <= 0 || Tf <= 0) { h->err = "fac_redecoder_decode: bad arguments"; return FAC_ERR_INVALID; }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* zcl = c.alloc<float>((size_t)B * Tf * LATENT);
        if (!c.dry) c.check(launch_transpose(z, zcl, B, LATENT, Tf, c.st), "red.dec.z_transpose");
        decoder_forward(c, h->dec2, zcl, B, Tf, y);
    });
}

int fac_voice_convert(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, const float* timbre, int B,
                      int T, int use_p_code, int use_c_code, int n_c, float* y, void* stream) {
    int rc = check_ready(h, FAC_REDECODER);
    if (!rc) rc = check_ready(h, FAC_REDECODER_DECODER);
    if (rc) return rc;
    if (!codes_p || !codes_c || !timbre || !y || B <= 0 || T <= 0 || n_c < 0 || n_c > 2 || n_c > n_c_rows) {
        h->err = "fac_voice_convert: bad arguments";
        return FAC_ERR_INVALID;
    }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* zcl = redecoder_forward(c, codes_p, codes_c, n_c_rows, timbre, B, T, use_p_code, use_c_code, n_c);
        decoder_forward(c, h->dec2, zcl, B, T, y);
    });
}

static bool dequant_args_ok(const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, int n_c, const int64_t* codes_r,
                            int n_r_rows, int n_r, const float* timbre, int B, int T) {
    return codes_p && codes_c && timbre && B > 0 && T > 0 && n_c >= 1 && n_c <= n_c_rows && n_c_rows <= 2 && n_r >= 0 &&
           n_r <= n_r_rows && n_r_rows <= 3 && (n_r == 0 || codes_r);
}

int fac_dequantize(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, int n_c, const int64_t* codes_r,
                   int n_r_rows, int n_r, const float* timbre, int B, int T, float* outs, float* zp, float* zc, float* zr,
                   void* stream) {
    int rc = check_ready(h, FAC_QUANTIZER);
    if (rc) return rc;
    if (!outs || !dequant_args_ok(codes_p, codes_c, n_c_rows, n_c, codes_r, n_r_rows, n_r, timbre, B, T)) {
        h->err = "fac_dequantize: bad arguments (1 <= n_c <= rows of codes_c <= 2, n_r <= rows of codes_r <= 3, B, T > 0)";
        return FAC_ERR_INVALID;
    }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* zp_cl = zp ? c.alloc<float>((size_t)B * T * LATENT) : nullptr;
        float* zc_cl = zc ? c.alloc<float>((size_t)B * T * LATENT) : nullptr;
        float* zr_cl = zr ? c.alloc<float>((size_t)B * T * LATENT) : nullptr;
        float* ocl = dequantize_forward(c, codes_p, codes_c, n_c_rows, n_c, codes_r, n_r_rows, n_r, timbre, B, T, zp_cl, zc_cl, zr_cl);
        if (c.dry) return;
        c.check(launch_transpose(ocl, outs, B, T, LATENT, c.st), "dq.outs_T");
        if (zp) c.check(launch_transpose(zp_cl, zp, B, T, LATENT, c.st), "dq.zp_T");
        if (zc) c.check(launch_transpose(zc_cl, zc, B, T, LATENT, c.st), "dq.zc_T");
        if (zr) c.check(launch_transpose(zr_cl, zr, B, T, LATENT, c.st), "dq.zr_T");
    });
}

int fac_decode_codes(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, int n_c, const int64_t* codes_r,
                     int n_r_rows, int n_r, const float* timbre, int B, int T, float* y, void* stream) {
    int rc = check_ready(h, FAC_QUANTIZER);
    if (!rc) rc = check_ready(h, FAC_DECODER);
    if (rc) return rc;
    if (!y || !dequant_args_ok(codes_p, codes_c, n_c_rows, n_c, codes_r, n_r_rows, n_r, timbre, B, T)) {
        h->err = "fac_decode_codes: bad arguments (1 <= n_c <= rows of codes_c <= 2, n_r <= rows of codes_r <= 3, B, T > 0)";
        return FAC_ERR_INVALID;
    }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        float* ocl = dequantize_forward(c, codes_p, codes_c, n_c_rows, n_c, codes_r, n_r_rows, n_r, timbre, B, T, nullptr, nullptr,
                                        nullptr);
        decoder_forward(c, h->dec, ocl, B, T, y);
    });
}

// ---- streaming (SURVEY.md 8f rank 4): chunked encoder / decoder with LSTM-state carry and conv halos ----
// Left context of the encoder's conv stack: 5581 samples (conv0 6 + stage 1 78 + down 3 + stage 2 156 + down 18 + stage 3 780
// + down 90 + stage 4 3900 + down 550) -> 6000 (20 frames); of the decoder's stack after the LSTM: < 18 latent frames -> 20.
constexpr int kEncCtx = 6000, kDecCtx = 20, kStreamMinFirst = 10;

int fac_stream_begin(fac_handle* h, int B) {
    if (!h || B < 1 || B > 32) { if (h) h->err = "fac_stream_begin: 1 <= B <= 32"; return FAC_ERR_INVALID; }
    if (!h->finalized) { h->err = "module weights not loaded/finalized"; return FAC_ERR_STATE; }
    cudaSetDevice(h->device);
    auto* s = new fac_handle::Stream();
    s->B = B;
    const size_t sizes[12] = {
        sizeof(float) * (size_t)B * kEncCtx, sizeof(float) * (size_t)B * 2 * LATENT, sizeof(float) * (size_t)B * 6 * LATENT,
        sizeof(float) * (size_t)B * kDecCtx * 1536,
        sizeof(uint32_t) * 2 * 512 * 32, sizeof(uint32_t) * 2 * 512 * 32, sizeof(float) * 128 * 32 * 8, sizeof(float) * 128 * 32 * 8,
        sizeof(uint32_t) * 768 * 32, sizeof(uint32_t) * 768 * 32, sizeof(float) * 128 * 32 * 12, sizeof(float) * 128 * 32 * 12};
    for (int i = 0; i < 12; ++i) {
        cudaError_t e = cudaMalloc(&s->all[i], sizes[i]);
        if (e == cudaSuccess) e = cudaMemset(s->all[i], 0, sizes[i]);
        if (e != cudaSuccess) {
            h->err = std::string("fac_stream_begin: ") + cudaGetErrorString(e);
            cudaGetLastError();
            for (void* p : s->all) if (p) cudaFree(p);
            delete s;
            return FAC_ERR_CUDA;
        }
    }
    s->x_hist = (float*)s->all[0]; s->ey_hist = (float*)s->all[1]; s->z_hist = (float*)s->all[2]; s->dy_hist = (float*)s->all[3];
    s->enc_h[0] = (uint32_t*)s->all[4]; s->enc_h[1] = (uint32_t*)s->all[5]; s->enc_c[0] = (float*)s->all[6]; s->enc_c[1] = (float*)s->all[7];
    s->dec_h[0] = (uint32_t*)s->all[8]; s->dec_h[1] = (uint32_t*)s->all[9]; s->dec_c[0] = (float*)s->all[10]; s->dec_c[1] = (float*)s->all[11];
    s->alive = true;
    h->streams.push_back(s);
    return (int)h->streams.size() - 1;
}

int fac_stream_end(fac_handle* h, int stream_id) {
    if (!h || stream_id < 0 || stream_id >= (int)h->streams.size()) return FAC_ERR_INVALID;
    fac_handle::Stream* s = h->streams[stream_id];
    if (s->alive) {
        cudaSetDevice(h->device);
        cudaDeviceSynchronize();
        for (void*& p : s->all) { if (p) cudaFree(p); p = nullptr; }
        s->alive = false;
    }
    return FAC_OK;
}

namespace {
// dst[b][0..n) = src[b][off..off+n) for rows of `w` floats each (row pitches in rows)
void copy_rows(Ctx& c, float* dst, int dst_pitch_rows, const float* src, int src_pitch_rows, int off_rows, int n_rows, int w, int B,
               const char* what) {
    if (c.dry || n_rows <= 0) return;
    c.check_nk(cudaMemcpy2DAsync(dst, sizeof(float) * (size_t)dst_pitch_rows * w, src + (size_t)off_rows * w,
                                 sizeof(float) * (size_t)src_pitch_rows * w, sizeof(float) * (size_t)n_rows * w, B,
                                 cudaMemcpyDeviceToDevice, c.st), what);
}
}  // namespace

int fac_stream_encode(fac_handle* h, int stream_id, const float* x, int T, float* z, void* stream) {
    int rc = check_ready(h, FAC_ENCODER);
    if (rc) return rc;
    if (stream_id < 0 || stream_id >= (int)h->streams.size() || !h->streams[stream_id]->alive || !x || !z) { h->err = "fac_stream_encode: bad arguments"; return FAC_ERR_INVALID; }
    fac_handle::Stream& s = *h->streams[stream_id];
    if (T <= 0 || T % HOP != 0 || (s.enc_samples == 0 && T < kStreamMinFirst * HOP)) {
        h->err = "fac_stream_encode: chunks must be multiples of 300 samples, the first one at least 3000";
        return FAC_ERR_INVALID;
    }
    if (!h->lstm_v2 || !h->enc.lstm.has2[1]) { h->err = "fac_stream_encode: needs the resident-W LSTM kernel"; return FAC_ERR_UNSUPPORTED; }
    const int B = s.B, hist = s.x_hist_len, Tw = hist + T, Fc = T / HOP, Fh = hist / HOP;
    rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        const EncW& e = h->enc;
        c.vq_critical = true;
        float* xw = c.alloc<float>((size_t)B * Tw);
        copy_rows(c, xw, Tw, s.x_hist, kEncCtx, 0, hist, 1, B, "stream.xh");
        copy_rows(c, xw + hist, Tw, x, T, 0, T, 1, B, "stream.xc");
        int Fw = 0;
        float* feats = encoder_front(c, xw, B, Tw, &Fw);                    // [B][Fw][1024], Fw == Fh + Fc
        float* fnew = c.alloc<float>((size_t)B * Fc * LATENT);
        copy_rows(c, fnew, Fc, feats, Fw, Fh, Fc, LATENT, B, "stream.fnew");
        const int yh = s.ey_hist_len;
        float* yw = c.alloc<float>((size_t)B * (yh + Fc) * LATENT);        // [hist | new] LSTM outputs
        float* ynew = c.alloc<float>((size_t)B * Fc * LATENT);
        LstmState st;
        st.h[0] = s.enc_h[0]; st.h[1] = s.enc_h[1]; st.c[0] = s.enc_c[0]; st.c[1] = s.enc_c[1];
        slstm(c, e.lstm, fnew, ynew, B, Fc, &st);
        copy_rows(c, yw, yh + Fc, s.ey_hist, 2, 0, yh, LATENT, B, "stream.yh");
        copy_rows(c, yw + (size_t)yh * LATENT, yh + Fc, ynew, Fc, 0, Fc, LATENT, B, "stream.yc");
        float* zw = c.alloc<float>((size_t)B * (yh + Fc) * LATENT);
        float* znew = c.alloc<float>((size_t)B * Fc * LATENT);
        ConvOpts o;
        o.in_snake = &e.snake;
        sconv(c, e.conv_out, yw, zw, B, yh + Fc, 1, 1, o, "enc.conv_out");
        copy_rows(c, znew, Fc, zw, yh + Fc, yh, Fc, LATENT, B, "stream.znew");
        if (!c.dry) c.check(launch_transpose(znew, z, B, Fc, LATENT, c.st), "enc.z_T");
        // new histories: the last kEncCtx samples / 2 LSTM-output frames of what has been seen so far
        const int nh = Tw < kEncCtx ? Tw : kEncCtx, nyh = yh + Fc < 2 ? yh + Fc : 2;
        float* tmpx = c.alloc<float>((size_t)B * kEncCtx);
        copy_rows(c, tmpx, kEncCtx, xw, Tw, Tw - nh, nh, 1, B, "stream.xh2");
        copy_rows(c, s.x_hist, kEncCtx, tmpx, kEncCtx, 0, nh, 1, B, "stream.xh3");
        copy_rows(c, s.ey_hist, 2, yw, yh + Fc, yh + Fc - nyh, nyh, LATENT, B, "stream.yh2");
        c.vq_critical = false;
    });
    if (rc == FAC_OK) {
        s.x_hist_len = Tw < kEncCtx ? Tw : kEncCtx;
        s.ey_hist_len = s.ey_hist_len + Fc < 2 ? s.ey_hist_len + Fc : 2;
        s.enc_samples += T;
    }
    return rc;
}

int fac_stream_decode(fac_handle* h, int stream_id, const float* z, int Fc, float* y, void* stream) {
    int rc = check_ready(h, FAC_DECODER);
    if (rc) return rc;
    if (stream_id < 0 || stream_id >= (int)h->streams.size() || !h->streams[stream_id]->alive || !z || !y) { h->err = "fac_stream_decode: bad arguments"; return FAC_ERR_INVALID; }
    fac_handle::Stream& s = *h->streams[stream_id];
    if (Fc <= 0 || (s.dec_frames == 0 && Fc < kStreamMinFirst)) { h->err = "fac_stream_decode: the first chunk needs at least 10 frames"; return FAC_ERR_INVALID; }
    if (!h->lstm_v2 || !h->dec_bf16 || !h->dec_lstm_fp16 || !h->dec.lstm.has2[0]) { h->err = "fac_stream_decode: needs the resident-W LSTM kernel"; return FAC_ERR_UNSUPPORTED; }
    const int B = s.B, zh = s.z_hist_len, dh = s.dy_hist_len;
    rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        const DecW& d = h->dec;
        float* znew = c.alloc<float>((size_t)B * Fc * LATENT);
        if (!c.dry) c.check(launch_transpose(z, znew, B, LATENT, Fc, c.st), "dec.z_transpose");
        float* zw = c.alloc<float>((size_t)B * (zh + Fc) * LATENT);
        copy_rows(c, zw, zh + Fc, s.z_hist, 6, 0, zh, LATENT, B, "stream.zh");
        copy_rows(c, zw + (size_t)zh * LATENT, zh + Fc, znew, Fc, 0, Fc, LATENT, B, "stream.zc");
        float* c0w = c.alloc<float>((size_t)B * (zh + Fc) * 1536);
        sconv(c, d.conv0, zw, c0w, B, zh + Fc, 1, 1, ConvOpts(), "dec.conv0");
        float* c0new = c.alloc<float>((size_t)B * Fc * 1536);
        copy_rows(c, c0new, Fc, c0w, zh + Fc, zh, Fc, 1536, B, "stream.c0new");
        float* ynew = c.alloc<float>((size_t)B * Fc * 1536);
        LstmState st;
        st.h[0] = s.dec_h[0]; st.h[1] = s.dec_h[1]; st.c[0] = s.dec_c[0]; st.c[1] = s.dec_c[1];
        slstm(c, d.lstm, c0new, ynew, B, Fc, &st);
        const int Fw = dh + Fc;
        const size_t stage = decoder_stage_floats(B, Fw);
        float* buf[3] = {c.alloc<float>(stage), c.alloc<float>(stage), c.alloc<float>(stage)};
        float* yw_in = c.alloc<float>((size_t)B * Fw * 1536);
        copy_rows(c, yw_in, Fw, s.dy_hist, kDecCtx, 0, dh, 1536, B, "stream.dh");
        copy_rows(c, yw_in + (size_t)dh * 1536, Fw, ynew, Fc, 0, Fc, 1536, B, "stream.dc");
        float* yw = c.alloc<float>((size_t)B * Fw * HOP);
        decoder_stack(c, d, yw_in, -1, buf, B, Fw, yw);
        copy_rows(c, y, Fc * HOP, yw, Fw * HOP, dh * HOP, Fc * HOP, 1, B, "stream.ynew");
        const int nzh = zh + Fc < 6 ? zh + Fc : 6, ndh = Fw < kDecCtx ? Fw : kDecCtx;
        float* tz = c.alloc<float>((size_t)B * 6 * LATENT);
        float* td = c.alloc<float>((size_t)B * kDecCtx * 1536);
        copy_rows(c, tz, 6, zw, zh + Fc, zh + Fc - nzh, nzh, LATENT, B, "stream.zh2");
        copy_rows(c, s.z_hist, 6, tz, 6, 0, nzh, LATENT, B, "stream.zh3");
        copy_rows(c, td, kDecCtx, yw_in, Fw, Fw - ndh, ndh, 1536, B, "stream.dh2");
        copy_rows(c, s.dy_hist, kDecCtx, td, kDecCtx, 0, ndh, 1536, B, "stream.dh3");
    });
    if (rc == FAC_OK) {
        s.z_hist_len = zh + Fc < 6 ? zh + Fc : 6;
        s.dy_hist_len = dh + Fc < kDecCtx ? dh + Fc : kDecCtx;
        s.dec_frames += Fc;
    }
    return rc;
}

// meldataset.py:37-47 preprocess: torchaudio MelSpectrogram(n_mels=80, n_fft=2048, win_length=1200, hop_length=300) with
// its DEFAULT sample_rate = 16000 (HTK filterbank over [0, 8000] Hz -- not the quantizer's 24 kHz one), centre = True
// (T/300 + 1 frames), then (log(1e-5 + mel) + 4) / 4.
int fac_dataset_mel(fac_handle* h, const float* wave, int B, int T, float* mel, void* stream) {
    if (!h || !wave || !mel || B <= 0) return FAC_ERR_INVALID;
    if (T <= N_FFT / 2) { h->err = "fac_dataset_mel: wave shorter than the STFT reflect padding (1024), as torch.stft"; return FAC_ERR_INVALID; }
    cudaSetDevice(h->device);
    if (!h->mel16_arena) {
        fac_handle tmp;
        tmp.device = h->device;
        std::vector<float> win(WIN), fb((size_t)N_BINS * N_MELS);
        for (int i = 0; i < WIN; ++i) win[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * (double)i / (double)WIN));   // periodic Hann
        // torchaudio.functional.melscale_fbanks(n_freqs=1025, f_min=0, f_max=8000, n_mels=80, sample_rate=16000, norm=None, "htk")
        const double sr = 16000.0, f_max = 8000.0;
        auto hz2mel = [](double f) { return 2595.0 * std::log10(1.0 + f / 700.0); };
        auto mel2hz = [](double m) { return 700.0 * (std::pow(10.0, m / 2595.0) - 1.0); };
        std::vector<double> fpts(N_MELS + 2);
        for (int i = 0; i < N_MELS + 2; ++i) fpts[i] = mel2hz(hz2mel(0.0) + (hz2mel(f_max) - hz2mel(0.0)) * i / (N_MELS + 1));
        for (int k = 0; k < N_BINS; ++k) {
            const double f = (sr / 2.0) * k / (N_BINS - 1);
            for (int m = 0; m < N_MELS; ++m) {
                const double down = (f - fpts[m]) / (fpts[m + 1] - fpts[m]), up = (fpts[m + 2] - f) / (fpts[m + 2] - fpts[m + 1]);
                fb[(size_t)k * N_MELS + m] = (float)std::max(0.0, std::min(down, up));
            }
        }
        try { pack_mel_frontend(&tmp, h->mel16_dft, h->mel16_dft_tc, h->mel16_fb, win.data(), fb.data()); }
        catch (const PackError& e) { h->err = e.msg; return FAC_ERR_STATE; }
        cudaError_t e = cudaMalloc(&h->mel16_arena, (tmp.pack.size() + 64) * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpy(h->mel16_arena, tmp.pack.data(), tmp.pack.size() * sizeof(float), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); h->mel16_arena = nullptr; return FAC_ERR_CUDA; }
    }
    float* saved = h->warena;
    h->warena = h->mel16_arena;
    const int F = T / HOP + 1;
    int rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        MelW mw{&h->mel16_dft, &h->mel16_dft_tc, h->mel16_fb};
        c.vq_critical = true;                        // fp32-faithful DFT (the promoted tensor-core kernel)
        float* mel_cl = mel_forward(c, wave, B, T, F, &mw);
        c.vq_critical = false;
        if (!c.dry) c.check(launch_transpose(mel_cl, mel, B, F, N_MELS, c.st), "mel16.T");
    });
    h->warena = saved;
    return rc;
}

// ---- losses.py:65-89 reconstruction_loss (SURVEY.md 8f rank 3: the loss forward of the training step) ----
// L = 100 * mse(x, G_x) + sum_{s = 64..2048} (l1_s + sqrt(s/2) * l2_s) over 64-band mel spectrograms
// (torchaudio MelSpectrogram(sample_rate=16000, n_fft=max(s,512), win_length=s, hop_length=s/4, n_mels=64): periodic Hann
// window of s samples centred in the n_fft frame, centre = True reflect padding, power 2, HTK bands over [0, 8000] Hz).
// Per scale: frame gather of both signals -> one GEMM against the window-folded DFT basis (fp32-faithful tensor-core class)
// -> mel_loss_terms_kernel -> fp64 sums in a fixed order.
int fac_reconstruction_loss(fac_handle* h, const float* x, const float* gx, int B, int T, float* loss, float* terms, void* stream) {
    if (!h || !x || !gx || !loss || B <= 0 || T <= 0) return FAC_ERR_INVALID;
    if (T <= 1024) { h->err = "fac_reconstruction_loss: signals must be longer than the largest STFT reflect padding (1024), as torch.stft"; return FAC_ERR_INVALID; }
    if (B > 32767) { h->err = "fac_reconstruction_loss: B > 32767"; return FAC_ERR_UNSUPPORTED; }
    cudaSetDevice(h->device);
    if (!h->loss_arena) {
        fac_handle tmp;
        tmp.device = h->device;
        const int NM = 64;
        auto hz2mel = [](double f) { return 2595.0 * std::log10(1.0 + f / 700.0); };
        auto mel2hz = [](double m) { return 700.0 * (std::pow(10.0, m / 2595.0) - 1.0); };
        std::vector<double> fpts(NM + 2);
        for (int i = 0; i < NM + 2; ++i) fpts[i] = mel2hz(hz2mel(0.0) + (hz2mel(8000.0) - hz2mel(0.0)) * i / (NM + 1));
        try {
            for (int i = 0; i < 6; ++i) {
                fac_handle::LossScale& L = h->loss_scale[i];
                L.s = 64 << i; L.nfft = L.s < 512 ? 512 : L.s; L.nb = L.nfft / 2 + 1;
                L.ld = (2 * L.nb + 127) / 128 * 128;            // zero columns beyond 2 * nb: whole 128-channel MMA tiles
                ConvW& d = L.dft;
                d = ConvW();
                d.Cin = L.s; d.Cout = L.ld; d.K = 1; d.ldw = L.ld;
                d.w = pack_alloc(&tmp, (size_t)L.s * L.ld);
                d.b = pack_alloc(&tmp, L.ld);
                const int left = (L.nfft - L.s) / 2;
                for (int n = 0; n < L.s; ++n) {
                    const double w = 0.5 - 0.5 * std::cos(2.0 * M_PI * (double)n / (double)L.s);       // periodic Hann(s)
                    for (int k = 0; k < L.nb; ++k) {
                        const long long ph = ((long long)k * (n + left)) % L.nfft;
                        const double ang = 2.0 * M_PI * (double)ph / (double)L.nfft;
                        tmp.pack[d.w + (size_t)n * L.ld + 2 * k] = (float)(w * std::cos(ang));
                        tmp.pack[d.w + (size_t)n * L.ld + 2 * k + 1] = (float)(-w * std::sin(ang));
                    }
                }
                attach_tc(&tmp, d, 1, true);
                // torchaudio.functional.melscale_fbanks(n_freqs, 0, 8000, 64, sample_rate=16000, norm=None, "htk")
                L.fb = pack_alloc(&tmp, (size_t)L.nb * NM);
                for (int k = 0; k < L.nb; ++k) {
                    const double f = 8000.0 * k / (L.nb - 1);
                    for (int m = 0; m < NM; ++m) {
                        const double down = (f - fpts[m]) / (fpts[m + 1] - fpts[m]), up = (fpts[m + 2] - f) / (fpts[m + 2] - fpts[m + 1]);
                        tmp.pack[L.fb + (size_t)k * NM + m] = (float)std::max(0.0, std::min(down, up));
                    }
                }
            }
        } catch (const PackError& e) { h->err = e.msg; return FAC_ERR_STATE; }
        cudaError_t e = cudaMalloc(&h->loss_arena, (tmp.pack.size() + 64) * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpy(h->loss_arena, tmp.pack.data(), tmp.pack.size() * sizeof(float), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); h->loss_arena = nullptr; return FAC_ERR_CUDA; }
    }
    float* saved = h->warena;
    h->warena = h->loss_arena;
    int rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        double* sums = c.alloc<double>(16);
        const int nblk = 1024;
        float* part = c.alloc<float>(nblk);
        if (!c.dry) {
            c.check(launch_sqdiff_partial(x, gx, (long long)B * T, part, nblk, c.st), "loss.mse");
            c.check(launch_strided_sum(part, nblk, 1, 1.0 / ((double)B * T), sums, c.st), "loss.mse.sum");
        }
        const size_t mark = c.off;                                   // the scales run one after another on one stream:
        size_t peak = c.off;                                         // they share the scratch above this mark
        c.vq_critical = true;                                        // fp32-faithful DFT (promoted tensor-core class)
        for (int i = 0; i < 6; ++i) {
            c.off = mark;
            const fac_handle::LossScale& L = c.h->loss_scale[i];
            const int hop = L.s / 4, F = T / hop + 1;
            const size_t rows = (size_t)2 * B * F;
            float* frames = c.alloc<float>(rows * L.s);
            float* spec = c.alloc<float>(rows * L.ld);
            float* tr = c.alloc<float>((size_t)B * F * 2);
            if (!c.dry) {
                c.check(launch_stft_frames(x, frames, B, T, F, hop, L.s, L.s / 2, c.st), "loss.frames");
                c.check(launch_stft_frames(gx, frames + (size_t)B * F * L.s, B, T, F, hop, L.s, L.s / 2, c.st), "loss.frames");
            }
            run_conv(c, L.dft, frames, spec, 1, (int)rows, (int)rows, ConvOpts(), "loss.dft");
            if (!c.dry) {
                c.check(launch_mel_loss_terms(spec, L.ld, L.nb, c.W(L.fb), B, F, 1e-7f, tr, c.st), "loss.mel");
                c.check(launch_strided_sum(tr, (long long)B * F, 2, 1.0 / ((double)B * F * 64.0), sums + 1 + 2 * i, c.st), "loss.l1");
                c.check(launch_strided_sum(tr + 1, (long long)B * F, 2, 1.0 / ((double)B * F), sums + 2 + 2 * i, c.st), "loss.l2");
            }
            if (c.off > peak) peak = c.off;
        }
        c.vq_critical = false;
        c.off = peak;
        if (!c.dry) c.check(launch_loss_combine(sums, loss, terms, c.st), "loss.combine");
    });
    h->warena = saved;
    return rc;
}

// ---- dac/nn/loss.py:142-327 MultiScaleSTFTLoss / MelSpectrogramLoss, :11-47 L1Loss (forward values) ----
// The reference computes them on audiotools AudioSignal objects (AudioSignal.stft / .magnitude / .mel_spectrogram; the
// package is not vendored: SURVEY.md 8c, parity unpinned).  Restated semantics: torch.stft(n_fft = window_length, hop =
// window_length / 4, periodic Hann window (scipy.signal.get_window("hann")), centre = True, reflect padding), magnitude =
// |stft|; mel_spectrogram = magnitude @ librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax)^T (Slaney scale, Slaney area
// normalisation).  loss = sum over scales of log_weight * L1(log10(clamp(v, eps)^pow)) + mag_weight * L1(v).
namespace {
void slaney_mel_fb(double sr, int n_fft, int n_mels, double fmin, double fmax, std::vector<float>& fb /* [nb][n_mels] */) {
    const int nb = n_fft / 2 + 1;
    const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp, logstep = std::log(6.4) / 27.0;
    auto hz2mel = [&](double f) { return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp; };
    auto mel2hz = [&](double m) { return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m; };
    std::vector<double> mf(n_mels + 2);
    const double m0 = hz2mel(fmin), m1 = hz2mel(fmax);
    for (int i = 0; i < n_mels + 2; ++i) mf[i] = mel2hz(m0 + (m1 - m0) * i / (n_mels + 1));
    fb.assign((size_t)nb * n_mels, 0.f);
    for (int k = 0; k < nb; ++k) {
        const double f = (sr / 2.0) * k / (nb - 1);
        for (int m = 0; m < n_mels; ++m) {
            const double lower = (f - mf[m]) / (mf[m + 1] - mf[m]), upper = (mf[m + 2] - f) / (mf[m + 2] - mf[m + 1]);
            const double w = std::max(0.0, std::min(lower, upper)) * (2.0 / (mf[m + 2] - mf[m]));
            fb[(size_t)k * n_mels + m] = (float)w;
        }
    }
}
}  // namespace

int fac_spectral_loss(fac_handle* h, const float* x, const float* y, int B, int T, int sample_rate, int n_scales, const int* window_lengths,
                      const int* n_mels, const float* mel_fmin, const float* mel_fmax, float clamp_eps, float mag_weight, float log_weight,
                      float pw, float* loss, void* stream) {
    if (!h || !x || !y || !loss || !window_lengths || B <= 0 || T <= 0 || n_scales < 1 || n_scales > 16 || sample_rate <= 0) return FAC_ERR_INVALID;
    if (B > 32767) { h->err = "fac_spectral_loss: B > 32767"; return FAC_ERR_UNSUPPORTED; }
    std::vector<double> key{(double)sample_rate, (double)n_scales};
    for (int i = 0; i < n_scales; ++i) {
        const int w = window_lengths[i];
        if (w < 16 || w > 4096 || (w & (w - 1)) != 0) { h->err = "fac_spectral_loss: window lengths must be powers of two in [16, 4096]"; return FAC_ERR_UNSUPPORTED; }
        if (T <= w / 2) { h->err = "fac_spectral_loss: signals must be longer than half the largest window (reflect padding), as torch.stft"; return FAC_ERR_INVALID; }
        const int nm = n_mels ? n_mels[i] : 0;
        if (nm < 0 || nm > 1024) return FAC_ERR_INVALID;
        const double f0 = (n_mels && mel_fmin) ? mel_fmin[i] : 0.0;
        const double f1 = (n_mels && mel_fmax && mel_fmax[i] > 0.f) ? mel_fmax[i] : sample_rate / 2.0;
        key.push_back(w); key.push_back(nm); key.push_back(f0); key.push_back(f1);
    }
    cudaSetDevice(h->device);
    if (!h->spec_arena || h->spec_key != key) {
        fac_handle tmp;
        tmp.device = h->device;
        std::vector<fac_handle::SpecScale> scales(n_scales);
        try {
            for (int i = 0; i < n_scales; ++i) {
                fac_handle::SpecScale& L = scales[i];
                L.w = window_lengths[i]; L.nb = L.w / 2 + 1; L.ld = (2 * L.nb + 127) / 128 * 128;
                const int nm = (int)key[2 + 4 * i + 1];
                L.mel = nm > 0; L.n_out = L.mel ? nm : L.nb;
                ConvW& d = L.dft;
                d = ConvW();
                d.Cin = L.w; d.Cout = L.ld; d.K = 1; d.ldw = L.ld;
                d.w = pack_alloc(&tmp, (size_t)L.w * L.ld);
                d.b = pack_alloc(&tmp, L.ld);
                for (int n = 0; n < L.w; ++n) {
                    const double wv = 0.5 - 0.5 * std::cos(2.0 * M_PI * (double)n / (double)L.w);      // periodic Hann
                    for (int k = 0; k < L.nb; ++k) {
                        const long long ph = ((long long)k * n) % L.w;
                        const double ang = 2.0 * M_PI * (double)ph / (double)L.w;
                        tmp.pack[d.w + (size_t)n * L.ld + 2 * k] = (float)(wv * std::cos(ang));
                        tmp.pack[d.w + (size_t)n * L.ld + 2 * k + 1] = (float)(-wv * std::sin(ang));
                    }
                }
                attach_tc(&tmp, d, 1, true);
                if (L.mel) {
                    std::vector<float> fb;
                    slaney_mel_fb((double)sample_rate, L.w, nm, key[2 + 4 * i + 2], key[2 + 4 * i + 3], fb);
                    L.fb = pack_alloc(&tmp, fb.size());
                    for (size_t j = 0; j < fb.size(); ++j) tmp.pack[L.fb + j] = fb[j];
                }
            }
        } catch (const PackError& e) { h->err = e.msg; return FAC_ERR_STATE; }
        if (h->spec_arena) { cudaDeviceSynchronize(); cudaFree(h->spec_arena); h->spec_arena = nullptr; }
        cudaError_t e = cudaMalloc(&h->spec_arena, (tmp.pack.size() + 64) * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpy(h->spec_arena, tmp.pack.data(), tmp.pack.size() * sizeof(float), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); h->spec_arena = nullptr; return FAC_ERR_CUDA; }
        h->spec_scales = scales;
        h->spec_key = key;
    }
    float* saved = h->warena;
    h->warena = h->spec_arena;
    int rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        double* sums = c.alloc<double>(2 * 16 + 2);
        const size_t mark = c.off;
        size_t peak = c.off;
        c.vq_critical = true;                                        // fp32-faithful DFT (promoted tensor-core class)
        for (int i = 0; i < n_scales; ++i) {
            c.off = mark;
            const fac_handle::SpecScale& L = c.h->spec_scales[i];
            const int hop = L.w / 4, F = T / hop + 1;
            const size_t rows = (size_t)2 * B * F;
            float* frames = c.alloc<float>(rows * L.w);
            float* spec = c.alloc<float>(rows * L.ld);
            float* tr = c.alloc<float>((size_t)B * F * 2);
            if (!c.dry) {
                c.check(launch_stft_frames(x, frames, B, T, F, hop, L.w, L.w / 2, c.st), "spec.frames");
                c.check(launch_stft_frames(y, frames + (size_t)B * F * L.w, B, T, F, hop, L.w, L.w / 2, c.st), "spec.frames");
            }
            run_conv(c, L.dft, frames, spec, 1, (int)rows, (int)rows, ConvOpts(), "spec.dft");
            if (!c.dry) {
                const double inv = 1.0 / ((double)B * F * L.n_out);
                c.check(launch_spec_loss_terms(spec, L.ld, L.nb, L.mel ? c.W(L.fb) : nullptr, L.n_out, B, F, clamp_eps, pw, tr, c.st), "spec.terms");
                c.check(launch_strided_sum(tr, (long long)B * F, 2, inv, sums + 2 * i, c.st), "spec.mag");
                c.check(launch_strided_sum(tr + 1, (long long)B * F, 2, inv, sums + 2 * i + 1, c.st), "spec.log");
            }
            if (c.off > peak) peak = c.off;
        }
        c.vq_critical = false;
        c.off = peak;
        if (!c.dry) c.check(launch_spec_loss_combine(sums, n_scales, mag_weight, log_weight, loss, c.st), "spec.combine");
    });
    h->warena = saved;
    return rc;
}

// dac/nn/loss.py:11-47 L1Loss on the waveforms: mean |x - y| over n floats
int fac_l1_loss(fac_handle* h, const float* x, const float* y, long long n, float* loss, void* stream) {
    if (!h || !x || !y || !loss || n <= 0) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        double* sum = c.alloc<double>(2);
        const int nblk = 1024;
        float* part = c.alloc<float>(nblk);
        if (!c.dry) {
            c.check(launch_absdiff_partial(x, y, n, part, nblk, c.st), "l1.partial");
            c.check(launch_strided_sum(part, nblk, 1, 1.0 / (double)n, sum, c.st), "l1.sum");
            c.check(launch_spec_loss_combine(sum, 0, 0.f, 0.f, loss, c.st), "l1.out");
        }
    });
}

// ---- predictor heads (SURVEY.md 8f rank 1; training-side in the reference, forward only here) ----
int fac_head_begin(fac_handle* h) {
    if (!h) return FAC_ERR_INVALID;
    h->heads.push_back(new fac_handle::HeadSet());
    return (int)h->heads.size() - 1;
}

int fac_head_tensor(fac_handle* h, int head_id, const char* key, const float* data_host, const int64_t* shape, int ndim) {
    if (!h || head_id < 0 || head_id >= (int)h->heads.size() || !key || !data_host || ndim < 0 || ndim > 4) return FAC_ERR_INVALID;
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; ++i) { if (shape[i] < 0) return FAC_ERR_INVALID; t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.data.assign(data_host, data_host + n);
    h->heads[head_id]->staged[key] = std::move(t);
    h->heads[head_id]->ready = false;
    return FAC_OK;
}

int fac_head_finalize(fac_handle* h, int head_id, int indim, int outdim, int nheads, int global_pred) {
    if (!h || head_id < 0 || head_id >= (int)h->heads.size() || indim <= 0 || outdim <= 0 || nheads < 1 || nheads > 8) return FAC_ERR_INVALID;
    if (indim % 16 != 0) { h->err = "fac_head_finalize: indim must be a multiple of 16"; return FAC_ERR_UNSUPPORTED; }
    fac_handle::HeadSet& hs = *h->heads[head_id];
    fac_handle tmp;                          // staging handle: reuses pack_conv / folded_weight on hs.staged
    tmp.device = h->device;
    tmp.host[0] = hs.staged;
    hs.indim = indim; hs.outdim = outdim; hs.nheads = nheads; hs.global_pred = global_pred;
    try {
        if (global_pred == 2) {
            // kind "linear": a plain nn.Linear(indim, outdim) staged as linear.weight [outdim][indim] / linear.bias
            // (FApredictors.timbre_predictor under timbre_norm, modules/quantize.py:470-473)
            if (nheads != 1) throw PackError{"a linear head has exactly one output"};
            hs.lin[0] = pack_conv(&tmp, 0, "linear");
            if (hs.lin[0].Cin != indim || hs.lin[0].Cout != outdim) throw PackError{"Linear geometry"};
        } else {
        auto expv = [&](const std::string& key) {
            const HostTensor& t = need(&tmp, 0, key);
            if ((int)t.numel() != indim) throw PackError{"shape of " + key};
            size_t off = pack_alloc(&tmp, indim);
            for (int i = 0; i < indim; ++i) tmp.pack[off + i] = expf(t.data[i]);     // alpha_logscale=True: exp() of the parameter
            return off;
        };
        const int dils[3] = {1, 2, 3};
        for (int j = 0; j < 3; ++j) {
            const std::string p = "model." + std::to_string(j);
            auto& u = hs.unit[j];
            u.dil = dils[j];
            u.a1 = expv(p + ".block.0.act.alpha"); u.b1 = expv(p + ".block.0.act.beta");
            u.c7 = pack_conv(&tmp, 0, p + ".block.1");
            u.a2 = expv(p + ".block.2.act.alpha"); u.b2 = expv(p + ".block.2.act.beta");
            u.c1 = pack_conv(&tmp, 0, p + ".block.3");
            if (u.c7.Cin != indim || u.c7.Cout != indim || u.c7.K != 7 || u.c1.K != 1) throw PackError{"head ResidualUnit geometry"};
        }
        hs.af = expv("model.3.act.alpha"); hs.bf = expv("model.3.act.beta");
        for (int i = 0; i < nheads; ++i) {
            hs.lin[i] = pack_conv(&tmp, 0, "heads." + std::to_string(i));
            if (hs.lin[i].Cin != indim || hs.lin[i].Cout != outdim) throw PackError{"head Linear geometry"};
        }
        }
    } catch (const PackError& e) {
        h->err = e.msg;
        return FAC_ERR_STATE;
    }
    cudaSetDevice(h->device);
    if (hs.arena) { cudaDeviceSynchronize(); cudaFree(hs.arena); hs.arena = nullptr; }
    cudaError_t e = cudaMalloc(&hs.arena, (tmp.pack.size() + 64) * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(hs.arena, tmp.pack.data(), tmp.pack.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    hs.staged.clear();
    hs.ready = true;
    return FAC_OK;
}

static int ensure_aa_filter(fac_handle* h);

int fac_head_forward(fac_handle* h, int head_id, const float* x, int B, int T, float* const* outs, void* stream) {
    if (!h || head_id < 0 || head_id >= (int)h->heads.size() || !x || !outs || B <= 0 || T <= 0) return FAC_ERR_INVALID;
    fac_handle::HeadSet& hs = *h->heads[head_id];
    if (!hs.ready) { h->err = "fac_head_forward: head not finalized"; return FAC_ERR_STATE; }
    int rc = ensure_aa_filter(h);
    if (rc) return rc;
    // the conv launch helpers read weights through h->warena: point it at this head's arena for the duration of the call
    float* saved = h->warena;
    h->warena = hs.arena;
    const int C = hs.indim;
    if (hs.global_pred == 2) {
        // kind "linear": x [B*T rows][indim] -> outs[0] [B*T][outdim]
        rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
            run_conv(c, hs.lin[0], x, outs[0], 1, B * T, B * T, ConvOpts(), "head.linear");
        });
        h->warena = saved;
        return rc;
    }
    rc = two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        const size_t n = (size_t)B * T * C;
        float* a_nct = c.alloc<float>(n);
        float* a_cl = c.alloc<float>(n);
        float* c7_cl = c.alloc<float>(n);
        float* c7_nct = c.alloc<float>(n);
        float* x_cl[2] = {c.alloc<float>(n), c.alloc<float>(n)};
        float* x_nct = c.alloc<float>(n);
        float* pooled = c.alloc<float>((size_t)B * C);
        auto act = [&](const float* src, float* dst, size_t al, size_t be, const char* nm) {
            if (!c.dry) c.check(launch_alias_free_act(src, dst, B, C, T, h->aa_filter, c.W(al), c.W(be), c.st), nm);
        };
        auto tr = [&](const float* src, float* dst, int R, int Cc, const char* nm) {     // [B][R][Cc] -> [B][Cc][R]
            if (!c.dry) c.check(launch_transpose(src, dst, B, R, Cc, c.st), nm);
        };
        tr(x, x_cl[0], C, T, "head.x_T");                                              // NCT -> channels-last
        const float* cur_nct = x;
        int cur = 0;
        for (int j = 0; j < 3; ++j) {
            const auto& u = hs.unit[j];
            act(cur_nct, a_nct, u.a1, u.b1, "head.act1");
            tr(a_nct, a_cl, C, T, "head.a_T");
            ConvOpts o7;
            o7.dil = u.dil; o7.pad_left = 3 * u.dil; o7.pad_right = 3 * u.dil; o7.reflect = 0;     // padding = ((7-1)*d)//2, zeros
            run_conv(c, u.c7, a_cl, c7_cl, B, T, T, o7, "head.conv7");
            tr(c7_cl, c7_nct, T, C, "head.c7_T");
            act(c7_nct, a_nct, u.a2, u.b2, "head.act2");
            tr(a_nct, a_cl, C, T, "head.b_T");
            ConvOpts o1;
            o1.res = x_cl[cur];
            run_conv(c, u.c1, a_cl, x_cl[cur ^ 1], B, T, T, o1, "head.conv1");
            cur ^= 1;
            tr(x_cl[cur], x_nct, T, C, "head.y_T");
            cur_nct = x_nct;
        }
        act(cur_nct, a_nct, hs.af, hs.bf, "head.act_final");
        tr(a_nct, a_cl, C, T, "head.f_T");                                             // Rearrange("b c t -> b t c")
        for (int i = 0; i < hs.nheads; ++i) {
            if (hs.global_pred) {
                if (!c.dry) c.check(launch_mean_pool(a_cl, pooled, B, T, C, nullptr, c.st), "head.mean");
                run_conv(c, hs.lin[i], pooled, outs[i], 1, B, B, ConvOpts(), "head.linear");
            } else {
                run_conv(c, hs.lin[i], a_cl, outs[i], 1, B * T, B * T, ConvOpts(), "head.linear");
            }
        }
    });
    h->warena = saved;
    return rc;
}

// out = a + b (+ c): the latent sums FApredictors.forward_v2 feeds its reversal heads (modules/quantize.py:571-586), in the
// reference's left-to-right order
int fac_add3(fac_handle* h, const float* a, const float* b, const float* c3, long long n, float* out, void* stream) {
    if (!h || !a || !b || !out || n <= 0) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaError_t e = launch_add3(a, b, c3, n, out, (cudaStream_t)stream);
    if (e != cudaSuccess) { h->err = std::string("CUDA error at add3: ") + cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_rvq_create(fac_handle* h, int nq, const float* const* in_w, const float* const* in_b, const float* const* out_w,
                   const float* const* out_b, const float* const* codebook) {
    if (!h || nq < 1 || nq > 8) return FAC_ERR_INVALID;
    std::vector<float> pack;
    RvqSet s;
    s.nq = nq;
    for (int q = 0; q < nq; ++q) s.vq[q] = pack_vq_raw(pack, in_w[q], in_b[q], out_w[q], out_b[q], codebook[q]);
    cudaSetDevice(h->device);
    float* dev = nullptr;
    cudaError_t e = cudaMalloc(&dev, (pack.size() + 64) * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(dev, pack.data(), pack.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    h->rvqs.push_back(s);
    h->rvq_arenas.push_back(dev);
    return (int)h->rvqs.size() - 1;
}

// Frees the device arena of one fac_rvq_create set (ids of other sets stay valid; the id is not reused).
int fac_rvq_destroy(fac_handle* h, int rvq_id) {
    if (!h || rvq_id < 0 || rvq_id >= (int)h->rvqs.size()) return FAC_ERR_INVALID;
    if (h->rvq_arenas[rvq_id]) {
        cudaSetDevice(h->device);
        cudaDeviceSynchronize();
        cudaFree(h->rvq_arenas[rvq_id]);
        h->rvq_arenas[rvq_id] = nullptr;
        h->rvqs[rvq_id].nq = 0;
    }
    return FAC_OK;
}

int fac_rvq_forward(fac_handle* h, int rvq_id, const float* x, int B, int T, int x_channels_last, float* quantized_out,
                    int64_t* indices, float* all_quantized, void* stream) {
    if (!h || rvq_id < 0 || rvq_id >= (int)h->rvqs.size() || !x || !quantized_out || !indices || B <= 0 || T <= 0) return FAC_ERR_INVALID;
    const RvqSet& s = h->rvqs[rvq_id];
    const float* base = h->rvq_arenas[rvq_id];
    if (!base || s.nq < 1) { h->err = "fac_rvq_forward: set was destroyed"; return FAC_ERR_STATE; }
    return two_pass(h, (cudaStream_t)stream, [&](Ctx& c) {
        size_t n = (size_t)B * T * 1024;
        float* xcl = x_channels_last ? nullptr : c.alloc<float>(n);
        float* qcl = x_channels_last ? nullptr : c.alloc<float>(n);
        float* acl = (x_channels_last || !all_quantized) ? nullptr : c.alloc<float>(n * s.nq);
        if (c.dry) return;
        RvqParams p;
        if (!x_channels_last) c.check(launch_transpose(x, xcl, B, 1024, T, c.st), "rvq.xT");
        p.x = x_channels_last ? x : xcl;
        p.qout = x_channels_last ? quantized_out : qcl;
        p.allq = all_quantized ? (x_channels_last ? all_quantized : acl) : nullptr;
        p.idx = indices;
        p.nq = s.nq; p.B = B; p.T = T;
        for (int q = 0; q < s.nq; ++q) {
            const VqW& v = s.vq[q];
            p.vq[q] = VqWeights{base + v.w_in, base + v.b_in, base + v.cb, base + v.cbn, base + v.cbn2, base + v.w_out, base + v.b_out};
        }
        c.check(launch_rvq(p, c.st), "rvq");
        if (!x_channels_last) {
            c.check(launch_transpose(qcl, quantized_out, B, T, 1024, c.st), "rvq.qT");
            if (all_quantized) c.check(launch_transpose(acl, all_quantized, B * s.nq, T, 1024, c.st), "rvq.aT");
        }
    });
}

static int ensure_aa_filter(fac_handle* h) {
    cudaSetDevice(h->device);
    if (!h->aa_filter) {
        // kaiser_sinc_filter1d(cutoff=0.25, half_width=0.3, kernel_size=12), alias_free_torch/filter.py:27-58
        const int ks = 12, half = 6;
        const double cutoff = 0.25, half_width = 0.3;
        double delta_f = 4 * half_width;
        double A = 2.285 * (half - 1) * M_PI * delta_f + 7.95;
        double beta_k = A > 50.0 ? 0.1102 * (A - 8.7) : (A >= 21.0 ? 0.5842 * std::pow(A - 21, 0.4) + 0.07886 * (A - 21.0) : 0.0);
        auto i0 = [](double v) { double s = 1, t = 1; for (int k = 1; k < 60; ++k) { t *= (v / (2 * k)) * (v / (2 * k)); s += t; } return s; };
        float f[12];
        double sum = 0;
        double tmp[12];
        for (int i = 0; i < ks; ++i) {
            double r = 2.0 * i / (ks - 1) - 1.0;                       // torch.kaiser_window(periodic=False)
            double w = i0(beta_k * std::sqrt(std::max(0.0, 1 - r * r))) / i0(beta_k);
            double tm = (i - half) + 0.5;
            double xx = 2 * cutoff * tm;
            double sinc = xx == 0 ? 1.0 : std::sin(M_PI * xx) / (M_PI * xx);
            tmp[i] = 2 * cutoff * w * sinc;
            sum += tmp[i];
        }
        for (int i = 0; i < ks; ++i) f[i] = (float)(tmp[i] / sum);
        cudaError_t e = cudaMalloc(&h->aa_filter, sizeof(f));
        if (e == cudaSuccess) e = cudaMemcpy(h->aa_filter, f, sizeof(f), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    }
    return FAC_OK;
}

int fac_alias_free_act(fac_handle* h, const float* x, int B, int C, int T, int act, const float* alpha,
                       const float* beta, float* y, void* stream) {
    if (!h || !x || !y || B <= 0 || C <= 0 || T <= 0 || (act == 1 && (!alpha || !beta))) return FAC_ERR_INVALID;
    int rc0 = ensure_aa_filter(h);
    if (rc0) return rc0;
    cudaError_t e = launch_alias_free_act(x, y, B, C, T, h->aa_filter, act == 1 ? alpha : nullptr, act == 1 ? beta : nullptr,
                                          (cudaStream_t)stream);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_conv(fac_handle* h, const float* x, const float* w_host, const float* bias_host, int B, int Tin, int Cin,
                   int Cout, int K, int dil, int stride, int pad_left, int pad_right, int reflect,
                   const float* in_alpha_host, const float* out_alpha_host, int act, const float* res, float* y,
                   int Tout, void* stream) {
    if (!h || !x || !w_host || !y) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    int ldw = (Cout + 3) / 4 * 4;
    std::vector<float> pk((size_t)K * Cin * ldw + Cout + 2 * Cin + 2 * Cout + 96, 0.f);
    for (int co = 0; co < Cout; ++co)
        for (int ci = 0; ci < Cin; ++ci)
            for (int k = 0; k < K; ++k) pk[((size_t)k * Cin + ci) * ldw + co] = w_host[((size_t)co * Cin + ci) * K + k];
    auto al4 = [](size_t v) { return (v + 3) / 4 * 4; };
    size_t o_b = (size_t)K * Cin * ldw, o_ia = al4(o_b + Cout), o_iia = al4(o_ia + Cin), o_oa = al4(o_iia + Cin), o_oia = al4(o_oa + Cout);
    for (int i = 0; i < Cout; ++i) pk[o_b + i] = bias_host ? bias_host[i] : 0.f;
    for (int i = 0; i < Cin; ++i) { pk[o_ia + i] = in_alpha_host ? in_alpha_host[i] : 1.f; pk[o_iia + i] = 1.0f / (pk[o_ia + i] + 1e-9f); }
    for (int i = 0; i < Cout; ++i) { pk[o_oa + i] = out_alpha_host ? out_alpha_host[i] : 1.f; pk[o_oia + i] = 1.0f / (pk[o_oa + i] + 1e-9f); }
    float* d = nullptr;
    cudaError_t e = cudaMalloc(&d, pk.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(d, pk.data(), pk.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    ConvParams p;
    p.x = x; p.y = y; p.w = d; p.bias = bias_host ? d + o_b : nullptr;
    if (in_alpha_host) { p.in_alpha = d + o_ia; p.in_inv_alpha = d + o_iia; }
    p.out_act = act;
    if (out_alpha_host) { p.out_act = ACT_SNAKE; p.out_alpha = d + o_oa; p.out_inv_alpha = d + o_oia; }
    p.res = res;
    p.B = B; p.Tin = Tin; p.Cin = Cin; p.Tout = Tout; p.Cout = Cout; p.K = K; p.dil = dil; p.stride = stride;
    p.pad_left = pad_left; p.pad_right = pad_right; p.pad_reflect = reflect;
    p.ldw = ldw; p.ldy = Cout; p.ldx = Cin;
    p.x_bstride = (size_t)Tin * Cin; p.y_bstride = (size_t)Tout * Cout;
    e = launch_conv(p, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) { h->err = std::string("fac_debug_conv: ") + cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_slstm(fac_handle* h, const float* x, const float* const* w_host, int B, int T, int H, float* y, void* stream) {
    if (!h || !x || !w_host || !y || B <= 0 || T <= 0) return FAC_ERR_INVALID;
    // build a private handle holding only this LSTM, reuse the packing + slstm code path
    fac_handle tmp;
    tmp.device = h->device;
    const char* names[8] = {"weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0", "weight_ih_l1", "weight_hh_l1", "bias_ih_l1", "bias_hh_l1"};
    for (int i = 0; i < 8; ++i) {
        HostTensor t;
        bool mat = (i % 4) < 2;
        if (mat) t.shape = {4 * H, H}; else t.shape = {4 * H};
        t.data.assign(w_host[i], w_host[i] + t.numel());
        tmp.host[0][std::string("l.") + names[i]] = std::move(t);
    }
    tmp.dec_bf16 = h->dec_bf16;     // decoder-class precision (bf16 hi/lo) unless the caller switched it off
    tmp.lstm_v2 = h->lstm_v2; tmp.dec_lstm_fp16 = h->dec_lstm_fp16;
    LstmW L;
    try { L = pack_lstm(&tmp, 0, "l"); } catch (const PackError& e) { h->err = e.msg; return FAC_ERR_UNSUPPORTED; }
    cudaSetDevice(h->device);
    cudaError_t e = cudaMalloc(&tmp.warena, (tmp.pack.size() + 64) * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(tmp.warena, tmp.pack.data(), tmp.pack.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    Ctx dry{&tmp, st, true};
    slstm(dry, L, x, y, B, T);
    int rc = ensure_ws(&tmp, dry.off);
    if (rc == FAC_OK) {
        Ctx c{&tmp, st, false};
        slstm(c, L, x, y, B, T);
        rc = finish(&tmp, c);
        cudaStreamSynchronize(st);
    }
    if (rc != FAC_OK) h->err = tmp.err;
    cudaFree(tmp.warena);
    if (tmp.ws) cudaFree(tmp.ws);
    return rc;
}

int fac_set_option(fac_handle* h, const char* name, int value) {
    if (!h || !name) return FAC_ERR_INVALID;
    if (std::string(name) == "fuse_resunit") { h->fuse_res = value < 0 ? 0 : (value > 2 ? 2 : value); return FAC_OK; }
    if (std::string(name) == "tc_dbg") { g_tc_dbg = value; return FAC_OK; }
    if (std::string(name) == "tc_slot_issue") { g_tc_slot_issue = value != 0; return FAC_OK; }
    if (std::string(name) == "tt_pair") { g_tt_pair_ok = value != 0; return FAC_OK; }
    if (std::string(name) == "tc_groups") { g_tc_groups_ok = value != 0; return FAC_OK; }
    if (std::string(name) == "tc_wide") { g_tc_wide_ok = value != 0; return FAC_OK; }
    if (std::string(name) == "tc_occ2_maxn") { h->tc_occ2 = value < 0 ? 0 : value; return FAC_OK; }
    if (std::string(name) == "encoder_f16x2") { h->enc_f16 = value != 0; return FAC_OK; }
    if (std::string(name) == "decoder_conv7_fp16") { h->dec_c7_f16 = value != 0; return FAC_OK; }
    if (std::string(name) == "encoder_tt") { h->enc_tt = value != 0; return FAC_OK; }
    if (std::string(name) == "encoder_snake_mufu") { h->enc_mufu = value != 0; return FAC_OK; }
    if (std::string(name) == "overlap_front") { h->overlap_front = value != 0; return FAC_OK; }
    if (std::string(name) == "lstm_v2") { h->lstm_v2 = value != 0; return FAC_OK; }
    if (std::string(name) == "decoder_lstm_fp16") { h->dec_lstm_fp16 = value != 0; return FAC_OK; }
    if (std::string(name) == "tt_probe") { g_tt_probe_on = value != 0; return FAC_OK; }
    if (std::string(name) == "attention_stream") { h->attn_stream = value != 0; return FAC_OK; }
    if (std::string(name) == "decoder_bf16") { h->dec_bf16 = value != 0; return FAC_OK; }
    if (std::string(name) == "tensor_cores") { h->use_tc = value < 0 ? 0 : (value > 2 ? 2 : value); return FAC_OK; }
    h->err = std::string("unknown option ") + name;
    return FAC_ERR_INVALID;
}

int fac_debug_conv_tc(fac_handle* h, const float* x, const float* w_host, const float* bias_host, int B, int Tin, int Cin,
                      int Cout, int K, int dil, int stride, int pad_left, int pad_right, int reflect,
                      const float* in_alpha_host, const float* out_alpha_host, int act, const float* res, float* y,
                      int Tout, int promoted, void* stream) {
    if (!h || !x || !w_host || !y) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    TcConvParams tp;
    tp.Cin = Cin; tp.Cout = Cout; tp.promoted = (promoted == 1 || promoted == 3) ? 1 : 0; tp.bf16 = (promoted == 2 || promoted == 5) ? 1 : 0;
    tp.f16x2 = promoted == 3 ? 1 : 0;
    tp.g1f16 = promoted == 5 ? 1 : 0;      // 5 = the one-pass fp16 class of conv_tc_kernel
    const bool use_tt = promoted == 4;
    tp.occ2_maxn = h->tc_occ2;
    tp.Tout = Tout;
    if (stride == 1) { tp.vf = 1; tp.Kr = K; tp.dil = dil; }
    else if (K == 2 * stride && dil == 1) { tp.vf = stride; tp.Kr = 2; tp.dil = 1; }
    else { h->err = "fac_debug_conv_tc: unsupported stride/kernel"; return FAC_ERR_UNSUPPORTED; }
    if (!(use_tt ? tt_conv_plan(tp) : tc_conv_plan(tp))) { h->err = "fac_debug_conv_tc: layer not eligible for the tensor-core path"; return FAC_ERR_UNSUPPORTED; }
    int ldw = (Cout + 3) / 4 * 4;
    std::vector<float> gen((size_t)K * Cin * ldw, 0.f);
    for (int co = 0; co < Cout; ++co)
        for (int ci = 0; ci < Cin; ++ci)
            for (int k = 0; k < K; ++k) gen[((size_t)k * Cin + ci) * ldw + co] = w_host[((size_t)co * Cin + ci) * K + k];
    size_t nb = use_tt ? tt_blob_floats(tp) : tc_blob_floats(tp);
    auto al4 = [](size_t v) { return (v + 3) / 4 * 4; };
    size_t o_b = al4(nb), o_ia = al4(o_b + Cout), o_iia = al4(o_ia + Cin), o_oa = al4(o_iia + Cin), o_oia = al4(o_oa + Cout);
    std::vector<float> pk(o_oia + Cout + 16, 0.f);
    if (use_tt) tt_pack_blob(tp, gen.data(), ldw, pk.data());
    else tc_pack_blob(tp, gen.data(), ldw, pk.data());
    for (int i = 0; i < Cout; ++i) pk[o_b + i] = bias_host ? bias_host[i] : 0.f;
    for (int i = 0; i < Cin; ++i) { pk[o_ia + i] = in_alpha_host ? in_alpha_host[i] : 1.f; pk[o_iia + i] = 1.0f / (pk[o_ia + i] + 1e-9f); }
    for (int i = 0; i < Cout; ++i) { pk[o_oa + i] = out_alpha_host ? out_alpha_host[i] : 1.f; pk[o_oia + i] = 1.0f / (pk[o_oa + i] + 1e-9f); }
    float* d = nullptr;
    cudaError_t e = cudaMalloc(&d, pk.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(d, pk.data(), pk.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    tp.x = x; tp.y = y; tp.wblob = d; tp.bias = d + o_b;
    if (in_alpha_host) { tp.in_alpha = d + o_ia; tp.in_inv_alpha = d + o_iia; }
    tp.out_act = act;
    if (out_alpha_host) { tp.out_act = ACT_SNAKE; tp.out_alpha = d + o_oa; tp.out_inv_alpha = d + o_oia; }
    tp.res = res;
    tp.B = B; tp.Tin = Tin; tp.ldx = Cin;
    tp.PLr = pad_left / tp.vf;
    tp.pad_left_s = pad_left; tp.pad_right_s = pad_right; tp.reflect = reflect;
    tp.Tout = Tout; tp.ldy = Cout;
    tp.x_bstride = (size_t)Tin * Cin; tp.y_bstride = (size_t)Tout * Cout;
    e = use_tt ? launch_conv_tt(tp, st) : launch_conv_tc(tp, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) { h->err = std::string("fac_debug_conv_tc: ") + cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_resunit(fac_handle* h, const float* x, const float* w7_host, const float* b7_host, const float* w1_host,
                      const float* b1_host, const float* alpha1_host, const float* alpha2_host, int B, int T, int C,
                      int dil, int mode, float* y, void* stream) {
    if (!h || !x || !y || !w7_host || !w1_host) return FAC_ERR_INVALID;
    fac_handle tmp;
    tmp.device = h->device;
    tmp.use_tc = mode == 0 ? 0 : 1;          // 0: fp32 FMA, 1: two tcgen05 launches, 2: fused launch; 3/4 = 1/2 with bf16 split;
                                             // 5/6 = 3/4 with the k = 7 conv in one fp16 pass
    tmp.fuse_res = (mode == 2 || mode == 4 || mode == 6) ? 1 : 0;
    tmp.dec_bf16 = mode >= 3;
    tmp.dec_c7_f16 = mode >= 5;
    tmp.tc_occ2 = h->tc_occ2;
    auto put = [&](const char* key, const float* d, std::vector<int64_t> shp) {
        HostTensor t;
        t.shape = shp;
        t.data.assign(d, d + t.numel());
        tmp.host[0][key] = std::move(t);
    };
    put("u.block.0.alpha", alpha1_host, {1, C, 1});
    put("u.block.1.conv.conv.weight", w7_host, {C, C, 7});
    put("u.block.1.conv.conv.bias", b7_host, {C});
    put("u.block.2.alpha", alpha2_host, {1, C, 1});
    put("u.block.3.conv.conv.weight", w1_host, {C, C, 1});
    put("u.block.3.conv.conv.bias", b1_host, {C});
    ResW r;
    try { r = pack_res(&tmp, 0, "u", dil, false); } catch (const PackError& e) { h->err = e.msg; return FAC_ERR_STATE; }
    cudaSetDevice(h->device);
    cudaError_t e = cudaMalloc(&tmp.warena, (tmp.pack.size() + 64) * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(tmp.warena, tmp.pack.data(), tmp.pack.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); cudaGetLastError(); return FAC_ERR_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    float* scratch = nullptr;
    e = cudaMalloc(&scratch, sizeof(float) * (size_t)B * T * C);
    int rc = FAC_OK;
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); rc = FAC_ERR_CUDA; }
    if (rc == FAC_OK) {
        Ctx c{&tmp, st, false};
        residual_unit(c, r, x, scratch, y, B, T);
        rc = finish(&tmp, c);
        cudaError_t e2 = cudaStreamSynchronize(st);
        if (rc == FAC_OK && e2 != cudaSuccess) { tmp.err = cudaGetErrorString(e2); rc = FAC_ERR_CUDA; }
        if (rc == FAC_OK && (mode == 2 || mode == 4 || mode == 6) && tmp.launches != 1) { tmp.err = "fused path not taken for this geometry"; rc = FAC_ERR_UNSUPPORTED; }
    }
    if (rc != FAC_OK) h->err = tmp.err;
    if (scratch) cudaFree(scratch);
    cudaFree(tmp.warena);
    return rc;
}

// Host-only: the recurrent-weight packing of lstm_rec_kernel for one nn.LSTM weight_hh [4H][H]:
// bf16 = 0 -> fp32 [G][H][4U] (row r = gate*U + u of CTA g); bf16 = 1 -> [G][H/16][hi|lo][8 k-pairs][4U] 32-bit words.
// Returns the number of 32-bit words (G*H*4U); info3 = {U, G, 4U}.
long long fac_debug_lstm_pack(const float* whh_host, int H, int bf16, float* out, long long capacity_floats, int* info3) {
    if (!whh_host || H <= 0) return FAC_ERR_INVALID;
    fac_handle tmp;
    const char* names[8] = {"weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0", "weight_ih_l1", "weight_hh_l1", "bias_ih_l1", "bias_hh_l1"};
    for (int i = 0; i < 8; ++i) {
        HostTensor t;
        const bool mat = (i % 4) < 2;
        if (mat) t.shape = {4 * H, H}; else t.shape = {4 * H};
        if (i == 1) t.data.assign(whh_host, whh_host + (size_t)4 * H * H);
        else t.data.assign(t.numel(), 0.f);
        tmp.host[0][std::string("l.") + names[i]] = std::move(t);
    }
    LstmW L;
    try { L = pack_lstm(&tmp, 0, "l"); } catch (const PackError&) { return FAC_ERR_UNSUPPORTED; }
    if (info3) { info3[0] = L.U; info3[1] = L.G; info3[2] = 4 * L.U; }
    if (bf16 == 2 || bf16 == 3) {
        // lstm2.cu layouts: 2 = one fp16 pass [G][H/16][8][4U] words, 3 = fp16 hi + scaled lo [G][H/16][hi|lo][8][4U]
        const int p3 = bf16 == 3;
        const long long n2 = (long long)lstm2_pack_words(H, L.U, p3);
        if (!out || capacity_floats < n2) return n2;
        lstm2_pack(whh_host, H, L.U, p3, reinterpret_cast<uint32_t*>(out));
        return n2;
    }
    const long long n = (long long)L.G * H * 4 * L.U;
    if (bf16 && !L.has16) return FAC_ERR_UNSUPPORTED;
    if (!out || capacity_floats < n) return n;
    memcpy(out, tmp.pack.data() + (bf16 ? L.whh16[0] : L.whh[0]), sizeof(float) * (size_t)n);
    return n;
}

// Host-only: the conv form of nn.ConvTranspose1d(k = 2s, stride s) weights [Cin][Cout][2s] (HOST, already weight-normed):
// causal != 0 -> 2 taps (x[t-1], x[t]); causal == 0 -> 3 taps (x[t-1], x[t], x[t+1]) (encodec.py:248-270 trims).  out is
// [taps][Cin][s*Cout] (phase-major output channels r*Cout + co); returns the number of floats.
long long fac_debug_convtr_pack(const float* w_host, int Cin, int Cout, int stride, int causal, float* out, long long capacity_floats) {
    if (!w_host || Cin <= 0 || Cout <= 0 || stride <= 0) return FAC_ERR_INVALID;
    fac_handle tmp;
    HostTensor t, b;
    t.shape = {Cin, Cout, 2 * stride};
    t.data.assign(w_host, w_host + (size_t)Cin * Cout * 2 * stride);
    b.shape = {Cout};
    b.data.assign(Cout, 0.f);
    tmp.host[0]["c.weight"] = std::move(t);
    tmp.host[0]["c.bias"] = std::move(b);
    ConvW c;
    try { c = causal ? pack_convtr(&tmp, 0, "c", stride) : pack_convtr_noncausal(&tmp, 0, "c", stride); }
    catch (const PackError&) { return FAC_ERR_UNSUPPORTED; }
    const long long n = (long long)c.K * Cin * c.Cout;
    if (!out || capacity_floats < n) return n;
    for (int k = 0; k < c.K; ++k)
        for (int ci = 0; ci < Cin; ++ci)
            for (int co = 0; co < c.Cout; ++co) out[((size_t)k * Cin + ci) * c.Cout + co] = tmp.pack[c.w + ((size_t)k * Cin + ci) * c.ldw + co];
    return n;
}

// Host-only: the padding index map every conv kernel uses (common.cuh PadMap): out[i] = source row of padded position
// i - pad_left, or -1 where the padded value is zero.
int fac_debug_pad_map(int L, int pad_left, int pad_right, int reflect, int* out, int n) {
    if (!out || L < 0 || pad_left < 0 || pad_right < 0 || n != pad_left + L + pad_right) return FAC_ERR_INVALID;
    const PadMap pm = PadMap::make(L, pad_left, pad_right, reflect);
    for (int i = 0; i < n; ++i) out[i] = pm.src(i - pad_left);
    return FAC_OK;
}

// Host-only: the tile plan the tcgen05 conv kernels would use for a layer geometry (no GPU, no handle).
int fac_debug_tc_plan(int Cin, int Cout, int K, int dil, int stride, int Tout, int mode, int occ2_maxn, int* out8) {
    if (!out8 || Cin <= 0 || Cout <= 0 || K <= 0 || dil <= 0 || stride <= 0 || mode < 0 || mode > 6) return FAC_ERR_INVALID;
    TcConvParams tp;
    tp.Cin = Cin; tp.Cout = Cout; tp.Tout = Tout; tp.occ2_maxn = occ2_maxn;
    tp.promoted = (mode == 1 || mode == 3) ? 1 : 0;
    tp.bf16 = (mode == 2 || mode == 4) ? 1 : 0;
    tp.f16x2 = mode == 3 ? 1 : 0;
    tp.fused = (mode == 4 || mode == 5) ? 1 : 0;
    if (stride == 1) { tp.vf = 1; tp.Kr = K; tp.dil = dil; }
    else if (K == 2 * stride && dil == 1) { tp.vf = stride; tp.Kr = 2; tp.dil = 1; }
    else return FAC_ERR_UNSUPPORTED;
    if (mode == 6) {
        tp.promoted = 0; tp.bf16 = 0; tp.f16x2 = 0; tp.fused = 0;
        if (!tt_conv_plan(tp)) return FAC_ERR_UNSUPPORTED;
        out8[0] = tp.N * (tp.pair ? 2 : 1);   // output channels per CTA tile: 128, or 256 in PAIR mode (two weight tiles)
        out8[1] = tp.NT; out8[2] = tp.nchunk; out8[3] = tp.stagesB; out8[4] = tp.tmem_cols;
        out8[5] = (int)tp.smem_bytes; out8[6] = tp.Rpad; out8[7] = tp.promote_every;
        return FAC_OK;
    }
    if (!tc_conv_plan(tp)) return FAC_ERR_UNSUPPORTED;
    out8[0] = tp.N; out8[1] = tp.MT; out8[2] = tp.nchunk; out8[3] = tp.stagesB; out8[4] = tp.tmem_cols;
    out8[5] = (int)tp.smem_bytes; out8[6] = tp.Rpad; out8[7] = tp.promote_every;
    return FAC_OK;
}

// Host-only: the tensor-core weight blob (tc_pack_blob) for nn.Conv1d weights [Cout][Cin][K]; returns the number of
// floats (32-bit words) of the blob, writes it when blob_out has room.
long long fac_debug_tc_pack(const float* w_host, int Cin, int Cout, int K, int stride, int mode, float* blob_out,
                            long long capacity_floats) {
    if (!w_host || Cin <= 0 || Cout <= 0 || K <= 0 || stride <= 0 || mode < 0 || mode > 4) return FAC_ERR_INVALID;
    TcConvParams tp;
    tp.Cin = Cin; tp.Cout = Cout; tp.dil = 1;
    tp.promoted = (mode == 1 || mode == 3) ? 1 : 0; tp.bf16 = mode == 2 ? 1 : 0; tp.f16x2 = mode == 3 ? 1 : 0;
    if (stride == 1) { tp.vf = 1; tp.Kr = K; }
    else if (K == 2 * stride) { tp.vf = stride; tp.Kr = 2; }
    else return FAC_ERR_UNSUPPORTED;
    const bool use_tt = mode == 4;
    if (use_tt) { tp.promoted = 0; tp.bf16 = 0; tp.f16x2 = 0; }
    if (!(use_tt ? tt_conv_plan(tp) : tc_conv_plan(tp))) return FAC_ERR_UNSUPPORTED;
    const long long n = (long long)(use_tt ? tt_blob_floats(tp) : tc_blob_floats(tp));
    if (!blob_out || capacity_floats < n) return n;
    const int ldw = (Cout + 3) / 4 * 4;
    std::vector<float> gen((size_t)K * Cin * ldw, 0.f);      // generic packed layout [K*Cin][ldw]
    for (int co = 0; co < Cout; ++co)
        for (int ci = 0; ci < Cin; ++ci)
            for (int k = 0; k < K; ++k) gen[((size_t)k * Cin + ci) * ldw + co] = w_host[((size_t)co * Cin + ci) * K + k];
    if (use_tt) tt_pack_blob(tp, gen.data(), ldw, blob_out);
    else tc_pack_blob(tp, gen.data(), ldw, blob_out);
    return n;
}

int fac_debug_tc_phase_clocks(fac_handle* h, long long* out8) {
    if (!h || !out8) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    cudaError_t e = g_tt_probe_on ? tt_read_probe(out8) : tc_read_phase_clocks(out8);

    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_tc_trace(fac_handle* h, long long* out80) {
    if (!h || !out80) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    cudaError_t e = tc_read_trace(out80);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_tc_producer_clocks(fac_handle* h, long long* out4) {
    if (!h || !out4) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    cudaError_t e = tc_read_producer_clocks(out4);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_lstm_phase_clocks(fac_handle* h, long long* out4) {
    if (!h || !out4) return FAC_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    cudaError_t e = h->lstm_v2 ? lstm2_read_phase_clocks(out4) : lstm_read_phase_clocks(out4);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return FAC_ERR_CUDA; }
    return FAC_OK;
}

int fac_debug_tap(fac_handle* h, const char* name, float* dst, size_t capacity_floats) {
    if (!h || !name) return FAC_ERR_INVALID;
    if (!dst) h->taps.erase(name);
    else h->taps[name] = std::make_pair(dst, capacity_floats);
    return FAC_OK;
}

int fac_profile_enable(fac_handle* h, int on) {
    if (!h) return FAC_ERR_INVALID;
    h->profiling = on != 0;
    return FAC_OK;
}

// Resolves pending event pairs (synchronises the device) and folds them into per-family totals.
static void profile_collect(fac_handle* h) {
    if (h->prof.empty()) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (auto& r : h->prof) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        auto& a = h->prof_agg[r.name];
        a.ms += ms; a.flops += r.flops; a.bytes += r.bytes; a.launches++;
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    h->prof.clear();
}

int fac_profile_reset(fac_handle* h) {
    if (!h) return FAC_ERR_INVALID;
    profile_collect(h);
    h->prof_agg.clear();
    return FAC_OK;
}

int fac_profile_get(fac_handle* h, const char* family, double* ms, double* flops, double* bytes, long long* launches) {
    if (!h || !family) return FAC_ERR_INVALID;
    profile_collect(h);
    std::string fam(family);
    fac_handle::ProfAgg t;
    for (auto& kv : h->prof_agg) {
        if (kv.first == fam || (kv.first.size() > fam.size() && kv.first.compare(0, fam.size(), fam) == 0 && kv.first[fam.size()] == ':')) {
            t.ms += kv.second.ms; t.flops += kv.second.flops; t.bytes += kv.second.bytes; t.launches += kv.second.launches;
        }
    }
    if (ms) *ms = t.ms;
    if (flops) *flops = t.flops;
    if (bytes) *bytes = t.bytes;
    if (launches) *launches = t.launches;
    return FAC_OK;
}

// Text dump "key\tms\tgflop\tgbytes\tlaunches\n" of every profiled call site; returns bytes needed.
size_t fac_profile_dump(fac_handle* h, char* buf, size_t cap) {
    if (!h) return 0;
    profile_collect(h);
    std::string out;
    char line[256];
    for (auto& kv : h->prof_agg) {
        snprintf(line, sizeof line, "%s\t%.4f\t%.3f\t%.4f\t%ld\n", kv.first.c_str(), kv.second.ms, kv.second.flops / 1e9,
                 kv.second.bytes / 1e9, kv.second.launches);
        out += line;
    }
    if (buf && cap > 0) {
        size_t n = out.size() < cap - 1 ? out.size() : cap - 1;
        memcpy(buf, out.data(), n);
        buf[n] = 0;
    }
    return out.size() + 1;
}

size_t fac_workspace_bytes(const fac_handle* h) { return h ? h->ws_bytes : 0; }
int fac_last_launch_count(const fac_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
