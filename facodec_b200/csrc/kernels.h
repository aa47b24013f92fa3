// Internal kernel launch interfaces (C++ only; the public C-ABI is include/facodec_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fac {

struct ConvParams {
    const float* x = nullptr;          // [B][Tin][Cin]
    const float* w = nullptr;          // [K*Cin][ldw]
    const float* bias = nullptr;       // [Cout] or null
    const float* in_alpha = nullptr;   // [Cin] snake on input, or null
    const float* in_inv_alpha = nullptr;
    const float* out_alpha = nullptr;  // [Cout] when out_act == ACT_SNAKE
    const float* out_inv_alpha = nullptr;
    const float* res = nullptr;        // residual, same layout as y, or null
    const int* valid_len = nullptr;    // [B] rows >= valid_len[b] are written as 0, or null
    float* y = nullptr;                // [B][Tout][ldy] (or [B][Cout][Tout] when y_transposed)
    int B = 0, Tin = 0, Cin = 0, Tout = 0, Cout = 0;
    int K = 1, dil = 1, stride = 1, pad_left = 0, pad_right = 0, pad_reflect = 0;
    int ldw = 0, ldy = 0, ldx = 0;   // ldx = input row stride (>= Cin)
    int out_act = 0;
    int y_transposed = 0;
    size_t x_bstride = 0, y_bstride = 0;
};
cudaError_t launch_conv(const ConvParams& p, cudaStream_t st);

// ---- tcgen05 tensor-core conv (conv_tc.cu) ---------------------------------------------------
struct TcConvParams {
    const float* x = nullptr;          // [B][Tin][ldx] channels-last samples
    const float* wblob = nullptr;      // [ntile][chunk][tap][hi|lo][4][N][4] (tc_pack_blob)
    const float* bias = nullptr;
    const float* in_alpha = nullptr;   // [Cin] Snake on the input or null
    const float* in_inv_alpha = nullptr;
    const float* out_alpha = nullptr;  // [Cout] when out_act == ACT_SNAKE
    const float* out_inv_alpha = nullptr;
    const float* res = nullptr;        // [B][Tout][ldy] or null
    float* y = nullptr;                // [B][Tout][ldy]
    int B = 0, Tin = 0, Cin = 0, ldx = 0;
    int vf = 1;                        // samples per A row (down-conv stride; 1 otherwise)
    int Kr = 1, dil = 1, PLr = 0;      // taps / dilation / left pad, in rows
    int pad_left_s = 0, pad_right_s = 0, reflect = 0;   // sample-level padding (PadMap)
    int Tout = 0, Cout = 0, ldy = 0;
    int out_act = 0;
    int promoted = 0;                  // 1 = conv_tcp_kernel (register-promoted accumulation)
    int bf16 = 0;                      // 1 = bf16 hi/lo split (kind::f16, K = 16) instead of tf32 hi/lo; decoder only
    int g1f16 = 0;                     // with bf16 = 1 (downstream only): the layer's own GEMM (the k-tap conv; GEMM 1 of a fused unit) takes
                                       // ONE fp16 pass (10-bit operands, fp32 accumulation) instead of the 3-pass bf16 hi/lo split
    int f16x2 = 0;                     // promoted only: fp16 hi + 2^11-scaled fp16 lo split (kind::f16, K = 16) instead of tf32 hi/lo
    int tt = 0;                        // 1 = conv_tt_kernel: transposed formulation (weights = MMA A operand, M = 128 output
                                       // channels; time = N = NT <= 256), fp16 hi + scaled-lo split, promoted (tt_conv_plan)
    int pair = 0;                      // tt (plan): 1 = PAIR mode, a CTA tile is two 128-channel weight tiles x NT <= 128 time steps
    int NT = 0;                        // tt: time steps per tile
    int snake_mufu = 0;                // tt, EXPERIMENT: Snake via the SFU sine (abs error ~4e-7 instead of 2.5e-7)
    int fused = 0;                     // 1 = whole ResidualUnit: conv7 -> +b7 -> Snake -> 1x1 conv -> +b1 -> +x
    const float* wblob2 = nullptr;     // 1x1 conv weight blob (same tile N), when fused
    const float* bias2 = nullptr;
    int nchunk2 = 0;
    int occ2_maxn = 0;                 // > 0: tiles with N <= occ2_maxn are planned for TWO resident CTAs per SM
                                       // (<= 256 TMEM columns, <= 112 KB smem each) so one CTA's MMAs overlap the other's
                                       // produce / epilogue phases
    // plan (tc_conv_plan)
    int promote_every = 1;
    int N = 0, MT = 0, nchunk = 0, Rpad = 0, stagesB = 0, tmem_cols = 0;
    int cps = 0;                       // conv_tc_kernel: > 0 = a weight-ring slot holds every tap of `cps` consecutive chunks (tpt = Kr * cps)
    int tpt = 1, tpt2 = 1;             // conv_tc_kernel: weight tiles ((chunk, tap) / GEMM-2 chunk) per bulk copy into one ring slot
    int b_slot = 0;                    // bytes of one weight-ring slot
    int R2pad = 0;                     // fused: row pitch (rows) of the resident GEMM-2 operand chunks
    int dbg = 0;                       // conv_tc_kernel timing experiments (g_tc_dbg); results are wrong when non-zero
    int ng = 1;                        // conv_tc_kernel: producer groups (2 = alternate chunks over a 4-deep operand ring)
    int wide = 0;                      // conv_tc_kernel: 1 = 16 worker warps (tile planned for one CTA per SM), 0 = 8
    size_t smem_bytes = 0;
    size_t x_bstride = 0, y_bstride = 0;
};
bool tc_conv_plan(TcConvParams& p);
size_t tc_blob_floats(const TcConvParams& p);
void tc_pack_blob(const TcConvParams& p, const float* wp, int ldw, float* blob);
cudaError_t launch_conv_tc(const TcConvParams& p, cudaStream_t st);
bool tt_conv_plan(TcConvParams& p);                 // conv_tt.cu
size_t tt_blob_floats(const TcConvParams& p);
void tt_pack_blob(const TcConvParams& p, const float* wp, int ldw, float* blob);
cudaError_t launch_conv_tt(const TcConvParams& p, cudaStream_t st);
extern int g_tc_dbg;
extern int g_tc_slot_issue;
extern int g_tc_groups_ok;
extern int g_tc_wide_ok;                             // conv_tc.cu: 0 = never plan 16-worker tiles (A/B aid)
extern int g_tt_pair_ok;                             // conv_tt.cu: 0 = never plan PAIR-mode tiles
extern int g_tt_probe_on;                            // 1 = launch the probing variant (process-wide test aid)
cudaError_t tt_read_probe(long long* out8);
cudaError_t tc_read_trace(long long* out80);          // per-chunk timeline of the probe CTA (conv_tc.cu g_tc_trace)
cudaError_t tc_read_producer_clocks(long long* out4); // probe producer thread of the last conv_tc_kernel
cudaError_t tc_read_phase_clocks(long long* out8);   // probe-CTA phase timestamps of the last conv_tc_kernel

// ---- LSTM recurrence (lstm.cu) -----------------------------------------------------------
// One nn.LSTM layer over all T steps for up to 32 sequences (dac/model/encodec.py:272-288).
struct LstmParams {
    const float* xg = nullptr;    // [B][T][4H] = x W_ih^T + b_ih + b_hh, gate order i,f,g,o
    const float* whh_p = nullptr; // packed per CTA: [G][H][4U]  (r = gate*U + u)
    const float* whh_p16 = nullptr; // bf16 split: [G][H/16][hi|lo][8 k-pairs][4U] 32-bit words (k even in the low half)
    int bf16 = 0;                 // 1 = bf16 hi/lo recurrence (downstream of the VQ only)
    // second-generation kernel (lstm2.cu): W_hh resident in shared memory as fp16 words, h exchanged pre-split
    const uint32_t* whh_p2 = nullptr;   // lstm2_pack layout
    uint32_t* h16 = nullptr;            // scratch [2 parities][planes][H/2][32] words
    int pass3 = 0;                      // 1 = fp16 hi + scaled-lo 3-pass (upstream of the VQ); 0 = one fp16 pass
    // streaming (lstm2 only): state carried between chunks, updated in place; null = zero initial state, nothing saved
    uint32_t* state_h = nullptr;        // [planes][H/2][32] words (h in the published fp16 layout)
    float* state_c = nullptr;           // [G][32][U] cell state
    const float* skip = nullptr;  // [B][T][H] added to the output (SLSTM skip) or null
    float* y = nullptr;           // [B][T][H]
    float* hT = nullptr;          // scratch [2][H][32]
    unsigned int* bar = nullptr;  // grid barrier counter (zeroed by the launcher)
    int B = 0, T = 0, H = 0, U = 0, G = 0;
};
cudaError_t launch_lstm_layer(const LstmParams& p, cudaStream_t st);
cudaError_t launch_lstm2_layer(const LstmParams& p, cudaStream_t st);   // lstm2.cu
size_t lstm2_pack_words(int H, int U, int pass3);
void lstm2_pack(const float* whh, int H, int U, int pass3, uint32_t* out);
size_t lstm2_smem_bytes(int H, int U, int pass3);
cudaError_t lstm2_read_phase_clocks(long long* out4);
int lstm_units_per_cta(int H);
cudaError_t lstm_read_phase_clocks(long long* out4);   // CTA-0 accumulated phase clocks of the last launch  // U such that H % U == 0 and H / U <= resident CTAs

// ---- mel front-end (frontend.cu) -----------------------------------------------------------
// spec [B][F][ldspec] (re at 2*bin, im at 2*bin+1) -> mel [B][Tm][80] = (log(1e-5 + |.|^2 fb)+4)/4
cudaError_t launch_stft_frames(const float* wave, float* frames /*[B][F][win]*/, int B, int T, int F, int hop, int win, int pad,
                               cudaStream_t st);
cudaError_t launch_mel_from_spec(const float* spec, int ldspec, const float* fb /*[1025][80]*/, float* mel,
                                 int B, int F, int Tm, cudaStream_t st);

// ---- quantizer-side kernels (quant.cu) -----------------------------------------------------
struct VqWeights {           // one dac/nn/quantize.py VectorQuantize, folded
    const float* w_in;       // [8][1024]
    const float* b_in;       // [8]
    const float* cb;         // [1024][8] raw codebook
    const float* cbn;        // [1024][8] F.normalize(codebook)
    const float* cbn2;       // [1024] sum(cbn^2)
    const float* w_out;      // [8][1024]  (transposed for coalescing: w_out_t[k][c])
    const float* b_out;      // [1024]
};
struct FaqParams {
    const float* f0 = nullptr;   // [B][Tq][1024] prosody features (channels-last)
    const float* z = nullptr;    // [B][Tz][1024] encoder latents (channels-last)
    VqWeights vq[6];             // prosody, content0, content1, residual0..2
    int n_c = 1;
    const float* gamma_beta = nullptr;  // [B][2048] timbre_linear(timbre)
    float* outs = nullptr;       // [B][Tq][1024]
    float* zp = nullptr, *zc = nullptr, *zr = nullptr;  // [B][Tq][1024] each (may be null)
    int64_t* codes_p = nullptr;  // [B][1][Tq]
    int64_t* codes_c = nullptr;  // [B][n_c][Tq]
    int64_t* codes_r = nullptr;  // [B][3][Tq]
    float* sqerr = nullptr;      // [6][B*Tq] per-frame sum (z_e - z_q)^2
    int B = 0, Tq = 0, Tz = 0, Tf0 = 0;   // Tz / Tf0 = frames per utterance of z / f0 (>= Tq)
};
cudaError_t launch_fa_quantize(const FaqParams& p, cudaStream_t st);
// codes -> outs (ResidualVectorQuantize.from_codes per group + the forward_v2 AdaLN tail); indices outside [0, 1024) are
// never dereferenced and make every channel of that frame's outs NaN
struct DequantParams {
    const int64_t* codes_p = nullptr;   // [B][1][T]
    const int64_t* codes_c = nullptr;   // [B][n_c_rows][T]; rows 0 .. n_c - 1 are used
    const int64_t* codes_r = nullptr;   // [B][n_r_rows][T]; rows 0 .. n_r - 1 are used (null when n_r = 0)
    int n_c_rows = 0, n_c = 1, n_r_rows = 0, n_r = 0;
    VqWeights vq[6];                    // prosody, content0, content1, residual0..2
    const float* gamma_beta = nullptr;  // [B][2048] timbre_linear(timbre)
    float* outs = nullptr;              // [B][T][1024]
    float* zp = nullptr, *zc = nullptr, *zr = nullptr;  // [B][T][1024] each (may be null)
    int B = 0, T = 0;
};
cudaError_t launch_dequantize(const DequantParams& p, cudaStream_t st);
// losses[0] = commitment, losses[1] = codebook (identical in forward), from sqerr
cudaError_t launch_vq_loss_reduce(const float* sqerr, int nq, int B, int Tq, float* losses2, cudaStream_t st);

// generic residual VQ over [N frames][D] with D == 1024, codebook_dim == 8 (quantize/rvq.py)
struct RvqParams {
    const float* x = nullptr;    // [B][T][1024] channels-last
    VqWeights vq[8];
    int nq = 0;
    float* qout = nullptr;       // [B][T][1024] quantized_out
    float* allq = nullptr;       // [nq][B][T][1024] or null
    int64_t* idx = nullptr;      // [nq][B][T]
    int B = 0, T = 0;
};
cudaError_t launch_rvq(const RvqParams& p, cudaStream_t st);

// elementwise / small ops
// losses.py:65-89 reconstruction_loss tail (frontend.cu)
cudaError_t launch_mel_loss_terms(const float* spec, int ldspec, int nb, const float* fb /*[nb][64]*/, int B, int F, float eps,
                                  float* terms /*[B*F][2]*/, cudaStream_t st);
cudaError_t launch_strided_sum(const float* in, long long n, int stride, double scale, double* out, cudaStream_t st);
cudaError_t launch_sqdiff_partial(const float* a, const float* b, long long n, float* part, int nblocks, cudaStream_t st);
// dac/nn/loss.py:142-327 spectral losses (frontend.cu)
cudaError_t launch_spec_loss_terms(const float* spec, int ldspec, int nb, const float* fb /*[nb][n_out] or null*/, int n_out, int B, int F,
                                   float eps, float pw, float* terms /*[B*F][2]*/, cudaStream_t st);
cudaError_t launch_absdiff_partial(const float* a, const float* b, long long n, float* part, int nblocks, cudaStream_t st);
cudaError_t launch_spec_loss_combine(const double* v, int n, float mag_weight, float log_weight, float* loss, cudaStream_t st);
cudaError_t launch_add3(const float* a, const float* b, const float* c /* or null */, long long n, float* out, cudaStream_t st);
cudaError_t launch_loss_combine(const double* v13, float* loss, float* terms, cudaStream_t st);
cudaError_t launch_transpose(const float* in, float* out, int B, int R, int C, cudaStream_t st);  // [B][R][C]->[B][C][R]
// tanh(a + g_a) * sigmoid(b + g_b); g = null or one [2*hidden] conditioning row per utterance (rows_per_utt rows each, g_stride floats apart)
cudaError_t launch_wn_gate(const float* xin, float* acts, size_t n_rows, int hidden, cudaStream_t st, const float* g = nullptr,
                           size_t rows_per_utt = 0, size_t g_stride = 0);
cudaError_t launch_wn_update(const float* rs, float* x, float* out, size_t n_rows, int hidden, int last, cudaStream_t st);
cudaError_t launch_glu_res(const float* y, float* x, int B, int T, int C, const int* valid_len, cudaStream_t st);  // x = x + y1*sig(y2) (masked)
cudaError_t launch_attention(const float* q, const float* k, const float* v, float* o, int B, int T, int heads,
                             int dk, const int* valid_len, cudaStream_t st, int force_stream = 0);
cudaError_t launch_mean_pool(const float* x, float* out, int B, int T, int C, const int* valid_len, cudaStream_t st);
cudaError_t launch_fill_u32(unsigned int* p, unsigned int v, size_t n, cudaStream_t st);

// alias-free activation (alias_free_torch/act.py:24-29): up x2 -> snake-beta/identity -> down x2
cudaError_t launch_alias_free_act(const float* x, float* y, int B, int C, int T, const float* filt12,
                                  const float* alpha, const float* inv_beta, cudaStream_t st);

}  // namespace fac
