/* facodec_b200 -- C-ABI of the B200-native FAcodec encode -> quantize -> decode hot path.
 *
 * The reference (Plachtaa/FAcodec) has no FFI layer: its boundary is the Python nn.Module call
 * surface  model.encoder(x) / model.quantizer(z, wave, ...) / model.decoder(z)  on the Munch
 * returned by build_model (modules/commons.py:283-348).  Each entry point below names the
 * reference interface it replaces; facodec_b200/modules.py is the thin ctypes shim that puts the
 * nn.Module surface back on top (INTEGRATION.md shows the binding).
 *
 * Conventions: plain pointers and sizes only; every tensor argument is a DEVICE pointer in the
 * reference's own layout (float32 [B, C, T] contiguous, int64 codes) unless the name ends in
 * _host; outputs are caller-allocated; `stream` is a cudaStream_t (0 = legacy default stream);
 * calls on one handle must be serialised by the caller.  Every function returns 0 on success or
 * a negative fac_status; fac_last_error() gives the text.  No exceptions cross the ABI.
 * Scratch memory is a grow-only device arena owned by the handle (fac_workspace_bytes).
 */
#ifndef FACODEC_B200_H
#define FACODEC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fac_handle fac_handle;

enum fac_status {
    FAC_OK = 0,
    FAC_ERR_INVALID = -1,   /* bad argument / shape */
    FAC_ERR_STATE = -2,     /* weights missing or not finalized */
    FAC_ERR_CUDA = -3,      /* CUDA runtime error (text in fac_last_error) */
    FAC_ERR_UNSUPPORTED = -4
};

/* FAC_REDECODER / FAC_REDECODER_DECODER: the voice-conversion model of build_model(args, stage='redecoder')
 * (modules/commons.py:385-412): modules/redecoder.py Redecoder (wavenet) and its Decoder(causal=False, lstm=0). */
enum fac_module { FAC_ENCODER = 0, FAC_QUANTIZER = 1, FAC_DECODER = 2, FAC_REDECODER = 3, FAC_REDECODER_DECODER = 4,
                  FAC_NUM_MODULES = 5 };

/* Library/ABI version (bumped on any signature change). */
int fac_abi_version(void);

/* Create / destroy an engine bound to CUDA device `device`. */
int fac_create(fac_handle** out, int device);
int fac_destroy(fac_handle* h);
const char* fac_last_error(const fac_handle* h);

/* Checkpoint loading.  Replaces  model[key].load_state_dict(ckpt[key])  (reconstruct.py:30-34,
 * modules/commons.py:446-471): feed every tensor of the reference state_dict of `module`
 * (reference key names, e.g. "block.1.block.0.block.1.conv.conv.weight_v"), HOST float32 data,
 * then call fac_finalize once.  fac_finalize folds weight-norm (g * v / ||v||, encodec.py:42-51),
 * Snake 1/(alpha+1e-9), LSTM biases, normalises the VQ codebooks, builds the STFT basis from
 * "to_mel.spectrogram.window", packs everything into kernel layouts and uploads it.
 * Modules whose tensors were never loaded stay unavailable (their entry points return
 * FAC_ERR_STATE). */
int fac_load_tensor(fac_handle* h, int module, const char* key, const float* data_host,
                    const int64_t* shape, int ndim);
int fac_finalize(fac_handle* h);

/* Replicated deployment (one process per GPU): rank 0 reads the checkpoint and broadcasts the raw
 * tensors as ONE flat fp32 buffer (ncclBroadcast through torch.distributed, see
 * facodec_b200/distributed.py); every rank then runs fac_load_tensor + fac_finalize locally.
 * There is no collective on the hot path. */

/* model.encoder(x): dac/model/dac.py:103-104 Encoder.forward.
 * x [B,1,T] -> z [B,1024,ceil(T/300)]. */
int fac_encode(fac_handle* h, const float* x, int B, int T, float* z, void* stream);
int fac_encode_frames(int T);   /* ceil-div chain of the strided convs = output frames */

/* model.quantizer(z, wave, n_c, n_t, full_waves, wave_lens, return_codes):
 * modules/quantize.py:375-454 FAquantizer.forward_v2 in eval mode.
 * z [B,1024,Tz], wave [B,1,T]; Tq = min(T/300, Tz).  full_waves [B,T_full] + wave_lens[B]
 * (int64, device) may be NULL (then the timbre comes from `wave`).  Outputs (any of zp/zc/zr/
 * codes_* may be NULL): outs, zp, zc, zr [B,1024,Tq]; losses2[2] = {commitment, codebook};
 * timbre [B,1024]; codes_p [B,1,Tq], codes_c [B,n_c,Tq], codes_r [B,3,Tq] int64. */
int fac_quantize(fac_handle* h, const float* z, const float* wave, int B, int T, int Tz, int n_c,
                 const float* full_waves, int T_full, const int64_t* wave_lens,
                 float* outs, float* zp, float* zc, float* zr, float* losses2, float* timbre,
                 int64_t* codes_p, int64_t* codes_c, int64_t* codes_r, void* stream);

/* model.decoder(z): dac/model/dac.py:164-165 Decoder.forward.  z [B,1024,Tf] -> y [B,1,300*Tf]. */
int fac_decode(fac_handle* h, const float* z, int B, int Tf, float* y, void* stream);

/* reconstruct.py:56-61 in one call, device buffers: encoder -> quantizer(n_c) -> decoder with the
 * latents kept channels-last on the device (no boundary transposes).  codes_* / timbre may be NULL. */
int fac_codec_forward(fac_handle* h, const float* x, int B, int T, int n_c, float* y,
                      int64_t* codes_p, int64_t* codes_c, int64_t* codes_r, float* timbre, void* stream);

/* Same, HOST buffers (pinned recommended): H2D of x, forward, D2H of y + codes, stream sync. */
int fac_codec_forward_host(fac_handle* h, const float* x_host, int B, int T, int n_c, float* y_host,
                           int64_t* codes_p_host, int64_t* codes_c_host, int64_t* codes_r_host, void* stream);

/* Voice conversion (reconstruct_redecoder.py:108-122, webui.py:68-81).
 * fac_redecode = model.encoder(p_code, c_code, timbre, use_p_code, use_c_code, n_c) of the redecoder model,
 * modules/redecoder.py:35-48: codes_p [B,1,T], codes_c [B,n_c_rows,T] int64 (device; the codec's codes[0], codes[1]),
 * timbre [B,1024] -> z [B,1024,T].  n_c <= n_c_rows <= 2 content codebooks are summed.
 * fac_redecoder_decode = that model's decoder (non-causal, no SLSTM: config_redecoder.yml decoder_causal / decoder_lstm),
 * z [B,1024,Tf] -> y [B,1,300*Tf].  fac_voice_convert runs both with the latents kept channels-last on the device. */
int fac_redecode(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, const float* timbre,
                 int B, int T, int use_p_code, int use_c_code, int n_c, float* z, void* stream);
int fac_redecoder_decode(fac_handle* h, const float* z, int B, int Tf, float* y, void* stream);
int fac_voice_convert(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, const float* timbre,
                      int B, int T, int use_p_code, int use_c_code, int n_c, float* y, void* stream);

/* Decoding from codes: the codes and timbre a forward returned (or a .dac file holds, plus a timbre) back to latents /
 * audio.  Per group (prosody, content, residual) this is ResidualVectorQuantize.from_codes (dac/nn/quantize.py:200-220):
 * z_g = 0 + sum_q out_proj_q(codebook_q[codes[:, q]]) on the raw codebook rows; then the FAquantizer.forward_v2 tail
 * (modules/quantize.py:435-449): outs = LayerNorm(z_p + z_c + z_r, no affine, eps 1e-5) * gamma + beta with
 * (gamma, beta) = timbre_linear(timbre).  (The reference's own FAquantizer.decode, modules/quantize.py:244-254, expects
 * the layout without timbre_norm and cannot run under configs/config.yml.)
 * codes_p [B,1,T], codes_c [B,n_c_rows,T], codes_r [B,n_r_rows,T] int64 (device); the first 1 <= n_c <= n_c_rows <= 2
 * content and 0 <= n_r <= n_r_rows <= 3 residual codebooks are used (fewer = a lower bitrate; codes_r may be NULL when
 * n_r = 0, and then z_r = 0); timbre [B,1024].  A code outside [0, 1024) is never dereferenced: every channel of that
 * frame's outs is NaN.  Needs the quantizer weights only.
 * fac_dequantize: outs [B,1024,T] and (each may be NULL) zp, zc, zr [B,1024,T].
 * fac_decode_codes: the same, then model.decoder (dac/model/dac.py:164-165) with the latents kept channels-last on the
 * device: y [B,1,300*T].  Needs the quantizer and decoder weights. */
int fac_dequantize(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, int n_c, const int64_t* codes_r,
                   int n_r_rows, int n_r, const float* timbre, int B, int T, float* outs, float* zp, float* zc, float* zr,
                   void* stream);
int fac_decode_codes(fac_handle* h, const int64_t* codes_p, const int64_t* codes_c, int n_c_rows, int n_c, const int64_t* codes_r,
                     int n_r_rows, int n_r, const float* timbre, int B, int T, float* y, void* stream);

/* Streaming (SURVEY.md section 8f rank 4; README.md:105-107 "causal ... can be used for streaming"): the encoder and the codec's
 * decoder are causal, so a long utterance can be processed in chunks with the SAME results as one offline call
 * (dac/model/dac.py:103-104, :164-165).  The reference ships no streaming driver; these entry points carry what the
 * causal graph needs between chunks on the device: the conv stacks' left context (6000 samples / 20 latent frames) and the
 * SLSTM (h, c) states (dac/model/encodec.py:272-288: the SLSTM itself keeps none; it is explicit here).
 * fac_stream_begin(B <= 32) -> stream id (>= 0) or a negative status; one stream holds one encoder and one decoder state.
 * fac_stream_encode: x_chunk [B,1,T] (device; T a multiple of 300, the first chunk >= 3000) -> z_chunk [B,1024,T/300].
 * fac_stream_decode: z_chunk [B,1024,Fc] (device; first chunk >= 10 frames) -> y_chunk [B,1,300*Fc].
 * The quantizer is not part of the stream: its timbre branch pools over the whole utterance (modules/quantize.py:375-454),
 * the VQ lookups themselves are per frame (fac_quantize on each z chunk is exact for the codes). */
int fac_stream_begin(fac_handle* h, int B);
int fac_stream_encode(fac_handle* h, int stream_id, const float* x, int T, float* z, void* stream);
int fac_stream_decode(fac_handle* h, int stream_id, const float* z, int Fc, float* y, void* stream);
int fac_stream_end(fac_handle* h, int stream_id);

/* quantize/rvq.py:27-75 ResidualVQ.forward (eval) over quantize/fvq.py FactorizedVectorQuantize,
 * dim=1024, codebook_dim=8, 2^10 entries (BASELINE configs[3]).  Parameters are passed directly
 * (already weight-normed, HOST): per quantizer q: in_w [8,1024], in_b [8], out_w [1024,8],
 * out_b [1024], codebook [1024,8].  fac_rvq_create returns an id usable with fac_rvq_forward:
 * x [B,1024,T] -> quantized_out [B,1024,T], indices [nq,B,T] int64, all_quantized [nq,B,1024,T]
 * (may be NULL).  x_channels_last != 0 means x / outputs are [B,T,1024] (no transposes). */
int fac_rvq_create(fac_handle* h, int nq, const float* const* in_w, const float* const* in_b,
                   const float* const* out_w, const float* const* out_b, const float* const* codebook);
int fac_rvq_destroy(fac_handle* h, int rvq_id);   /* frees that set's device arena (e.g. before re-creating it with new weights) */
int fac_rvq_forward(fac_handle* h, int rvq_id, const float* x, int B, int T, int x_channels_last,
                    float* quantized_out, int64_t* indices, float* all_quantized, void* stream);

/* alias_free_torch/act.py:24-29 Activation1d.forward with up/down ratio 2, 12-tap Kaiser-sinc
 * filters (filter.py:27-58).  x, y [B,C,T].  act: 0 = identity, 1 = SnakeBeta with per-channel
 * alpha / beta given as already-exponentiated values (modules/quantize.py:29-79). */
int fac_alias_free_act(fac_handle* h, const float* x, int B, int C, int T, int act,
                       const float* alpha, const float* beta, float* y, void* stream);

/* Dataset-side mel: meldataset.py:37-47 preprocess (PseudoDataset.__getitem__ :64-71) -- torchaudio MelSpectrogram(n_mels=80,
 * n_fft=2048, win_length=1200, hop_length=300) with its default sample_rate=16000 filterbank, centre=True, then
 * (log(1e-5 + mel) + 4) / 4.  wave [B,T] (device, T > 1024) -> mel [B,80,T/300+1]. */
int fac_dataset_mel(fac_handle* h, const float* wave, int B, int T, float* mel, void* stream);

/* Training-side reconstruction loss, forward only: losses.py:65-89 reconstruction_loss(x, G_x) =
 * 100 * mse(x, G_x) + sum over s in {64, 128, ..., 2048} of (l1_s + sqrt(s/2) * l2_s) between the 64-band mel spectrograms
 * torchaudio MelSpectrogram(sample_rate=16000, n_fft=max(s,512), win_length=s, hop_length=s/4, n_mels=64) gives for x and G_x:
 * l1 = mean |S_x - S_G|, l2 = mean over (utterance, frame) of sqrt(mean over bands of (log(|S_x|+1e-7) - log(|S_G|+1e-7))^2).
 * x, gx [B,T] (device, T > 1024).  loss: 1 float (device).  terms: NULL or 13 floats (device): mse, then (l1, l2) per scale. */
int fac_reconstruction_loss(fac_handle* h, const float* x, const float* gx, int B, int T, float* loss, float* terms, void* stream);

/* dac/nn/loss.py:142-327 MultiScaleSTFTLoss (n_mels = NULL) / MelSpectrogramLoss and :11-47 L1Loss, forward values.  The
 * reference evaluates them on audiotools AudioSignal objects; audiotools / librosa are not vendored (SURVEY.md 8c: parity
 * UNPINNED), so their published semantics are restated: torch.stft(n_fft = window_length, hop = window_length/4, periodic Hann,
 * centre = True, reflect), magnitude = |stft|, mel = magnitude @ librosa.filters.mel(sample_rate, n_fft, n_mels, fmin, fmax)^T
 * (Slaney scale + area normalisation); loss = sum over scales of log_weight * mean|log10(clamp(v,eps)^pow) differences| +
 * mag_weight * mean|v differences|.  x, y [B,T] (device).  window_lengths: powers of two in [16, 4096]; mel_fmax[i] <= 0 means
 * sample_rate / 2.  loss: 1 float (device).  The (sample_rate, scales) configuration is cached on the handle. */
int fac_spectral_loss(fac_handle* h, const float* x, const float* y, int B, int T, int sample_rate, int n_scales,
                      const int* window_lengths, const int* n_mels, const float* mel_fmin, const float* mel_fmax, float clamp_eps,
                      float mag_weight, float log_weight, float pow, float* loss, void* stream);
int fac_l1_loss(fac_handle* h, const float* x, const float* y, long long n, float* loss, void* stream);

/* Predictor heads: modules/quantize.py:106-125 CNNLSTM(indim, outdim, head, global_pred) forward (3 ResidualUnits of
 * alias-free SnakeBeta + weight-normed Conv1d k7 (dilation 1, 2, 3, zero padding) / k1, a final alias-free SnakeBeta,
 * `nheads` nn.Linear layers; mean over time first when global_pred).  fac_head_begin returns a head id; feed the reference
 * state_dict tensors (keys "model.0.block.0.act.alpha", "model.0.block.1.weight_g", ..., "heads.0.weight"; the registered
 * filter buffers are ignored) with fac_head_tensor, then fac_head_finalize.  fac_head_forward: x [B,indim,T] (device) ->
 * outs[i] [B,T,outdim] (or [B,outdim] when global_pred), i < nheads, caller-allocated device buffers.
 * global_pred = 2 makes the head a plain nn.Linear(indim, outdim) (FApredictors.timbre_predictor under timbre_norm,
 * modules/quantize.py:470-473): stage "linear.weight" [outdim][indim] and "linear.bias", nheads = 1; fac_head_forward then
 * takes x as [B*T rows][indim] and writes outs[0] [B*T][outdim].
 * fac_add3: out = a + b (+ c when c is not NULL), n floats on the device: the latent sums FApredictors.forward_v2 feeds
 * its gradient-reversal heads (modules/quantize.py:571-586). */
int fac_head_begin(fac_handle* h);
int fac_head_tensor(fac_handle* h, int head_id, const char* key, const float* data_host, const int64_t* shape, int ndim);
int fac_head_finalize(fac_handle* h, int head_id, int indim, int outdim, int nheads, int global_pred);
int fac_head_forward(fac_handle* h, int head_id, const float* x, int B, int T, float* const* outs, void* stream);
int fac_add3(fac_handle* h, const float* a, const float* b, const float* c, long long n, float* out, void* stream);

/* Engine options.  "tensor_cores": 0 = fp32 FMA kernels everywhere; 1 = tcgen05 3xTF32
 * kernel for every eligible layer downstream of the VQ (decoder, timbre branch), fp32 FMA upstream
 * (encoder, prosody branch); 2 (default) = tcgen05 everywhere, with the register-promoted accumulation
 * variant upstream of the VQ where the bit-exact argmin needs fp32-grade sums.
 * "fuse_resunit": 1 (default) runs each decoder ResidualUnit whose channels fit one CTA tile as a single
 * fused launch (conv7 -> Snake -> 1x1 conv -> +x with the intermediate kept in TMEM/SMEM); 0 = two launches;
 * 2 = fuse only units of at most 128 channels (the ones whose fused tile still allows two CTAs per SM).
 * "decoder_bf16": 1 (default) = layers downstream of the VQ split operands into bf16 hi + bf16 lo
 * (tcgen05.mma.kind::f16, K = 16: half the MMAs and half the operand bytes of the TF32 split; waveform error
 * ~1e-5 RMS against the 1e-4 bar), evaluate Snake with the SFU sine and run the LSTM recurrence on bf16 hi/lo
 * mma.sync tiles; 0 = TF32 hi/lo everywhere.  Never applied upstream of the VQ.
 * "encoder_f16x2": 0 (default) / 1 = EXPERIMENTAL: layers upstream of the VQ split operands into fp16 hi + fp16 lo
 * scaled by 2^11 (kind::f16, K = 16, cross terms in their own TMEM accumulator, scaled back at promotion) instead of
 * the TF32 pair: same 22 mantissa bits and bit-exact codes on every fixture, but operands must stay below fp16's
 * 65504, and the measured gain is only 5-11 % on the k=7 encoder convs (one MMA stream per SM runs kind::f16 at
 * about half rate for N <= 128), so it is off by default.
 * "tc_occ2_maxn": channel tiles of at most this width (default 256; 0 = off) are planned for TWO resident CTAs per
 * SM (<= 256 TMEM columns, <= 112 KB shared memory each) so one CTA's MMAs overlap the other's produce/epilogue. */
int fac_set_option(fac_handle* h, const char* name, int value);

size_t fac_workspace_bytes(const fac_handle* h);
/* number of kernel launches issued by the last forward call (bench.py "gpu_launches") */
int fac_last_launch_count(const fac_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* FACODEC_B200_H */
