/*
 * ovc.h -- C ABI of libovc_b200.so: the tone-colour-converter hot path of OpenVoice
 * (ToneColorConverter.convert -> SynthesizerTrn.voice_conversion) as hand-written
 * sm_100a CUDA kernels.
 *
 * The reference has no FFI / plugin interface (it is pure Python; SURVEY.md section 8b).  The
 * boundary this library replaces is the Python seam
 *
 *     model.voice_conversion(y, y_lengths, sid_src, sid_tgt, tau)
 *         -> (o_hat[B,1,256T], y_mask[B,1,T], (z, z_p, z_hat))      openvoice/models.py:492-499
 *
 * called from openvoice/api.py:154, plus checkpoint loading (openvoice/api.py:35-39) and model
 * construction from the JSON hparams (openvoice/api.py:21-28).  Entry points take plain
 * pointers and sizes only -- no torch types.  All functions return 0 on success and a negative
 * status otherwise; ovc_last_error() gives the message.  Nothing here ever falls back to a CPU
 * path: without a CUDA device every compute entry point fails.
 */
#ifndef OVC_B200_H
#define OVC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OVC_ABI_VERSION 4   /* 2: ovc_graph_replays, OVC_OPT_PDL .. OVC_OPT_PAIR; 3: OVC_OPT_ACT_TMA, OVC_OPT_TUNE and
                             * OVC_OPT_WIDE_VARIANT 1 retired (ovc_set_option refuses them); 4: precision mode 3 */

#if defined(__GNUC__)
#define OVC_API __attribute__((visibility("default")))
#else
#define OVC_API
#endif

enum {
  OVC_OK = 0,
  OVC_ERR_INVALID = -1,     /* bad argument / unsupported hyper-parameter               */
  OVC_ERR_CUDA = -2,        /* CUDA runtime error (message has cudaGetErrorString)      */
  OVC_ERR_STATE = -3,       /* call order violated (e.g. convert before finalize)       */
  OVC_ERR_MISSING = -4,     /* a checkpoint tensor needed by the hot path is missing    */
  OVC_ERR_NOMEM = -5
};

typedef struct ovc_ctx ovc_ctx;

/* Mirrors the `model` / `data` sections of the converter config.json that
 * OpenVoiceBaseClass.__init__ splats into SynthesizerTrn (openvoice/api.py:21-28,
 * openvoice/models.py:404-465).  The kernels are specialised for the released family
 * (SURVEY.md appendix A.1); anything else is refused by ovc_create with OVC_ERR_INVALID. */
typedef struct ovc_hparams {
  int32_t spec_channels;            /* filter_length/2+1 = 513          api.py:25            */
  int32_t inter_channels;           /* 192                              models.py:408        */
  int32_t hidden_channels;          /* 192                              models.py:409        */
  int32_t gin_channels;             /* 256                              models.py:422        */
  int32_t resblock;                 /* 1 (ResBlock1)                    models.py:242        */
  int32_t n_resblock_kernels;       /* 3                                                     */
  int32_t resblock_kernel_sizes[4]; /* 3,7,11                           models.py:261-264    */
  int32_t resblock_dilations[4][3]; /* {1,3,5} each                                          */
  int32_t n_upsamples;              /* 4                                                     */
  int32_t upsample_rates[4];        /* 8,8,2,2                          models.py:245-256    */
  int32_t upsample_kernel_sizes[4]; /* 16,16,4,4                                             */
  int32_t upsample_initial_channel; /* 512                                                   */
  int32_t zero_g;                   /* V2: g zeroed for enc_q and dec   models.py:423,495,498*/
  int32_t hop_length;               /* 256 (= product of upsample_rates)                     */
} ovc_hparams;

/* ABI version of the loaded library (== OVC_ABI_VERSION it was built with). */
OVC_API int ovc_abi_version(void);

/* Last error message of this thread ("" if none). Never NULL. */
OVC_API const char* ovc_last_error(void);

/* Build a converter context on CUDA device `device` (replaces SynthesizerTrn construction,
 * openvoice/api.py:23-30).  Fails with OVC_ERR_CUDA when no usable sm_100 device exists. */
OVC_API int ovc_create(const ovc_hparams* hp, int device, ovc_ctx** out);
OVC_API void ovc_destroy(ovc_ctx* ctx);

/* Feed one checkpoint tensor under its reference state-dict key, fp32, C-contiguous, host
 * memory (replaces load_state_dict(strict=False), openvoice/api.py:35-39; key schema in
 * SURVEY.md appendix A.2, weight-norm stored un-folded as weight_g / weight_v).  Keys that the
 * hot path does not use (ref_enc.*, enc_p.*, ...) are accepted and ignored (returns 1). */
OVC_API int ovc_load_tensor(ovc_ctx* ctx, const char* key, const float* data, const int64_t* shape, int ndim);

/* Fold weight-norm (g*v/||v||, per dim-0 slice), absorb the channel Flips of the flow into the
 * coupling weights, repack every conv for the kernels and upload.  The first bad tensor fails the
 * call and the message names its key: OVC_ERR_MISSING when it is missing, OVC_ERR_INVALID when
 * its shape is wrong. */
OVC_API int ovc_finalize_weights(ovc_ctx* ctx);

/* Number of floats of device workspace a call with (B, Tmax) needs (informational; the arena
 * grows on demand and is reused, so steady-state calls do not allocate). */
OVC_API size_t ovc_workspace_floats(const ovc_ctx* ctx, int B, int Tmax);

/* The hot path.  All pointers are DEVICE pointers on the context's device; the call only
 * enqueues work on `stream` (a cudaStream_t; NULL = default stream) and returns.
 *
 *   spec     [B, spec_channels, Tmax]  linear magnitude spectrogram            (api.py:150-152)
 *   lengths  [B] int64, valid frames per item (1 <= len <= Tmax)               (api.py:153)
 *   g_src    [B, gin] source tone-colour embedding (sid_src, [B,gin,1])        (models.py:493)
 *   g_tgt    [B, gin] target tone-colour embedding (sid_tgt)
 *   noise    [B, inter, Tmax] N(0,1) draws standing in for randn_like at models.py:220,
 *            or NULL: the kernel then draws Philox4x32-10 normals from `seed`
 *   tau      scales the noise term only                                        (models.py:220)
 *   ragged   0: reference batch semantics -- the (unmasked) generator runs over all Tmax frames
 *               of every item exactly as SynthesizerTrn.voice_conversion does on a padded batch
 *            1: every item is converted at its own exact length, i.e. what
 *               ToneColorConverter.convert (batch 1, api.py:148-154) produces per utterance
 *   o_hat    [B, hop*Tmax] waveform out (zero past hop*len when ragged)        (models.py:498)
 *   z, z_p, z_hat  [B, inter, Tmax] latents, masked like the reference; each may be NULL
 */
OVC_API int ovc_voice_conversion(ovc_ctx* ctx, const float* spec, const int64_t* lengths,
                         const float* g_src, const float* g_tgt, const float* noise,
                         uint64_t seed, float tau, int B, int Tmax, int ragged,
                         float* o_hat, float* z, float* z_p, float* z_hat, void* stream);

/* Front end of convert (row a2): linear magnitude spectrogram, replaces spectrogram_torch
 * (openvoice/mel_processing.py:40-75; call sites api.py:126-128,150-152) for n_fft = win = 1024,
 * hop 256: reflect-pad 384 at both ends of each item's own length, periodic hann, centre=False,
 * sqrt(re^2 + im^2 + 1e-6).
 *   wav          [B, Lmax] fp32 (device), rows zero padded past wav_lengths[b]
 *   wav_lengths  [B] int64 samples (device), each > 384 (reflect padding) and <= Lmax
 *   spec         [B, spec_channels, Tmax] out; frames >= wav_lengths[b]/hop are written as zeros
 *   frames       [B] int64 out (nullable): min(Tmax, wav_lengths[b] / hop)                          */
OVC_API int ovc_spectrogram(ovc_ctx* ctx, const float* wav, const int64_t* wav_lengths, int B, int Lmax,
                            int Tmax, float* spec, int64_t* frames, void* stream);

/* ToneColorConverter.convert's device work in one call (openvoice/api.py:148-155, batch of B):
 * spectrogram -> voice_conversion with per-item exact lengths (ragged).  Tmax = Lmax / hop.
 *   o_hat   [B, hop*Tmax] out; item b holds hop*frames[b] samples, zeros after
 *   frames  [B] int64 out (nullable)                                                               */
OVC_API int ovc_convert_waveform(ovc_ctx* ctx, const float* wav, const int64_t* wav_lengths, int B, int Lmax,
                                 const float* g_src, const float* g_tgt, const float* noise, uint64_t seed,
                                 float tau, float* o_hat, int64_t* frames, void* stream);

/* Tone-colour embedding of extract_se (row f2): ReferenceEncoder.forward (openvoice/models.py:339-359; call site
 * openvoice/api.py:130) on device -- LayerNorm over frequency, 6 x (Conv2d 3x3 s2 + ReLU), GRU(128) last state,
 * Linear.  Needs the checkpoint's ref_enc.* tensors (OVC_ERR_MISSING otherwise).
 *   spec  [N, spec_channels, T] magnitude spectrogram as written by ovc_spectrogram (all N items T frames)
 *   out   [N, gin]                                                                                          */
OVC_API int ovc_reference_encoder(ovc_ctx* ctx, const float* spec, int N, int T, float* out, void* stream);

/* ---- V1 base-speaker TTS front half: SynthesizerTrn.infer (openvoice/models.py:467-490), SURVEY.md section 8 row f3 ----
 * Available when the checkpoint passed through ovc_load_tensor holds enc_p.* / dp.* / sdp.* / emb_g.* (a V1 base
 * speaker, models.py:451-465); their hyper-parameters (n_vocab, heads, layers, window, filter sizes, n_speakers) are
 * read off the tensor shapes.  infer() is split where the reference itself synchronises (y_lengths -> mask sizes,
 * models.py:476-478):
 *
 *   ovc_tts_encode   x, m_p, logs_p = enc_p(tokens)                        models.py:468, 16-57; attentions.py:37-465
 *                    g = emb_g(sid)                                          models.py:470
 *                    logw = sdp(x, g, reverse) * ratio + dp(x, g) * (1 - ratio)   models.py:474-475, 60-180;
 *                                                                             modules.py:84-130, 459-516; transforms.py
 *                    w_ceil = ceil(exp(logw) * mask * length_scale); y_lengths = max(1, sum w_ceil)   models.py:477-479
 *   ovc_tts_decode   attn = generate_path(w_ceil); m_p, logs_p expanded; z_p = m_p + noise * exp(logs_p) * noise_scale;
 *                    z = flow(z_p, g, reverse); o = dec(z * y_mask, g)       models.py:480-490; commons.py:128-142
 *
 * tokens [B][T] int64 (padded), x_lengths [B] int64, sid [B] int64, noise_w [B][2][T] or NULL (Philox from `seed`);
 * y_lengths [B] int64 out; w_ceil / logw [B][T] optional outs.  All device pointers.  ovc_tts_decode uses the state the
 * last ovc_tts_encode left in the context: noise [B][inter][Ymax] or NULL (Philox), Ymax = max(y_lengths) (the
 * caller reads y_lengths back, as the reference does), max_len = the reference's max_len (0: none; the flow still runs
 * on all Ymax frames, only the generator is cut, models.py:489), ragged as in ovc_voice_conversion;
 * o [B][min(Ymax, max_len)*hop], z / z_p [B][inter][Ymax] optional.  ovc_tts_info: out8 = {has_tts, n_vocab, n_speakers, n_heads, n_layers, window, filter_channels, dp_filter}. */
OVC_API int ovc_tts_info(const ovc_ctx* ctx, int32_t* out8);
OVC_API int ovc_tts_encode(ovc_ctx* ctx, const int64_t* tokens, const int64_t* x_lengths, const int64_t* sid,
                           const float* noise_w, uint64_t seed, float noise_scale_w, float length_scale, float sdp_ratio,
                           int B, int T, int64_t* y_lengths, float* w_ceil, float* logw, void* stream);
OVC_API int ovc_tts_decode(ovc_ctx* ctx, const float* noise, uint64_t seed, float noise_scale, int B, int Ymax, int max_len,
                           int ragged, float* o, float* z, float* z_p, void* stream);

/* Arithmetic of the convolutions (generator ResBlocks = 90 % of the FLOPs, WaveNet stacks, upsamplers):
 *   0            fp32 FFMA2 on the CUDA cores
 *   1 (default of the Python surface)  split-precision "3xFP16" on the 5th-gen tensor cores (tcgen05 + TMEM):
 *                x = hi + lo / 2^11 with hi = fp16(x), lo = fp16((x - hi) * 2^11); every product is
 *                a_hi*b_hi + (a_lo*b_hi + a_hi*b_lo) / 2^11, fp32 accumulation, cross terms in their own
 *                accumulator -- fp32-grade error, same parity gate as mode 0.  Operands must be < 65504 in magnitude.
 *   2            single-pass fp16 on the tensor cores (11-bit operands): the precision class the REFERENCE itself
 *                gets on a GPU by default (cuDNN TF32, torch.backends.cudnn.allow_tf32 = True); own looser gate
 *   3            fp16 storage in the generator ("f16s"): everything before the generator runs as in mode 1, so z, z_p and
 *                z_hat are bit-identical to mode 1.  From conv_pre's output to conv_post's input every activation is
 *                fp16 in memory (channels-last) and every conv is one fp16 pass with fp32 accumulation; bias, residual,
 *                MRF sum and the 1/3 are fp32 math, each store rounds to fp16.  conv_post reads fp16 and writes fp32.
 *                Half the generator's HBM traffic and workspace; o_hat SNR >= 50 dB against fp32.  Activations must
 *                stay below 65504 in magnitude (no saturation).  OVC_OPT_PAIR and OVC_OPT_WIDE_VARIANT have no effect
 *                on the generator in this mode. */
OVC_API int ovc_set_precision(ovc_ctx* ctx, int mode);

/* Tuning / diagnostics switches (never change results beyond fp32 reordering):
 *   OVC_OPT_WIDE_VARIANT  kernel of the 128-column tensor-core layers: 0 the persistent kernel (one CTA per SM,
 *                         TMA-staged activations, overlapped epilogue); 2: one 128-step tile per CTA, two CTAs per SM;
 *                         3 (default): 2 for k >= 7 at Cin >= 256, else 0.  (1, 256-step tiles, is retired.)
 *   OVC_OPT_TTS_SIMPLE    1: one-thread-per-element text-side kernels (the CPU-checked element functions) instead of
 *                         the warp-cooperative LayerNorm / fused attention
 *   OVC_OPT_GRAPH         1 (default): replay the launch sequence of a repeated (shape, buffers) call from a CUDA graph
 *   OVC_OPT_PDL           programmatic stream serialization of the tensor-core conv launches (the prologue of kernel n+1 --
 *                         barriers, TMEM, weight TMA -- overlaps the drain of kernel n): 0 off, 1 all of them, 2 (default)
 *                         the WaveNet stacks only.  Measured on a B200: 2 saves 0.5-0.8 % at batch 32 and 2.4 % at batch 1;
 *                         1 costs 3 % at batch 32
 * Keys 4 (OVC_OPT_ACT_TMA) and 6 (OVC_OPT_TUNE) are retired: ovc_set_option returns OVC_ERR_INVALID for them. */
#define OVC_OPT_WIDE_VARIANT 1
#define OVC_OPT_TTS_SIMPLE 2
#define OVC_OPT_GRAPH 3
#define OVC_OPT_PDL 5
#define OVC_OPT_BRANCHES 7   /* 1 (default): latency-bound calls (B * Tmax <= 512 frames) run the three ResBlock branches of an
                              * MRF stage concurrently (three streams, a third of the SMs per kernel); results are bit-identical */
#define OVC_OPT_PAIR 8       /* 1 (default): the HBM-bound ResBlock conv pairs (C <= 64, k = 3) run as ONE kernel each
                              * (ovc_tcpair.cuh): the intermediate activation stays in shared memory; same bits as two launches */
OVC_API int ovc_set_option(ovc_ctx* ctx, int key, int value);

/* Number of kernels the last ovc_voice_conversion / ovc_convert_waveform call launched. */
OVC_API int ovc_last_launch_count(const ovc_ctx* ctx);

/* Number of ovc_voice_conversion / ovc_convert_waveform calls served by replaying a captured CUDA graph (OVC_OPT_GRAPH)
 * since the context was created.  A (shapes, buffers, options) signature is captured the second time it is seen and
 * replayed from the third call on; results are bit-identical to the directly launched sequence. */
OVC_API int ovc_graph_replays(const ovc_ctx* ctx);

/* Per-call timing hook for bench.py's roofline: when enabled, the dominant kernel family
 * (generator ResBlock convolutions) is bracketed with CUDA events on `stream`.  After the
 * stream has been synchronised, ovc_profile_read returns the accumulated milliseconds, the
 * number of launches, their algorithmic FLOPs and their algorithmic (layer-granular) bytes
 * since the last reset. */
OVC_API int ovc_profile_enable(ovc_ctx* ctx, int enable);
OVC_API int ovc_profile_read(ovc_ctx* ctx, double* ms, int64_t* launches, double* flops, double* bytes);
/* Per-launch detail of every conv kernel since the last reset (call before ovc_profile_read):
 * kernel-variant name (16 bytes each), milliseconds, algorithmic FLOPs / bytes, family (1 = generator
 * ResBlock convs).  Returns the number of entries written (<= max). */
OVC_API int ovc_profile_detail(ovc_ctx* ctx, int max, char* names, double* ms, double* flops, double* bytes,
                               int* family);

/* Debug taps (tests only): when enabled, named intermediate tensors of the next call are
 * copied aside; ovc_debug_fetch copies one to host memory.  Names: "enc.pre", "enc.wn",
 * "dec.pre", "dec.ups0".."dec.ups3", "dec.stage0".."dec.stage3", "cond". */
OVC_API int ovc_debug_enable(ovc_ctx* ctx, int enable);
OVC_API int ovc_debug_fetch(ovc_ctx* ctx, const char* name, float* host_out, size_t max_floats,
                    int64_t* shape4 /* B, C, T, pitch */);

#ifdef __cplusplus
}
#endif
#endif /* OVC_B200_H */
