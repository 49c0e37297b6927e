/*
 * dfb200.h -- C ABI of libdfb200.so: the B200 (sm_100a) implementation of DeepFilterNet's
 * per-frame enhancement path (STFT -> ERB / complex features -> encoder / GRUs / decoders ->
 * gain mask + deep filter -> ISTFT).
 *
 * The reference has NO C ABI for this batched path: its boundary is the PyO3 module `libdf`
 * (pyDF/src/lib.rs) plus the Python functions in DeepFilterNet/df/enhance.py.  Each entry point
 * below names the reference interface it replaces; INTEGRATION.md shows the binding a reference
 * maintainer would add (ctypes stubs that stand in for pyDF's #[pymethods]).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / numpy types cross this boundary.
 *   - every function returns 0 on success or a negative dfb_status; dfb_last_error() returns a
 *     thread-local human readable message for the last failure.
 *   - "_host" entry points take HOST pointers and do the host<->device copies themselves (on the
 *     handle's stream, synchronised before returning); the others take DEVICE pointers valid on
 *     the handle's device and are asynchronous on `stream` (a cudaStream_t passed as void*).
 *   - complex data are interleaved (re, im) float pairs, exactly numpy complex64 / Rust Complex32.
 *   - there is no CPU fallback: every function fails with DFB_ERR_CUDA when no sm_100 device is
 *     usable.
 */
#ifndef DFB200_H
#define DFB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    DFB_OK = 0,
    DFB_ERR_INVALID = -1,     /* bad argument (shape, null pointer, unsupported size) */
    DFB_ERR_CUDA = -2,        /* CUDA runtime / launch failure, or no usable device    */
    DFB_ERR_UNSUPPORTED = -3, /* configuration outside the built kernels               */
    DFB_ERR_OOM = -4
} dfb_status;

const char *dfb_last_error(void);
/* ABI / build info: "dfb200 <version> sm_100a" */
const char *dfb_version(void);
/* number of CUDA kernels this library has launched in the calling process (all handles) */
int64_t dfb_kernel_launches(void);

/* Per-kernel timing with CUDA events on the launching stream (used by bench.py for the roofline
 * numbers).  on != 0 enables it; only_kernel (may be NULL) restricts it to one kernel name.
 * dfb_profile_report synchronises the device, writes "name count total_ms\n" lines for everything
 * recorded since the previous report into buf and returns the number of bytes written. */
int dfb_profile_enable(int on, const char *only_kernel);
int64_t dfb_profile_report(char *buf, int64_t buflen);

/* ------------------------------------------------------------------ DSP state ------------
 * Replaces libDF `DFState` as exposed by pyDF `DF` (pyDF/src/lib.rs:14-136,
 * libDF/src/lib.rs:104-154).  Holds the vorbis window, FFT twiddles and ERB tables on the device.
 * The analysis / synthesis memories (lib.rs:60-62) are carried by the *_host_ex entry points exactly as
 * pyDF does with `reset=False`; the device-pointer entry points and the fused enhance path always start
 * each channel from the reset state (pyDF's default `reset=True`, pyDF/src/lib.rs:56-58, 91-93). */
typedef struct dfb_state dfb_state;

/* pyDF DF.__new__ (pyDF/src/lib.rs:22-39) -> DFState::new (libDF/src/lib.rs:104-154).
 * device: CUDA ordinal.  STFT geometries: fft_size 960 / hop_size 480 (all shipped models) runs specialised
 * kernels; any other even fft_size with 32 <= fft_size <= 4096 whose half has no prime factor above 7 (320, 384,
 * 512, 640, 882, 1024, 1920, 4096, ...) runs runtime mixed-radix kernels, at any hop_size <= fft_size / 2 for
 * analysis / synthesis / features / forward / apply.  Other sizes: DFB_ERR_UNSUPPORTED; hop_size * 2 > fft_size:
 * DFB_ERR_INVALID.  dfb_enhance* and dfb_stream_* need hop_size == fft_size / 2 (DFB_ERR_UNSUPPORTED otherwise);
 * a model whose nb_df exceeds fft_size / 2 + 1 is rejected with DFB_ERR_INVALID. */
int dfb_state_create(dfb_state **out, int device, int sr, int fft_size, int hop_size, int nb_erb,
                     int min_nb_erb_freqs);
void dfb_state_free(dfb_state *st);
/* pyDF erb_widths / fft_window / sr / fft_size / hop_size / nb_erb (pyDF/src/lib.rs:109-131) */
int dfb_state_erb_widths(const dfb_state *st, int64_t *widths /* [nb_erb] host */);
int dfb_state_fft_window(const dfb_state *st, float *window /* [fft_size] host */);
int dfb_state_params(const dfb_state *st, int *sr, int *fft_size, int *hop_size, int *nb_erb);
/* ERB band widths only, no device needed: libDF erb_fb (libDF/src/lib.rs:68-100) */
int dfb_erb_widths(int sr, int fft_size, int nb_erb, int min_nb_freqs, int64_t *widths);

/* pyDF DF.analysis (pyDF/src/lib.rs:41-72) -> frame_analysis (libDF/src/lib.rs:356-394).
 * audio f32[C, T] (row stride T) -> spec c64[C, T / hop, F].  Trailing partial frame dropped. */
int dfb_analysis(dfb_state *st, const float *d_audio, int64_t C, int64_t T, float *d_spec, void *stream);
int dfb_analysis_host(dfb_state *st, const float *h_audio, int64_t C, int64_t T, float *h_spec);
/* same with pyDF's `reset` argument: reset == 0 carries the STFT memory across calls and channels exactly like
 * the shared DFState of the reference (channel 0 continues the previous call, channel c continues c - 1) */
int dfb_analysis_host_ex(dfb_state *st, const float *h_audio, int64_t C, int64_t T, int reset, float *h_spec);
/* pyDF DF.reset (pyDF/src/lib.rs:133-135): zero the carried analysis / synthesis memories */
int dfb_state_reset(dfb_state *st);

/* pyDF DF.synthesis (pyDF/src/lib.rs:74-107) -> frame_synthesis (libDF/src/lib.rs:396-427).
 * spec c64[C, Tf, F] -> audio f32[C, Tf * hop].  Does NOT clobber its input (the reference does). */
int dfb_synthesis(dfb_state *st, const float *d_spec, int64_t C, int64_t Tf, float *d_audio, void *stream);
int dfb_synthesis_host(dfb_state *st, const float *h_spec, int64_t C, int64_t Tf, float *h_audio);
int dfb_synthesis_host_ex(dfb_state *st, const float *h_spec, int64_t C, int64_t Tf, int reset, float *h_audio);

/* libdf.erb (pyDF/src/lib.rs:142-192) -> compute_band_corr (+dB) (libDF/src/lib.rs:280-295,
 * transforms.rs:236-253).  spec c64[n_frames, F] -> f32[n_frames, E]; widths host int64[E]. */
int dfb_erb_host(int device, const float *h_spec, int64_t n_frames, int64_t F, const int64_t *widths, int E,
                 int db, float *h_out);
/* libdf.erb_inv (pyDF/src/lib.rs:194-250) -> interp_band_gain (libDF/src/lib.rs:328-337). */
int dfb_erb_inv_host(int device, const float *h_gains, int64_t n_frames, const int64_t *widths, int E,
                     float *h_out /* [n_frames, sum(widths)] */);
/* libdf.erb_norm (pyDF/src/lib.rs:252-274) -> band_mean_norm_erb (libDF/src/lib.rs:244-251).
 * erb f32[C, T, E] -> out f32[C, T, E]; state f32[C, E] or NULL (linspace(-60,-90,E)). */
int dfb_erb_norm_host(int device, const float *h_erb, int64_t C, int64_t T, int64_t E, float alpha,
                      const float *h_state, float *h_out);
/* libdf.unit_norm (pyDF/src/lib.rs:276-298) -> band_unit_norm (libDF/src/lib.rs:253-259).
 * spec c64[C, T, F] -> out c64[C, T, F]; state f32[C, F] or NULL (linspace(1e-3,1e-4,F)). */
int dfb_unit_norm_host(int device, const float *h_spec, int64_t C, int64_t T, int64_t F, float alpha,
                       const float *h_state, float *h_out);
/* libdf.unit_norm_init (pyDF/src/lib.rs:300-307) */
int dfb_unit_norm_init(int64_t n, float *h_out);

/* df.enhance.df_features (DeepFilterNet/df/enhance.py:190-203) as ONE fused device pass:
 * audio f32[C,T] -> spec c64[C,Tf,F], feat_erb f32[C,Tf,E], feat_spec c64[C,Tf,nb_df]. */
int dfb_features(dfb_state *st, const float *d_audio, int64_t C, int64_t T, int nb_df, float alpha,
                 float *d_spec, float *d_feat_erb, float *d_feat_spec, void *stream);
int dfb_features_host(dfb_state *st, const float *h_audio, int64_t C, int64_t T, int nb_df, float alpha,
                      float *h_spec, float *h_feat_erb, float *h_feat_spec);

/* df.io.resample (DeepFilterNet/df/io.py:107-129 -> torchaudio.functional.resample): polyphase sinc resampling on the
 * device.  h_kernel f32[new][2 * width + orig] are the taps of torchaudio's _get_sinc_resample_kernel for the gcd-reduced
 * rates (orig, new); audio f32[C][T] -> out f32[C][T_out], T_out = ceil(new * T / orig). */
int dfb_resample_host(int device, const float *h_audio, int64_t C, int64_t T, const float *h_kernel, int orig, int new_rate,
                      int width, float *h_out, int64_t T_out);

/* ------------------------------------------------------------------ metrics ----------------
 * Speech-quality metrics of B (clean, degraded) pairs, the device counterpart of the reference's evaluation metrics
 * (df/stoi.py, df/sepm.py, df/evaluation_utils.py).  One bit per metric; d_out f32[B][popcount(which)] holds the selected
 * metrics in bit order:
 *   STOI   df.stoi.stoi at 10 kHz (inputs resampled like df.io.resample); NaN when fewer than 512 samples remain after
 *          the silent-frame removal (the reference leaves the entry uninitialised)
 *   SISDR  df.evaluation_utils.si_sdr_speechmetrics at the input rate
 *   SSNR / LLR / WSS   df.sepm.SNRseg / llr / wss at 16 kHz (inputs resampled to 16 kHz unless sr == 16000, as
 *          CompositeMetric does); NaN when the 16 kHz signal has fewer than 600 samples (no frame to score) */
enum {
    DFB_METRIC_STOI = 1,
    DFB_METRIC_SISDR = 2,
    DFB_METRIC_SSNR = 4,
    DFB_METRIC_LLR = 8,
    DFB_METRIC_WSS = 16
};
/* d_clean / d_deg f32[B][T] (device); lengths: HOST int64[B] (NULL: all T), 1 <= lengths[b] <= T; pair b is scored on its
 * first lengths[b] samples exactly as if it were scored alone.  sr: 8000, 16000, 22050, 24000, 32000, 44100 or 48000.
 * Asynchronous on `stream` (device scratch is stream-ordered).  DFB_ERR_INVALID for a bad length, sr or bit. */
int dfb_metrics(int device, const float *d_clean, const float *d_deg, const int64_t *lengths, int64_t B, int64_t T, int sr,
                unsigned which, float *d_out, void *stream);
int dfb_metrics_host(int device, const float *h_clean, const float *h_deg, const int64_t *lengths, int64_t B, int64_t T,
                     int sr, unsigned which, float *h_out);

/* ------------------------------------------------------------------ model ------------------
 * Replaces the forward pass of DeepFilterNet/df/deepfilternet3.py (DfNet :334-456) and
 * deepfilternet2.py (DfNet :374-505) for the shipped DeepFilterNet2 / 3 / 3_ll topologies. */
typedef struct dfb_model dfb_model;

typedef struct {
    int32_t model_kind;      /* 2 = DeepFilterNet2, 3 = DeepFilterNet3 (incl. _ll)          */
    int32_t nb_erb, nb_df, df_order, df_lookahead, conv_lookahead;
    int32_t conv_ch;         /* 64                                                           */
    int32_t conv_kt;         /* time taps of the `conv_kernel` layers (1; _ll: 2)            */
    int32_t inp_kt;          /* time taps of conv_kernel_inp (3)                             */
    int32_t emb_hidden, df_hidden;
    int32_t enc_gru_layers, erb_gru_layers, df_gru_layers;
    int32_t df_pathway_kt;   /* 5 */
    int32_t enc_concat;      /* DFN2: 1 */
    int32_t g_df_fc_emb, g_enc_in, g_enc_out, g_erb_in, g_erb_out, g_df_in, g_df_skip, g_df_out;
    float lsnr_scale, lsnr_offset;
    float norm_alpha;        /* feature normalisation decay, df/utils.py:108-124 (0.99) */
} dfb_model_config;

/* One named fp32 tensor of the packed weight set (BatchNorm already folded, layouts as documented
 * in deepfilternet_b200/weights.py).  `data` is a HOST pointer; it is copied to the device. */
typedef struct {
    const char *name;
    const float *data;
    int64_t numel;
} dfb_tensor;

/* Replaces init_model + load_state_dict (deepfilternet3.py:80-87, checkpoint.py:46-104). */
int dfb_model_create(dfb_model **out, int device, const dfb_model_config *cfg, const dfb_tensor *tensors,
                     int n_tensors, const int64_t *erb_widths);
void dfb_model_free(dfb_model *m);

/* DfNet.forward without the spectral apply (deepfilternet3.py:407-441): features -> ERB mask m,
 * DF coefficients and local SNR.  feat_erb f32[B,T,E], feat_spec c64[B,T,nb_df]
 * -> m f32[B,T,E], coefs f32[B,T,nb_df,2*order], lsnr f32[B,T] (may be NULL), alpha f32[B,T]
 * (DeepFilterNet2's df_fc_a output, deepfilternet2.py:368; may be NULL, ignored for kind 3). */
int dfb_model_forward(dfb_model *m, const float *d_feat_erb, const float *d_feat_spec, int64_t B, int64_t T,
                      float *d_m, float *d_coefs, float *d_lsnr, float *d_alpha, void *stream);

/* Mask.forward + MF.DF.forward (modules.py:248-269, multiframe.py:169-180,
 * deepfilternet3.py:431-443 / deepfilternet2.py:494-503): spec c64[B,T,F], m, coefs -> spec_e. */
int dfb_apply(dfb_model *m, dfb_state *st, const float *d_spec, const float *d_m, const float *d_coefs,
              int64_t B, int64_t T, float *d_spec_e, void *stream);

/* DfNet.forward (deepfilternet3.py:389-456): (spec, feat_erb, feat_spec) -> (spec_e, m, lsnr, coefs);
 * any of d_m / d_lsnr / d_coefs / d_alpha may be NULL. */
int dfb_model_forward_full(dfb_model *m, dfb_state *st, const float *d_spec, const float *d_feat_erb,
                           const float *d_feat_spec, int64_t B, int64_t T, float *d_spec_e, float *d_m,
                           float *d_lsnr, float *d_coefs, float *d_alpha, void *stream);

/* df.enhance.enhance (DeepFilterNet/df/enhance.py:206-250), the whole path in one call:
 * audio f32[B,T] -> enhanced f32[B,T_out].  pad != 0: zero-pad fft_size samples at the end and
 * crop the STFT delay (T_out = T); pad == 0: T_out = (T / hop) * hop, delayed by fft - hop.
 * atten_lim_db <= 0 disables the attenuation limit (enhance.py:238-240).
 * The apply + ISTFT stage is one fused kernel (gain x spectrum + deep filter + irFFT + OLA).
 * The signal is processed in time chunks with carried state (see "streaming" below), so the device workspace does
 * not grow with T; dfb_enhance_host additionally overlaps the H2D / D2H copies of neighbouring chunks with the compute. */
int dfb_enhance(dfb_model *m, dfb_state *st, const float *d_audio, int64_t B, int64_t T, int pad,
                float atten_lim_db, float *d_out, void *stream);
int dfb_enhance_host(dfb_model *m, dfb_state *st, const float *h_audio, int64_t B, int64_t T, int pad,
                     float atten_lim_db, float *h_out);
/* output length of dfb_enhance for a given input length */
int64_t dfb_enhance_out_len(const dfb_state *st, int64_t T, int pad);
/* ------------------------------------------------------------------ streaming -----------------
 * Frame-incremental processing with carried per-stream state: the batched counterpart of the reference's
 * single-stream runtime `DfTract::process` (libDF/src/tract.rs:509-642) and its C ABI (libDF/src/capi.rs:83-253:
 * df_create / df_get_frame_length / df_process_frame / df_free).  The state carried between calls is SURVEY.md
 * Appendix D: STFT / ISTFT memories, normalisation EMAs, GRU hidden states, conv / deep-filter history.
 * Every call feeds n >= 1 hops per stream and returns n hops; the output trails the input by
 * dfb_stream_latency_frames() hops (the model's look-ahead) on top of the STFT's fft - hop samples: the concatenated
 * output equals dfb_enhance(pad = 0) of the concatenated input, delayed by latency * hop samples.  dfb_enhance itself
 * runs on the same time-chunked executor.  Optional stages: the post filter (dfb_model_set_options) and the Rust
 * runtime's LSNR stage gating (dfb_stream_set_lsnr_thresholds); not built: its silent-frame skip (tract.rs:516-525). */
typedef struct dfb_stream dfb_stream;
/* capi.rs df_create: B independent streams on the model's device; atten_lim_db <= 0 disables the limit */
int dfb_stream_create(dfb_stream **out, dfb_model *m, dfb_state *st, int64_t B, float atten_lim_db);
void dfb_stream_free(dfb_stream *s);                       /* capi.rs df_free */
int dfb_stream_reset(dfb_stream *s);                       /* back to the initial state (all memories zero) */
int64_t dfb_stream_frame_length(const dfb_stream *s);      /* capi.rs df_get_frame_length: hop size in samples */
int64_t dfb_stream_latency_frames(const dfb_stream *s);    /* hops the output trails the input by */
/* LSNR stage gating (libDF/src/tract.rs:658-672 apply_stages; defaults -10 / 30 / 20 dB, tract.rs:180-185): per frame,
 * lsnr < min_db_thresh -> zero gains, no deep filter; > max_db_erb_thresh -> the frame passes unprocessed;
 * > max_db_df_thresh -> ERB gains only; else gains + deep filter.  Off by default (the Python path never gates);
 * DeepFilterNet3 topologies only. */
int dfb_stream_set_lsnr_thresholds(dfb_stream *s, int enable, float min_db_thresh, float max_db_erb_thresh,
                                   float max_db_df_thresh);
/* capi.rs df_process_frame, batched and for n_frames hops at once: d_in / d_out f32[B][n_frames * hop] (device) */
int dfb_stream_process(dfb_stream *s, const float *d_in, int64_t n_frames, float *d_out, void *stream);
/* end of stream: the latency frames still in flight, d_out f32[B][latency * hop]; reset before feeding again */
int dfb_stream_flush(dfb_stream *s, float *d_out, void *stream);
/* host pointers, synchronous; h_in == NULL flushes into h_out f32[B][latency * hop] */
int dfb_stream_process_host(dfb_stream *s, const float *h_in, int64_t n_frames, float *h_out);

/* Arithmetic of the dense contractions -- a bit mask; everything that is not a contraction is always IEEE fp32:
 *   bit 1 (2): GRU recurrence W_hh h on tcgen05 with BF16 hi/lo split operands (3 MMAs per product, fp32 accumulate)
 *   bit 2 (4): GRU input projections W_ih x on the BF16x3 tcgen05 GEMM
 *   bit 3 (8): 1x1 convs of the separable conv blocks and the grouped linears on the BF16x3 tcgen05 kernels
 * 0 = FFMA everywhere; 14 = the default of the Python mirror (deepfilternet_b200/model.py set_precision).
 * BF16x3 is ~2^-17 relative per product: 1e-7 .. 4e-7 RMS end to end against the fp32 oracle (bound 1e-4). */
int dfb_model_set_precision(dfb_model *m, int mode);
/* Chunk pipeline of dfb_enhance (device_chunks) / dfb_enhance_host (host_chunks): a signal of >= 64 * chunks frames is cut
 * into at least that many time chunks; lanes = 2 overlaps the encoder phase of chunk c + 1 with the decoder phase (the
 * recurrences) of chunk c on a second set of streams and a second workspace, lanes = 1 runs them back to back.
 * Defaults 0 (auto: 3 chunks up to 8 streams, 2 up to 256, else 1) / 4 / 2, from the measured sweep in profiles/.  The output
 * does not depend on these settings beyond fp32 reduction order (tests compare them). */
int dfb_model_set_chunking(dfb_model *m, int device_chunks, int host_chunks, int lanes);
/* init_df(post_filter=..., mask_only=...) (DeepFilterNet/df/enhance.py:101-187).  post_filter: Valin's post filter -- for
 * DeepFilterNet3 on the enhanced spectrum with beta = pf_beta (deepfilternet3.py:448-454), for DeepFilterNet2 on the ERB
 * gains with beta = 0.02 (Mask.pf, modules.py:234-245).  mask_only: the model as built with run_df = False
 * (checkpoint.py:32): no deep-filter stage, every bin takes the ERB gain. */
int dfb_model_set_options(dfb_model *m, int post_filter, float pf_beta, int mask_only);
/* Cap (bytes) of the per-call device workspace of dfb_enhance: the batch is processed in time chunks (and, for very
 * large batches, stream groups) that fit below it (default 64 GB, or DFB_MAX_WORKSPACE_MB in the environment at
 * dfb_model_create). */
int dfb_model_set_max_workspace(dfb_model *m, int64_t bytes);
/* Debug aid: steps > 0 with h_out == NULL arms clock64() phase stamps ([steps][8]) for the following
 * GRU launches; a second call with h_out != NULL copies the stamps of the last launch and disarms. */
int dfb_debug_gru_timing(dfb_model *m, int steps, long long *h_out);
/* Debug aid for parity tests: copies the named activation of the LAST forward pass on this handle
 * (e0,e1,e2,e3,c0,c1,emb_in,emb,dec_emb,d3,d2,d1,dfc) to the host; returns the element count
 * (or a negative dfb_status).  Valid until the next call on the handle. */
int64_t dfb_model_debug_fetch(dfb_model *m, const char *name, float *h_out, int64_t max_numel);
/* bytes of device workspace the model handle currently owns (grow-only arena) */
int64_t dfb_model_workspace_bytes(const dfb_model *m);

#ifdef __cplusplus
}
#endif
#endif /* DFB200_H */
