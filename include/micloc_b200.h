/*
 * micloc_b200.h -- C-ABI of the B200-native micloc SNN-localisation hot path.
 *
 * Drop-in boundary for the reference's Python entry points (all paths under
 * /root/reference):
 *   SNNBeamformer.apply_to_signal      micloc/snn_beamformer.py:283-370
 *   + callers' mean-power / argmax     paper_plots/target_snn_localization.py:462-464
 *   ZeroCrossingSpikeEncoder.evolve    micloc/spike_encoder.py:115-137
 *   Beamformer.apply_to_signal         micloc/beamformer.py:260-292
 *   Demo.spike_encoding / xylo_process micloc/xylo_snn_localization.py:315-377
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in signatures
 *     (`stream` is a cudaStream_t passed as void*; NULL = default stream).
 *   - *_dev pointers are device pointers on the context's device; *_host are
 *     host pointers.  Optional outputs may be NULL.
 *   - every function returns 0 on success or a negative micloc_status;
 *     micloc_last_error() gives the message of the calling thread's last failure.
 *   - launches are stream-ordered; no internal threads; one context per GPU.
 *   - ONE STREAM PER CONTEXT AT A TIME: a context owns scratch buffers and the fused kernel's work counter, so
 *     calls on the same context must be issued on one stream (or be ordered by the caller); use one context per
 *     concurrent stream.  micloc_snn_run_host orders itself behind the context's previous device-side call.
 *   - audio layout is the reference's: [B][T][M] row-major, mics interleaved
 *     (micloc/snn_beamformer.py:298 `T x num_mic`; micloc/record.py:54-75 wav frames).
 */
#ifndef MICLOC_B200_H_
#define MICLOC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MICLOC_VERSION 100 /* 0.1.0 */

typedef enum {
    MICLOC_OK = 0,
    MICLOC_ERR_SHAPE = -1,       /* reference raises ValueError (snn_beamformer.py:303-306) */
    MICLOC_ERR_CONFIG = -2,      /* reference raises ValueError/AssertionError at construction */
    MICLOC_ERR_CUDA = -3,
    MICLOC_ERR_UNSUPPORTED = -4,
    MICLOC_ERR_OVERFLOW = -5     /* reserved (RZCC overflow is reported per clip in `flags` and healed by the library) */
} micloc_status;

typedef enum { MICLOC_F32 = 0, MICLOC_I16 = 1, MICLOC_I32 = 2 /* streams only: wav frames of micloc/record.py */ } micloc_dtype;

typedef struct micloc_snn micloc_snn;   /* float SNN chain   */
typedef struct micloc_xylo micloc_xylo; /* Xylo integer chain */
typedef struct micloc_stream micloc_stream; /* stateful frames of one continuous recording */

/* ---- float SNN chain ------------------------------------------------------ */
typedef struct {
    int32_t num_mic;            /* M                                   geometry            */
    int32_t kernel_len;         /* K = int(fs*kernel_duration)         snn_beamformer.py:49 */
    const double *stht_kernel;  /* [K] fftshift(imag(hilbert(delta)))  snn_beamformer.py:50-53 */
    int32_t n_sections;         /* biquads of the band-pass (2)        snn_beamformer.py:68-72 */
    const double *sos;          /* [n_sections][6] b0 b1 b2 1 a1 a2                           */
    int32_t robust_width;       /* ceil(distance) >= 1                 snn_beamformer.py:75-80 */
    int32_t bipolar;            /* 0: +1 spikes only, 1: +1/-1         spike_encoder.py:130-135 */
    double neuron_decay;        /* a = exp(-1/(tau*fs))                snn_beamformer.py:342-361 */
    double neuron_scale;        /* c: h[n] = c*n*a^n, n < neuron_len                          */
    int32_t neuron_len;         /* L = effective_length                                       */
    int32_t num_doa;            /* G                                                          */
    const double *bf_mat;       /* [2M][G] row-major                   snn_beamformer.py:368  */
} micloc_snn_config;

/* Build a context on `device`.  Copies every array; the config may be freed. */
int micloc_snn_create(const micloc_snn_config *cfg, int device, micloc_snn **out);
int micloc_snn_destroy(micloc_snn *ctx);

/* Replace the beamforming matrix (bf_mat is a per-call argument in the reference). */
int micloc_snn_set_bf(micloc_snn *ctx, const double *bf_mat, int32_t num_doa);

/* Hot path, device buffers: audio -> spikes, power, DoA index.
 *   audio_dev  [B][T][M] float32 or int16
 *   spikes_dev [B][T][2M] int8 in {-1,0,+1}       (nullable)
 *   power_dev  [B][G] float32 = mean_t y[t,g]^2   (nullable)
 *   doa_dev    [B] int32 = argmax_g power (first maximum) (nullable)
 *   flags_dev  [B] int32, bit0 = RZCC overflow of the fused kernel's bounded streaming encoder (a cluster of more
 *              than 8 candidates or a flat top of more than 16 exact zeros, e.g. digital silence): the clip's results
 *              are then not the reference's until micloc_snn_refine has redone it (nullable)
 * `fused` != 0 runs the single fused kernel, 0 the staged kernels (same results; they heal overflowed clips
 * themselves with the unbounded float64 encoder, at the price of one stream synchronisation). */
int micloc_snn_run(micloc_snn *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T,
                   int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, int32_t *flags_dev,
                   int fused, void *stream);

/* Synchronising companion of the fused micloc_snn_run (which stays stream-ordered): reads flags_dev back, reruns every
 * clip with bit0 set through the staged kernels + the unbounded float64 RZCC encoder (spike_encoder.py:115-137 has no
 * cluster bound), overwrites that clip's rows of the (nullable) outputs and clears the bit.  Same arguments as the run
 * it follows; n_refined (nullable) = clips redone.  micloc_snn_run_host does this on its own. */
int micloc_snn_refine(micloc_snn *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T,
                      int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, int32_t *flags_dev,
                      int64_t *n_refined, void *stream);
/* clips this context has redone with the unbounded encoder since it was created (all entry points) */
int64_t micloc_snn_refined_count(micloc_snn *ctx);

/* Same with per-stage debug taps (all nullable, all device):
 *   q_dev [B][T][M] f32 (STHT quadrature), z_dev [B][T][2M] f32 (post band-pass,
 *   hstack(real, imag)), vmem_dev [B][T][2M] f32, y_dev [B][T][G] f32 (dense
 *   beamformed signal = apply_to_signal's return value). Always staged. */
int micloc_snn_run_taps(micloc_snn *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T,
                        float *q_dev, float *z_dev, int8_t *spikes_dev, float *vmem_dev,
                        float *y_dev, float *power_dev, int32_t *doa_dev, int32_t *flags_dev,
                        void *stream);

/* End-to-end with HOST buffers: chunks the batch, copies H2D from pinned staging,
 * runs the hot path, copies results D2H, redoes RZCC-overflowed clips (micloc_snn_refine).  Outputs nullable as above. */
int micloc_snn_run_host(micloc_snn *ctx, const void *audio_host, int dtype, int64_t B, int64_t T,
                        int8_t *spikes_host, float *power_host, int32_t *doa_host,
                        int32_t *flags_host, int fused);

/* Design-time helper (SNNBeamformer.design_from_template, snn_beamformer.py:158-191):
 * front end + neuron filter, then gram_dev[b][i][j] = sum_{t >= t_start} v[t][i] v[t][j]
 * (float64, [B][2M][2M]); the caller divides by T - t_start and runs the SVD. */
int micloc_snn_gram(micloc_snn *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T,
                    int64_t t_start, double *gram_dev, void *stream);

/* hist_dev[g] += #{b : doa_dev[b] == g}; hist_dev is int64[G] on `device`, accumulated
 * (zero it first).  The per-GPU histograms are what the Monte-Carlo driver sums across
 * GPUs (paper_plots/target_snn_localization.py:447-467 keeps per-trial DoA errors). */
int micloc_doa_histogram(const int32_t *doa_dev, int64_t B, int32_t G, int64_t *hist_dev, int device,
                         void *stream);

/* ---- stateful frames + Envelope tracker (SURVEY.md 8f) -------------------------- */
/* The live loop of micloc/localization_demo_snn.py:125-193 records a frame, runs the chain from ZERO state and
 * repeats.  A stream carries the state instead (STHT history, band-pass, RZCC running sum and open clusters, neuron,
 * envelope): N pushed frames give exactly what one clip of their concatenation gives.  By nature of a stream the
 * in-phase branch is the causal delay x[t - K/2] (np.roll's wrap-around needs the clip's end; identical whenever the
 * last K/2 samples of the clip are zero) and results lag the input by micloc_snn_stream_latency() samples (the RZCC
 * distance rule decides a spike only that much later).
 *   frame_dev  [n][in_channels] interleaved float32 / int16 / int32 PCM (the recorder's `T x 8` int32 wav frames with
 *              in_channels = 8: channels >= num_mic are dropped, localization_demo_snn.py:145); n <= max_frame_len
 *   outputs describe the n_out samples that became final with this call (all nullable, device pointers):
 *     spikes_dev [n_out][2M] int8;  power_dev [G] = mean over those samples of y^2, doa_dev [1] its first argmax;
 *     env_dev [n_out][G] = Envelope(rise_time, fall_time, fs).evolve(y) continued across calls (micloc/utils.py:15-81),
 *     doa_t_dev [n_out] = per-sample argmax of the envelope (tests/test_snn_hilbert_localization.py:284-293)
 *   buffers must hold max_frame_len + latency rows.  micloc_snn_stream_flush ends the stream like a clip end and
 *   returns the remaining samples (+ the RZCC overflow flag); after it only micloc_snn_stream_reset is allowed.
 * The stream uses its parent context's constants: destroy it before the context, re-create it after micloc_snn_set_bf. */
int micloc_snn_stream_create(micloc_snn *ctx, int64_t max_frame_len, double fs, double rise_time, double fall_time,
                             micloc_stream **out);
int micloc_snn_stream_destroy(micloc_stream *s);
int micloc_snn_stream_reset(micloc_stream *s, void *stream);
int micloc_snn_stream_latency(micloc_stream *s);
int micloc_snn_stream_push(micloc_stream *s, const void *frame_dev, int dtype, int64_t n, int32_t in_channels,
                           int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev, int32_t *doa_t_dev,
                           int64_t *n_out, void *stream);
int micloc_snn_stream_flush(micloc_stream *s, int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev,
                            int32_t *doa_t_dev, int64_t *n_out, int32_t *flags_host, void *stream);

/* ---- stream batches: many live recordings, one push per frame tick ---------------------------------------------- */
/* A stream batch holds S independent slots on one context; each slot is one continuous recording with the semantics
 * of a micloc_stream above (N pushed frames = one clip of their concatenation, causal in-phase delay, results lag the
 * input by micloc_snn_streams_latency() = D samples).  A single micloc_stream is a batch of one slot.
 *   - Slots are independent: reset and flush act on the listed slots only (slots_host [n_slots], NULL = every slot).
 *     A flushed slot ignores its rows of later pushes (n_out = 0, state untouched) until it is reset, so one slot can be
 *     recycled while the others keep running; a push after every slot was flushed is no error (all n_out = 0).
 *   - Positions are per slot: a slot reset mid-run restarts at sample 0 while the others go on.  n_out_host[s] is the
 *     number of samples of slot s that became final with this call (N_s - D - F_s for a push, the rest at a flush); the
 *     library computes it on the host, without a device synchronisation.
 *   - push: frames_dev [S][n][in_channels] float32 / int16 / int32 (one frame of n samples per slot, the same n for all
 *     slots, 1 <= n <= max_frame_len; channels >= num_mic are dropped).  Outputs, all nullable device pointers:
 *       spikes_dev [S][n + D][2M] int8, power_dev [S][G] (mean over the slot's final samples of y^2), doa_dev [S] (its
 *       first argmax), env_dev [S][n + D][G] (Envelope continued across calls), doa_t_dev [S][n + D] (per-sample argmax
 *       of the envelope).  Slot s fills its first n_out_host[s] rows; the other rows, and power / doa of a slot with
 *       n_out = 0, are NOT written.
 *   - flush closes the listed slots like a clip end; outputs as in push with [S][max_frame_len + D] rows;
 *     flags_host [S] (nullable, host): bit 0 = RZCC overflow anywhere in that slot's recording (synchronises).
 *   - reset and flush synchronise `stream` (reset with slots_host NULL too); a push does not synchronise.  This holds
 *     for every stream batch kind: micloc_snn_streams_*, micloc_snn_mb_streams_* and micloc_xylo_streams_*.
 * Kernel launches per push, whatever S: 5 (frame assembly, STHT, band-pass + RZCC + neuron, Gram, power), of which Gram
 * and power only when power_dev or doa_dev is given; +2 (dense y, envelope) when env_dev or doa_t_dev is given, +1
 * (argmax) when doa_t_dev is given.  The envelope scratch (S (n + D) G floats, twice when env_dev is NULL) is allocated
 * on the first call that asks for it.  1 <= num_streams <= 65535.  Same lifetime rules as micloc_stream. */
typedef struct micloc_stream_batch micloc_stream_batch;
int micloc_snn_streams_create(micloc_snn *ctx, int32_t num_streams, int64_t max_frame_len, double fs,
                              double rise_time, double fall_time, micloc_stream_batch **out);
int micloc_snn_streams_destroy(micloc_stream_batch *sb);
int micloc_snn_streams_latency(micloc_stream_batch *sb);
int micloc_snn_streams_reset(micloc_stream_batch *sb, const int32_t *slots_host, int32_t n_slots, void *stream);
int micloc_snn_streams_push(micloc_stream_batch *sb, const void *frames_dev, int dtype, int64_t n, int32_t in_channels,
                            int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev, int32_t *doa_t_dev,
                            int64_t *n_out_host, void *stream);
int micloc_snn_streams_flush(micloc_stream_batch *sb, const int32_t *slots_host, int32_t n_slots,
                             int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev, int32_t *doa_t_dev,
                             int64_t *n_out_host, int32_t *flags_host, void *stream);

/* ---- multi-band stream batches: the live localiser, continuous, over many arrays -------------------------------- */
/* The multi-band localiser of micloc/localization_demo_snn.py:125-193 (filterbank, one chain per band, power summed
 * over the bands, estimators) with the state carried across pushes.  A batch holds S independent slots over F contexts
 * ctxs[F] (one per band, 1 <= F <= 8, same device, M and G) and the F band-pass filters of the filterbank
 * (sos [F][n_sections][6], host; the sections of micloc_filterbank).
 *   - Concatenation rule: N pushed frames give, for every band f, what micloc_filterbank of the concatenation followed
 *     by band f's stream batch gives.  The filterbank state carries over, so band f's chain input is bit for bit the
 *     filterbank output of the whole recording; the chain has the semantics of a stream batch slot.
 *   - One latency for all bands: D = micloc_snn_mb_streams_latency() = max_f rzcc_lag(w_f).  Every band finalises
 *     the same samples [F_s, N_s - D) of slot s in a push, and the rest at a flush, so n_out_host[s] is one number per
 *     slot (computed on the host, no synchronisation).  A band with a smaller lag finalises later than it could; its
 *     spikes are unchanged by that.
 *   - push: frames_dev [S][n][in_channels] float32 / int16 / int32, as for micloc_snn_streams_push.  Outputs, all
 *     nullable device pointers, over the n_out_host[s] final samples of slot s:
 *       spikes_dev [F][S][n + D][2M] int8;  power_dev [F][S][G] float32 (per band, mean of y^2);  power_grid_dev [S][G]
 *       float32 (sum over the bands in band order, float64, as micloc_power_fuse);  doa_dev [S] (first argmax);
 *       periodic_ml_dev / trimmed_ml_dev [S] float64 (the estimators of micloc_power_fuse; they need doa_list);
 *       flags_dev [S]: bit 0 = RZCC overflow so far in any band of the slot, bit 1 = the trimmed estimator's
 *       IndexError case (estimate NaN).  A slot with n_out = 0 (a first push shorter than D, a flushed slot) gets none
 *       of these written.
 *       sumsq_dev [S] float64 = sum of x^2 over the kept channels of the frame just pushed, every slot (activity
 *       detection, localization_demo_snn.py:151-163): float32 partials of 256 samples added in float64, so it equals
 *       micloc_filterbank's sumsq of that frame up to the order in which the microphones are added.  The gate looks
 *       at the newest frame, D samples ahead of the samples the power describes.
 *   - flush closes the listed slots (slots_host [n_slots], NULL = every slot) like a clip end; outputs as in push with
 *     [max_frame_len + D] rows; flags_host [S] (nullable, host): bit 0 = RZCC overflow anywhere in that slot's
 *     recording, any band.  reset / flush / flushed slots and synchronisation behave as in micloc_snn_streams_*;
 *     reset also restarts the filterbank of the listed slots from zero state.
 * Kernel launches per push, whatever S: 4 F + 2 (filterbank + frame assembly; per band STHT, band-pass + RZCC +
 * neuron, Gram, power; the sum over bands with its estimators), 2 F + 1 when no power, fused output or flags are
 * requested.  1 <= num_streams <= 65535; doa_list [G] (host, nullable: no ML estimators).  The contexts' constants
 * are used: destroy the batch before any of its contexts, re-create it after micloc_snn_set_bf. */
typedef struct micloc_mb_streams micloc_mb_streams;
int micloc_snn_mb_streams_create(micloc_snn *const *ctxs, int32_t F, int32_t n_sections, const double *sos,
                                 const double *doa_list, int32_t num_streams, int64_t max_frame_len,
                                 micloc_mb_streams **out);
int micloc_snn_mb_streams_destroy(micloc_mb_streams *mb);
int micloc_snn_mb_streams_latency(micloc_mb_streams *mb);
int micloc_snn_mb_streams_reset(micloc_mb_streams *mb, const int32_t *slots_host, int32_t n_slots, void *stream);
int micloc_snn_mb_streams_push(micloc_mb_streams *mb, const void *frames_dev, int dtype, int64_t n, int32_t in_channels,
                               int8_t *spikes_dev, float *power_dev, float *power_grid_dev, int32_t *doa_dev,
                               double *periodic_ml_dev, double *trimmed_ml_dev, double *sumsq_dev, int32_t *flags_dev,
                               int64_t *n_out_host, void *stream);
int micloc_snn_mb_streams_flush(micloc_mb_streams *mb, const int32_t *slots_host, int32_t n_slots, int8_t *spikes_dev,
                                float *power_dev, float *power_grid_dev, int32_t *doa_dev, double *periodic_ml_dev,
                                double *trimmed_ml_dev, int32_t *flags_dev, int64_t *n_out_host, int32_t *flags_host,
                                void *stream);

/* Envelope.evolve on a whole device array x_dev [T][C] float32 (fresh state) -> env_dev [T][C]; argmax_dev [T]
 * (nullable) = first argmax over the C channels of every row. */
int micloc_envelope(const float *x_dev, int64_t T, int32_t C, double fs, double rise_time, double fall_time,
                    float *env_dev, int32_t *argmax_dev, int device, void *stream);

/* ---- multi-band localiser: filterbank, power summed over bands, estimators (SURVEY.md 8f) ---- */
/* ButterworthFilterbank.evolve (micloc/filterbank.py:25-46) on raw frames: F band-pass filters given as SOS sections
 * (sos [F][n_sections][6], host) on every microphone channel, zero state.
 *   audio_dev [B][T][in_channels] float32 / int16 / int32 (wav frames: channels >= M are dropped,
 *             micloc/localization_demo_snn.py:145);  out_dev [F][B][T][M] float32: band f is the [B][T][M] batch a
 *             per-band context's micloc_snn_run takes;  sumsq_dev [B] float64 (nullable) = sum of x^2 over the kept
 *             channels of a clip (activity detection, localization_demo_snn.py:151-163). */
int micloc_filterbank(const void *audio_dev, int dtype, int64_t B, int64_t T, int32_t in_channels, int32_t M,
                      int32_t F, int32_t n_sections, const double *sos, float *out_dev, double *sumsq_dev,
                      int device, void *stream);
/* power_grid = sum over bands (micloc/localization_demo_snn.py:172-189) + the estimators of
 * micloc/xylo_snn_localization.py:400-444 on it:
 *   power_dev [F][B][G] float32 (the per-band power outputs of micloc_snn_run);  doa_list_dev [G] float64 (nullable
 *   when no ML estimate is wanted);  outputs, all nullable: power_sum_dev [B][G] float32, doa_dev [B] first argmax
 *   ("peak"), periodic_ml_dev [B] float64 = angle(mean(p e^{j doa})), trimmed_ml_dev [B] float64 = the same over the
 *   reference's window around the peak; where the reference's indexing raises IndexError (peak index > 3G/4) the
 *   estimate is NaN and flags_dev [B] gets bit 1. */
int micloc_power_fuse(const float *power_dev, int32_t F, int64_t B, int32_t G, const double *doa_list_dev,
                      float *power_sum_dev, int32_t *doa_dev, double *periodic_ml_dev, double *trimmed_ml_dev,
                      int32_t *flags_dev, int device, void *stream);

/* ---- Monte-Carlo input synthesis (SURVEY.md 8f) ------------------------------ */
/* Synthetic array clips on the device, as the reference builds them on the host:
 *   mode 0  SNNBeamformer.apply_to_template (micloc/snn_beamformer.py:243-275): per-microphone delays
 *           -r cos(theta_m - doa)/c minus their minimum, x[t][m] = interp(t - delay_m) clamped at t_min
 *   mode 1  signal_multiple_targets (paper_plots/multiple_targets_snn.py:87-159): x[t][m] = sum_k gain_k
 *           interp(t + delay_{k,m}), un-normalised delays, np.interp's clamping at both ends
 * followed by AWGN of sigma = sqrt(mean(x^2)) / sqrt(snr) per clip (snn_beamformer.py:270-275).
 *   source_kind 0: table src_dev [S][clip_len] f32 on the clip's own sample grid (chirp, filtered noise, ...);
 *                  clip b uses row src_index_dev[b] (row 0 when src_index_dev is NULL)
 *   source_kind 1: sine of sine_freq sampled at fs (paper_plots/target_snn_localization.py:439-441)
 *   doa_dev [B][n_targets] f64 rad; gain_dev [B][n_targets] f32 (NULL = 1); snr_lin_dev [B] f32 linear SNR (NULL = no noise)
 *   out_f32_dev [B][clip_len][num_mic] always written; out_i16_dev (nullable) = round(x * int16_peak / max|x|) per clip
 *   scratch_dev: B * 12 bytes (8-byte aligned).  B <= 65535 per call.  Noise: Philox4x32-10, `seed`. */
typedef struct {
    int32_t num_mic;
    const double *r_vec;        /* [num_mic] radius of every microphone   array_geometry.py:32-37 */
    const double *theta_vec;    /* [num_mic] angle of every microphone                            */
    double fs;
    double speed;               /* 340 m/s                                array_geometry.py:14    */
    int64_t clip_len;           /* T */
    int32_t n_targets;
    int32_t mode;               /* 0 apply_to_template, 1 signal_multiple_targets */
    int32_t source_kind;        /* 0 table, 1 sine */
    double sine_freq;
} micloc_synth_config;

int micloc_synth_clips(const micloc_synth_config *cfg, int64_t B, const float *src_dev,
                       const int32_t *src_index_dev, const double *doa_dev, const float *gain_dev,
                       const float *snr_lin_dev, uint64_t seed, float *out_f32_dev, int16_t *out_i16_dev,
                       float int16_peak, double *scratch_dev, int device, void *stream);

/* ---- stand-alone stages ---------------------------------------------------- */
/* ZeroCrossingSpikeEncoder.evolve on arbitrary float64 input, exact find_peaks
 * semantics (unbounded clusters).  sig_dev [B][T][C] f64 -> spikes_dev [B][T][C] int8. */
int micloc_rzcc_encode_f64(const double *sig_dev, int64_t B, int64_t T, int32_t C,
                           int32_t robust_width, int32_t bipolar, int8_t *spikes_dev,
                           int device, void *stream);

/* Beamformer.apply_to_signal: STHT + band-pass + complex projection.
 *   bf_re/bf_im [M][G] (host, float64); y_dev [B][T][G][2] f32 (re, im interleaved),
 *   power_dev [B][G] = mean_t |y|^2 (nullable), doa_dev [B] (nullable). */
int micloc_hilbert_beamform(micloc_snn *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T,
                            const double *bf_re_host, const double *bf_im_host, int32_t G,
                            float *y_dev, float *power_dev, int32_t *doa_dev, void *stream);

/* Beamformer at batch scale.  The complex steering matrix of Beamformer.apply_to_signal, bf = bf_re + i bf_im,
 * [M][G] host float64, kept by the context beside (not instead of) the SNN bf_mat: its own G, its own buffers;
 * micloc_snn_set_bf is unaffected.  Waits for the device (calls in flight may read the old matrix). */
int micloc_hilbert_set_bf(micloc_snn *ctx, const double *bf_re_host, const double *bf_im_host, int32_t G);
/* s_t = analytic signal of clip b: band-passed (bandpass != 0, beamformer.py:281-287) or roll(x, K/2) + j STHT(x)
 * (bandpass == 0, the form design_from_template uses).  All outputs nullable, device:
 *   z_dev     [B][T][2M] f32   s_t as (real | imag), debug tap;
 *   cov_dev   [B][M][M][2] f64 sum_{t >= t_start} conj(s_t[i]) s_t[j]  (re, im);
 *   power_dev [B][G] f32       mean_{t >= t_start} |sum_m s_t[m] conj(bf[m][g])|^2, as (u^T G u + v^T G v) / (T - t_start)
 *                              of the real Gram matrix G of (real | imag), u = [Re bf; Im bf], v = [-Im bf; Re bf];
 *   doa_dev   [B] int32        first argmax of power.
 * Never forms the dense T x G output.  Stream-ordered (no synchronisation), any B (chunks of <= 65535 clips whose
 * scratch stays within ~1 GB), f32 / i16 audio, 0 <= t_start < T.  Kernels per chunk: 3 for M <= 8 (STHT, band-pass +
 * float64 Gram on chip, Gram reduce + cov + power + argmax), 4 for M > 8 (STHT, band-pass -> z, tiled float32 Gram over
 * 1024-sample slabs, the same last kernel).  power / doa before micloc_hilbert_set_bf -> MICLOC_ERR_CONFIG. */
int micloc_hilbert_localize(micloc_snn *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T, int64_t t_start,
                            int bandpass, float *z_dev, double *cov_dev, float *power_dev, int32_t *doa_dev,
                            void *stream);

/* ---- design_from_template on the device ----------------------------------- */
/* The template of SNNBeamformer / Beamformer.design_from_template after its resampling onto the fs grid (the host
 * keeps that O(T) np.interp).  num_mic <= 64 (MICLOC_ERR_UNSUPPORTED beyond), T >= 2. */
typedef struct {
    int32_t num_mic;
    const double *r_vec, *theta_vec;    /* [num_mic] host, float64 (array_geometry.py) */
    double speed;
    int64_t T;
    const double *time_dev, *sig_dev;   /* [T] device, float64: the fs grid and the template on it */
} micloc_design_template;
/* clips_dev [G][T][M] f32: the template delayed for every doa_dev [G] (device, f64 rad), exactly as
 * SNNBeamformer._delayed_template and the Hilbert design loop compute it (float64 delays normalised to start at 0,
 * td clamped below at time[0], np.interp's formula, one rounding to float32).  1 launch per 65535 DoAs. */
int micloc_design_templates(const micloc_design_template *tp, const double *doa_dev, int64_t G, float *clips_dev,
                            int device, void *stream);
/* SNNBeamformer.design_from_template on the device, mode 0 (unipolar) or 1 (bipolar) from the context's encoder.
 * C_g = Gram of the membrane signals from t_start = T / 4 on, / (T - t_start), of the context's chain (built for
 * the template's own time grid).  bf_dev [2M][G] f64 (the micloc_snn_config.bf_mat layout); cov_dev [G][2M][2M] f64,
 * nullable.  Per chunk of DoAs whose clips and front-end scratch stay within ~1 GB: templates, the staged front end
 * of micloc_snn_gram (STHT, band-pass + RZCC, neuron filter) and the Gram matrix; per call: 1 scale + 1 solver launch.
 * The front end reads its overflow flags back once per chunk (as micloc_snn_gram does), which synchronises the
 * stream; nothing else does. */
int micloc_snn_design(micloc_snn *ctx, const micloc_design_template *tp, const double *doa_dev, int64_t G,
                      double *bf_dev, double *cov_dev, void *stream);
/* Beamformer.design_from_template on the device: cov_g = micloc_hilbert_localize's cov (bandpass = 0,
 * t_start = min(K, T / 2)) / (T - t_start); mode 2, or mode 3 with interference_removal.  bf_dev [M][G][2] f64
 * (re, im); cov_dev [G][M][M][2] f64, nullable.  Per chunk of DoAs (clips within ~0.5 GB): templates + the 3 or 4
 * launches of micloc_hilbert_localize; per call: 1 scale + the solver's launches.  Stream-ordered, no
 * synchronisation. */
int micloc_hilbert_design(micloc_snn *ctx, const micloc_design_template *tp, const double *doa_dev, int64_t G,
                          int interference_removal, double *bf_dev, double *cov_dev, void *stream);
/* The batched float64 solver alone (cyclic Jacobi, one CTA per matrix, n = 2M <= 128), on device inputs:
 *   mode 0 (SNN unipolar): cov [G][2M][2M] real PSD -> _find_dc_removed_sing_vec(C, rel_prec = 1e-8): theta = U^T 1,
 *          bisection between the two largest singular values, U theta / (D - root) normalised; value = root.
 *          Independent of the eigenvectors' signs, so it needs no phase rule.
 *   mode 1 (SNN bipolar):  the same cov -> top left singular vector u of (C11 + C22)/2 + i (C12 + C21^T)/2, as the
 *          column [Re u; Im u]; value = its singular value.
 *   mode 2 (Hilbert):      cov [G][M][M][2] Hermitian PSD -> top eigenvector; value = its eigenvalue.
 *   mode 3 (Hilbert, interference removal): the same cov -> C_sum = sum_g C_g + diag(mean(diag(C_sum))) / 10, then
 *          the top generalised eigenvector of (C_g, C_sum - C_g) (Cholesky of C_sum - C_g), normalised;
 *          value = the generalised eigenvalue.
 * bf_dev: [2M][G] for modes 0 and 1, [M][G][2] for modes 2 and 3.  value_dev [G], nullable.
 * Phase rule (modes 1-3): every complex column is rotated so that its entry of largest modulus (the first such index)
 * is real and positive.  numpy's SVD leaves an arbitrary LAPACK phase, so device and host columns agree up to a
 * phase.  The SNN bipolar chain is not exactly invariant under a phase rotation of [Re u; Im u]: device- and
 * host-designed bipolar matrices can give slightly different SNN power.
 * Launches: 1 (modes 0-2) or 3 (mode 3: C_sum, Cholesky + whitening, solver).  Stream-ordered, no synchronisation.
 * M > 64 -> MICLOC_ERR_UNSUPPORTED; G < 1 or a null pointer -> MICLOC_ERR_SHAPE; a mode outside 0..3 ->
 * MICLOC_ERR_CONFIG. */
int micloc_design_vectors(int mode, const double *cov_dev, int32_t M, int64_t G, double *bf_dev, double *value_dev,
                          int device, void *stream);

/* ---- Xylo integer chain ---------------------------------------------------- */
/* Network constants are what rockpool's mapper + global_quantize + config_from_specification
 * hand to XyloSim (micloc/xylo_snn_localization.py:268-290); the host package restates that
 * quantisation (haghighatshoarmuir2024_b200/xylo_snn_localization.py: quantize_network). */
typedef struct {
    int32_t num_mic;            /* M                                                      */
    int32_t kernel_len;         /* K                                                      */
    const double *stht_kernel;  /* [K]                       xylo_snn_localization.py:327  */
    int32_t num_bands;          /* F                         xylo_snn_localization.py:148-152 */
    int32_t n_sections;         /* biquads per band filter (order 1 -> 1, order 2 -> 2): float32 front end */
    const double *sos;          /* [F][n_sections][6]        filterbank.py:79-81           */
    int32_t n_ba;               /* len(b) == len(a) per band (2*order + 1): float64 exact front end; 0 = none */
    const double *ba_b;         /* [F][n_ba]                 filterbank.py:79-81 (output="ba") */
    const double *ba_a;         /* [F][n_ba], a[0] == 1                                    */
    int32_t robust_width;       /* band-0 width for all bands  xylo_snn_localization.py:346 */
    int32_t bipolar;            /* 1: inputs = [pos | neg]   xylo_snn_localization.py:350-354 */
    int32_t num_hidden;         /* N = G*F hidden neurons                                  */
    int32_t num_doa;            /* G                                                       */
    const int8_t *w_in;         /* [N_in][N] int8, N_in = 2M*F*(bipolar?2:1)               */
    const int8_t *w_rec;        /* [N][N] int8 or NULL; must be all-zero on the device     */
    const int16_t *threshold;   /* [N] >= 1                                                */
    const int8_t *dash_syn;     /* [N] bit-shift decay of I_syn                            */
    const int8_t *dash_mem;     /* [N] bit-shift decay of V_mem                            */
    const int16_t *bias;        /* [N] or NULL                                             */
    int32_t weight_shift_in;    /* left shift applied to input weights (0 in the reference) */
    int32_t weight_shift_rec;   /* left shift applied to recurrent weights                 */
    int32_t max_spikes;         /* spikes per hidden neuron per step (31)                  */
} micloc_xylo_config;

int micloc_xylo_create(const micloc_xylo_config *cfg, int device, micloc_xylo **out);
int micloc_xylo_destroy(micloc_xylo *ctx);

/* audio -> input spikes (Demo.spike_encoding) -> hidden spike counts -> DoA.
 *   exact != 0: float64 front end with scipy's operation order (spikes bit-identical to the
 *               reference's numpy/scipy path); 0: float32 front end (float-path tolerance).
 *   spikes_in_dev [B][T][N_in] int8 in {0,1}      (nullable)
 *   raster_dev    [B][T][N] uint8 hidden spikes per step = rec["Spikes"] (nullable)
 *   counts_dev    [B][N] int32 = sum_t raster     (nullable)
 *   doa_dev       [B] int32: first argmax over g of the band-summed counts (nullable)
 *   doa_peak_dev  [B] int32: utils.find_peak_location(counts, peak_win) (nullable; win odd)
 *   flags_dev     [B] int32, bit0 = RZCC cluster overflow of the float32 front end (nullable) */
int micloc_xylo_run(micloc_xylo *ctx, const void *audio_dev, int dtype, int64_t B, int64_t T, int exact,
                    int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev,
                    int32_t *doa_dev, int32_t *doa_peak_dev, int32_t peak_win,
                    int32_t *flags_dev, void *stream);

/* Integer network only (Demo.xylo_process): spikes_in_dev [B][T][N_in] int8 {0,1}. */
int micloc_xylo_process(micloc_xylo *ctx, const int8_t *spikes_in_dev, int64_t B, int64_t T,
                        uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                        int32_t *doa_peak_dev, int32_t peak_win, void *stream);

/* ---- Xylo stream batches: many live recordings through the bit-exact integer chain ------------------------------ */
/* A Xylo stream batch holds S independent slots (1 <= S <= 65535) on one micloc_xylo context; each slot is one
 * continuous recording through the EXACT (float64) front end and the integer network.
 *   - Concatenation rule: N pushed frames plus a flush give, for every slot, what micloc_xylo_run(exact = 1) gives on
 *     one clip of their concatenation -- signed input spikes, hidden raster and (summed over the calls) hidden spike
 *     counts, bit for bit -- with the usual stream differences: the in-phase branch is the causal delay x[t - K/2]
 *     (zeros before the slot starts; identical to np.roll whenever the clip's last K/2 samples are zero), and results
 *     lag the input by D = micloc_xylo_streams_latency() samples.  Band-filter delays, running sum, flat-top starts,
 *     open candidate clusters (kF64Cluster = 32 per polarity) and I_syn / V_mem carry over.  The sample path is float64
 *     from the frame on, so int32 wav samples beyond 2^24 are taken exactly.
 *   - Latency: D = (kF64Cluster - 1)(w - 1) + w + 64 + 32 with w = robust_width: a cluster of up to 32 candidates
 *     spaced by at most w - 1, the distance w that closes it, the 64-sample tile of the chain kernel and a flat-top
 *     allowance of 64 samples (a candidate sits at the midpoint of its flat top).  At the end of a push, every spike at
 *     a position below N_s - D has been emitted, or the slot's flags bit 0 is set: the kernel checks the earliest
 *     position a spike can still take (the first candidate of an open cluster, the midpoint of an open flat top or
 *     bottom) against N_s - D, and sets the bit as well when a cluster overflows its 32 candidates (where the one-shot
 *     path redoes the clip with the unbounded kernels).  Bit 0 stays set until the slot is reset.
 *     INVARIANT: bit 0 clear => the slot's results are the clip's bits.  A push never synchronises nor redoes anything.
 *   - Slots, positions, flushed slots, n_out_host and unwritten rows as in micloc_snn_streams_*: slots_host [n_slots]
 *     (NULL = every slot); a slot reset mid-run restarts at 0 while the others go on; a flushed slot ignores later pushes
 *     (n_out = 0, state untouched) until it is reset; n_out_host[s] (host, computed without a synchronisation) is the
 *     number of samples of slot s that became final with this call; synchronisation as there; a push that would take
 *     a slot's position to 2^31 - 4096 samples or beyond is refused.
 *   - push: frames_dev [S][n][in_channels] float32 / int16 / int32, 1 <= n <= max_frame_len (channels >= num_mic are
 *     dropped).  Outputs, all nullable device pointers, over the n_out_host[s] final samples of slot s:
 *       spikes_in_dev [S][n + D][N_in] int8 {0,1} (Demo.spike_encoding's layout);  raster_dev [S][n + D][N] uint8;
 *       counts_dev [S][N] int32 hidden spikes over those samples;  doa_dev / doa_peak_dev [S] int32: first argmax of the
 *       band-summed counts / utils.find_peak_location of them (peak_win odd, at most G / 2);  flags_dev [S] int32 bit 0
 *       as above.  Rows past n_out_host[s], and counts / doa / doa_peak of a slot with n_out = 0, are NOT written.
 *   - flush closes the listed slots like a clip end; outputs as in push with [S][max_frame_len + D] rows; flags_host [S]
 *     (nullable, host, synchronises) = the flags after the flush.
 *   - create: MICLOC_ERR_CONFIG without the b/a band filters (n_ba == 0); MICLOC_ERR_UNSUPPORTED where the fast exact
 *     front end does not apply (a Hilbert kernel with every other tap zero and K a multiple of 8, n_ba <= 5,
 *     2 M F <= 64, M <= 32).
 * Kernel launches per push, whatever S: 4 (frame assembly, STHT of the frame rows, band filters + cumsum + find_peaks,
 * integer network), +1 (DoA) when doa_dev or doa_peak_dev is given, +1 (pos / neg split) when spikes_in_dev is given.
 * Device memory: 3 S (K - 1 + max_frame_len) M float64 (two assembly buffers and the STHT), S 2 M F x 856 bytes of chain
 * state, S N x 8 bytes of neuron state, S 2 M F (R + max_frame_len + D) bytes of spike ring and raster (R = the
 * power of two >= max_frame_len + D, at least 64), S N x 4 bytes of counts.  The batch uses its context's constants:
 * destroy it before the context. */
typedef struct micloc_xylo_streams micloc_xylo_streams;
int micloc_xylo_streams_create(micloc_xylo *ctx, int32_t num_streams, int64_t max_frame_len, micloc_xylo_streams **out);
int micloc_xylo_streams_destroy(micloc_xylo_streams *xs);
int micloc_xylo_streams_latency(micloc_xylo_streams *xs);
int micloc_xylo_streams_reset(micloc_xylo_streams *xs, const int32_t *slots_host, int32_t n_slots, void *stream);
int micloc_xylo_streams_push(micloc_xylo_streams *xs, const void *frames_dev, int dtype, int64_t n, int32_t in_channels,
                             int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                             int32_t *doa_peak_dev, int32_t peak_win, int32_t *flags_dev, int64_t *n_out_host, void *stream);
int micloc_xylo_streams_flush(micloc_xylo_streams *xs, const int32_t *slots_host, int32_t n_slots,
                              int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                              int32_t *doa_peak_dev, int32_t peak_win, int32_t *flags_dev, int64_t *n_out_host,
                              int32_t *flags_host, void *stream);

/* ---- Hilbert stream batches: the Hilbert beamformer over many live recordings ---------------------------------- */
/* The live Hilbert beamformer (the baseline of every SNN localiser) with its state carried across pushes.  A batch
 * holds S independent slots (1 <= S <= 65535) over F contexts ctxs[F] (one per band, 1 <= F <= 8, same device, same M),
 * each with its Hilbert steering matrix set (micloc_hilbert_set_bf) and the same hG; otherwise create returns
 * MICLOC_ERR_CONFIG (no steering matrix, a device or F out of range, a NULL context) or MICLOC_ERR_SHAPE (M or G differ).
 *   - sos [F][n_sections][6] (host) != NULL: a Butterworth filterbank (the sections of micloc_filterbank) runs in front
 *     of the band chains, its state carried: the live multi-band localiser.  sos == NULL: F must be 1 (MICLOC_ERR_CONFIG
 *     otherwise) and the raw frame goes straight into the band's chain, Beamformer.apply_to_signal's own band-pass
 *     chain made continuous.
 *   - Band f's chain is micloc_hilbert_localize's with bandpass = 1: STHT, the context's band-pass, the Gram matrix of
 *     the analytic signal.  The batch COPIES every band's complex steering matrix at create time (a later
 *     micloc_hilbert_set_bf leaves the batch as it was); the STHT taps and the band-pass sections are the context's,
 *     fixed for its lifetime: destroy the batch before its contexts.
 *   - Concatenation rule: N pushed frames give band f's analytic signal z of the whole recording bit for bit: with a
 *     filterbank, micloc_filterbank of the concatenation followed by band f's chain; without, the chain on the
 *     concatenation itself.  As in every stream, the in-phase branch is the causal delay x[t - K/2] (zeros before the
 *     slot starts; identical to np.roll whenever the recording's last K/2 samples are zero).  On wide arrays (M > 8) the
 *     STHT runs on the tensor cores, which scale each 256-sample tile by its own largest magnitude: q, and with it z, then
 *     agrees with the one-shot chain to the tensor-core STHT's tolerance (5e-6 of max |z| measured) rather than bit
 *     for bit
 *     (bit for bit again with MICLOC_STHT_FP32 set).
 *   - Latency 0: every pushed sample is final at once, n_out_host[s] = n for every slot; there is no flush.  reset takes
 *     a slot list (slots_host [n_slots], NULL = every slot): the listed slots restart at sample 0 with zero filterbank,
 *     band-pass and STHT history.  reset synchronises `stream`; a push does not.
 *   - push: frames_dev [S][n][in_channels] float32 / int16 / int32 (int32 wav frames with the recorder's extra channel:
 *     channels >= M are dropped), 1 <= n <= max_frame_len, in_channels >= M; a push that would take a slot's position to
 *     2^31 - 4096 samples or beyond is refused.  Outputs, all nullable device pointers, over the n rows of this push:
 *       z_dev          [F][S][n][2M] f32   s_t as (real | imag), debug tap;
 *       cov_dev        [F][S][M][M][2] f64 sum_t conj(s_t[i]) s_t[j], not normalised (micloc_hilbert_localize's cov);
 *       power_dev      [F][S][G] f32       mean_t |s_t . conj(bf_g)|^2;
 *       power_grid_dev [S][G] f32, doa_dev [S]: the sum over the bands and its first argmax (micloc_power_fuse, for every
 *                      F);  periodic_ml_dev / trimmed_ml_dev [S] f64: its estimators (need doa_list, MICLOC_ERR_SHAPE
 *                      otherwise; NaN and flags bit 1 in the reference's IndexError case);
 *       sumsq_dev      [S] f64: sum of x^2 over the kept channels of the frame, as micloc_snn_mb_streams_push (needs the
 *                      filterbank: MICLOC_ERR_SHAPE without one);
 *       flags_dev      [S]: bit 1 as above (there is no RZCC: bit 0 is never set).
 * Kernel launches per push, whatever S: 1 (frame assembly, with the filterbank when there is one); per band, 2 (STHT,
 * band-pass + float64 Gram) for M <= 8 or 3 (STHT, band-pass -> z, tiled Gram) for M > 8, +1 (Gram -> cov, power) when
 * cov, power or a fused output is asked for; +1 (sum over bands, argmax, estimators) when power_grid, doa, the
 * estimators or flags are asked for.  doa_list [G] (host, nullable).  Device memory: 3 S (K - 1 + max_frame_len) M
 * floats and S 2M biquad states per band, S G F floats of power scratch, S (2M)^2 doubles of Gram partials per
 * 1024-sample slab (one slab for M <= 8), S max_frame_len 2M floats of z scratch for M > 8. */
typedef struct micloc_hilbert_streams micloc_hilbert_streams;
int micloc_hilbert_streams_create(micloc_snn *const *ctxs, int32_t F, int32_t n_sections, const double *sos,
                                  const double *doa_list, int32_t num_streams, int64_t max_frame_len,
                                  micloc_hilbert_streams **out);
int micloc_hilbert_streams_destroy(micloc_hilbert_streams *hs);
/* always 0 */
int micloc_hilbert_streams_latency(micloc_hilbert_streams *hs);
int micloc_hilbert_streams_reset(micloc_hilbert_streams *hs, const int32_t *slots_host, int32_t n_slots, void *stream);
int micloc_hilbert_streams_push(micloc_hilbert_streams *hs, const void *frames_dev, int dtype, int64_t n,
                                int32_t in_channels, float *z_dev, double *cov_dev, float *power_dev,
                                float *power_grid_dev, int32_t *doa_dev, double *periodic_ml_dev, double *trimmed_ml_dev,
                                double *sumsq_dev, int32_t *flags_dev, int64_t *n_out_host, void *stream);

/* ---- misc ------------------------------------------------------------------ */
const char *micloc_last_error(void);
int micloc_version(void);
/* kernels launched by this library since load (claim for bench.py's gpu_launches) */
int64_t micloc_launch_count(void);
/* With timing enabled every micloc_snn_run / run_taps brackets its kernels with a pair
 * of CUDA events on the caller's stream.  micloc_snn_last_kernel_ms waits for them and
 * returns the SUM of those durations (ms) since the previous read, with the number of
 * runs summed in n_runs, then forgets them. */
int micloc_snn_last_kernel_ms(micloc_snn *ctx, float *ms, int32_t *n_runs);
int micloc_snn_enable_timing(micloc_snn *ctx, int enable);
/* Debug counters of the fused kernel (MICLOC_ROLE_TIMING builds only, zeros otherwise): out[0..7] = busy
 * cycles summed per warp role (FIR clip 0 half 0/1, FIR clip 1 half 0/1, band-pass, RZCC, neuron, Gram),
 * out[8..15] = number of warps that reported each, out[16] / out[17] = clock64 cycles / nanoseconds of CTA 0.
 * Synchronises the device. */
int micloc_snn_debug_counters(micloc_snn *ctx, uint64_t out[32]);
/* Debug: out[16*i .. 16*i+15] = (start ns, end ns, SM id, role map: byte w = role | smsp << 3 of warp w, busy
 * cycles of the eight roles, unused) of CTA i of the last fused launch, i < n <= 512 (MICLOC_ROLE_TIMING builds only). */
int micloc_snn_debug_cta_times(micloc_snn *ctx, uint64_t *out, int32_t n);
/* FP32 FMA-pipe micro-benchmark on `device` (the measured denominator of the
 * roofline in bench.py): variant 0 = scalar FFMA, 1 = packed fma.rn.f32x2, 2 = FP64 DFMA (FP64 TFLOP/s).
 * Any other variant returns MICLOC_ERR_CONFIG. */
int micloc_fp32_peak(int device, int variant, double *tflops);

#ifdef __cplusplus
}
#endif
#endif /* MICLOC_B200_H_ */
