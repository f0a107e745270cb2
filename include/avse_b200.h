/* avse_b200.h -- C ABI of the B200-native spectral front/back end.
 *
 * Drop-in boundary for ONE hot path of melspectrum007/audio-visual-speech-enhancement:
 * the audio half of data_processor.py (mix at SNR -> STFT -> mel -> dB -> AV-aligned slices,
 * and mel -> linear -> ISTFT at predict time).  The reference has no FFI; its boundary is the
 * set of Python functions in /root/reference/data_processor.py.  Each entry point below names
 * the reference function(s) (file:line) whose arithmetic it replaces; the Python mirror of
 * those signatures lives in audio-visual-speech-enhancement_b200/data_processor.py and binds
 * this library with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - All data pointers are DEVICE pointers unless the name says host; float32 unless stated.
 *  - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream and
 *    allocates nothing (the context owns only small constant tables).
 *  - Return value: 0 ok; < 0 bad arguments (AVSE_E_*); > 0 a cudaError_t.  Nothing throws.
 *    avse_last_error() returns a thread-local description of the last failure.
 *  - Geometry: the reference's hard-coded one (dp:44-45, dp:83-89: n_fft 640, hop 160, 321 bins, 80 mel bands,
 *    20 spectrogram frames per 200 ms slice at 16 kHz / 25 fps) is the specialised hot path; the shapes in the
 *    comments below ([80][20], [321], 160 ...) read as [n_mels][spss], [bins], hop ... for avse_create_ex contexts.
 */
#ifndef AVSE_B200_H
#define AVSE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define AVSE_N_FFT 640
#define AVSE_HOP 160
#define AVSE_N_BINS 321
#define AVSE_N_MELS 80
#define AVSE_SPSS 20 /* spectrogram frames per slice: int(3200 / 160), dp:49 */

#define AVSE_E_ARG (-1)
#define AVSE_E_CONFIG (-2)
#define AVSE_E_NOCUDA (-3)

#define AVSE_SAMPLE_F32 0 /* float32 samples */
#define AVSE_SAMPLE_I16 1 /* raw int16 WAV samples (AudioSignal.from_wav_file, dp:122-123): decode fused into the kernels' loads;
                             encode = clip to [-32768, 32767] + truncate (AudioSignal.save_to_wav_file, se:176-177) fused into the stores */

#define AVSE_LAYOUT_SLICES 0 /* [B][n_slices][80][20]  (np.stack of dp:52-57) */
#define AVSE_LAYOUT_SPEC 1   /* [B][80][ld_t]          (dp:96 magnitude, time minor) */

typedef struct avse_ctx avse_ctx;

/* Builds the constant tables (periodic Hann, FFT twiddles, librosa.filters.mel(sr, 640, 80,
 * fmin, fmax) in banded form, tridiagonal factors of F F^T) in float64 on the host and uploads
 * them to `device`.  Replaces the per-call rebuilds at dp:83-89, dp:104-112.
 * Returns AVSE_E_CONFIG for a bank the specialised kernels cannot serve: an empty or non-contiguous band, a band wider than
 * the banded tables hold, a band touching the DC or Nyquist bin, a filterbank column with more than two taps or whose taps
 * are not adjacent bands (the inverse's walk tables; e.g. 80 / 3000 Hz or 980 / 6200 Hz at 16 kHz, 50 / 8000 Hz at 24 kHz),
 * or a 1-norm cond(F F^T) above 1e5 (the float32 tridiagonal solve would drift from pinv(F); e.g. 550 / 4600 Hz at
 * 16 kHz).  avse_create_ex serves every such bank with the generic kernels. */
int avse_create(int sample_rate, double fmin, double fmax, int device, avse_ctx** out);

/* Any geometry the reference derives from (sample rate, video frame rate, slice duration): n_fft = int(sr / fps) (dp:44),
 * hop = int(n_fft / 4) (dp:45), spss = int(samples_per_slice / hop) (dp:49), n_mels (dp:86).  (640, 160, 80, 20) gives the
 * specialised kernels (same as avse_create); anything else -- 320 @ 50 fps, 666 @ 24 fps, odd sizes like 533 @ 30 fps,
 * 1764 @ 44.1 kHz -- runs the generic kernels (two-level DFT with run-time factors, dense filterbank / pinv tables): same
 * entry points, same argument structs, correct but several times slower.  For odd n_fft the inverse uses librosa.istft's
 * inferred size 2 * (bins - 1), as the reference does (dp:114).  Limits: n_fft <= 4096, n_mels <= 256. */
int avse_create_ex(int sample_rate, int n_fft, int hop, int n_mels, int spss, double fmin, double fmax, int device,
                   avse_ctx** out);

/* out6 = { n_fft, hop, bins, n_mels, spss, generic (1: fallback kernels, 0: specialised) } of the context. */
int avse_get_geometry(const avse_ctx* ctx, int* out6);
void avse_destroy(avse_ctx* ctx);
const char* avse_last_error(void);
const char* avse_version(void);

/* Host copy of the dense filterbank, float64 [n_mels][bins] ([80][321] for avse_create; == librosa.filters.mel, dp:83-89). */
int avse_get_filterbank(const avse_ctx* ctx, double* host_out);

/* AudioMixer.snr_factor (dp:130): factor[u] = sqrt(var(speech_u) / var(noise_u)) * 10^(-snr_db[u]/20),
 * population variance over the first lengths[u] samples (lengths == NULL: L for all; values are clamped to [0, L]).
 * Accumulates in float64.  snr_db == NULL means 0 dB for every utterance (the reference).
 * noise_period (may be NULL): [B] own length Ln of each noise file.  Where Ln < lengths[u] the noise is the periodic tiling
 *   noise[i] = nz[i mod Ln] -- what the reference's "double until long enough, then truncate" loop builds (dp:125-128) --
 *   and only the first Ln samples of the noise row are read.
 * equalizer_out (may be NULL): [B] sqrt(sum s^2 / sum n^2), the ratio of the RAW powers (mean included) of speech and noise
 *   over exactly the samples the factor uses (the first lengths[u], the weighted period of a tiled noise, the window of a
 *   pooled row); hand it to avse_forward (avse_forward_args::equalizer).  0 where lengths[u] == 0; finite for a constant
 *   non-zero noise, whose factor is non-finite.
 * lengths[u] == 0 gives factor 0 (the reference mixes two empty arrays and zero-pads them, dp:39-40); a silent noise
 * (variance 0) gives inf / nan like numpy, and so does everything computed from it.
 * Also resets max_key[u][0..2] (the running dB maxima used by avse_forward / avse_floor_*) and, when
 * given, min_key[u][0..2] (the running minima of the stored values).
 * speech/noise: [B][stride] with stride >= L, float32 or int16 (sample_format = AVSE_SAMPLE_*). */
int avse_snr_factor(avse_ctx* ctx, const void* speech, const void* noise, int sample_format, long long stride,
                    const int* lengths, const int* noise_period, int B, int L, const float* snr_db,
                    float* factor_out, float* equalizer_out, int* max_key, int* min_key, void* stream);

typedef struct avse_forward_args {
    /* inputs */
    const void* speech;      /* [B][in_stride], float32 or int16 (see sample_format) */
    const void* noise;       /* [B][in_stride]; covers the speech length unless noise_period says otherwise; NULL: single signal */
    long long in_stride;     /* elements between consecutive utterances */
    const int* len_speech;   /* [B] samples present (zeros beyond: pad_with_zeros dp:40); NULL: L */
    const int* len_noise;    /* [B]; NULL: same as len_speech */
    const float* factor;     /* [B] from avse_snr_factor; NULL: 1.0 (noise used as given) */
    int B;
    int L;                   /* signal_length = samples_per_slice * n_video_slices (dp:37); frames T = 1 + L/160 */
    /* outputs: un-floored dB log-mel (amplitude_to_db before its top_db clip, dp:94) */
    int layout;              /* AVSE_LAYOUT_SLICES or AVSE_LAYOUT_SPEC */
    int n_slices;            /* slices kept per utterance: min(video, audio) (dp:164); layout SLICES only */
    int ld_t;                /* leading dimension (>= T) for layout SPEC */
    float* out_speech;       /* any of the three may be NULL */
    float* out_noise;
    float* out_mixed;
    long long out_stride;    /* elements between utterances in each output */
    float* mixed_pcm;        /* [B][pcm_stride] s + f*n padded/truncated to L (dp:133, dp:39-42); may be NULL */
    long long pcm_stride;
    int* max_key;            /* [B][3] running maxima (speech, noise, mixed) as ordered-int keys; required */
    float* stft_speech;      /* optional complex64 [B][T][321] (re, im interleaved): librosa.stft of `speech` (dp:79), frame-major */
    int* min_key;            /* optional [B][3] running minima of the STORED dB values (same key encoding): lets avse_floor_*
                                skip every utterance whose minimum is already >= max - 80 (nothing to clip) */
    int sample_format;       /* AVSE_SAMPLE_F32 (0) or AVSE_SAMPLE_I16: element type of speech / noise.  int16 is supported
                                for pair batches (noise != NULL) without stft_speech */
    const float* equalizer;  /* [B] from avse_snr_factor (equalizer_out), or NULL.  Numerical conditioning only: results are the
                                reference's s + factor * n either way.  The float32 kernels carry speech and noise through ONE
                                packed complex FFT, where float32 rounding of each channel leaks into the other in proportion to
                                its raw power; with the noise pre-scaled by equalizer[u] = sqrt(sum s^2 / sum n^2) both channels
                                have equal raw power whatever the levels and DC offsets of the two files (a float WAV next to an
                                int16 one ...), and the remaining factor[u] / equalizer[u] is applied by STFT linearity.
                                NULL: the whole factor is applied before the transform */
    const int* noise_period; /* [B] or NULL: own length Ln of each noise file; where Ln < len_noise[u] the kernels read
                                noise[i mod Ln] (dp:125-128) and only the first Ln samples of the noise row need to exist */
} avse_forward_args;

/* preprocess_audio_pair's arithmetic (dp:130-137) / signal_to_spectrogram (dp:77-96) for a batch:
 * one fused kernel: framing + reflect pad + Hann + packed 640-point FFT + |.| + mel + dB. */
int avse_forward(avse_ctx* ctx, const avse_forward_args* args, void* stream);

/* amplitude_to_db's top_db floor (dp:94): x = max(x, max_u - 80), in place on a SLICES or SPEC
 * output of avse_forward.  which: 0 speech, 1 noise, 2 mixed (selects the key column).
 * min_key (may be NULL): minima written by avse_forward; utterances with min >= max - 80 are skipped unread. */
int avse_floor_inplace(avse_ctx* ctx, float* data, long long stride, long long n_per_utt, int B,
                       const int* max_key, const int* min_key, int which, void* stream);

/* The same floor for the three outputs of a pair batch (speech, noise, mixed: max_key columns 0, 1, 2) in one launch. */
int avse_floor_inplace3(avse_ctx* ctx, float* speech, float* noise, float* mixed, long long stride, long long n_per_utt,
                        int B, const int* max_key, const int* min_key, void* stream);

/* Dynamic mixing for training: preprocess_audio_pair (dp:119-139) of pairings drawn from two device-resident clip pools,
 * without materialising them.  Output row b < B mixes s = the first Ls = speech_len[speech_index[b]] samples of that speech
 * clip with the noise n[i] = z[(off + i) mod Ln], i < Ls, where z = the first Ln = noise_len[noise_index[b]] samples of that
 * noise clip and off = noise_offset[b]: off = 0 is the reference's own rule (tile a short noise, dp:125-126, truncate a long
 * one, dp:128).  factor = sqrt(var(s) / var(n)) * 10^(-snr_db[b]/20) over the Ls samples (dp:130, float64 sums); the speech
 * always starts at its sample 0 (its video slices are aligned to it, dp:164) and is zero padded / truncated to L (dp:36-42).
 * A row is INVALID when an index is out of range or off is outside [0, Ln) (so every empty noise clip): it reads no sample,
 * is processed as an empty pair (factor 0, every slice at the amin floor -100 dB, PCM zeros) and sets *bad_row_flag.
 * A silent noise window gives inf / nan like numpy (avse_snr_factor).
 * Enqueues the statistics pass, the forward pass and avse_floor_inplace3 on `stream`; allocates nothing.  Works on every
 * context avse_forward serves pair batches on (F4, 2-frame and generic-geometry kernels), float32 or int16 pools under the
 * same rules as avse_forward. */
typedef struct avse_pool_mix_args {
    /* pools */
    const void* speech_pool;        /* [n_speech][speech_stride], float32 or int16 (sample_format) */
    const int* speech_len;          /* [n_speech] clip lengths; clamped to [0, speech_stride] */
    long long speech_stride;        /* elements between consecutive clips */
    long long n_speech;
    const void* noise_pool;         /* [n_noise][noise_stride], same sample format */
    const int* noise_len;           /* [n_noise]; clamped to [0, noise_stride] */
    long long noise_stride;
    long long n_noise;
    int sample_format;              /* AVSE_SAMPLE_F32 or AVSE_SAMPLE_I16 */
    /* pairing of each output row b < B */
    const long long* speech_index;  /* [B] int64 */
    const long long* noise_index;   /* [B] int64 */
    const int* noise_offset;        /* [B] int32 phase of the noise, NULL: 0 for every row */
    const float* snr_db;            /* [B] or NULL: 0 dB */
    int B;
    int L;                          /* signal_length = samples_per_slice * n_video_slices (dp:37) */
    int n_slices;                   /* slices kept per row, 1 <= n_slices <= int(T / 20) (dp:50, dp:164) */
    /* outputs */
    float* out_speech;              /* SLICES [B][n_slices][80][20], floored dB (all three required, 16-byte aligned) */
    float* out_noise;
    float* out_mixed;
    long long out_stride;           /* elements between rows, multiple of 4 */
    float* mixed_pcm;               /* [B][pcm_stride] s + factor * n zero padded / truncated to L, or NULL */
    long long pcm_stride;
    float* factor_out;              /* [B] SNR factor, required */
    float* equalizer_out;           /* [B] sqrt(sum s^2 / sum n^2), or NULL (see avse_forward_args::equalizer) */
    int* max_key;                   /* [B][3] caller scratch (running dB maxima), required */
    int* min_key;                   /* [B][3] caller scratch (running minima: lets the floor skip rows), or NULL */
    int* bad_row_flag;              /* device int the caller zeroed; set to 1 when any row is invalid; required */
} avse_pool_mix_args;

int avse_mix_pooled(avse_ctx* ctx, const avse_pool_mix_args* args, void* stream);

/* dp:49-57 segment gather with the floor applied: SPEC [B][80][ld_t] -> SLICES [B][n_slices][80][20]. */
int avse_floor_gather(avse_ctx* ctx, const float* spec, long long spec_stride, int ld_t,
                      float* slices, long long slices_stride, int n_slices, int B,
                      const int* max_key, int which, void* stream);

typedef struct avse_inverse_args {
    const float* mel_db;     /* dB log-mel: SLICES [B][n_slices][80][20] (np.concatenate(list(slices), axis=1), dp:66) or SPEC [B][80][ld_t] */
    int layout;
    int n_slices;            /* layout SLICES */
    int n_frames;            /* layout SPEC: frames held in mel_db */
    int ld_t;                /* layout SPEC: leading dimension */
    long long mel_stride;    /* elements between utterances */
    const float* mixed_pcm;  /* [B][pcm_stride] mixture waveform whose STFT phase is re-used (dp:64) */
    long long pcm_stride;
    const int* len_pcm;      /* [B] samples present (zeros beyond); NULL: L */
    int B;
    int L;                   /* mixture length; T = 1 + L/160 frames; frames used = min(mel frames, T) (dp:68) */
    void* out_pcm;           /* [B][out_stride] reconstructed PCM, 160 * (frames_used - 1) samples each (librosa.istft, dp:114) */
    long long out_stride;
    float* work;             /* scratch [B][work_stride], work_stride >= avse_inverse_work_elems(frames_used).  Only the generic-geometry
                                kernels (avse_create_ex contexts) and the 4-frame kernel kept for A/B runs (AVSE_INV4=1) use it; the
                                specialised I8 kernel keeps the coefficients on chip and accepts NULL */
    long long work_stride;
    const float* phase;      /* optional complex64 [B][phase_frames][321] (re, im): explicit phase (dp:99 signature); when set,
                                mixed_pcm / L are ignored and frames used = min(mel frames, phase_frames) */
    long long phase_stride;  /* complex elements between utterances */
    int phase_frames;
    int out_format;          /* AVSE_SAMPLE_F32 (0): out_pcm is float32; AVSE_SAMPLE_I16: out_pcm is int16 [B][out_stride],
                                clipped to the int16 range and truncated like AudioSignal.save_to_wav_file (se:176-177) */
} avse_inverse_args;

/* reconstruct_speech_signal / reconstruct_signal_from_spectrogram (dp:60-74, dp:99-116) for a batch:
 * db_to_amplitude -> pinv(mel fb) as a tridiagonal solve + 2-tap F^T -> x phase of the mixture's STFT (recomputed
 * on the fly) -> irfft + Hann + overlap-add / window sum-square, centre trim.  One kernel on `stream` (two for generic geometries). */
int avse_inverse(avse_ctx* ctx, const avse_inverse_args* args, void* stream);

/* Scratch floats per utterance needed by avse_inverse for `n_frames_use` reconstructed frames (specialised geometry). */
int avse_inverse_work_elems(int n_frames_use, long long* per_utterance);
/* The same for the geometry of `ctx` (use this one with avse_create_ex contexts). */
int avse_inverse_work_elems_ctx(const avse_ctx* ctx, int n_frames_use, long long* per_utterance);

/* Sets n running-max keys to "minus infinity" (and, when min_key != NULL, n running-min keys to "plus infinity") (needed before avse_forward when avse_snr_factor,
 * which also resets them, is not part of the sequence, e.g. single-signal spectrograms). */
int avse_reset_max(avse_ctx* ctx, int* max_key, int* min_key, int n, void* stream);

/* Decodes max_key[u][which] to float dB on the host side convention (device -> device). */
int avse_max_db(avse_ctx* ctx, const int* max_key, int n, float* out_db, void* stream);

/* make_sample_set (speech_enhancer.py:241-262): the np.concatenate over samples followed by ONE shared random
 * permutation, as a device row gather: dstK[i][0..row_elems) = srcK[index[i]][0..row_elems) for K = 0..2 (src1/dst1 and
 * src2/dst2 optional, given in order).  Rows are dense (row stride == row_elems, a multiple of 4 floats; a slice is
 * 80 * 20 = 1600).  index: int64 [n_out] on the device, values in [0, src_rows); an out-of-range value sets
 * *bad_index_flag (device int the caller zeroed) and leaves that output row untouched. */
int avse_gather_rows(avse_ctx* ctx, const float* src0, const float* src1, const float* src2, long long src_rows,
                     long long row_elems, const long long* index, long long n_out, float* dst0, float* dst1, float* dst2,
                     int* bad_index_flag, void* stream);

/* VideoNormalizer.__init__ (dp:201-205): per-pixel mean and population std over (slices, frames) of the mouth-crop tensor
 * video [n_slices][hw][frames] float32 (hw = height * width, e.g. 128 * 128; frames = 5).  scratch: 2 * hw doubles
 * (device).  mean_out / std_out: [hw] float32.  Float64 accumulation. */
int avse_video_stats(avse_ctx* ctx, const float* video, long long n_slices, int hw, int frames, double* scratch,
                     float* mean_out, float* std_out, void* stream);

/* VideoNormalizer.normalize (dp:207-212): video[s][p][f] = (video[s][p][f] - mean[p]) / std[p], in place, no epsilon. */
int avse_video_normalize(avse_ctx* ctx, float* video, long long n_slices, int hw, int frames, const float* mean,
                         const float* stdv, void* stream);

/* Mean squared error over n elements (the loss network.evaluate reports on log-mel slices, network.py:214-220).
 * scratch: 1 double (device); out: 1 float (device). */
int avse_mse(avse_ctx* ctx, const float* a, const float* b, long long n, double* scratch, float* out, void* stream);

/* librosa.core.magphase (dp:80) on the complex STFT that avse_forward writes (stft_speech, frame-major [n_utt][n_frames][n_bins],
 * re / im interleaved): mag_out [n_utt][n_bins][n_frames] = |D| and phase_out (same shape, complex64) = D / |D|, with 1 + 0j where
 * D == 0 -- i.e. in the reference's (freq, time) orientation (dp:96).  Either output may be NULL. */
int avse_magphase(avse_ctx* ctx, const float* stft, long long n_utt, int n_frames, int n_bins, float* mag_out, float* phase_out,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVSE_B200_H */
