/*
 * audiocalm_b200.h -- C ABI of the B200-native (sm_100a) log-mel front-end for Audio-CALM.
 *
 * Drop-in boundary.  The reference has no FFI: its boundary is the Python symbols of
 * preprocess/core.py and preprocess/compute_mel_stats.py.  Every entry point below names the reference
 * lines it replaces; the Python shims in audio-calm_b200/preprocess/ keep the reference's call
 * signatures and bind these functions with ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - plain C types only; every pointer marked "device" is a CUDA device pointer owned by the caller
 *     (the Python side allocates with torch); nothing is allocated or freed across the ABI except the
 *     opaque front-end handle (constant tables) created/destroyed explicitly.
 *   - all work is enqueued on the caller's `stream` (a cudaStream_t passed as void*); no call
 *     synchronises the device unless stated.
 *   - return value: 0 = ACB_OK, negative = error; acb_last_error() returns a thread-local message.
 *     No exception ever crosses the ABI.
 */
#ifndef AUDIOCALM_B200_H_
#define AUDIOCALM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACB_OK 0
#define ACB_ERR_INVALID (-1)      /* bad argument (null pointer, unsupported preset, clip too short ...) */
#define ACB_ERR_CUDA (-2)         /* a CUDA runtime call failed; message carries cudaGetErrorString */
#define ACB_ERR_UNSUPPORTED (-3)  /* valid request this build has no kernel for */

#define ACB_ABI_VERSION 2

/* output element type */
#define ACB_F32 0
#define ACB_BF16 1
/* output layout of one clip: MEL_MAJOR = [n_mels][frame_capacity] (what the saved {"mel"} payload and the
 * VAE consume, preprocess/process_dataset.py:155); TIME_MAJOR = [frame_capacity][n_mels], the physical
 * layout torchaudio's MelScale returns as a transposed view (SURVEY.md 8a4). */
#define ACB_MEL_MAJOR 0
#define ACB_TIME_MAJOR 1
/* log kind */
#define ACB_LOG_NATURAL 0         /* preprocess/core.py:60 */
#define ACB_LOG_10 1

typedef struct acb_frontend acb_frontend; /* opaque: device-resident tables for one (device, preset) */

int acb_abi_version(void);
const char* acb_last_error(void);

/* Frames tile: the hot kernel processes clips in tiles of this many frames. */
int acb_frames_per_tile(void);

/* T = 1 + L / hop of torch.stft(center=True) as called through preprocess/core.py:55; returns -1 when
 * L <= n_fft/2 (the reference raises RuntimeError: reflect padding needs a longer input). */
int64_t acb_frames_for_length(int64_t length, int n_fft, int hop);
/* Frame count after the reflect pad to a multiple (preprocess/process_dataset.py:146-150). */
int64_t acb_padded_frames(int64_t frames, int multiple);

/* Host-side planning: exclusive prefix of per-clip tile counts for acb_logmel_forward.
 * lengths_host[n_clips] in samples; frame_capacity > 0 asks for tiles covering the whole row (used with
 * fill_tail), 0 covers only the frames that exist.  Writes tile_start_host[n_clips + 1]; returns the
 * total tile count or a negative error (a clip shorter than n_fft/2 + 1 samples). */
int64_t acb_plan_tiles(const int64_t* lengths_host, int32_t n_clips, int n_fft, int hop,
                       int64_t frame_capacity, int32_t* tile_start_host);

/* Build the device tables (replaces MelExtractor.__init__, preprocess/core.py:33-48).
 * window_host[n_fft] and fb_host[(n_fft/2+1) * n_mels] (row-major [freq][mel]) are the fp32 tables the
 * host derived with the reference's torch calls.  This build has kernels for n_fft = 1024, hop = 256,
 * n_mels <= 128; anything else returns ACB_ERR_UNSUPPORTED.  So does a window without the periodic-Hann property
 * |w[n + 512] - (1 - w[n])| <= 1e-6 (the kernel computes the second half of the window from the first), a filterbank with
 * weight on the Nyquist bin, or one with more than 4096 banded weights. */
int acb_frontend_create(acb_frontend** out, int device, int n_fft, int hop, int n_mels,
                        const float* window_host, const float* fb_host, float clamp_min, int log_kind);
int acb_frontend_destroy(acb_frontend* fe);
/* Which implementation of the fused log-mel kernel acb_logmel_forward launches.  This build has one, with the mel projection
 * on the CUDA cores: 0 = automatic and 1 = CUDA-core mel projection both select it and return ACB_OK.  2 = the warp-specialised
 * kernel with the mel projection on the tensor pipe (mma.sync TF32 pairs) returns ACB_ERR_UNSUPPORTED: it was measured on B200
 * at 1.80 ms against 0.466 ms for the CUDA-core kernel (256 x 30 s) and removed.  Any other kind returns ACB_ERR_INVALID. */
int acb_frontend_set_kernel(acb_frontend* fe, int kind);
/* bytes of device workspace acb_logmel_forward needs when moments are requested */
int64_t acb_moments_workspace_bytes(const acb_frontend* fe);

typedef struct acb_logmel_args {
    /* ---- input: a flat device buffer of fp32 samples holding n_clips clips ---- */
    const float* wav;            /* device */
    const int64_t* clip_offset;  /* device [n_clips]: first sample of clip i in wav; NULL => i * clip_stride */
    const int64_t* clip_length;  /* device [n_clips]: samples in clip i;            NULL => uniform_length */
    int64_t clip_stride;         /* used when clip_offset is NULL */
    int64_t uniform_length;      /* used when clip_length is NULL */
    const int32_t* tile_start;   /* device [n_clips + 1] from acb_plan_tiles;        NULL => uniform clips, or ragged clips
                                  * with fill_tail (every clip then covers ceil(frame_capacity / tile) tiles) */
    int32_t n_clips;
    int32_t n_tiles;             /* total tiles (last entry of tile_start) */
    /* ---- optional fused peak normalisation (preprocess/core.py:108-110) ---- */
    const float* clip_peak;      /* device [n_clips] max|x| per clip from acb_peak_abs, or NULL */
    /* ---- output ---- */
    void* out;                   /* device; NULL = statistics-only launch (needs moments != NULL): nothing is stored */
    int32_t out_dtype;           /* ACB_F32 | ACB_BF16 */
    int32_t out_layout;          /* ACB_MEL_MAJOR | ACB_TIME_MAJOR */
    const int64_t* out_offset;   /* device [n_clips] element offset of clip i in out; NULL => i * out_clip_stride */
    int64_t out_clip_stride;     /* elements */
    int64_t frame_capacity;      /* frames per clip row in `out` (row pitch of MEL_MAJOR; >= padded frames) */
    const int64_t* frame_capacity_per_clip; /* device [n_clips] overrides frame_capacity (packed outputs) or NULL */
    int32_t pad_multiple;        /* 1 = none, 4 = reflect-pad the time axis (process_dataset.py:146-150) */
    int32_t fill_tail;           /* !=0: frames [padded, frame_capacity) are set to fill_value (ragged batches); with a tile plan
                                  * (tile_start) the clip's last tile fills the rest of its row in one sweep */
    float fill_value;
    /* ---- optional fused affine normalisation (models/modeling_vae.py:317-319) ---- */
    int32_t affine;              /* 0 none, 1 scalar (affine_mean/affine_std), 2 per-bin arrays */
    float affine_mean;
    float affine_std;
    const float* bin_mean;       /* device [n_mels] when affine == 2 */
    const float* bin_std;        /* device [n_mels] when affine == 2 */
    /* ---- optional fused per-bin moments of the un-normalised log-mel (compute_mel_stats.py:26-27) ---- */
    double* moments;             /* device [2 * n_mels]: sum then sum of squares, ACCUMULATED into; or NULL */
    void* moments_workspace;     /* device, acb_moments_workspace_bytes() bytes, when moments != NULL */
} acb_logmel_args;

/* Fused reflect-pad + framing + Hann window + STFT + power + mel projection + clamp + log
 * (+ pad-to-4, + affine normalisation, + per-bin moments): replaces MelExtractor.forward
 * (preprocess/core.py:50-61) and the torchaudio/torch.stft calls below it. */
int acb_logmel_forward(const acb_frontend* fe, const acb_logmel_args* args, void* stream);
/* Synchronises `stream` and reports (ACB_ERR_CUDA) whether a sample-tile copy failed to complete inside a launch since the last
 * check: the kernel's barrier waits are bounded so that a faulted copy cannot hang the device; the host-buffer entry points
 * below run this check themselves.  The reference's counterpart is the exception a failed torch.stft launch raises. */
int acb_frontend_check(const acb_frontend* fe, void* stream);

/* Per-clip max|x| (preprocess/core.py:108). peak_out: device [n_clips] fp32. */
int acb_peak_abs(const float* wav, const int64_t* clip_offset, const int64_t* clip_length, int64_t clip_stride,
                 int64_t uniform_length, int32_t n_clips, float* peak_out, void* stream);

/* process_audio_chunk (preprocess/core.py:93-112): wav_cl device [channels][length] -> out device [length]:
 * channel mean when channels > 1, then x / (peak + 1e-8) * 0.95 when peak > 0 (division first).
 * scratch_peak: device [1] fp32 workspace. */
int acb_process_audio_chunk(const float* wav_cl, int32_t channels, int64_t length, float* out,
                            float* scratch_peak, void* stream);
/* First half of process_audio_chunk only (preprocess/core.py:102-108): channel mean -> out device [length] and, when peak_out
 * (device [1]) is given, max|mean|.  The scaling is then fused into the log-mel kernel through acb_logmel_args.clip_peak, which
 * saves the second pass over the waveform for multi-channel clips too. */
int acb_mixdown_peak(const float* wav_cl, int32_t channels, int64_t length, float* out, float* peak_out, void* stream);

/* Per-bin moments of already-extracted features (compute_mel_stats.py:19-28 over saved files):
 * feat device, MEL_MAJOR [n_clips][n_mels][frame_capacity] fp32 or bf16, frames[i] valid frames of clip i
 * (device [n_clips]; NULL => all frame_capacity).  Accumulates into moments[2 * n_mels] (device, fp64).
 * workspace: device scratch of acb_moments_accumulate_workspace_bytes(n_mels) bytes owned by the caller, or NULL
 * (a stream-ordered allocation is made and freed inside the call). */
int64_t acb_moments_accumulate_workspace_bytes(int32_t n_mels);
int acb_moments_accumulate(const void* feat, int32_t dtype, int32_t n_clips, int32_t n_mels, int64_t frame_capacity,
                           int64_t clip_stride, const int64_t* frames, double* moments, void* workspace, void* stream);

/* Finalise on the host (compute_mel_stats.py:30-33): per-bin mean/std and the reference's global scalars.
 * moments_host[2 * n_mels], frames = total frame count (all clips).  var floor as in the reference (1e-8). */
int acb_moments_finalize(const double* moments_host, int32_t n_mels, int64_t frames, double var_floor,
                         double* bin_mean, double* bin_std, double* global_mean, double* global_std);

/* Per-utterance, per-bin normalisation used by eval (eval/eval_vae.py:80-82): (x - mean_t) / max(std_t, 1e-5)
 * with the unbiased std over time.  feat/out device MEL_MAJOR fp32 [n_clips][n_mels][frame_capacity]. */
int acb_normalize_per_utterance(const float* feat, float* out, int32_t n_clips, int32_t n_mels,
                                int64_t frame_capacity, const int64_t* frames, float min_std, void* stream);

/* Crop / zero-pad of stored features to a fixed number of frames, stacked: MelDataset.__getitem__ + data_collator
 * (train/train_vae.py:83-116).  feat device MEL_MAJOR [n_clips][n_mels][frame_capacity] fp32 or bf16 (clip_stride elements
 * between clips), frames[i] valid frames (device, NULL => frame_capacity), start[i] first frame of the crop (device, NULL => 0;
 * the caller draws random starts for training and (T - crop) / 2 for eval, like the reference).
 * out device [n_clips][n_mels][out_frames], same dtype: out[i][b][t] = feat[i][b][start[i] + t] inside the clip, else pad_value. */
int acb_crop_pad(const void* feat, int32_t dtype, int32_t n_clips, int32_t n_mels, int64_t frame_capacity, int64_t clip_stride,
                 const int64_t* frames, const int64_t* start, void* out, int64_t out_frames, float pad_value, void* stream);

/* Ragged collation to a channels-first padded batch: CalmCollator's pad_sequence(batch_first) + transpose(1, 2)
 * (train/train_calm.py:205-215), with the optional time mask of _apply_spec_augment (:184-191).
 * feat_tm device, time-major rows [sum lens][dim] fp32 or bf16; row_offset[i] first row of clip i, lens[i] its rows (device);
 * out device [n_clips][dim][out_frames], same dtype, pad_value beyond lens[i]; mask_start/mask_len (device, both or neither):
 * rows [mask_start[i], mask_start[i] + mask_len[i]) of clip i are written as 0. */
int acb_pad_transpose(const void* feat_tm, int32_t dtype, const int64_t* row_offset, const int64_t* lens, int32_t n_clips,
                      int32_t dim, void* out, int64_t out_frames, float pad_value, const int64_t* mask_start,
                      const int64_t* mask_len, void* stream);

/* Host-buffer convenience path (pinned or pageable host memory): H2D copy, acb_logmel_forward on uniform
 * clips [n_clips][length], D2H copy, chunked over `n_chunks` so copies overlap compute.  dev_in/dev_out
 * are caller-provided device staging buffers (n_clips*length floats / n_clips*n_mels*frame_capacity
 * elements).  out_host == NULL keeps the features on the device (dev_out) and skips the D2H copies: the training-feed
 * case, where the consumer is a model on the same GPU.  Synchronises `stream` before returning. */
int acb_logmel_forward_host(const acb_frontend* fe, const float* wav_host, int32_t n_clips, int64_t length,
                            void* out_host, acb_logmel_args* args_template, float* dev_in, void* dev_out,
                            int32_t n_chunks, void* stream);

/* 16-bit PCM transport (an extension: the reference moves fp32 over PCIe, preprocess/process_dataset.py:135-140).
 * int16 samples are widened on the device to x / 32768, exactly the values torchaudio.load(normalize=True) produces for
 * 16-bit files, so every result is bit-identical to the fp32 path; host->device traffic halves. */
int acb_pcm16_to_float(const int16_t* pcm, float* out, int64_t n, void* stream);                       /* pcm, out: device */
int acb_logmel_forward_host_pcm16(const acb_frontend* fe, const int16_t* pcm_host, int32_t n_clips, int64_t length,
                                  void* out_host, acb_logmel_args* args_template, int16_t* dev_pcm, float* dev_in,
                                  void* dev_out, int32_t n_chunks, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Tensor-core route (DFT-as-GEMM on tcgen05, split-fp16 operands, fp32 accumulation in TMEM) for the "Whisper-style"
 * preset BASELINE.json's north star names: n_fft 400, hop 160, reflect-padded centred frames, periodic Hann window,
 * the 80-band bank of models/mel_filters.npz, log10(clamp(., 1e-10)), max - 8 dynamic-range floor, (x + 4) / 4.
 * Replaces transformers.WhisperFeatureExtractor._np_extract_fbank_features, which the reference reaches through the
 * Hugging Face ASR pipeline it scores generated speech with (eval/eval_calm.py:548-552); the reference's own extractor
 * (preprocess/core.py, n_fft 1024) stays on acb_logmel_forward.  Input domain: |x| <= 2 (fp16 operand range after the
 * internal 2^12 pre-scale; audio is in [-1, 1]).
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct acb_dftgemm acb_dftgemm; /* opaque: DFT matrices, window halves and the streaming mel program */

/* Frames of one clip: 1 + L / 160 (torch.stft center=True), minus the last one when drop_last_frame (Whisper drops it:
 * stft[..., :-1]); -1 when L <= 200 (reflect padding needs a longer input). */
int64_t acb_dftgemm_frames(int64_t length, int drop_last_frame);

/* window_host[400] (must be symmetric: w[n] == w[400 - n]) and fb_host[201 * n_mels] (row-major [freq][mel]; used in banded
 * form: at most 3072 weights between the first and last non-zero bin of every band) as fp32.  Only n_fft = 400, hop = 160 is built. */
int acb_dftgemm_create(acb_dftgemm** out, int device, int n_fft, int hop, int n_mels, const float* window_host,
                       const float* fb_host, float clamp_min, int log_kind);
int acb_dftgemm_destroy(acb_dftgemm* fe);
/* int32 elements of the `clip_max` workspace for n_clips clips of `length` samples: n_clips * (1 + tiles per clip) */
int64_t acb_dftgemm_workspace_ints(int64_t length, int drop_last_frame, int32_t n_clips);

typedef struct acb_dftgemm_args {
    const float* wav;          /* device: n_clips uniform clips, clip i at wav + i * clip_stride (16-byte aligned rows take the bulk-copy path) */
    int64_t clip_stride;       /* samples */
    int64_t length;            /* samples per clip (Whisper pads / trims to 480000 on the host side) */
    int32_t n_clips;
    int32_t drop_last_frame;   /* !=0: store frames [0, L / 160) */
    void* out;                 /* device fp32 or bf16 [n_clips][n_mels][frame_capacity] */
    int64_t out_clip_stride;   /* elements */
    int64_t frame_capacity;    /* >= frames */
    float dyn_range;           /* > 0: out = max(out, max over the clip - dyn_range) (Whisper: 8.0); <= 0: none */
    int32_t affine;            /* 1: out = (out - affine_mean) / affine_std afterwards (Whisper: mean -4, std 4); 2: per band with bin_mean / bin_std */
    float affine_mean;
    float affine_std;
    int32_t* clip_max;         /* device workspace of acb_dftgemm_workspace_ints() int32 (per-clip maximum and per-tile minimum keys),
                                * needed when dyn_range > 0 */
    int32_t out_dtype;         /* ACB_F32 | ACB_BF16 (the affine is applied in fp32 before the single rounding) */
    /* ---- the fields below mirror acb_logmel_args (ABI version 2) ---- */
    const int64_t* clip_length;  /* device [n_clips]: samples of clip i (200 < clip_length[i] <= length; rows are padded to `length` with
                                  * finite values); reflection happens at each clip's own end, frames beyond a clip's count get
                                  * fill_value; NULL => every clip has `length` samples */
    const float* clip_peak;      /* device [n_clips] max|x| (acb_peak_abs) or NULL.  Given: every clip is pre-scaled by the power of two
                                  * that brings its peak into [0.5, 1) and the mel powers are scaled back exactly, so ANY amplitude fits the
                                  * fp16 operands.  NULL: the caller vouches for |x| <= 2; acb_dftgemm_check reports violations. */
    int32_t peak_norm;           /* !=0 (needs clip_peak): fused process_audio_chunk gain 0.95 / (peak + 1e-8) (preprocess/core.py:108-110) */
    float fill_value;            /* frames [frames of the clip, frames of `length`) of a shorter clip */
    const float* bin_mean;       /* device [n_mels] when affine == 2 (the stored per-bin statistics) */
    const float* bin_std;
    double* moments;             /* device [2 * n_mels], ACCUMULATED into: per-bin sum and sum of squares of the un-normalised log-mel over
                                  * the frames that exist (compute_mel_stats.py:26-27).  Only with dyn_range <= 0: the per-clip floor is
                                  * applied after the kernel; floored features go through acb_moments_accumulate. */
    void* moments_workspace;     /* device, acb_dftgemm_moments_workspace_bytes() bytes, when moments != NULL */
} acb_dftgemm_args;
/* bytes of device workspace the fused moments of acb_dftgemm_forward need */
int64_t acb_dftgemm_moments_workspace_bytes(const acb_dftgemm* fe);

/* One persistent tcgen05 launch on `stream`, plus -- when dyn_range > 0 -- a pass that rewrites only the tiles holding values below
 * their clip's floor (the kernel records every tile's minimum). */
int acb_dftgemm_forward(const acb_dftgemm* fe, const acb_dftgemm_args* args, void* stream);
/* Synchronises `stream` and reports what the launches since the last check flagged: ACB_ERR_CUDA when an in-kernel pipeline barrier
 * timed out, ACB_ERR_INVALID when features came out non-finite (a sample beyond the fp16 operand range without clip_peak, or NaN input). */
int acb_dftgemm_check(const acb_dftgemm* fe, void* stream);

/* ---------------------------------------------------------------------------------------------
 * VAE-side spectral op (SURVEY.md 8f rank 4): short-time Fourier magnitudes over the time axis of features.
 * Replaces AcousticVAE._stft_mag (models/modeling_vae.py:271-289: torch.stft(n_fft, hop, window = periodic Hann(n_fft),
 * center=False, onesided, normalized=False) + torch.abs), which stft_loss (:291-305) calls with (n_fft, hop) = (256, 64),
 * (128, 32), (64, 16) on [B, 80, T] features.
 *   x      device [rows][length] fp32 (rows = B * C, contiguous)
 *   window device [n_fft] fp32 (torch.hann_window(n_fft), passed by the host so that it is bit-identical)
 *   out    device [rows][n_fft / 2 + 1][frames] fp32, frames = acb_stft_mag_frames(length, n_fft, hop) = 1 + (length - n_fft) / hop
 * n_fft in {64, 128, 256, 512, 1024}; length < n_fft returns ACB_ERR_INVALID (torch.stft raises for center=False). */
int64_t acb_stft_mag_frames(int64_t length, int n_fft, int hop);
int acb_stft_mag(const float* x, int64_t rows, int64_t length, int n_fft, int hop, const float* window, float* out, void* stream);
/* Its adjoint (what autograd computes through torch.stft + abs in stft_loss, models/modeling_vae.py:291-305): given grad_mag (device
 * [rows][n_fft / 2 + 1][frames]) writes grad_x (device [rows][length]).  X is recomputed, not stored; a bin with |X| = 0 passes no
 * gradient (torch's abs does the same). */
int acb_stft_mag_backward(const float* x, const float* grad_mag, int64_t rows, int64_t length, int n_fft, int hop, const float* window,
                          float* grad_x, void* stream);

/* Griffin-Lim building blocks: the vocoder fallback of eval/eval_calm.py:184-208 runs torchaudio.transforms.GriffinLim(n_fft=1024)
 * (torchaudio.functional.griffinlim: n_iter x [torch.istft, torch.stft(center=True, reflect), phase update with momentum]).
 *   acb_stft_complex: x device [rows][length] -> spec device complex64 [rows][n_fft/2+1][1 + length/hop] (interleaved re, im), frames
 *     centred with reflect padding like torch.stft(center=True).  With gl_previous / gl_magnitude (same shape as spec: complex /
 *     real) the epilogue applies one Griffin-Lim update instead: rebuilt = STFT; angles = rebuilt - gl_momentum * gl_previous;
 *     gl_previous = rebuilt; spec = angles / (|angles| + 1e-16) * gl_magnitude.
 *   acb_istft: spec -> out device [rows][length] like torch.istft(center=True, length=length): inverse transform, window,
 *     overlap-add, division by the window envelope, n_fft/2 trimmed at the start.
 * n_fft in {256, 512, 1024}; window device [n_fft]. */
int acb_stft_complex(const float* x, int64_t rows, int64_t length, int n_fft, int hop, const float* window, float* spec, float* gl_previous,
                     const float* gl_magnitude, float gl_momentum, void* stream);
int acb_istft(const float* spec, int64_t rows, int64_t n_frames, int n_fft, int hop, const float* window, float* out, int64_t length, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Resampling to the front-end's rate: torchaudio.transforms.Resample(orig_freq, new_freq) with the default "sinc_interp_hann"
 * method, which the reference runs on the host for every file that is not 16 kHz (preprocess/process_dataset.py:135-137).
 * With (O, N) = (orig_freq, new_freq) / gcd, output y[b * N + j] = sum_k kernel[j][k] * xpad[b * O + k], xpad = the clip zero-padded
 * by `width` samples on the left and width + O on the right (at each clip's own ends), over the band of non-zero coefficients of
 * each phase.  Skipped coefficients are exact zeros, so finite input gives torchaudio's result up to fp32 summation order; a
 * non-finite sample does not reach outputs through zero coefficients, as it does through torchaudio's dense conv1d.
 * ------------------------------------------------------------------------------------------------------------------ */
#define ACB_I16 2                 /* input element type of acb_resample: int16 samples, widened on the device to x / 32768 */

typedef struct acb_resampler acb_resampler; /* opaque: banded per-phase coefficient table for one (device, O, N) */

/* torchaudio's output length for `length` input samples: ceil(torch.as_tensor(N * length / O)) -- the quotient is rounded to fp32
 * before the ceiling, so beyond 2^24 outputs it can differ from the exact ceiling (24 kHz -> 16 kHz: 30000001 -> 20000000) -- capped
 * by the conv1d length (length / O + 1) * N.  orig_freq == new_freq returns length.  Host only; -1 for a negative length or rate. */
int64_t acb_resampled_length(int64_t length, int orig_freq, int new_freq);
/* kernel_host[N * (2 * width + O)]: the fp32 table transforms.Resample holds (row-major [N][K]).  Tables with more than 32768 banded
 * coefficients or a band wider than 512 taps return ACB_ERR_UNSUPPORTED (8-192 kHz <-> 16 kHz at lowpass_filter_width <= 16 fit). */
int acb_resampler_create(acb_resampler** out, int device, int orig_freq, int new_freq, int width, const float* kernel_host);
int acb_resampler_destroy(acb_resampler* rs);
/* Resamples n_rows rows in one launch.  in: device samples of in_dtype (ACB_F32 | ACB_I16); row i starts at element in_offset[i]
 * (device; NULL => i * in_stride) and has in_length[i] samples (device; NULL => uniform_length).  out: device fp32; row i's
 * acb_resampled_length(len_i) outputs start at out_offset[i] (device; NULL => i * out_stride).  Nothing outside a row is read. */
int acb_resample(const acb_resampler* rs, const void* in, int32_t in_dtype, const int64_t* in_offset, const int64_t* in_length,
                 int64_t in_stride, int64_t uniform_length, int32_t n_rows, float* out, const int64_t* out_offset,
                 int64_t out_stride, void* stream);

/* ---------------------------------------------------------------------------------------------
 * FLAC decoding (RFC 9639) for the dataset driver: LibriSpeech ships as 16 kHz, 16-bit mono FLAC.  The host parses the stream
 * header (section 8: "fLaC", STREAMINFO first, the other metadata blocks skipped); the device decodes the audio frames of many
 * streams in one call, bit-exact:
 *   - frame headers (9.1): both blocking strategies, block-size codes 1-15 including the 8- and 16-bit uncommon forms, sample-rate
 *     codes 0-14 including the uncommon forms, channel assignments 0-10, bit-depth codes, coded numbers of up to 7 bytes, CRC-8;
 *   - subframes (9.2): CONSTANT, VERBATIM, FIXED orders 0-4, LPC orders 1-32, wasted bits, residual coding methods 0 and 1 with
 *     partition orders 0-15 and escaped partitions; left/side, side/right and mid/side stereo (9.2 / 4.2);
 *   - the frame footer (9.3): byte-alignment padding and CRC-16.
 * Rejected: 32-bit samples (the host parse returns ACB_ERR_UNSUPPORTED), negative LPC shifts, coefficient precision 16, reserved
 * codes.  The STREAMINFO MD5 is not verified (it is sequential over the whole stream); every frame's CRC-16 is.
 * Frames are found by searching every byte of a clip's region for a sync whose header has a valid CRC-8 and agrees with STREAMINFO;
 * a candidate is accepted only when it decodes and its CRC-16 matches, and the accepted frames must tile [0, total_samples) in byte
 * order with contiguous byte ranges.  A clip that fails any of this gets a non-zero status; the other clips of the call are decoded.
 * ------------------------------------------------------------------------------------------------------------------ */
#define ACB_FLAC_OK 0
#define ACB_FLAC_BAD_CLIP 1               /* descriptor out of range (channels 1-8, bps 4-24, max_block 1-65536, region < 2 GiB) */
#define ACB_FLAC_TOO_MANY_CANDIDATES 2    /* more sync candidates than acb_flac_candidate_capacity(byte_length) */
#define ACB_FLAC_NOT_TILED 3              /* accepted frames do not tile [0, total_samples): corrupt, truncated or missing frames */

typedef struct acb_flac_clip {     /* one stream, in device memory (72 bytes) */
    int64_t byte_offset;           /* first byte of the stream's audio-frame region in `data` */
    int64_t byte_length;           /* bytes of the region; nothing outside [byte_offset, byte_offset + byte_length) is read */
    int64_t total_samples;         /* samples per channel (STREAMINFO, or recovered by the host when STREAMINFO says 0) */
    int64_t out_offset;            /* element of `out` where channel 0 starts */
    int64_t out_stride;            /* elements between channel rows */
    int64_t cand_offset;           /* first candidate slot: exclusive prefix over clips of acb_flac_candidate_capacity(byte_length) */
    int32_t channels, bps, sample_rate, max_block;   /* STREAMINFO */
    int32_t variable;              /* blocking strategy of the stream's frames: 0 fixed (0xFFF8), 1 variable (0xFFF9) */
    int32_t reserved;
} acb_flac_clip;

/* Candidate slots one clip needs: byte_length / 8 + 16 (a frame takes at least 9 bytes). */
int64_t acb_flac_candidate_capacity(int64_t byte_length);
/* Bytes of device workspace for total_candidates slots (the sum of the capacities) and n_clips clips. */
int64_t acb_flac_workspace_bytes(int64_t total_candidates, int32_t n_clips);
/* Decodes n_clips streams: data (device bytes), clips (device [n_clips]).  out: device int16 (ACB_I16, only for bps = 16 streams:
 * the samples themselves) or fp32 (ACB_F32: x / 2^(bps - 1), exact for bps <= 24 and what torchaudio.load returns).  status: device
 * int32 [n_clips], ACB_FLAC_*.  Only frames that pass their CRC-16 are written; a clip with a non-zero status may be partly written.
 * workspace: 16-byte aligned, acb_flac_workspace_bytes(total_candidates, n_clips) bytes.  Three launches on `stream`. */
int acb_flac_decode(const uint8_t* data, const acb_flac_clip* clips, int32_t n_clips, int32_t out_dtype, void* out, int32_t* status,
                    void* workspace, int64_t total_candidates, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AUDIOCALM_B200_H_ */
