/*
 * b200audio.h -- C ABI of libb200audio.so, the sm_100a implementation of torchaudio's DSP
 * front-end hot path (STFT -> |.|^p -> mel -> dB/log -> DCT, and the polyphase sinc resampler).
 *
 * This is the drop-in boundary.  pytorch/audio has no native op for this path (it is Python
 * over ATen: torch.stft / matmul / conv1d); the entry points below are what a native op for it
 * would bind, following the convention of the reference's own native ops
 * (src/libtorchaudio/lfilter.cpp:54-138, src/libtorchaudio/iir_cuda.cu:41-78):
 *   - the caller allocates every buffer, outputs included (Tensor(a!) style);
 *   - kernels are enqueued on the stream the caller passes (cuda_utils.h:9-15), never synchronise;
 *   - arguments are validated and an error CODE is returned (the reference throws via
 *     STD_TORCH_CHECK; a C ABI cannot, and it never aborts -- contrast rnnt/gpu/gpu_transducer.h:20-31).
 * No torch/ATen type crosses this boundary: plain pointers, sizes and one POD descriptor.
 *
 * Rules for every function taking a stream:
 *   - all data pointers are DEVICE pointers on the current device, fp32 unless noted, and 4-byte aligned;
 *     complex64 buffers (marked "8-byte aligned" below) are read and written as float2 and must be 8-byte
 *     aligned -- a misaligned one is B200A_EINVAL, before anything is enqueued.  Every other buffer may sit at
 *     any float offset; kernels that vectorise check the alignment of the pointer they were given;
 *   - the library never allocates, frees or copies device memory behind the caller's back, and
 *     keeps no mutable global state except one-time cudaFuncSetAttribute calls;
 *   - calls are asynchronous; return value 0 (B200A_OK) means "enqueued", a negative value is
 *     one of the B200A_E* codes and nothing was enqueued;
 *   - re-entrant and thread-safe for distinct streams/workspaces.
 *
 * Layouts: spectra and features are FRAME-MAJOR, out[b][t][bin], which is the physical layout of
 * the tensors the reference returns (logical (..., bin, t) with strides (.., 1, n_bins):
 * functional.py:123-137 and transforms/_transforms.py:413 produce transposed views).
 *
 * Citations below are relative to /root/reference/src/torchaudio/.
 */
#ifndef B200AUDIO_H
#define B200AUDIO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200A_VERSION 100 /* 0.1.0 */

typedef void* b200a_stream; /* cudaStream_t */

enum b200a_status {
  B200A_OK = 0,
  B200A_EINVAL = -1,       /* bad argument (null pointer, non-positive size, bad enum) */
  B200A_EUNSUPPORTED = -2, /* valid in the reference, not implemented here (documented) */
  B200A_ESHORT = -3,       /* signal too short: reflect/circular pad needs n_fft/2 < length, or < n_fft samples */
  B200A_EWORKSPACE = -4,   /* workspace too small / not prepared for this descriptor */
  B200A_ECUDA = -5         /* CUDA runtime reported an error at launch (cudaGetLastError) */
};

enum b200a_pad_mode { /* torch.nn.functional.pad modes accepted by torch.stft(center=True) */
  B200A_PAD_REFLECT = 0,
  B200A_PAD_CONSTANT = 1,
  B200A_PAD_REPLICATE = 2,
  B200A_PAD_CIRCULAR = 3
};

/* What the fused front-end kernel writes. */
enum b200a_stage {
  B200A_STAGE_COMPLEX = 0, /* power=None: complex64 STFT, out[b][t][bin][2]        (functional.py:145) */
  B200A_STAGE_POWER = 1,   /* |X|^power,            out[b][t][n_bins]               (functional.py:141-144) */
  B200A_STAGE_MEL = 2,     /* (|X|^power) @ fb,     out[b][t][n_mels]               (transforms/_transforms.py:413) */
  B200A_STAGE_FEAT = 3     /* dB (unclamped) or log(mel+1e-6), out[b][t][n_mels]    (_transforms.py:701-705) */
};

/* One descriptor for Spectrogram / MelSpectrogram / MFCC (the three share the STFT stage). */
typedef struct b200a_frontend_desc {
  int32_t n_fft;             /* FFT size, 2..8192 (any integer; powers of two take the register-FFT path) */
  int32_t win_length;        /* window length <= n_fft; centred zero padding as at::stft does */
  int32_t hop;               /* hop length >= 1 */
  int32_t pad;               /* two-sided constant pre-padding (functional.py:112-114) */
  int32_t center;            /* torch.stft center */
  int32_t pad_mode;          /* enum b200a_pad_mode (only read when center != 0) */
  int32_t onesided;          /* 1: n_bins = n_fft/2+1, 0: n_bins = n_fft */
  int32_t frame_length_norm; /* normalized == "frame_length": X *= n_fft^-1/2 (functional.py:116,131) */
  int32_t window_norm;       /* normalized == True/"window": X /= sqrt(sum w^2)   (functional.py:139-140) */
  float power;               /* exponent > 0; ignored for B200A_STAGE_COMPLEX */
  int32_t n_mels;            /* 0 when no mel stage */
  int32_t n_mfcc;            /* 0 when no DCT stage */
  int32_t log_mels;          /* MFCC: 1 -> log(mel + 1e-6); 0 -> 10*log10(max(mel,1e-10))   */
  float db_multiplier;       /* AmplitudeToDB: 10 (power) or 20 (magnitude) */
  float db_amin;             /* 1e-10 */
  float db_offset;           /* multiplier * log10(max(amin, ref)); 0 for ref = 1 */
} b200a_frontend_desc;

/* ---- library ---------------------------------------------------------------------------- */
int b200a_version(void);
const char* b200a_strerror(int status);

/* ---- integer bookkeeping (host, bit-exact with the reference's shapes) -------------------- */
/* Frames torch.stft yields (functional.py:123-134); -1 when the padded signal is shorter than n_fft. */
int64_t b200a_num_frames(int64_t length, int32_t n_fft, int32_t hop, int32_t center, int32_t pad);
/* Source index in [0,n) for index i of a padded signal, -1 for "zero" (torch/functional.py:675-680). */
int64_t b200a_pad_index(int64_t i, int64_t n, int32_t pad_mode);
/* n_fft/2+1 or n_fft. */
int32_t b200a_num_bins(int32_t n_fft, int32_t onesided);
/* FIR half-width ceil(lpw*orig'/(min(orig',new')*rolloff)) (functional.py:1359). */
int32_t b200a_resample_width(int32_t orig_r, int32_t new_r, int32_t lowpass_filter_width, double rolloff);
/* ceil(new'*L/orig') evaluated as the reference does (functional.py:1427). */
int64_t b200a_resample_len(int64_t length, int32_t orig_r, int32_t new_r);
/* Live taps [first, first + count) of output phase `phase` of the (new', 2*width+orig') sinc kernel: the taps whose
 * window argument lies strictly inside +-lowpass_filter_width (functional.py:1376-1400); every other tap of the row
 * is (numerically) zero.  ~2*lpw*orig'/min(orig',new') taps.  Returns 0 or B200A_EINVAL. */
int b200a_resample_support(int32_t orig_r, int32_t new_r, int32_t lowpass_filter_width, double rolloff, int32_t phase,
                           int32_t* first, int32_t* count);
/* Which kernel b200a_resample_run launches for a ratio, decided on the host from (orig', new', width) alone (never from
 * the batch: a row's result does not depend on what it is batched with).  info[0] = 1 tcgen05 banded product (odd
 * orig', taps and bands fit shared memory), 2 mma.sync TF32x3, 3 direct; info[1] = bytes of the tcgen05 plan's banded
 * bf16 tap blocks, info[2] = its dynamic shared memory, info[3] = tcgen05.mma instructions per 32-frame tile.
 * No reference counterpart (conv1d picks its own algorithm, functional.py:1421).  Returns 0 or B200A_EINVAL. */
int b200a_resample_plan_info(int32_t orig_r, int32_t new_r, int32_t width, int32_t* info);
/* The live-tap band [first, last] the tcgen05 plan assumes for output phase `phase`: (phase*orig'/new',
 * phase*orig'/new' + 2*width), a superset of b200a_resample_support for kernels built like functional.py:1359-1400
 * (checked on the device against the caller's kernel by b200a_resample_prepare).  Returns 0 or B200A_EINVAL. */
int b200a_resample_tc_band(int32_t orig_r, int32_t new_r, int32_t width, int32_t phase, int32_t* first, int32_t* last);

/* ---- fused front end -------------------------------------------------------------------- */
/* Bytes of caller-owned device workspace that b200a_frontend_prepare fills for this descriptor. */
size_t b200a_frontend_workspace_bytes(const b200a_frontend_desc* desc);

/*
 * Build the device-side constant tables (centre-padded window, twiddles, normalisation scale,
 * filterbank band table + copy, DCT copy) from the module's buffers.  Must be re-run whenever
 * `window`, `fb` or `dct` change (the Python modules track tensor versions).
 *   window : [win_length]           Spectrogram.window           (_transforms.py:86-87)
 *   fb     : [n_bins][n_mels] or NULL   MelScale.fb              (_transforms.py:400-401)
 *   dct    : [n_mels][n_mfcc] or NULL   MFCC.dct_mat             (_transforms.py:688-689)
 */
int b200a_frontend_prepare(const b200a_frontend_desc* desc, const float* window, const float* fb,
                           const float* dct, void* workspace, size_t workspace_bytes,
                           b200a_stream stream);

/*
 * Fused STFT front end: replaces F.spectrogram (functional.py:54-145) [+ MelScale.forward
 * (_transforms.py:403-415)] [+ the dB/log step of MFCC.forward (_transforms.py:701-705)].
 *   wave        : [rows] utterances of `length` samples, row r at wave + r*row_stride
 *   stage       : enum b200a_stage
 *   out         : [rows][T][n_bins] (POWER), [rows][T][n_bins][2] (COMPLEX, 8-byte aligned), [rows][T][n_mels] (MEL/FEAT)
 *   group_max   : FEAT only, may be NULL: [ceil(rows/rows_per_group)] running maxima of the dB
 *                 features, combined with atomic max -- the caller initialises them to -inf
 *                 (b200a_fill_f32).  This is the `amax` of functional.py:399; rows_per_group
 *                 encodes the reference's packing rule (functional.py:395-397).
 */
int b200a_frontend_run(const b200a_frontend_desc* desc, const void* workspace, int32_t stage,
                       const float* wave, int64_t rows, int64_t length, int64_t row_stride,
                       float* out, float* group_max, int64_t rows_per_group, b200a_stream stream);

/*
 * Second MFCC stage: top_db clamp + DCT-II, replaces functional.py:399 + _transforms.py:708.
 *   feat      : [rows][T][n_mels] from B200A_STAGE_FEAT
 *   group_max : [groups] maxima (after any cross-rank all-reduce), NULL or top_db < 0 => no clamp
 *   out       : [rows][T][n_mfcc]
 * With a clamp the product runs on the tensor pipe in error-compensated TF32 (~2^-21 relative to sum |feat * dct|, inside
 * the 1e-4 bar of the dB path); without one (log-mel MFCC, Kaldi MFCC) in FP32 FMAs.
 */
int b200a_mfcc_finish(const b200a_frontend_desc* desc, const void* workspace, const float* feat,
                      int64_t rows, int64_t frames, const float* group_max, int64_t rows_per_group,
                      float top_db, float* out, b200a_stream stream);

/* ---- stand-alone stages (MelScale / AmplitudeToDB modules used on their own) ---------------- */
/*
 * out[r][t][m] = sum_k spec[r][k][t] * fb[k][m] for a spectrogram given in the reference's LOGICAL
 * layout (.., n_bins, T) with arbitrary element strides (MelScale.forward, _transforms.py:403-415).
 */
int b200a_apply_fbank(const float* spec, int64_t rows, int64_t n_bins, int64_t frames,
                      int64_t stride_row, int64_t stride_bin, int64_t stride_frame, const float* fb,
                      int32_t n_filters, float* out, b200a_stream stream);

/*
 * F.amplitude_to_DB (functional.py:356-404) over `groups` contiguous chunks of `group_elems` floats:
 * y = mult*log10(max(x, amin)) - offset; if top_db >= 0, y = max(y, max_over_group(y) - top_db).
 * `scratch` holds `groups` floats.
 */
int b200a_amplitude_to_db(const float* x, int64_t groups, int64_t group_elems, float multiplier,
                          float amin, float offset, float top_db, float* scratch, float* out,
                          b200a_stream stream);

int b200a_fill_f32(float* dst, int64_t n, float value, b200a_stream stream);

/*
 * out[i] = pairs[i][0] / pairs[i][1]; `pairs` 8-byte aligned.  Last step of F.spectral_centroid (functional.py:1257-1299): the
 * fused front end is run with the two-column "filterbank" [bin frequency | 1] on the magnitude
 * spectrogram, which yields (sum_k f_k |X_k|, sum_k |X_k|) per frame; this divides them.
 */
int b200a_ratio_f32(const float* pairs, int64_t n, float* out, b200a_stream stream);

/* ---- inverse STFT ---------------------------------------------------------------------------- */
/*
 * torch.istft as F.inverse_spectrogram calls it (functional/functional.py:148-225): Hermitian inverse FFT of every
 * frame (C2R: the imaginary parts of bins 0 and n_fft/2 are ignored), x window, overlap-add, division by the
 * overlap-added squared window, for the output positions [start, start + out_len) of the n_fft + hop*(frames-1)
 * long signal (start = n_fft/2 when center).  The workspace is the one b200a_frontend_prepare built for the same
 * descriptor (window, twiddles, normalisation: `normalized` modes are undone here).  onesided descriptors only.
 *   spec      : complex64, logical [rows][n_fft/2+1][frames], strides in complex elements, 8-byte aligned
 *   frame_buf : caller-owned scratch of rows * frames * n_fft floats (the windowed time frames)
 *   out       : [rows] signals of out_len samples, row r at out + r*out_row_stride
 * The caller checks the window envelope (NOLA) -- torch raises when its minimum is < 1e-11; this library divides.
 */
int b200a_istft_run(const b200a_frontend_desc* desc, const void* workspace, const float* spec, int64_t rows,
                    int64_t frames, int64_t stride_row, int64_t stride_bin, int64_t stride_frame,
                    float* frame_buf, float* out, int64_t out_row_stride, int64_t start, int64_t out_len,
                    b200a_stream stream);

/*
 * One phase step of F.griffinlim (functional/functional.py:330-341):
 *   proj = mag^inv_power * angles,  angles = d / (|d| + 1e-16),  d = rebuilt - momentum * tprev
 * with angles = 1 when rebuilt is NULL (the first inversion, rand_init = False), d = rebuilt when tprev is NULL, and
 * angles = rebuilt as is when normalize == 0 (the first inversion with a random initial phase, :310-311).
 *   mag                   : |X|^power, logical [rows][bins][frames] with element strides (the user's tensor)
 *   rebuilt, tprev, proj  : complex64 frame-major [rows][frames][bins] (what b200a_frontend_run(COMPLEX) writes and
 *                           b200a_istft_run reads with strides (frames*bins, 1, bins)), 8-byte aligned
 */
int b200a_griffinlim_update(const float* mag, int64_t stride_row, int64_t stride_bin, int64_t stride_frame,
                            float inv_power, const float* rebuilt, const float* tprev, float momentum,
                            int32_t normalize, float* proj, int64_t rows, int64_t bins, int64_t frames,
                            b200a_stream stream);

/*
 * F.phase_vocoder (functional/functional.py:713-803): time-stretch a complex spectrogram by `rate` without changing
 * pitch.  Output frame t' interpolates the magnitudes of input frames trunc(ts), trunc(ts + 1), ts = float(rate * t'),
 * and carries the accumulated phase advance; frames_out = ceil(frames_in / rate) (torch.arange(0, frames_in, rate)).
 *   spec          : complex64, logical [rows][bins][frames_in], strides in complex elements, 8-byte aligned
 *   phase_advance : [bins] expected phase advance per hop (linspace(0, pi * hop, bins))
 *   out           : complex64 frame-major [rows][frames_out][bins], 8-byte aligned
 */
int b200a_phase_vocoder(const float* spec, int64_t stride_row, int64_t stride_bin, int64_t stride_frame, int64_t rows,
                        int64_t bins, int64_t frames_in, double rate, const float* phase_advance, float* out,
                        int64_t frames_out, b200a_stream stream);

/* ---- Kaldi-compatible features (compliance/kaldi.py: spectrogram :229-316, fbank :514-645, mfcc :669-813) -------- */
/*
 * Per-frame conditioning and output placement of the Kaldi front end; the transform itself (window, FFT size,
 * |X| or |X|^2, mel matrix) is described by a b200a_frontend_desc with center = 0, n_fft = win_length = padded_size,
 * hop = window_shift, and a workspace prepared by b200a_frontend_prepare from
 *   window : [padded_size]  the Kaldi window (_feature_window_function, :86-113) followed by zeros (:206-211)
 *   fb     : [padded_size/2+1][n_mels]  get_mel_banks(...) transposed, last row zero (:436-511, :623-624), or NULL.
 */
typedef struct b200a_kaldi_desc {
  int32_t window_size;      /* samples per frame, int(sample_frequency * frame_length * 0.001)          (:139) */
  int32_t window_shift;     /* int(sample_frequency * frame_shift * 0.001)                             (:138) */
  int32_t padded_size;      /* FFT size: next power of two of window_size, or window_size; even        (:140) */
  int32_t snip_edges;       /* 1: only frames inside the signal; 0: mirror-extended signal             (:44-83) */
  int32_t remove_dc_offset; /* subtract each frame's mean                                              (:181-184) */
  float preemphasis;        /* s[j] -= c * s[max(0, j-1)]; 0 disables                                  (:191-197) */
  int32_t energy_mode;      /* 0 none, 1 raw (after DC removal, before pre-emphasis), 2 after the window (:186-189,:213-215) */
  float energy_floor;       /* log energy >= log(energy_floor); 0: no floor                            (:116-123) */
  int32_t energy_col;       /* output column that receives the log energy, -1: none                   */
  int32_t out_width;        /* floats per output frame                                                 */
  int32_t out_col0;         /* output column of the first spectral / mel value                         */
  int32_t use_log;          /* log(max(v, FLT_EPSILON)) on the spectral / mel values                   (:310, :629-631) */
} b200a_kaldi_desc;

/* m of _get_strided (:62-68): 1 + (L - win)/shift (0 if L < win) when snip_edges, else (L + shift/2)/shift. */
int64_t b200a_kaldi_num_frames(int64_t length, int32_t window_size, int32_t window_shift, int32_t snip_edges);

/*
 * Fused Kaldi front end: frames -> DC removal -> [raw log energy] -> pre-emphasis -> window -> zero pad -> rFFT ->
 * |X|^power -> [mel] -> [log] for `rows` signals.  stage = B200A_STAGE_POWER (spectrogram) or B200A_STAGE_MEL (fbank).
 *   out : [rows][m][out_width]; spectral value k goes to column out_col0 + k unless that is energy_col.
 * Dither is not offered: the reference draws it with torch.randn per frame element (:176-178), which no
 * other generator reproduces; callers pass dither = 0.
 */
int b200a_kaldi_run(const b200a_kaldi_desc* kaldi, const b200a_frontend_desc* desc, const void* workspace,
                    int32_t stage, const float* wave, int64_t rows, int64_t length, int64_t row_stride,
                    float* out, b200a_stream stream);

/* x[r][t][c] -= mean_t x[r][t][c], in place, for each of `rows` feature matrices (_subtract_column_mean, :219-226). */
int b200a_subtract_column_mean(float* x, int64_t rows, int64_t frames, int64_t width, b200a_stream stream);

/* ---- polyphase sinc resampler ------------------------------------------------------------- */
/* Workspace bytes for b200a_resample_prepare (per-phase tap supports + compacted taps). */
size_t b200a_resample_workspace_bytes(int32_t new_r, int32_t taps);
/*
 * Analyse the cached kernel (Resample.kernel, _transforms.py:955-968; functional.py:1305-1402):
 * find each phase's contiguous non-negligible tap range and write the compacted table.
 *   kernel : [new_r][taps], taps = 2*width + orig_r
 */
int b200a_resample_prepare(const float* kernel, int32_t orig_r, int32_t new_r, int32_t width,
                           void* workspace, size_t workspace_bytes, b200a_stream stream);
/*
 * F._apply_sinc_resample_kernel (functional.py:1405-1432):
 *   out[r][f*new_r + j] = sum_i kernel[j][i] * xpad[r][f*orig_r + i],  xpad = width zeros | x | zeros,
 * for the first out_len = b200a_resample_len(length, orig_r, new_r) outputs of each row.
 */
int b200a_resample_run(const void* workspace, const float* kernel, int32_t orig_r, int32_t new_r,
                       int32_t width, const float* wave, int64_t rows, int64_t length,
                       int64_t row_stride, float* out, int64_t out_row_stride, int64_t out_len,
                       b200a_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B200AUDIO_H */
