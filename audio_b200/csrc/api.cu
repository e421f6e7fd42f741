// extern "C" surface of libb200audio.so -- see include/b200audio.h for the contract.
#include <cmath>

#include "common.cuh"

namespace b200a {
int validate_desc(const b200a_frontend_desc* d);
int frontend_prepare_impl(const b200a_frontend_desc*, const float*, const float*, const float*, void*, size_t, cudaStream_t);
int frontend_run_generic(const b200a_frontend_desc*, const void*, int, const float*, int64_t, int64_t, int64_t, int64_t,
                         float*, float*, int64_t, cudaStream_t, const b200a_kaldi_desc* = nullptr);
int subtract_column_mean_impl(float*, int64_t, int64_t, int64_t, cudaStream_t);
int phase_vocoder_impl(const float*, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, double, const float*, float*, int64_t,
                       cudaStream_t);
int griffinlim_update_impl(const float*, int64_t, int64_t, int64_t, float, const float*, const float*, float, int, float*,
                           int64_t, int64_t, int64_t, cudaStream_t);
int istft_run_impl(const b200a_frontend_desc*, const void*, const float*, int64_t, int64_t, int64_t, int64_t, int64_t, float*,
                   float*, int64_t, int64_t, int64_t, cudaStream_t);
int frontend_run_pow2(const b200a_frontend_desc*, const void*, int, const float*, int64_t, int64_t, int64_t, int64_t,
                      float*, float*, int64_t, cudaStream_t,
                      const b200a_kaldi_desc* = nullptr);  // returns B200A_EUNSUPPORTED when not applicable
size_t pow2_workspace_extra(const b200a_frontend_desc*);
int pow2_prepare(const b200a_frontend_desc*, void*, size_t, cudaStream_t);
int mfcc_finish_impl(const b200a_frontend_desc*, const void*, const float*, int64_t, int64_t, const float*, int64_t, float,
                     float*, cudaStream_t);
int fill_impl(float*, int64_t, float, cudaStream_t);
int ratio_impl(const float*, int64_t, float*, cudaStream_t);
int apply_fbank_impl(const float*, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, const float*, int, float*,
                     cudaStream_t);
int amplitude_to_db_impl(const float*, int64_t, int64_t, float, float, float, float, float*, float*, cudaStream_t);
size_t resample_workspace_bytes_impl(int, int);
int resample_plan_info_impl(int, int, int, int32_t*);
int resample_tc_band_impl(int, int, int, int, int32_t*, int32_t*);
int resample_prepare_impl(const float*, int, int, int, void*, size_t, cudaStream_t);
int resample_run_impl(const void*, const float*, int, int, int, const float*, int64_t, int64_t, int64_t, float*, int64_t,
                      int64_t, cudaStream_t);
}  // namespace b200a

using namespace b200a;

// complex64 data (and the (sum, count) pairs of b200a_ratio_f32) are read and written as float2: 8-byte alignment
static bool misaligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7) != 0; }

#pragma GCC visibility push(default)
extern "C" {

int b200a_version(void) { return B200A_VERSION; }

const char* b200a_strerror(int status) {
  switch (status) {
    case B200A_OK: return "ok";
    case B200A_EINVAL: return "invalid argument";
    case B200A_EUNSUPPORTED: return "configuration not supported by libb200audio";
    case B200A_ESHORT: return "signal too short for this n_fft / padding mode";
    case B200A_EWORKSPACE: return "workspace too small or not prepared";
    case B200A_ECUDA: return "CUDA launch failed";
    default: return "unknown status";
  }
}

int64_t b200a_num_frames(int64_t length, int32_t n_fft, int32_t hop, int32_t center, int32_t pad) {
  if (n_fft < 1 || hop < 1 || length < 0 || pad < 0) return -1;
  const int64_t span = length + 2 * (int64_t)pad + (center ? 2 * (int64_t)(n_fft / 2) : 0);
  if (span < n_fft) return -1;
  return 1 + (span - n_fft) / hop;
}

int64_t b200a_pad_index(int64_t i, int64_t n, int32_t pad_mode) {
  if (i >= 0 && i < n) return i;
  switch (pad_mode) {
    case B200A_PAD_CONSTANT: return -1;
    case B200A_PAD_REFLECT: return i < 0 ? -i : 2 * (n - 1) - i;
    case B200A_PAD_REPLICATE: return i < 0 ? 0 : n - 1;
    default: {
      int64_t j = i % n;
      return j < 0 ? j + n : j;
    }
  }
}

int32_t b200a_num_bins(int32_t n_fft, int32_t onesided) { return onesided ? n_fft / 2 + 1 : n_fft; }

int32_t b200a_resample_width(int32_t orig_r, int32_t new_r, int32_t lowpass_filter_width, double rolloff) {
  // python: base = min(o, n); base *= rolloff; ceil(lpw * o / base)   (functional.py:1346-1359)
  double base = (double)(orig_r < new_r ? orig_r : new_r);
  base *= rolloff;
  return (int32_t)std::ceil((double)lowpass_filter_width * (double)orig_r / base);
}

int64_t b200a_resample_len(int64_t length, int32_t orig_r, int32_t new_r) {
  // python: torch.ceil(torch.as_tensor(new * L / orig)): exact int product, true (double) division,
  // then as_tensor rounds the python float to the default dtype float32 BEFORE the ceil.
  const double q = (double)((int64_t)new_r * length) / (double)orig_r;
  return (int64_t)std::ceil((float)q);
}

int b200a_resample_support(int32_t orig_r, int32_t new_r, int32_t lowpass_filter_width, double rolloff, int32_t phase,
                           int32_t* first, int32_t* count) {
  // functional.py:1376-1400: tap i of phase j is the windowed sinc at t = (-j/new' + (i - width)/orig') * base,
  // clamped to +-lowpass_filter_width where the window is (numerically) zero: live taps have |t| < lpw.
  if (orig_r < 1 || new_r < 1 || lowpass_filter_width < 1 || !(rolloff > 0.0) || phase < 0 || phase >= new_r ||
      first == nullptr || count == nullptr)
    return B200A_EINVAL;
  const int32_t width = b200a_resample_width(orig_r, new_r, lowpass_filter_width, rolloff);
  const int32_t taps = 2 * width + orig_r;
  const double base = (double)(orig_r < new_r ? orig_r : new_r) * rolloff;
  int32_t lo = taps, hi = -1;
  for (int32_t i = 0; i < taps; ++i) {
    const double t = ((double)(i - width) / (double)orig_r - (double)phase / (double)new_r) * base;
    if (std::fabs(t) < (double)lowpass_filter_width) {
      if (i < lo) lo = i;
      hi = i;
    }
  }
  *first = hi < 0 ? 0 : lo;
  *count = hi < 0 ? 0 : hi - lo + 1;
  return B200A_OK;
}

size_t b200a_frontend_workspace_bytes(const b200a_frontend_desc* desc) {
  if (validate_desc(desc) != B200A_OK) return 0;
  return ws_layout(*desc).total + pow2_workspace_extra(desc);
}

int b200a_frontend_prepare(const b200a_frontend_desc* desc, const float* window, const float* fb, const float* dct,
                           void* workspace, size_t workspace_bytes, b200a_stream stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int rc = frontend_prepare_impl(desc, window, fb, dct, workspace, workspace_bytes, s);
  if (rc != B200A_OK) return rc;
  return pow2_prepare(desc, workspace, workspace_bytes, s);
}

int b200a_frontend_run(const b200a_frontend_desc* desc, const void* workspace, int32_t stage, const float* wave,
                       int64_t rows, int64_t length, int64_t row_stride, float* out, float* group_max,
                       int64_t rows_per_group, b200a_stream stream) {
  int rc = validate_desc(desc);
  if (rc != B200A_OK) return rc;
  if (rows == 0) return B200A_OK;  // empty batch: nothing to enqueue (pointers may be null)
  if (workspace == nullptr || wave == nullptr || out == nullptr) return B200A_EINVAL;
  if (rows < 0 || length < 0 || row_stride < length) return B200A_EINVAL;
  if (stage < B200A_STAGE_COMPLEX || stage > B200A_STAGE_FEAT) return B200A_EINVAL;
  if (stage == B200A_STAGE_COMPLEX && misaligned8(out)) return B200A_EINVAL;
  if (stage >= B200A_STAGE_MEL && desc->n_mels <= 0) return B200A_EINVAL;
  if (stage != B200A_STAGE_COMPLEX && !(desc->power > 0.f)) return B200A_EINVAL;
  const int64_t ext = length + 2 * (int64_t)desc->pad;
  if (desc->center && (desc->pad_mode == B200A_PAD_REFLECT || desc->pad_mode == B200A_PAD_CIRCULAR)) {
    // torch: "Padding size should be less than the corresponding input dimension" (reflect needs
    // pad < n, circular pad <= n); both are reported as ESHORT
    const int64_t half = desc->n_fft / 2;
    if (desc->pad_mode == B200A_PAD_REFLECT ? half >= ext : half > ext) return B200A_ESHORT;
  }
  const int64_t frames = b200a_num_frames(length, desc->n_fft, desc->hop, desc->center, desc->pad);
  if (frames < 1) return B200A_ESHORT;
  if (rows == 0) return B200A_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  rc = frontend_run_pow2(desc, workspace, stage, wave, rows, length, row_stride, frames, out, group_max,
                         rows_per_group, s);
  if (rc != B200A_EUNSUPPORTED) return rc;
  return frontend_run_generic(desc, workspace, stage, wave, rows, length, row_stride, frames, out, group_max,
                              rows_per_group, s);
}

int b200a_mfcc_finish(const b200a_frontend_desc* desc, const void* workspace, const float* feat, int64_t rows,
                      int64_t frames, const float* group_max, int64_t rows_per_group, float top_db, float* out,
                      b200a_stream stream) {
  int rc = validate_desc(desc);
  if (rc != B200A_OK) return rc;
  if (desc->n_mels <= 0 || desc->n_mfcc <= 0) return B200A_EINVAL;
  if (workspace == nullptr || feat == nullptr || out == nullptr || rows < 0 || frames < 0) return B200A_EINVAL;
  return mfcc_finish_impl(desc, workspace, feat, rows, frames, group_max, rows_per_group, top_db, out,
                          static_cast<cudaStream_t>(stream));
}

int b200a_apply_fbank(const float* spec, int64_t rows, int64_t n_bins, int64_t frames, int64_t stride_row,
                      int64_t stride_bin, int64_t stride_frame, const float* fb, int32_t n_filters, float* out,
                      b200a_stream stream) {
  if (spec == nullptr || fb == nullptr || out == nullptr) return B200A_EINVAL;
  if (rows < 0 || n_bins < 1 || frames < 0 || n_filters < 1) return B200A_EINVAL;
  return apply_fbank_impl(spec, rows, n_bins, frames, stride_row, stride_bin, stride_frame, fb, n_filters, out,
                          static_cast<cudaStream_t>(stream));
}

int b200a_amplitude_to_db(const float* x, int64_t groups, int64_t group_elems, float multiplier, float amin,
                          float offset, float top_db, float* scratch, float* out, b200a_stream stream) {
  if (x == nullptr || out == nullptr || groups < 0 || group_elems < 0) return B200A_EINVAL;
  return amplitude_to_db_impl(x, groups, group_elems, multiplier, amin, offset, top_db, scratch, out,
                              static_cast<cudaStream_t>(stream));
}

int b200a_istft_run(const b200a_frontend_desc* desc, const void* workspace, const float* spec, int64_t rows,
                    int64_t frames, int64_t stride_row, int64_t stride_bin, int64_t stride_frame, float* frame_buf,
                    float* out, int64_t out_row_stride, int64_t start, int64_t out_len, b200a_stream stream) {
  int rc = validate_desc(desc);
  if (rc != B200A_OK) return rc;
  if (!desc->onesided || desc->n_fft % 2 != 0) return B200A_EUNSUPPORTED;
  if (rows < 0 || frames < 1 || out_len < 0 || start < 0 || out_row_stride < out_len) return B200A_EINVAL;
  if (rows == 0 || out_len == 0) return B200A_OK;
  if (workspace == nullptr || spec == nullptr || frame_buf == nullptr || out == nullptr) return B200A_EINVAL;
  if (misaligned8(spec)) return B200A_EINVAL;
  return istft_run_impl(desc, workspace, spec, rows, frames, stride_row, stride_bin, stride_frame, frame_buf, out,
                        out_row_stride, start, out_len, static_cast<cudaStream_t>(stream));
}

int b200a_griffinlim_update(const float* mag, int64_t stride_row, int64_t stride_bin, int64_t stride_frame, float inv_power,
                            const float* rebuilt, const float* tprev, float momentum, int32_t normalize, float* proj,
                            int64_t rows, int64_t bins, int64_t frames, b200a_stream stream) {
  if (rows < 0 || bins < 1 || frames < 1 || !(inv_power > 0.f)) return B200A_EINVAL;
  if (rows == 0) return B200A_OK;
  if (mag == nullptr || proj == nullptr || (tprev != nullptr && rebuilt == nullptr)) return B200A_EINVAL;
  if (misaligned8(proj) || misaligned8(rebuilt) || misaligned8(tprev)) return B200A_EINVAL;
  return griffinlim_update_impl(mag, stride_row, stride_bin, stride_frame, inv_power, rebuilt, tprev, momentum, normalize,
                                proj, rows, bins, frames, static_cast<cudaStream_t>(stream));
}

int b200a_phase_vocoder(const float* spec, int64_t stride_row, int64_t stride_bin, int64_t stride_frame, int64_t rows,
                        int64_t bins, int64_t frames_in, double rate, const float* phase_advance, float* out,
                        int64_t frames_out, b200a_stream stream) {
  if (rows < 0 || bins < 1 || frames_in < 1 || frames_out < 0 || !(rate > 0.0)) return B200A_EINVAL;
  if (rows == 0 || frames_out == 0) return B200A_OK;
  if (spec == nullptr || phase_advance == nullptr || out == nullptr) return B200A_EINVAL;
  if (misaligned8(spec) || misaligned8(out)) return B200A_EINVAL;
  return phase_vocoder_impl(spec, stride_row, stride_bin, stride_frame, rows, bins, frames_in, rate, phase_advance, out,
                            frames_out, static_cast<cudaStream_t>(stream));
}

int64_t b200a_kaldi_num_frames(int64_t length, int32_t window_size, int32_t window_shift, int32_t snip_edges) {
  if (length < 0 || window_size < 1 || window_shift < 1) return -1;
  if (snip_edges) return length < window_size ? 0 : 1 + (length - window_size) / window_shift;
  return (length + window_shift / 2) / window_shift;
}

int b200a_kaldi_run(const b200a_kaldi_desc* kaldi, const b200a_frontend_desc* desc, const void* workspace,
                    int32_t stage, const float* wave, int64_t rows, int64_t length, int64_t row_stride,
                    float* out, b200a_stream stream) {
  if (kaldi == nullptr) return B200A_EINVAL;
  int rc = validate_desc(desc);
  if (rc != B200A_OK) return rc;
  if (kaldi->window_size < 2 || kaldi->window_shift < 1 || kaldi->padded_size < kaldi->window_size ||
      kaldi->padded_size % 2 != 0)
    return B200A_EINVAL;
  if (desc->n_fft != kaldi->padded_size || desc->win_length != kaldi->padded_size || desc->hop != kaldi->window_shift ||
      desc->center != 0 || desc->pad != 0 || !desc->onesided)
    return B200A_EINVAL;
  if (stage != B200A_STAGE_POWER && stage != B200A_STAGE_MEL) return B200A_EINVAL;
  if (stage == B200A_STAGE_MEL && desc->n_mels <= 0) return B200A_EINVAL;
  if (!(desc->power > 0.f) || !(kaldi->preemphasis >= 0.f && kaldi->preemphasis <= 1.f)) return B200A_EINVAL;
  if (kaldi->energy_mode < 0 || kaldi->energy_mode > 2 || kaldi->energy_floor < 0.f) return B200A_EINVAL;
  const int values = stage == B200A_STAGE_MEL ? desc->n_mels : desc->n_fft / 2 + 1;
  if (kaldi->out_col0 < 0 || kaldi->out_col0 + values > kaldi->out_width ||
      kaldi->energy_col >= kaldi->out_width)
    return B200A_EINVAL;
  if (rows == 0) return B200A_OK;
  if (workspace == nullptr || wave == nullptr || out == nullptr) return B200A_EINVAL;
  if (rows < 0 || length < 0 || row_stride < length) return B200A_EINVAL;
  if (length < kaldi->window_size) return B200A_ESHORT;  // kaldi.py:142-144
  const int64_t frames = b200a_kaldi_num_frames(length, kaldi->window_size, kaldi->window_shift, kaldi->snip_edges);
  if (frames < 1) return B200A_ESHORT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  rc = frontend_run_pow2(desc, workspace, stage, wave, rows, length, row_stride, frames, out, nullptr, 1, s, kaldi);
  if (rc != B200A_EUNSUPPORTED) return rc;
  return frontend_run_generic(desc, workspace, stage, wave, rows, length, row_stride, frames, out, nullptr, 1, s, kaldi);
}

int b200a_subtract_column_mean(float* x, int64_t rows, int64_t frames, int64_t width, b200a_stream stream) {
  if (rows < 0 || frames < 0 || width < 0) return B200A_EINVAL;
  if (rows == 0 || frames == 0 || width == 0) return B200A_OK;
  if (x == nullptr) return B200A_EINVAL;
  return subtract_column_mean_impl(x, rows, frames, width, static_cast<cudaStream_t>(stream));
}

int b200a_ratio_f32(const float* pairs, int64_t n, float* out, b200a_stream stream) {
  if (n < 0) return B200A_EINVAL;
  if (n == 0) return B200A_OK;
  if (pairs == nullptr || out == nullptr || misaligned8(pairs)) return B200A_EINVAL;
  return ratio_impl(pairs, n, out, static_cast<cudaStream_t>(stream));
}

int b200a_fill_f32(float* dst, int64_t n, float value, b200a_stream stream) {
  if (dst == nullptr || n < 0) return B200A_EINVAL;
  return fill_impl(dst, n, value, static_cast<cudaStream_t>(stream));
}

int b200a_resample_plan_info(int32_t orig_r, int32_t new_r, int32_t width, int32_t* info) {
  return resample_plan_info_impl(orig_r, new_r, width, info);
}

int b200a_resample_tc_band(int32_t orig_r, int32_t new_r, int32_t width, int32_t phase, int32_t* first, int32_t* last) {
  return resample_tc_band_impl(orig_r, new_r, width, phase, first, last);
}

size_t b200a_resample_workspace_bytes(int32_t new_r, int32_t taps) {
  if (new_r < 1 || taps < 1) return 0;
  return resample_workspace_bytes_impl(new_r, taps);
}

int b200a_resample_prepare(const float* kernel, int32_t orig_r, int32_t new_r, int32_t width, void* workspace,
                           size_t workspace_bytes, b200a_stream stream) {
  return resample_prepare_impl(kernel, orig_r, new_r, width, workspace, workspace_bytes,
                               static_cast<cudaStream_t>(stream));
}

int b200a_resample_run(const void* workspace, const float* kernel, int32_t orig_r, int32_t new_r, int32_t width,
                       const float* wave, int64_t rows, int64_t length, int64_t row_stride, float* out,
                       int64_t out_row_stride, int64_t out_len, b200a_stream stream) {
  return resample_run_impl(workspace, kernel, orig_r, new_r, width, wave, rows, length, row_stride, out,
                           out_row_stride, out_len, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
#pragma GCC visibility pop
