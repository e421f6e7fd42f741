// Generic (any n_fft) fused STFT front end + workspace preparation + MFCC second stage.
//
// One CTA turns `2*pairs` consecutive frames of one utterance into power / complex / mel / dB
// features without touching HBM in between:
//   gather frame samples (pad / reflect index math in registers) x window
//   -> two real frames packed as one complex signal (a + i b)
//   -> n_fft-point complex Stockham FFT in shared memory, mixed radix, one output per thread per stage
//   -> un-pack the two Hermitian spectra, scale, |.|^p into a shared power tile
//   -> banded mel projection (each filter only visits its non-zero bins) -> optional dB / log.
// Power-of-two n_fft take the register-FFT kernel in frontend_pow2.cu instead; this file is the
// always-correct path for every other size and for two-sided / complex output.
//
// Reference semantics: src/torchaudio/functional/functional.py:54-145 (spectrogram),
// transforms/_transforms.py:403-415 (MelScale), :701-705 (MFCC log/dB), functional.py:356-404.
#include "common.cuh"
#include "ptx.cuh"

namespace b200a {

// ------------------------------------------------------------------------------------------
// workspace preparation
// ------------------------------------------------------------------------------------------
__global__ void prepare_window_kernel(const float* __restrict__ window, int win_length, int n_fft,
                                      int n_bins, int n_mels, int n_mfcc, int frame_length_norm,
                                      int window_norm, WsHeader* hdr, float* padded) {
  __shared__ double partial[256];
  const int left = (n_fft - win_length) / 2;  // at::stft centres a short window
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_fft; i += blockDim.x) {
    const int j = i - left;
    const float w = (j >= 0 && j < win_length) ? window[j] : 0.f;
    padded[i] = w;
    acc += (double)w * (double)w;
  }
  partial[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) partial[threadIdx.x] += partial[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double scale = 1.0;
    if (frame_length_norm) scale *= 1.0 / sqrt((double)n_fft);
    if (window_norm) scale *= 1.0 / sqrt(partial[0]);
    hdr->magic = kWsMagic;
    hdr->n_fft = n_fft;
    hdr->n_bins = n_bins;
    hdr->n_mels = n_mels;
    hdr->n_mfcc = n_mfcc;
    hdr->scale = (float)scale;
  }
}

__global__ void prepare_twiddle_kernel(int n_fft, float2* tw) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < n_fft) {
    double s, c;
    sincospi(-2.0 * (double)q / (double)n_fft, &s, &c);
    tw[q] = make_float2((float)c, (float)s);
  }
}

// One thread per filter: copy the column and record its non-zero bin range [lo, hi).
__global__ void prepare_fbank_kernel(const float* __restrict__ fb, int n_bins, int n_mels,
                                     float* fb_copy, int2* bands) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_mels) return;
  int lo = n_bins, hi = 0;
  for (int k = 0; k < n_bins; ++k) {
    const float v = fb[(size_t)k * n_mels + m];
    fb_copy[(size_t)k * n_mels + m] = v;
    if (v != 0.f) {
      lo = min(lo, k);
      hi = k + 1;
    }
  }
  if (hi == 0) lo = 0;
  bands[m] = make_int2(lo, hi);
}

__global__ void copy_kernel(const float* __restrict__ src, float* dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

// ------------------------------------------------------------------------------------------
// generic fused kernel
// ------------------------------------------------------------------------------------------
struct GenericParams {
  const float* wave;
  int64_t length, row_stride;
  int64_t frames;         // T
  int64_t tiles_per_row;  // ceil(T / (2*pairs))
  float* out;
  float* group_max;
  int64_t rows_per_group;
  const float* window;  // [n_fft] centre padded
  const float2* twiddle;
  const int2* bands;
  const float* fb;
  const WsHeader* hdr;
  int n_fft, hop, pad, center, pad_mode, n_bins, n_mels;
  int pairs;
  int n_stages;
  int radix[kMaxStages];
  int stage;  // b200a_stage
  int log_mels;
  float power, db_mult, db_amin, db_offset;
  // output row geometry (Kaldi features put the frame energy next to the spectral values)
  int out_width, out_col0;
  // Kaldi framing and per-frame conditioning (compliance/kaldi.py:44-83, :153-226); kaldi == 0: torch.stft framing
  int kaldi, k_win, k_snip, k_dc, k_energy_mode, k_energy_col, k_log;
  float k_preemph, k_energy_floor;
};

constexpr float kKaldiEps = 1.1920928955078125e-07f;  // numeric_limits<float>::epsilon(), kaldi.py:21-22

// Sample n of Kaldi frame t (kaldi.py:_get_strided).  snip_edges: frames lie inside the signal.  Otherwise the
// signal is extended by its mirror image on both sides (x[-1-j] = x[j], x[L+j] = x[L-1-j]) and frame t starts
// at t*shift - (win/2 - shift/2).
__device__ __forceinline__ float kaldi_sample(const float* __restrict__ x, int64_t length, int64_t t, int n, int win,
                                              int shift, int snip) {
  int64_t j = t * shift + n;
  if (!snip) {
    j -= win / 2 - shift / 2;
    if (j < 0) j = -1 - j;
    if (j >= length) j = 2 * length - 1 - j;
    if (j < 0 || j >= length) return 0.f;  // only for signals shorter than half a frame
  }
  return x[j];
}

// ------------------------------------------------------------------------------------------
// Stockham autosort FFT of `pairs` signals of N points in shared memory (forward transform, twiddles W^q in tw[q]).
// Radix 2 / 3 / 4 / 5 stages: ONE BUTTERFLY PER THREAD -- R inputs are read once, twiddled (R-1 complex multiplies),
// passed through the radix's few-multiply DFT and written to their R outputs.  Any other prime radix: one OUTPUT per
// thread with the direct R-term sum.  Returns the buffer that holds the result (natural order); the other one is free.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 cmulf(float2 a, float2 b) {
  return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 mul_neg_i(float2 a) { return make_float2(a.y, -a.x); }  // a * (-i)

template <int R>
__device__ __forceinline__ void butterfly_stage(const float2* __restrict__ src, float2* __restrict__ dst,
                                                const float2* __restrict__ tw, int N, int Ns, int pairs, int tid,
                                                int nthr) {
  const int NR = N / R, span = Ns * R, step = N / span;
  for (int b = tid; b < pairs * NR; b += nthr) {
    const int pr = b / NR, j = b - pr * NR;
    const int blk = j / Ns, k = j - blk * Ns;
    const float2* in = src + (size_t)pr * N + j;
    float2 x[R];
    x[0] = in[0];
#pragma unroll
    for (int r = 1; r < R; ++r) x[r] = cmulf(in[(size_t)r * NR], tw[r * k * step]);
    float2* out = dst + (size_t)pr * N + blk * span + k;
    if constexpr (R == 2) {
      out[0] = cadd(x[0], x[1]);
      out[Ns] = csub(x[0], x[1]);
    } else if constexpr (R == 3) {
      const float2 s = cadd(x[1], x[2]), d = csub(x[1], x[2]);
      const float2 m = make_float2(fmaf(-0.5f, s.x, x[0].x), fmaf(-0.5f, s.y, x[0].y));
      const float2 n = make_float2(0.86602540378443865f * d.y, -0.86602540378443865f * d.x);
      out[0] = cadd(x[0], s);
      out[Ns] = cadd(m, n);
      out[2 * Ns] = csub(m, n);
    } else if constexpr (R == 4) {
      const float2 t0 = cadd(x[0], x[2]), t1 = csub(x[0], x[2]), t2 = cadd(x[1], x[3]), t3 = mul_neg_i(csub(x[1], x[3]));
      out[0] = cadd(t0, t2);
      out[Ns] = cadd(t1, t3);
      out[2 * Ns] = csub(t0, t2);
      out[3 * Ns] = csub(t1, t3);
    } else {  // R == 5
      constexpr float c1 = 0.30901699437494742f, c2 = -0.80901699437494742f;
      constexpr float s1 = 0.95105651629515357f, s2 = 0.58778525229247313f;
      const float2 a = cadd(x[1], x[4]), bb = cadd(x[2], x[3]), c = csub(x[1], x[4]), d = csub(x[2], x[3]);
      const float2 p1 = make_float2(fmaf(c1, a.x, fmaf(c2, bb.x, x[0].x)), fmaf(c1, a.y, fmaf(c2, bb.y, x[0].y)));
      const float2 p2 = make_float2(fmaf(c2, a.x, fmaf(c1, bb.x, x[0].x)), fmaf(c2, a.y, fmaf(c1, bb.y, x[0].y)));
      const float2 q1 = mul_neg_i(make_float2(fmaf(s1, c.x, s2 * d.x), fmaf(s1, c.y, s2 * d.y)));
      const float2 q2 = mul_neg_i(make_float2(fmaf(s2, c.x, -s1 * d.x), fmaf(s2, c.y, -s1 * d.y)));
      out[0] = cadd(x[0], cadd(a, bb));
      out[Ns] = cadd(p1, q1);
      out[2 * Ns] = cadd(p2, q2);
      out[3 * Ns] = csub(p2, q2);
      out[4 * Ns] = csub(p1, q1);
    }
  }
}

__device__ __forceinline__ float2* stockham_fft(float2* buf0, float2* buf1, const float2* tw, int N, int pairs,
                                                const int* radix, int n_stages, int tid, int nthr) {
  float2* src = buf0;
  float2* dst = buf1;
  int Ns = 1;
  for (int st = 0; st < n_stages; ++st) {
    const int R = radix[st];
    if (R == 4) butterfly_stage<4>(src, dst, tw, N, Ns, pairs, tid, nthr);
    else if (R == 2) butterfly_stage<2>(src, dst, tw, N, Ns, pairs, tid, nthr);
    else if (R == 5) butterfly_stage<5>(src, dst, tw, N, Ns, pairs, tid, nthr);
    else if (R == 3) butterfly_stage<3>(src, dst, tw, N, Ns, pairs, tid, nthr);
    else {
      const int span = Ns * R, NR = N / R;
      const int step_stage = N / span, step_dft = NR;
      for (int o = tid; o < pairs * N; o += nthr) {
        const int pr = o / N, i = o - pr * N;
        const int blk = i / span, rem = i - blk * span;
        const int q = rem / Ns, k = rem - q * Ns;
        const float2* in = src + (size_t)pr * N + blk * Ns + k;
        const int e1 = (k * step_stage + q * step_dft) % N;
        float2 acc = in[0];
        int e = e1;
        for (int r = 1; r < R; ++r) {
          const float2 v = in[(size_t)r * NR];
          const float2 w = tw[e];
          acc.x = fmaf(v.x, w.x, fmaf(-v.y, w.y, acc.x));
          acc.y = fmaf(v.x, w.y, fmaf(v.y, w.x, acc.y));
          e += e1;
          if (e >= N) e -= N;
        }
        dst[o] = acc;
      }
    }
    __syncthreads();
    float2* t = src;
    src = dst;
    dst = t;
    Ns *= R;
  }
  return src;
}

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}

__device__ __forceinline__ float spectral_power(float re, float im, float power) {
  if (power == 2.f) return fmaf(re, re, im * im);
  const float mag = hypotf(re, im);
  if (power == 1.f) return mag;
  return powf(mag, power);
}

__global__ void __launch_bounds__(256) stft_generic_kernel(const GenericParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.n_fft;
  const int pairs = p.pairs;
  float2* buf0 = reinterpret_cast<float2*>(smem_raw);
  float2* buf1 = buf0 + (size_t)pairs * N;
  float2* tw = buf1 + (size_t)pairs * N;

  const int tid = threadIdx.x;
  const int nthr = blockDim.x;
  const int64_t row = blockIdx.x / p.tiles_per_row;
  const int64_t tile = blockIdx.x - row * p.tiles_per_row;
  const int64_t t0 = tile * (2 * pairs);
  const float* __restrict__ x = p.wave + row * p.row_stride;
  const int half = p.center ? N / 2 : 0;

  for (int i = tid; i < N; i += nthr) tw[i] = p.twiddle[i];

  if (p.kaldi) {
    // ---- Kaldi conditioning: raw frames -> (DC removal) -> [raw energy] -> pre-emphasis -> window -> [energy] ----
    float* raw = reinterpret_cast<float*>(buf1);   // [pair][n][2]
    float* cond = reinterpret_cast<float*>(buf0);  // same layout: z[n] = frame_a[n] + i frame_b[n]
    const int win = p.k_win;
    for (int o = tid; o < pairs * N; o += nthr) {
      const int pr = o / N, n = o - pr * N;
      const int64_t ta = t0 + 2 * pr, tb = ta + 1;
      float a = 0.f, b = 0.f;
      if (n < win) {
        if (ta < p.frames) a = kaldi_sample(x, p.length, ta, n, win, p.hop, p.k_snip);
        if (tb < p.frames) b = kaldi_sample(x, p.length, tb, n, win, p.hop, p.k_snip);
      }
      buf1[o] = make_float2(a, b);
    }
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
    for (int f = warp; f < 2 * pairs; f += nwarps) {  // one warp per frame
      const float* fr = raw + (size_t)(f >> 1) * N * 2 + (f & 1);
      float* dstf = cond + (size_t)(f >> 1) * N * 2 + (f & 1);
      float mean = 0.f;
      if (p.k_dc) {
        float sum = 0.f;
        for (int n = lane; n < win; n += 32) sum += fr[2 * n];
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mean = sum / (float)win;
      }
      float energy = 0.f;
      if (p.k_energy_mode == 1)
        for (int n = lane; n < win; n += 32) {
          const float v = fr[2 * n] - mean;
          energy = fmaf(v, v, energy);
        }
      for (int n = lane; n < N; n += 32) {
        float v = 0.f;
        if (n < win) {
          const float cur = fr[2 * n] - mean, prev = fr[2 * (n > 0 ? n - 1 : 0)] - mean;
          v = (cur - p.k_preemph * prev) * p.window[n];
        }
        dstf[2 * n] = v;
        if (p.k_energy_mode == 2) energy = fmaf(v, v, energy);
      }
      const int64_t t = t0 + f;
      if (p.k_energy_mode != 0 && p.k_energy_col >= 0 && t < p.frames) {
        for (int o = 16; o > 0; o >>= 1) energy += __shfl_xor_sync(0xffffffffu, energy, o);
        float le = logf(fmaxf(energy, kKaldiEps));
        if (p.k_energy_floor > 0.f) le = fmaxf(le, logf(p.k_energy_floor));
        if (lane == 0) p.out[(row * p.frames + t) * p.out_width + p.k_energy_col] = le;
      }
    }
    __syncthreads();
  } else
  // ---- gather + window: z[n] = w[n] * (frame_a[n] + i frame_b[n]) --------------------------
  for (int o = tid; o < pairs * N; o += nthr) {
    const int pr = o / N, n = o - pr * N;
    const int64_t ta = t0 + 2 * pr, tb = ta + 1;
    const float w = p.window[n];
    float a = 0.f, b = 0.f;
    if (ta < p.frames) {
      const int64_t s = source_index(ta * p.hop + n, p.length, p.pad, half, p.pad_mode);
      if (s >= 0) a = x[s] * w;
    }
    if (tb < p.frames) {
      const int64_t s = source_index(tb * p.hop + n, p.length, p.pad, half, p.pad_mode);
      if (s >= 0) b = x[s] * w;
    }
    buf0[o] = make_float2(a, b);
  }
  __syncthreads();

  // ---- Stockham autosort FFT in shared memory ------------------------------------------------
  float2* src = stockham_fft(buf0, buf1, tw, N, pairs, p.radix, p.n_stages, tid, nthr);
  float2* dst = src == buf0 ? buf1 : buf0;
  // `src` now holds Z[k] = A[k] + i B[k] in natural order; `dst` is free.
  const float scale = p.hdr->scale;
  const int n_bins = p.n_bins;
  const float hs = 0.5f * scale;
  float* tile_pow = reinterpret_cast<float*>(dst);  // [2*pairs][n_bins] (n_bins <= N, fits)

  for (int o = tid; o < pairs * n_bins; o += nthr) {
    const int pr = o / n_bins, k = o - pr * n_bins;
    const float2 z = src[(size_t)pr * N + k];
    const float2 zm = src[(size_t)pr * N + (k == 0 ? 0 : N - k)];
    // A = (Z[k] + conj Z[N-k]) / 2,  B = (Z[k] - conj Z[N-k]) / (2i)
    const float are = (z.x + zm.x) * hs, aim = (z.y - zm.y) * hs;
    const float bre = (z.y + zm.y) * hs, bim = (zm.x - z.x) * hs;
    const int64_t ta = t0 + 2 * pr, tb = ta + 1;
    if (p.stage == B200A_STAGE_COMPLEX) {
      float2* o2 = reinterpret_cast<float2*>(p.out);
      if (ta < p.frames) o2[(row * p.frames + ta) * n_bins + k] = make_float2(are, aim);
      if (tb < p.frames) o2[(row * p.frames + tb) * n_bins + k] = make_float2(bre, bim);
    } else {
      float pa = spectral_power(are, aim, p.power);
      float pb = spectral_power(bre, bim, p.power);
      if (p.stage == B200A_STAGE_POWER) {
        if (p.k_log) {  // Kaldi spectrogram: log(max(|X|^2, eps)), kaldi.py:310
          pa = logf(fmaxf(pa, kKaldiEps));
          pb = logf(fmaxf(pb, kKaldiEps));
        }
        if (p.out_col0 + k != p.k_energy_col) {
          if (ta < p.frames) p.out[(row * p.frames + ta) * p.out_width + p.out_col0 + k] = pa;
          if (tb < p.frames) p.out[(row * p.frames + tb) * p.out_width + p.out_col0 + k] = pb;
        }
      } else {
        tile_pow[(size_t)(2 * pr) * n_bins + k] = pa;
        tile_pow[(size_t)(2 * pr + 1) * n_bins + k] = pb;
      }
    }
  }
  if (p.stage < B200A_STAGE_MEL) return;
  __syncthreads();

  // ---- banded mel projection (+ dB / log) ---------------------------------------------------
  const int lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
  float local_max = -CUDART_INF_F;
  for (int f = warp; f < 2 * pairs; f += nwarps) {
    const int64_t t = t0 + f;
    if (t >= p.frames) break;
    const float* pw = tile_pow + (size_t)f * n_bins;
    float* orow = p.out + (row * p.frames + t) * p.out_width + p.out_col0;
    for (int m = lane; m < p.n_mels; m += 32) {
      const int2 band = p.bands[m];
      float acc = 0.f;
      for (int k = band.x; k < band.y; ++k) acc = fmaf(pw[k], p.fb[(size_t)k * p.n_mels + m], acc);
      if (p.stage == B200A_STAGE_FEAT) {
        acc = p.log_mels ? logf(acc + 1e-6f) : p.db_mult * log10f(fmaxf(acc, p.db_amin)) - p.db_offset;
        local_max = fmaxf(local_max, acc);
      }
      if (p.k_log) acc = logf(fmaxf(acc, kKaldiEps));  // Kaldi fbank, kaldi.py:629-631
      orow[m] = acc;
    }
  }
  if (p.stage == B200A_STAGE_FEAT && p.group_max != nullptr) {
    local_max = warp_max(local_max);
    if (lane == 0 && local_max > -CUDART_INF_F) atomic_max_f32(p.group_max + row / p.rows_per_group, local_max);
  }
}

// ------------------------------------------------------------------------------------------
// MFCC second stage: clamp at (group max - top_db), multiply by the DCT matrix
// ------------------------------------------------------------------------------------------
constexpr int kDctRowsPerBlock = 32;

__global__ void __launch_bounds__(256)
mfcc_finish_kernel(const float* __restrict__ feat, int64_t total_rows, int64_t frames, int n_mels,
                   int n_mfcc, const float* __restrict__ dct, const float* __restrict__ group_max,
                   int64_t rows_per_group, float top_db, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_dct = reinterpret_cast<float*>(smem_raw);       // [n_mels][n_mfcc]
  float* s_feat = s_dct + (size_t)n_mels * n_mfcc;          // [rows][n_mels + 1]
  const int ld = n_mels + 1;
  const int64_t r0 = (int64_t)blockIdx.x * kDctRowsPerBlock;  // rows are (utterance, frame) pairs
  const int rows = (int)min((int64_t)kDctRowsPerBlock, total_rows - r0);
  for (int i = threadIdx.x; i < n_mels * n_mfcc; i += blockDim.x) s_dct[i] = dct[i];
  for (int i = threadIdx.x; i < rows * n_mels; i += blockDim.x) {
    const int r = i / n_mels, m = i - r * n_mels;
    float v = feat[(r0 + r) * n_mels + m];
    if (group_max != nullptr && top_db >= 0.f) {
      const int64_t utt = (r0 + r) / frames;
      v = fmaxf(v, group_max[utt / rows_per_group] - top_db);
    }
    s_feat[r * ld + m] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < rows * n_mfcc; i += blockDim.x) {
    const int r = i / n_mfcc, c = i - r * n_mfcc;
    float acc = 0.f;
    for (int m = 0; m < n_mels; ++m) acc = fmaf(s_feat[r * ld + m], s_dct[m * n_mfcc + c], acc);
    out[(r0 + r) * n_mfcc + c] = acc;
  }
}

// Register-tiled variant (n_mfcc <= 64, the usual case): a CTA walks tiles of 128 feature rows; each
// thread owns 4 rows x CPT coefficient columns (columns strided by 8 so that the DCT reads of a warp and
// its output stores are contiguous), features are clamped while they are staged into a padded tile.
constexpr int kFinRows = 128;

template <int CPT>
__global__ void __launch_bounds__(256)
mfcc_finish_tiled_kernel(const float* __restrict__ feat, int64_t total_rows, int64_t frames, int n_mels, int n_mfcc,
                         const float* __restrict__ dct, const float* __restrict__ group_max, int64_t rows_per_group,
                         float top_db, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_dct = reinterpret_cast<float*>(smem_raw);  // [n_mels][8 * CPT], zero padded columns
  const int dld = 8 * CPT;
  const int ld = n_mels + 1;
  float* s_feat = s_dct + (size_t)n_mels * dld;       // [kFinRows][n_mels + 1]
  float* s_floor = s_feat + (size_t)kFinRows * ld;    // [kFinRows] clamp floor of each row
  for (int i = threadIdx.x; i < n_mels * dld; i += blockDim.x) {
    const int m = i / dld, c = i - m * dld;
    s_dct[i] = c < n_mfcc ? dct[m * n_mfcc + c] : 0.f;
  }
  const bool clamp = group_max != nullptr && top_db >= 0.f;
  const int rg = threadIdx.x >> 3, cg = threadIdx.x & 7;  // 32 row groups of 4 rows, 8 column groups
  const int64_t n_tiles = (total_rows + kFinRows - 1) / kFinRows;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * kFinRows;
    const int rows = (int)min((int64_t)kFinRows, total_rows - r0);
    __syncthreads();  // the previous tile has been consumed (and s_dct is complete on the first pass)
    if (threadIdx.x < rows)  // one clamp floor per row (two 64-bit divisions per ROW, not per element)
      s_floor[threadIdx.x] =
          clamp ? group_max[((r0 + threadIdx.x) / frames) / rows_per_group] - top_db : -CUDART_INF_F;
    __syncthreads();
    if ((n_mels & 3) == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0) {
      const int q4 = n_mels >> 2;  // float4 per row
      const float4* src = reinterpret_cast<const float4*>(feat + r0 * n_mels);
      for (int i = threadIdx.x; i < rows * q4; i += blockDim.x) {
        const int r = i / q4, m = (i - r * q4) << 2;
        const float4 v = __ldg(src + i);
        const float fl = s_floor[r];
        float* d = s_feat + r * ld + m;
        d[0] = fmaxf(v.x, fl);
        d[1] = fmaxf(v.y, fl);
        d[2] = fmaxf(v.z, fl);
        d[3] = fmaxf(v.w, fl);
      }
    } else {
      for (int i = threadIdx.x; i < rows * n_mels; i += blockDim.x) {
        const int r = i / n_mels, m = i - r * n_mels;
        s_feat[r * ld + m] = fmaxf(feat[r0 * n_mels + i], s_floor[r]);
      }
    }
    __syncthreads();
    float acc[4][CPT];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int i = 0; i < CPT; ++i) acc[q][i] = 0.f;
    const float* f0 = s_feat + (size_t)(4 * rg) * ld;
#pragma unroll 4
    for (int m = 0; m < n_mels; ++m) {
      float dv[CPT];
#pragma unroll
      for (int i = 0; i < CPT; ++i) dv[i] = s_dct[m * dld + cg + 8 * i];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float a = f0[q * ld + m];
#pragma unroll
        for (int i = 0; i < CPT; ++i) acc[q][i] = fmaf(a, dv[i], acc[q][i]);
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int r = 4 * rg + q;
      if (r < rows) {
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
          const int c = cg + 8 * i;
          if (c < n_mfcc) out[(r0 + r) * n_mfcc + c] = acc[q][i];
        }
      }
    }
  }
}

// Tensor-pipe variant: out[128 rows x n_mfcc] = clamp(feat[128 x n_mels]) * dct on mma.sync m16n8k8 TF32 with
// error-compensated operands (A_hi B_hi + A_lo B_hi + A_hi B_lo, ~2^-21 relative to sum |a b|).  One warp per 16 rows,
// all column tiles; the DCT matrix is kept in shared memory pre-split in B-fragment order.  ~7x fewer issued
// instructions than the FP32 register-tiled kernel above, which is issue bound (54 % issue utilisation at 59 us):
// 59 -> 29 us at config 4.  Used for the dB path of MFCC / LFCC (top_db clamp requested; parity bar 1e-4 relative);
// un-clamped callers -- log-mel MFCC, and the Kaldi MFCC whose goldens hold cepstra (differences of ~20-valued log
// energies) to 1e-5 absolute -- keep the FP32 kernel: a six-product TF32 scheme that reaches fp32 accuracy was measured
// and is no faster than FP32 FMAs here.
constexpr int kMmaFinRows = 128;

__global__ void __launch_bounds__(256)
mfcc_finish_mma_kernel(const float* __restrict__ feat, int64_t total_rows, int64_t frames, int n_mels, int n_mfcc,
                       const float* __restrict__ dct, const float* __restrict__ group_max, int64_t rows_per_group,
                       float top_db, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int ksteps = (n_mels + 7) >> 3, ntiles = (n_mfcc + 7) >> 3;
  const int ldf = 8 * ksteps + 4;  // == 4 (mod 8): rows g, g + 8 x columns c, c + 4 of a fragment hit 32 distinct banks
  float4* s_frag = reinterpret_cast<float4*>(smem_raw);                        // [ksteps][ntiles][32] (b0h, b1h, b0l, b1l)
  float* s_feat = reinterpret_cast<float*>(s_frag + (size_t)ksteps * ntiles * 32);  // [128][ldf]
  float* s_floor = s_feat + (size_t)kMmaFinRows * ldf;                          // [128]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, c = lane & 3;
  for (int i = tid; i < ksteps * ntiles * 32; i += blockDim.x) {
    const int ln = i & 31, nt = (i >> 5) % ntiles, ks = (i >> 5) / ntiles;
    const int n = 8 * nt + (ln >> 2), k0 = 8 * ks + (ln & 3), k1 = k0 + 4;
    const float b0 = (n < n_mfcc && k0 < n_mels) ? dct[(size_t)k0 * n_mfcc + n] : 0.f;
    const float b1 = (n < n_mfcc && k1 < n_mels) ? dct[(size_t)k1 * n_mfcc + n] : 0.f;
    uint32_t h0, l0, h1, l1;
    split_tf32(b0, h0, l0);
    split_tf32(b1, h1, l1);
    s_frag[i] = make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
  }
  for (int i = tid; i < kMmaFinRows * (ldf - n_mels); i += blockDim.x) {  // K padding stays zero
    const int r = i / (ldf - n_mels), k = n_mels + i % (ldf - n_mels);
    s_feat[r * ldf + k] = 0.f;
  }
  const bool clamp = group_max != nullptr && top_db >= 0.f;
  const int64_t n_tiles = (total_rows + kMmaFinRows - 1) / kMmaFinRows;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * kMmaFinRows;
    const int rows = (int)min((int64_t)kMmaFinRows, total_rows - r0);
    __syncthreads();  // the previous tile has been consumed (and the tables are complete on the first pass)
    if (tid < kMmaFinRows)
      s_floor[tid] = (clamp && tid < rows) ? group_max[((r0 + tid) / frames) / rows_per_group] - top_db : -CUDART_INF_F;
    __syncthreads();
    if ((n_mels & 3) == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0) {
      const int q4 = n_mels >> 2;
      const float4* src = reinterpret_cast<const float4*>(feat + r0 * n_mels);
      for (int i = tid; i < kMmaFinRows * q4; i += blockDim.x) {
        const int r = i / q4, m = (i - r * q4) << 2;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < rows) v = __ldg(src + i);
        const float fl = s_floor[r];
        float* d = s_feat + r * ldf + m;
        d[0] = fmaxf(v.x, fl);
        d[1] = fmaxf(v.y, fl);
        d[2] = fmaxf(v.z, fl);
        d[3] = fmaxf(v.w, fl);
      }
    } else {
      for (int i = tid; i < kMmaFinRows * n_mels; i += blockDim.x) {
        const int r = i / n_mels, m = i - r * n_mels;
        s_feat[r * ldf + m] = r < rows ? fmaxf(feat[r0 * n_mels + i], s_floor[r]) : 0.f;
      }
    }
    __syncthreads();
    float acc[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[nt][q] = 0.f;
    const float* a_lo_row = s_feat + (size_t)(16 * warp + g) * ldf + c;
    const float* a_hi_row = a_lo_row + 8 * ldf;
#pragma unroll 2
    for (int ks = 0; ks < ksteps; ++ks) {
      const float av[4] = {a_lo_row[8 * ks], a_hi_row[8 * ks], a_lo_row[8 * ks + 4], a_hi_row[8 * ks + 4]};
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) split_tf32(av[q], hi[q], lo[q]);
      const float4* fr = s_frag + (size_t)ks * ntiles * 32 + lane;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        if (nt < ntiles) {
          const float4 bf = fr[nt * 32];
          mma_tf32(acc[nt], lo, __float_as_uint(bf.x), __float_as_uint(bf.y));
          mma_tf32(acc[nt], hi, __float_as_uint(bf.z), __float_as_uint(bf.w));
          mma_tf32(acc[nt], hi, __float_as_uint(bf.x), __float_as_uint(bf.y));
        }
      }
    }
    const int r_lo = 16 * warp + g, r_hi = r_lo + 8;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt < ntiles) {
        const int n0 = 8 * nt + 2 * c;
        if (r_lo < rows) {
          float* o = out + (r0 + r_lo) * n_mfcc + n0;
          if (n0 < n_mfcc) o[0] = acc[nt][0];
          if (n0 + 1 < n_mfcc) o[1] = acc[nt][1];
        }
        if (r_hi < rows) {
          float* o = out + (r0 + r_hi) * n_mfcc + n0;
          if (n0 < n_mfcc) o[0] = acc[nt][2];
          if (n0 + 1 < n_mfcc) o[1] = acc[nt][3];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int factorize(int n, int* radix) {
  int cnt = 0;
  while (n % 4 == 0) { radix[cnt++] = 4; n /= 4; if (cnt >= kMaxStages) return -1; }
  while (n % 2 == 0) { radix[cnt++] = 2; n /= 2; if (cnt >= kMaxStages) return -1; }
  for (int f = 3; f * f <= n; f += 2)
    while (n % f == 0) { radix[cnt++] = f; n /= f; if (cnt >= kMaxStages) return -1; }
  if (n > 1) { if (cnt >= kMaxStages) return -1; radix[cnt++] = n; }
  return cnt;
}

int validate_desc(const b200a_frontend_desc* d) {
  if (d == nullptr) return B200A_EINVAL;
  if (d->n_fft < 2 || d->hop < 1 || d->win_length < 1 || d->win_length > d->n_fft || d->pad < 0) return B200A_EINVAL;
  if (d->n_fft > kMaxFft) return B200A_EUNSUPPORTED;
  if (d->pad_mode < B200A_PAD_REFLECT || d->pad_mode > B200A_PAD_CIRCULAR) return B200A_EINVAL;
  if (d->n_mels < 0 || d->n_mfcc < 0 || (d->n_mfcc > 0 && d->n_mels == 0)) return B200A_EINVAL;  // LFCC allows n_lfcc > n_filter
  if (d->n_mels > 0 && !d->onesided) return B200A_EINVAL;
  return B200A_OK;
}

int frontend_prepare_impl(const b200a_frontend_desc* d, const float* window, const float* fb,
                          const float* dct, void* ws, size_t ws_bytes, cudaStream_t stream) {
  int rc = validate_desc(d);
  if (rc != B200A_OK) return rc;
  if (window == nullptr || ws == nullptr) return B200A_EINVAL;
  if (d->n_mels > 0 && fb == nullptr) return B200A_EINVAL;
  if (d->n_mfcc > 0 && dct == nullptr) return B200A_EINVAL;
  const WsLayout l = ws_layout(*d);
  if (ws_bytes < l.total) return B200A_EWORKSPACE;
  unsigned char* base = static_cast<unsigned char*>(ws);
  const int n_bins = d->onesided ? d->n_fft / 2 + 1 : d->n_fft;
  prepare_window_kernel<<<1, 256, 0, stream>>>(window, d->win_length, d->n_fft, n_bins, d->n_mels, d->n_mfcc,
                                               d->frame_length_norm, d->window_norm,
                                               reinterpret_cast<WsHeader*>(base + l.header),
                                               reinterpret_cast<float*>(base + l.window));
  prepare_twiddle_kernel<<<(d->n_fft + 255) / 256, 256, 0, stream>>>(d->n_fft, reinterpret_cast<float2*>(base + l.twiddle));
  if (d->n_mels > 0) {
    prepare_fbank_kernel<<<(d->n_mels + 63) / 64, 64, 0, stream>>>(fb, n_bins, d->n_mels,
                                                                  reinterpret_cast<float*>(base + l.fb),
                                                                  reinterpret_cast<int2*>(base + l.bands));
  }
  if (d->n_mfcc > 0) {
    const int64_t n = (int64_t)d->n_mels * d->n_mfcc;
    copy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(dct, reinterpret_cast<float*>(base + l.dct), n);
  }
  return launch_status();
}

int frontend_run_generic(const b200a_frontend_desc* d, const void* ws, int stage, const float* wave,
                         int64_t rows, int64_t length, int64_t row_stride, int64_t frames, float* out,
                         float* group_max, int64_t rows_per_group, cudaStream_t stream,
                         const b200a_kaldi_desc* kd) {
  const WsLayout l = ws_layout(*d);
  const unsigned char* base = static_cast<const unsigned char*>(ws);
  GenericParams p{};
  p.n_stages = factorize(d->n_fft, p.radix);
  if (p.n_stages < 0) return B200A_EUNSUPPORTED;
  p.wave = wave;
  p.length = length;
  p.row_stride = row_stride;
  p.frames = frames;
  p.out = out;
  p.group_max = group_max;
  p.rows_per_group = rows_per_group > 0 ? rows_per_group : 1;
  p.window = reinterpret_cast<const float*>(base + l.window);
  p.twiddle = reinterpret_cast<const float2*>(base + l.twiddle);
  p.bands = reinterpret_cast<const int2*>(base + l.bands);
  p.fb = reinterpret_cast<const float*>(base + l.fb);
  p.hdr = reinterpret_cast<const WsHeader*>(base + l.header);
  p.n_fft = d->n_fft;
  p.hop = d->hop;
  p.pad = d->pad;
  p.center = d->center;
  p.pad_mode = d->pad_mode;
  p.n_bins = d->onesided ? d->n_fft / 2 + 1 : d->n_fft;
  p.n_mels = d->n_mels;
  p.stage = stage;
  p.log_mels = d->log_mels;
  p.power = d->power;
  p.db_mult = d->db_multiplier;
  p.db_amin = d->db_amin;
  p.db_offset = d->db_offset;
  p.out_width = stage >= B200A_STAGE_MEL ? p.n_mels : p.n_bins;
  p.out_col0 = 0;
  p.k_energy_col = -1;
  if (kd != nullptr) {
    p.kaldi = 1;
    p.k_win = kd->window_size;
    p.k_snip = kd->snip_edges;
    p.k_dc = kd->remove_dc_offset;
    p.k_preemph = kd->preemphasis;
    p.k_energy_mode = kd->energy_col >= 0 ? kd->energy_mode : 0;
    p.k_energy_floor = kd->energy_floor;
    p.k_energy_col = kd->energy_col;
    p.k_log = kd->use_log;
    p.out_width = kd->out_width;
    p.out_col0 = kd->out_col0;
  }
  // frames per CTA: enough work for 256 threads, at most ~48 KB of ping-pong buffers
  int pairs = (int)(49152 / (16 * (size_t)d->n_fft));
  if (pairs < 1) pairs = 1;
  if (pairs > 8) pairs = 8;
  while (pairs > 1 && (int64_t)2 * (pairs - 1) >= frames) --pairs;
  p.pairs = pairs;
  p.tiles_per_row = (frames + 2 * pairs - 1) / (2 * pairs);
  const size_t smem = sizeof(float2) * (size_t)d->n_fft * (2 * pairs + 1);
  static_assert(kMaxFft * 8 * 3 <= 227 * 1024, "largest FFT must fit in shared memory");
  if (cudaFuncSetAttribute(stft_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
    return B200A_ECUDA;
  const int64_t grid = rows * p.tiles_per_row;
  if (grid <= 0 || grid > 0x7fffffffLL) return B200A_EUNSUPPORTED;
  stft_generic_kernel<<<(unsigned)grid, 256, smem, stream>>>(p);
  return launch_status();
}

// ------------------------------------------------------------------------------------------
// inverse STFT (torch.istft as called by F.inverse_spectrogram, functional/functional.py:198-218)
// ------------------------------------------------------------------------------------------
struct IstftParams {
  const float2* spec;  // logical [rows][n_bins][frames] complex64, element strides below
  int64_t stride_row, stride_bin, stride_frame;
  int64_t frames, tiles_per_row;
  float* frame_buf;  // [rows][frames][n_fft] windowed time frames
  const float* window;
  const float2* twiddle;
  const WsHeader* hdr;
  int n_fft, pairs, n_stages;
  int radix[kMaxStages];
};

// One CTA = 2*pairs frames of one row: Z = A + i B from the two Hermitian spectra, inverse FFT as
// conj(FFT(conj Z)) / n_fft with the forward Stockham stages, a = Re z, b = Im z, times the window and the
// inverse of the forward normalisation.  C2R semantics: the imaginary parts of bins 0 and n_fft/2 are ignored.
__global__ void __launch_bounds__(256) istft_frames_kernel(const IstftParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.n_fft, pairs = p.pairs, n_bins = N / 2 + 1;
  float2* buf0 = reinterpret_cast<float2*>(smem_raw);
  float2* buf1 = buf0 + (size_t)pairs * N;
  float2* tw = buf1 + (size_t)pairs * N;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int64_t row = blockIdx.x / p.tiles_per_row;
  const int64_t tile = blockIdx.x - row * p.tiles_per_row;
  const int64_t t0 = tile * (2 * pairs);
  const float2* __restrict__ sp = p.spec + row * p.stride_row;
  for (int i = tid; i < N; i += nthr) tw[i] = p.twiddle[i];
  // conj(Z[k]), Z[k] = A[k] + i B[k]; for k > N/2 the Hermitian mirror conj(A[N-k]) + i conj(B[N-k])
  for (int o = tid; o < pairs * N; o += nthr) {
    const int pr = o / N, k = o - pr * N;
    const int kk = k < n_bins ? k : N - k;
    const int64_t ta = t0 + 2 * pr, tb = ta + 1;
    float2 a = make_float2(0.f, 0.f), b = a;
    if (ta < p.frames) a = sp[kk * p.stride_bin + ta * p.stride_frame];
    if (tb < p.frames) b = sp[kk * p.stride_bin + tb * p.stride_frame];
    if (kk == 0 || 2 * kk == N) a.y = b.y = 0.f;
    if (k >= n_bins) {
      a.y = -a.y;
      b.y = -b.y;
    }
    // Z = (a.x - b.y) + i (a.y + b.x); store its conjugate
    buf0[o] = make_float2(a.x - b.y, -(a.y + b.x));
  }
  __syncthreads();
  float2* src = stockham_fft(buf0, buf1, tw, N, pairs, p.radix, p.n_stages, tid, nthr);
  const float gain = 1.f / ((float)N * p.hdr->scale);
  for (int o = tid; o < pairs * N; o += nthr) {
    const int pr = o / N, n = o - pr * N;
    const float2 z = src[o];  // FFT(conj Z): Re z = N a[n], Im z = -N b[n]
    const float w = p.window[n] * gain;
    const int64_t ta = t0 + 2 * pr, tb = ta + 1;
    if (ta < p.frames) p.frame_buf[((row * p.frames + ta) * N) + n] = z.x * w;
    if (tb < p.frames) p.frame_buf[((row * p.frames + tb) * N) + n] = -z.y * w;
  }
}

// Overlap-add and window-envelope normalisation: y[s'] = sum_t F[t][s - t hop] / sum_t w^2[s - t hop], s = s' + start,
// frames added in ascending t (deterministic).  Positions beyond the last frame are zero (torch pads, :warns).
__global__ void __launch_bounds__(256) istft_ola_kernel(const float* __restrict__ frame_buf, const float* __restrict__ window,
                                                        int n_fft, int hop, int64_t frames, int64_t start, int64_t out_len,
                                                        float* __restrict__ out, int64_t out_row_stride) {
  const int64_t row = blockIdx.y;
  const int64_t sp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (sp >= out_len) return;
  const int64_t s = sp + start;
  int64_t t_lo = s - n_fft + 1 <= 0 ? 0 : (s - n_fft + hop) / hop;  // ceil((s - n_fft + 1) / hop)
  int64_t t_hi = s / hop;
  if (t_hi > frames - 1) t_hi = frames - 1;
  const float* fb = frame_buf + row * frames * n_fft;
  float acc = 0.f, env = 0.f;
  for (int64_t t = t_lo; t <= t_hi; ++t) {
    const int n = (int)(s - t * hop);
    const float w = window[n];
    acc += fb[t * n_fft + n];
    env = fmaf(w, w, env);
  }
  out[row * out_row_stride + sp] = t_hi >= t_lo ? acc / env : 0.f;
}

int istft_frames_pow2(const b200a_frontend_desc*, const void*, const float*, int64_t, int64_t, int64_t, int64_t, int64_t, float*,
                      cudaStream_t);  // frontend_pow2.cu; B200A_EUNSUPPORTED when the size is not 256 / 512 / 1024

int istft_run_impl(const b200a_frontend_desc* d, const void* ws, const float* spec, int64_t rows, int64_t frames,
                   int64_t stride_row, int64_t stride_bin, int64_t stride_frame, float* frame_buf, float* out,
                   int64_t out_row_stride, int64_t start, int64_t out_len, cudaStream_t stream) {
  const WsLayout l = ws_layout(*d);
  const unsigned char* base = static_cast<const unsigned char*>(ws);
  IstftParams p{};
  p.n_stages = factorize(d->n_fft, p.radix);
  if (p.n_stages < 0) return B200A_EUNSUPPORTED;
  p.spec = reinterpret_cast<const float2*>(spec);
  p.stride_row = stride_row;
  p.stride_bin = stride_bin;
  p.stride_frame = stride_frame;
  p.frames = frames;
  p.frame_buf = frame_buf;
  p.window = reinterpret_cast<const float*>(base + l.window);
  p.twiddle = reinterpret_cast<const float2*>(base + l.twiddle);
  p.hdr = reinterpret_cast<const WsHeader*>(base + l.header);
  p.n_fft = d->n_fft;
  int pairs = (int)(49152 / (16 * (size_t)d->n_fft));
  if (pairs < 1) pairs = 1;
  if (pairs > 8) pairs = 8;
  while (pairs > 1 && (int64_t)2 * (pairs - 1) >= frames) --pairs;
  p.pairs = pairs;
  p.tiles_per_row = (frames + 2 * pairs - 1) / (2 * pairs);
  const size_t smem = sizeof(float2) * (size_t)d->n_fft * (2 * pairs + 1);
  if (cudaFuncSetAttribute(istft_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
    return B200A_ECUDA;
  const int64_t grid = rows * p.tiles_per_row;
  if (grid <= 0 || grid > 0x7fffffffLL || rows > 65535) return B200A_EUNSUPPORTED;
  int rc = istft_frames_pow2(d, ws, spec, rows, frames, stride_row, stride_bin, stride_frame, frame_buf, stream);
  if (rc == B200A_EUNSUPPORTED) {  // any other size: shared-memory Stockham
    istft_frames_kernel<<<(unsigned)grid, 256, smem, stream>>>(p);
    rc = launch_status();
  }
  if (rc != B200A_OK) return rc;
  const int64_t blocks = (out_len + 255) / 256;
  if (blocks > 0x7fffffffLL) return B200A_EUNSUPPORTED;
  istft_ola_kernel<<<dim3((unsigned)blocks, (unsigned)rows), 256, 0, stream>>>(frame_buf, p.window, d->n_fft, d->hop, frames,
                                                                               start, out_len, out, out_row_stride);
  return launch_status();
}

int mfcc_finish_impl(const b200a_frontend_desc* d, const void* ws, const float* feat, int64_t rows,
                     int64_t frames, const float* group_max, int64_t rows_per_group, float top_db,
                     float* out, cudaStream_t stream) {
  const WsLayout l = ws_layout(*d);
  const float* dct = reinterpret_cast<const float*>(static_cast<const unsigned char*>(ws) + l.dct);
  const int64_t total = rows * frames;
  if (total == 0) return B200A_OK;
  if (d->n_mfcc <= 64 && group_max != nullptr && top_db >= 0.f) {  // dB path: tensor-pipe kernel
    const int ksteps = (d->n_mels + 7) / 8, ntiles = (d->n_mfcc + 7) / 8;
    const size_t msmem = sizeof(float4) * (size_t)ksteps * ntiles * 32 + sizeof(float) * ((size_t)kMmaFinRows * (8 * ksteps + 4) + kMmaFinRows);
    if (msmem <= 200 * 1024) {
      if (cudaFuncSetAttribute(mfcc_finish_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
        return B200A_ECUDA;
      const int64_t tiles = (total + kMmaFinRows - 1) / kMmaFinRows;
      const int per_sm = msmem <= 72 * 1024 ? 3 : (msmem <= 110 * 1024 ? 2 : 1);
      const int64_t grid = tiles < 148 * per_sm ? tiles : 148 * per_sm;
      mfcc_finish_mma_kernel<<<(unsigned)grid, 256, msmem, stream>>>(feat, total, frames, d->n_mels, d->n_mfcc, dct, group_max,
                                                                   rows_per_group > 0 ? rows_per_group : 1, top_db, out);
      return launch_status();
    }
  }
  if (d->n_mfcc <= 64) {  // register-tiled persistent kernel
    const int cpt = d->n_mfcc <= 40 ? 5 : 8;
    const size_t tsmem = sizeof(float) * ((size_t)d->n_mels * 8 * cpt + (size_t)kFinRows * (d->n_mels + 2));
    if (tsmem <= 200 * 1024) {
      auto kern = cpt == 5 ? mfcc_finish_tiled_kernel<5> : mfcc_finish_tiled_kernel<8>;
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
        return B200A_ECUDA;
      const int64_t tiles = (total + kFinRows - 1) / kFinRows;
      const int64_t grid = tiles < 148 * 4 ? tiles : 148 * 4;
      kern<<<(unsigned)grid, 256, tsmem, stream>>>(feat, total, frames, d->n_mels, d->n_mfcc, dct, group_max,
                                                   rows_per_group > 0 ? rows_per_group : 1, top_db, out);
      return launch_status();
    }
  }
  const size_t smem = sizeof(float) * ((size_t)d->n_mels * d->n_mfcc + (size_t)kDctRowsPerBlock * (d->n_mels + 1));
  if (smem > 200 * 1024) return B200A_EUNSUPPORTED;
  if (cudaFuncSetAttribute(mfcc_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
    return B200A_ECUDA;
  const int64_t grid = (total + kDctRowsPerBlock - 1) / kDctRowsPerBlock;
  if (grid > 0x7fffffffLL) return B200A_EUNSUPPORTED;
  mfcc_finish_kernel<<<(unsigned)grid, 256, smem, stream>>>(feat, total, frames, d->n_mels, d->n_mfcc, dct, group_max,
                                                            rows_per_group > 0 ? rows_per_group : 1, top_db, out);
  return launch_status();
}

}  // namespace b200a
