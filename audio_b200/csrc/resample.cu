// Polyphase windowed-sinc resampler.
//
// The reference evaluates  y[r][f*new' + j] = sum_i k[j][i] * xpad[r][f*orig' + i]  as a dense
// conv1d with a (new', 1, 2*width+orig') filter and stride orig'
// (src/torchaudio/functional/functional.py:1405-1432).  Almost all of every filter row is
// (numerically) zero: row j only has a contiguous run of ~2*lowpass_width*orig'/min(orig',new')
// taps around the position of output phase j.
//
// The sum IS a banded matrix product
//     Y[f][j] = sum_i X[f][i] * K[j][i],   X[f][i] = x[f*orig' + i - width]  (a strided view of the signal)
// and three kernel families compute it.  rs_choose picks one from the ratio alone, never from the batch, so a row's
// result does not depend on what it is batched with; resample_run_impl adds only the per-call conditions (pointer
// alignment, the 2^31 index bound).
//
// resample_tc_kernel (odd orig', when the banded tcgen05 plan fits: new' <= 160, <= 30 16-tap k-steps, tap blocks
// in shared memory): convert warps build a K-major bf16 hi / lo operand per 32-frame tile, one thread issues
// tcgen05.mma over the phases with live taps in each k-step (bf16 x 3, FP32 accumulate).  The plan is computed on the
// host from (orig', new', width); the device checks it against the measured support of the caller's kernel, and if a
// tap lies outside the band the kernel leaves and resample_mma_kernel, always launched behind it, does the work.
//
// resample_mma_kernel (even orig', or odd orig' beyond the tcgen05 limits, while new' <= 1024 and two staging
// buffers fit): a CTA stages the samples of 32 output frames in shared memory with one bulk asynchronous copy
// (double buffered: the next tile lands while this one is multiplied), and its warps run mma.sync.m16n8k8 TF32 tiles
// of 16 frames x 8 phases over just the k-steps where those 8 phases have live taps, with error-compensated operands
// (X_hi*K_hi + X_lo*K_hi + X_hi*K_lo, ~2^-21 relative).
//
// resample_direct_kernel: one output per thread over the phase's live taps, for ratios whose tiles do not fit
// (new' > 1024, or orig' so large that two 32-frame staging buffers exceed shared memory) and for inputs that are not
// 4-byte aligned.
//
// No padded copy of the input, no (rows, new', frames) intermediate; the output is written already interleaved and
// truncated.  The two tensor-core kernels read each input sample from HBM once and write each output once.
#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace b200a {

namespace {

constexpr int kRsMaxWarps = 24;      // warps per CTA are chosen per ratio so the (half, group) items divide evenly
constexpr int kRsFrames = 32;        // frames per CTA tile (two 16-row MMA tiles)
constexpr int kRsMaxTiles = 128;     // groups of 8 phases  (new' <= 1024)
constexpr int kRsSmemBudget = 224 * 1024;

struct RsTile {  // one group of 8 phases
  int kstart;    // first tap of its first k-step (multiple of 8)
  int nsteps;    // 8-tap k-steps covering the union of the group's live taps
  int frag_off;  // first step in the TF32 fragment array
  int pad;
};
static_assert(sizeof(RsTile) == 16, "the mma kernel's shared-memory layout assumes 16-byte tiles");

struct RsHeader {
  uint32_t magic;
  int32_t orig_r, new_r, width, taps, max_support, n_tiles, total_steps;
  int32_t tc_ok;  // 1: the banded tcgen05 plan fits (resample_tc_kernel applies)
  int32_t reserved[7];
};
static_assert(sizeof(RsHeader) == 64, "header is 64 bytes");

struct RsLayout {
  size_t header, support, tiles, frags, tcblocks, total;
};

constexpr int kTcBBudgetBytes = 64 * 1024;  // banded tap blocks of the tcgen05 kernel

inline int rs_tiles(int new_r) { return (new_r + 7) / 8; }

inline RsLayout rs_layout(int new_r, int taps) {
  RsLayout l{};
  size_t off = 0;
  l.header = off;
  off = align_up(off + sizeof(RsHeader), 256);
  l.support = off;
  off = align_up(off + sizeof(int2) * (size_t)new_r, 256);
  l.tiles = off;
  off = align_up(off + sizeof(RsTile) * (size_t)rs_tiles(new_r), 256);
  l.frags = off;  // worst case: every group spans every tap
  const size_t nt = rs_tiles(new_r) <= kRsMaxTiles ? rs_tiles(new_r) : 0;
  off = align_up(off + sizeof(float4) * 32 * nt * ((size_t)taps / 8 + 2), 256);
  l.tcblocks = off;  // the banded bf16 tap blocks of resample_tc_kernel
  off = align_up(off + (size_t)kTcBBudgetBytes, 256);
  l.total = off;
  return l;
}

// One warp per phase: [first, last] index of taps with |k| > 1e-12 * max|k| of that row.
__global__ void resample_support_kernel(const float* __restrict__ kernel, int new_r, int taps, int orig_r,
                                        int width, RsHeader* hdr, int2* support) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    hdr->magic = kWsMagic;
    hdr->orig_r = orig_r;
    hdr->new_r = new_r;
    hdr->width = width;
    hdr->taps = taps;
  }
  if (j >= new_r) return;
  const float* row = kernel + (size_t)j * taps;
  float mx = 0.f;
  for (int i = lane; i < taps; i += 32) mx = fmaxf(mx, fabsf(row[i]));
  mx = warp_max(mx);
  const float thr = mx * 1e-12f;
  int lo = taps, hi = -1;
  for (int i = lane; i < taps; i += 32) {
    if (fabsf(row[i]) > thr) {
      lo = min(lo, i);
      hi = max(hi, i);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if (lane == 0) {
    if (hi < 0) { lo = 0; hi = -1; }
    support[j] = make_int2(lo, hi - lo + 1);
    atomicMax(&hdr->max_support, hi - lo + 1);
  }
}

// (x, y) -> packed bf16 pair (x in the low half) and the packed pair of the residuals
__device__ __forceinline__ void rs_split_bf16x2(float x, float y, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(y), "f"(x));
  const float rx = x - __uint_as_float(hi << 16), ry = y - __uint_as_float(hi & 0xffff0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(ry), "f"(rx));
}

// Per group of 8 phases: the k-steps its live taps span, and the taps split into TF32 hi/lo parts in
// mma.m16n8k8 B-fragment order (B[k][n] = K[8 t + n][kstart + k]).
__global__ void resample_plan_kernel(const float* __restrict__ kernel, const int2* __restrict__ support, int new_r,
                                     int taps, int n_tiles, RsHeader* hdr, RsTile* tiles, float4* frags) {
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int t = 0; t < n_tiles; ++t) {
      int lo = taps, hi = 0;
      for (int j = 8 * t; j < min(8 * t + 8, new_r); ++j) {
        const int2 sp = support[j];
        if (sp.y > 0) { lo = min(lo, sp.x); hi = max(hi, sp.x + sp.y); }
      }
      RsTile rt{0, 0, acc, 0};
      if (hi > lo) {
        rt.kstart = lo & ~7;
        rt.nsteps = (hi - rt.kstart + 7) / 8;
      }
      tiles[t] = rt;
      acc += rt.nsteps;
    }
    hdr->n_tiles = n_tiles;
    hdr->total_steps = acc;
  }
  __syncthreads();
  for (int t = 0; t < n_tiles; ++t) {
    const RsTile rt = tiles[t];
    for (int i = threadIdx.x; i < rt.nsteps * 32; i += blockDim.x) {
      const int s = i >> 5, lane = i & 31;
      const int j = 8 * t + (lane >> 2);
      const int k0 = rt.kstart + 8 * s + (lane & 3), k1 = k0 + 4;
      const float b0 = (j < new_r && k0 < taps) ? kernel[(size_t)j * taps + k0] : 0.f;
      const float b1 = (j < new_r && k1 < taps) ? kernel[(size_t)j * taps + k1] : 0.f;
      const float b0h = __uint_as_float(__float_as_uint(b0) & 0xffffe000u);
      const float b1h = __uint_as_float(__float_as_uint(b1) & 0xffffe000u);
      frags[(size_t)(rt.frag_off + s) * 32 + lane] = make_float4(b0h, b1h, b0 - b0h, b1 - b1h);
    }
  }
}

struct RsParams {
  const float* wave;
  int64_t rows, length, row_stride;
  float* out;
  int64_t out_row_stride, out_len;
  const RsHeader* hdr;
  const RsTile* tiles;
  const float4* frags;
  int orig_r, new_r, width, taps, n_tiles;
  int64_t frames;           // output frames per row = ceil(out_len / new_r)
  int64_t blocks_per_row;   // ceil(frames / kRsFrames)
  int64_t total_blocks;
  int xs_floats;            // floats per staging buffer
  int frag_smem_bytes;      // shared memory granted to the fragment copy (0: read them from global)
  int row_spread;           // 1, 2 or 4: frame distance of the 8 rows one A-fragment load touches
  int behind_tc;            // launched behind resample_tc_kernel: leave when the header says that kernel did the work
  int out_pair;             // new' and the row pitch are even and `out` is 8-byte aligned: phase pairs are one float2 store
};

// Fill one staging buffer with the samples frames [f0, f0 + 32) of `row` need:
// xs[q] = x[T0 + q - shift] (zero outside the signal), T0 = f0*orig' - width, shift = (-T0) mod 4 so that
// 16-byte aligned global addresses land on 16-byte aligned shared addresses for the bulk copy.
__device__ __forceinline__ int rs_fill(const RsParams& p, int64_t row, int64_t f0, float* xs, uint64_t* bar, int tid,
                                       int nthreads) {
  const int64_t T0 = f0 * p.orig_r - p.width;
  const float* x = p.wave + row * p.row_stride;
  // word address of sample g is a0 + g (mod 4): the bulk copy needs 16-byte aligned global AND shared
  // addresses, so the tile is shifted by 0..3 floats until the two alignments agree
  const int a0 = (int)((reinterpret_cast<uintptr_t>(x) >> 2) & 3);
  const int shift = (int)((((a0 + T0) % 4) + 4) % 4);  // xs index of sample g: q = g - T0 + shift == a0 + g (mod 4)
  const int64_t span = (int64_t)kRsFrames * p.orig_r + p.taps + 16;  // + the zero-tap tail of the last 16-tap step
  const int64_t lo = T0 < 0 ? 0 : T0;
  int64_t hi = T0 + span;
  if (hi > p.length) hi = p.length;
  if (hi < lo) hi = lo;
  const int64_t lo_a = lo + ((4 - ((a0 + lo) & 3)) & 3);  // first sample >= lo on a 16-byte boundary
  const int64_t hi_a = hi - ((a0 + hi) & 3);               // last 16-byte boundary <= hi; bulk part [lo_a, hi_a)
  const int q_lo = (int)(lo - T0) + shift, q_hi = (int)(hi - T0) + shift;
  // zeros where the tile sticks out of the signal (only edge tiles), scalar loads for the (< 4 sample)
  // unaligned head and tail of the bulk range
  if (q_lo > 0 && T0 < 0)
    for (int q = tid; q < q_lo; q += nthreads) xs[q] = 0.f;
  if (hi < T0 + span)
    for (int q = q_hi + tid; q < p.xs_floats; q += nthreads) xs[q] = 0.f;
  if (hi_a > lo_a) {
    const int head = (int)(lo_a - lo), tail = (int)(hi - hi_a);
    if (tid < head) xs[q_lo + tid] = x[lo + tid];
    else if (tid >= 32 && tid < 32 + tail) xs[(int)(hi_a - T0) + shift + (tid - 32)] = x[hi_a + (tid - 32)];
  } else {
    for (int q = q_lo + tid; q < q_hi; q += nthreads) xs[q] = x[T0 + q - shift];
  }
  if (tid == 0) {
    if (hi_a > lo_a) {
      const uint32_t bytes = (uint32_t)(hi_a - lo_a) * 4u;
      mbar_expect_tx(bar, bytes);
      bulk_g2s(xs + (lo_a - T0) + shift, x + lo_a, bytes, bar);
    } else {
      mbar_arrive(bar);  // nothing to copy: complete the phase
    }
  }
  return shift;
}

// Frame (0..31 within the tile) of MMA row rho (0..15) of 16-frame half h, for row spread S in {1, 2, 4}:
// rows rho%8 of one load instruction are S frames apart; the remaining frames fill the gaps.
__device__ __forceinline__ int frame_of(int spread, int h, int rho) {
  const int lo = rho & 7, hi = rho >> 3;
  if (spread == 4) return 4 * lo + hi + 2 * h;
  if (spread == 2) return 16 * h + 2 * lo + hi;
  return 16 * h + rho;
}

// m16n8k8 TF32 x 3 (2^-21 relative)
__global__ void __launch_bounds__(kRsMaxWarps * 32, 1) resample_mma_kernel(const RsParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* s_x = reinterpret_cast<float*>(smem_raw);                              // [2][xs_floats]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_x + 2 * (size_t)p.xs_floats);  // [2]
  RsTile* s_tiles = reinterpret_cast<RsTile*>(s_bar + 2);                       // [n_tiles]
  float4* s_frags = reinterpret_cast<float4*>(s_tiles + ((p.n_tiles + 3) & ~3));  // optional

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (p.behind_tc && p.hdr->tc_ok != 0) return;
  for (int i = tid; i < p.n_tiles; i += blockDim.x) s_tiles[i] = p.tiles[i];
  const int total_steps = p.hdr->total_steps;
  const bool frags_in_smem = (size_t)total_steps * 512 <= (size_t)p.frag_smem_bytes;
  if (frags_in_smem)
    for (int i = tid; i < total_steps * 32; i += blockDim.x) s_frags[i] = p.frags[i];
  if (tid == 0) {
    mbar_init(s_bar + 0, 1);
    mbar_init(s_bar + 1, 1);
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  int shift[2] = {0, 0};
  int64_t blk = blockIdx.x;
  if (blk < p.total_blocks) {
    const int64_t row = blk / p.blocks_per_row, fb = blk - row * p.blocks_per_row;
    shift[0] = rs_fill(p, row, fb * kRsFrames, s_x, s_bar + 0, tid, blockDim.x);
  }
  __syncthreads();  // the scalar part of the first fill is visible
  const int r = lane >> 2, c = lane & 3;
  const int n_warps = blockDim.x >> 5;
  for (int it = 0; blk < p.total_blocks; blk += gridDim.x, ++it) {
    const int b = it & 1;
    const int64_t nxt = blk + gridDim.x;
    if (nxt < p.total_blocks) {  // stage the next tile into the other buffer (its readers finished last iteration)
      const int64_t nrow = nxt / p.blocks_per_row, nfb = nxt - nrow * p.blocks_per_row;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      shift[b ^ 1] = rs_fill(p, nrow, nfb * kRsFrames, s_x + (size_t)(b ^ 1) * p.xs_floats, s_bar + (b ^ 1), tid,
                             blockDim.x);
    }
    // the bulk part of this tile has landed; its scalar part was written before the barrier that ended
    // the previous iteration (or the one after the prologue fill)
    mbar_wait(s_bar + b, (it >> 1) & 1);

    const int64_t row = blk / p.blocks_per_row, fb = blk - row * p.blocks_per_row;
    const int64_t f0 = fb * kRsFrames;
    const float* xs = s_x + (size_t)b * p.xs_floats + shift[b];
    float* orow = p.out + row * p.out_row_stride;
    for (int t = warp; t < p.n_tiles; t += n_warps) {  // one phase group, both 16-frame halves
      const RsTile rt = s_tiles[t];
      // A[f][i] = xs[f*orig' + i].  MMA row rho of 16-frame half h is frame_of(S, h, rho): the 8 rows one load
      // instruction touches are S frames apart so that their 4-word windows fall into different banks
      // (S*orig' == 4 (mod 8) words for odd orig').
      int fr[4];              // frames of rows (h=0: r, r+8), (h=1: r, r+8)
      const float* arow[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        fr[q] = frame_of(p.row_spread, q >> 1, r + 8 * (q & 1));
        arow[q] = xs + (size_t)fr[q] * p.orig_r + rt.kstart + c;
      }
      // per half: three independent accumulator chains (hi*hi, lo*hi, hi*lo), summed in a fixed order
      float d[2][3][4];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int ch = 0; ch < 3; ++ch)
#pragma unroll
          for (int q = 0; q < 4; ++q) d[h][ch][q] = 0.f;
      auto contract = [&](auto in_smem) {
        const float4* frg = (decltype(in_smem)::value ? s_frags : p.frags) + (size_t)rt.frag_off * 32 + lane;
#pragma unroll 2
        for (int s = 0; s < rt.nsteps; ++s) {
          float4 bf;
          if constexpr (decltype(in_smem)::value) bf = frg[(size_t)s * 32];
          else bf = __ldg(frg + (size_t)s * 32);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float av[4] = {arow[2 * h][8 * s], arow[2 * h + 1][8 * s], arow[2 * h][8 * s + 4],
                                 arow[2 * h + 1][8 * s + 4]};
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) split_tf32(av[q], hi[q], lo[q]);
            mma_tf32(d[h][0], hi, __float_as_uint(bf.x), __float_as_uint(bf.y));
            mma_tf32(d[h][1], lo, __float_as_uint(bf.x), __float_as_uint(bf.y));
            mma_tf32(d[h][2], hi, __float_as_uint(bf.z), __float_as_uint(bf.w));
          }
        }
      };
      if (frags_in_smem) contract(std::true_type{});
      else contract(std::false_type{});
      // D rows = frames; columns 2c, 2c+1 = phases 8t + 2c (+1): out index = f*new' + phase
      const int j0 = 8 * t + 2 * c;
      const bool pair_ok = j0 + 1 < p.new_r && p.out_pair != 0;
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int half_row = 0; half_row < 2; ++half_row) {
          const float v0 = d[h][0][2 * half_row] + (d[h][1][2 * half_row] + d[h][2][2 * half_row]);
          const float v1 = d[h][0][2 * half_row + 1] + (d[h][1][2 * half_row + 1] + d[h][2][2 * half_row + 1]);
          const int64_t m = (f0 + fr[2 * h + half_row]) * p.new_r + j0;
          if (pair_ok && m + 1 < p.out_len) {
            *reinterpret_cast<float2*>(orow + m) = make_float2(v0, v1);  // m even, row pitch even, out aligned: 8 bytes
          } else {
            if (j0 < p.new_r && m < p.out_len) orow[m] = v0;
            if (j0 + 1 < p.new_r && m + 1 < p.out_len) orow[m + 1] = v1;
          }
        }
    }
    __syncthreads();  // everyone is done with buffer b before it is refilled
  }
}

// Straightforward one-output-per-thread kernel (any ratio).  Consecutive threads are consecutive
// output samples, i.e. consecutive phases of the same input neighbourhood: input loads hit L1.
__global__ void __launch_bounds__(256)
resample_direct_kernel(const float* __restrict__ wave, int64_t length, int64_t row_stride,
                       const float* __restrict__ kernel, const int2* __restrict__ support, int orig_r,
                       int new_r, int width, int taps, float* __restrict__ out, int64_t out_row_stride,
                       int64_t out_len) {
  const int64_t row = blockIdx.y;
  const float* __restrict__ x = wave + row * row_stride;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < out_len; n += (int64_t)gridDim.x * blockDim.x) {
    const int64_t f = n / new_r;
    const int j = (int)(n - f * new_r);
    const int2 sp = support[j];
    const int64_t base = f * orig_r - width + sp.x;  // input index of the first live tap
    const float* __restrict__ k = kernel + (size_t)j * taps + sp.x;
    float acc = 0.f;
    for (int i = 0; i < sp.y; ++i) {
      const int64_t s = base + i;
      const float v = (s >= 0 && s < length) ? x[s] : 0.f;
      acc = fmaf(k[i], v, acc);
    }
    out[row * out_row_stride + n] = acc;
  }
}

// ================================================================================================
// tcgen05 kernel (resample_tc_kernel): the banded product  Y[f][j] = sum_i X[f][i] K[j][i]  on the 5th-generation
// tensor cores.
//   The strided view X[f][i] = xp[f orig' + i] cannot be described to the tensor core (its rows are orig' samples apart,
//   a K-major core matrix wants them 16 bytes apart), so twelve CONVERT warps materialise it per 32-frame tile as a
//   K-major bf16 operand in shared memory -- the error-compensated hi and lo planes of a frame being two ROWS of the
//   same M = 64 tile, like the mel contraction (frontend_pow2.cu, mel_body_tc2) -- from the tile's contiguous
//   samples, which a producer warp stages with bulk asynchronous copies in four 8-frame units (a unit's buffer is
//   re-filled with the next tile's unit as soon as its convert pass is over).  That is an 8 % expansion (475 taps per
//   441 new samples), read conflict free (lane = frame x 4 consecutive chunks; frames orig' words apart, orig' odd) and
//   written as whole 16-byte core-matrix rows.  The operand is double buffered: tile n + 1 is converted while the
//   tensor core multiplies tile n.
//   One thread issues, per 16-tap k-step, TWO tcgen05.mma (taps_hi, taps_lo accumulate into the same columns) whose
//   B operand holds only the phases that have live taps in that step, banded like the mel filterbank: 60 instructions
//   of N = 8..32 per tile instead of 960 legacy HMMAs.  The accumulator (<= 160 columns) is double buffered in tensor
//   memory; four epilogue warps (one per TMEM lane quadrant) read it (tcgen05.ld), add the hi / lo ROWS of a frame
//   with one shuffle and store 64 bytes per thread.
//   Shared memory at 441:160: 2 x 60 KB operand + 43 KB taps + 4 x 14 KB staged; HBM traffic = the algorithmic bytes.
//   Arithmetic: bf16 x 3 (x_hi k_hi + x_hi k_lo + x_lo k_hi + x_lo k_lo), FP32 accumulate: ~5e-6 of the peak.
// ================================================================================================
constexpr int kTcFrames = 32;          // frames per tile (x 2 planes = the 64 rows of one MMA)
constexpr int kTcUnit = 8;             // frames per staged unit
constexpr int kTcUnits = kTcFrames / kTcUnit;
constexpr int kTcSlots = kTcUnits;  // staged units: slot u holds unit u of the current / next tile
constexpr int kTcMaxKSteps = 30;       // 16-tap k-steps
constexpr int kTcAStride = 1024;       // bytes per 8-tap chunk: 8 row groups x 128 B ([hi | lo] of four 8-frame groups)
// Warp roles by scheduler (warp % 4): the issuer shares its scheduler with one epilogue warp and the (mostly
// sleeping) producer only -- a tcgen05.mma costs ~10 issue slots of that one thread, and behind five busy warps the 61
// instructions of a tile took 6100 cycles instead of 1800.
//   warps 0-3 epilogue (TMEM lane quadrant = warp), 7 issuer, 11 producer, the other warps with warp % 4 != 3 convert
//   (12 of them); warp 15 has no role
constexpr int kTcConvWarps = 12, kTcEpiWarps = 4;  // one epilogue warp per TMEM lane quadrant
constexpr int kTcWarps = kTcEpiWarps + 15;
constexpr int kTcThreads = kTcWarps * 32;
constexpr int kTcIssuerWarp = kTcEpiWarps + 3, kTcProducerWarp = kTcEpiWarps + 7;
constexpr int kTcMaxPhases = 160;     // columns of one accumulator
constexpr int kTcAccStride = 256;      // TMEM columns between the two accumulators
constexpr int kTcSmemLimit = 227 * 1024;
constexpr int kTcIssueBytes = 2 * (2 * kTcMaxKSteps + 2) * 16;  // per accumulator / operand buffer: one uint4 per MMA

struct RsTcSmem {  // byte offsets into dynamic shared memory
  int n_chunks, a_bytes, zero_off, b_off, b_room, x_off, slot_floats, issue_off, bar_off, total;
};
__host__ __device__ inline RsTcSmem rs_tc_smem(int orig_r, int taps) {
  RsTcSmem m;
  m.n_chunks = 2 * ((taps + 15) / 16);
  m.a_bytes = m.n_chunks * kTcAStride;  // one operand buffer; two of them at offset 0
  m.zero_off = 2 * m.a_bytes;           // one all-zero k-step (the accumulator is cleared by multiplying with it)
  m.b_off = m.zero_off + 2 * kTcAStride;
  m.slot_floats = ((kTcUnit - 1) * orig_r + 8 * m.n_chunks + 3 + 3 + 8 + 3) & ~3;  // span + shift + round-up + slack
  const int tail = kTcSlots * m.slot_floats * 4 + kTcIssueBytes + 256;  // + barriers and the unit records
  int room = (kTcSmemLimit - m.b_off - tail) & ~127;
  if (room > kTcBBudgetBytes) room = kTcBBudgetBytes;
  m.b_room = room;  // (<= 0: does not fit)
  m.x_off = m.b_off + (room > 0 ? room : 0);
  m.issue_off = m.x_off + kTcSlots * m.slot_floats * 4;
  m.bar_off = m.issue_off + kTcIssueBytes;
  m.total = m.bar_off + 256;
  return m;
}

struct RsTcStep {
  uint32_t b_off;  // byte offset of the step's tap blocks: [taps_hi: n rows][taps_lo: n rows], each K-major
  uint32_t n;      // phases covered (multiple of 8)
  uint32_t col;    // first phase (multiple of 8)
  uint32_t kstep;  // 16-tap step of the A operand
};
// The band structure, computed on the HOST from (orig', new', width) alone so that the issuing thread reads its
// descriptors from kernel parameters (uniform loads, no register -> uniform-register moves): phase j can have live
// taps only in (j orig'/new', j orig'/new' + 2 width) -- the window of the reference kernel is zero outside +-lowpass
// width and width = ceil(that width x orig'/cutoff) (functional.py:1467-1472, 1514-1519).  The plan kernel checks the
// measured support against this band and clears hdr->tc_ok when a caller's kernel does not honour it.
struct RsTcSteps {
  int ok, steps, b_bytes, n_pad;
  RsTcStep step[kTcMaxKSteps];
};
inline void rs_tc_band(int j, int orig_r, int new_r, int width, int& first, int& last) {  // live taps of phase j: [first, last]
  first = (int)(((int64_t)j * orig_r) / new_r);
  last = (int)(((int64_t)j * orig_r + new_r - 1) / new_r) + 2 * width;
}
inline RsTcSteps rs_tc_steps(int orig_r, int new_r, int width) {
  RsTcSteps t{};
  const int taps = 2 * width + orig_r, k_steps = (taps + 15) / 16;
  const RsTcSmem m = rs_tc_smem(orig_r, taps);
  if (k_steps > kTcMaxKSteps || new_r > kTcMaxPhases || m.b_room <= 0) return t;
  int off = 0;
  for (int s = 0; s < k_steps; ++s) {
    const int t0 = 16 * s, t1 = t0 + 16;
    int lo = new_r, hi = -1;
    for (int j = 0; j < new_r; ++j) {
      int first, last;
      rs_tc_band(j, orig_r, new_r, width, first, last);
      if (first < t1 && last >= t0) {
        if (j < lo) lo = j;
        hi = j;
      }
    }
    if (hi < 0) continue;
    const int n0 = lo / 8 * 8, n = (hi + 1 - n0 + 7) / 8 * 8;
    t.step[t.steps++] = RsTcStep{(uint32_t)off, (uint32_t)n, (uint32_t)n0, (uint32_t)s};
    off += n * 64;
  }
  t.b_bytes = off;
  t.n_pad = (new_r + 7) / 8 * 8;
  // the accumulator is cleared by multiplying an all-zero A k-step with the first n_pad rows of the tap blocks
  t.ok = (t.steps > 0 && off <= m.b_room && off >= t.n_pad * 32) ? 1 : 0;
  return t;
}

// One MMA of a tile as the issuing thread needs it (low descriptor words relative to the operand bases)
struct RsTcMma {
  uint32_t a_lo, b_lo, idesc, col;
};
struct RsTcIssueTab {
  int count, n_pad, b_bytes, count_lo;  // count_lo: MMAs of the low-K half (k-steps < lo_chunks / 2)
  int lo_chunks, pad0, pad1, pad2;
  RsTcMma clear;
  RsTcMma m[2 * kTcMaxKSteps];
};
constexpr uint32_t kTcDescHi = (128u >> 4) | (1u << 14);  // SBO = 128 bytes, descriptor version 1 (bit 46)
inline RsTcIssueTab rs_tc_issue_tab(const RsTcSteps& t, int n_chunks) {
  RsTcIssueTab tab{};
  tab.count = 2 * t.steps;
  tab.n_pad = t.n_pad;
  tab.b_bytes = t.b_bytes;
  tab.lo_chunks = (n_chunks / 4 + 1) / 2 * 4;  // whole items (4 chunks = 2 k-steps)
  tab.count_lo = 0;
  for (int s = 0; s < t.steps; ++s)
    if ((int)t.step[s].kstep * 2 < tab.lo_chunks) tab.count_lo = 2 * (s + 1);
  tab.clear = RsTcMma{(uint32_t)(kTcAStride >> 4) << 16, (uint32_t)((t.n_pad * 16) >> 4) << 16,
                      umma_idesc_bf16(64, t.n_pad), 0u};
  for (int s = 0; s < t.steps; ++s)
    for (int pl = 0; pl < 2; ++pl) {
      const RsTcStep& st = t.step[s];
      RsTcMma& e = tab.m[2 * s + pl];
      e.a_lo = ((st.kstep * 2 * kTcAStride) >> 4) | ((uint32_t)(kTcAStride >> 4) << 16);
      e.b_lo = ((st.b_off + pl * st.n * 32) >> 4) | ((uint32_t)((st.n * 16) >> 4) << 16);
      e.idesc = umma_idesc_bf16(64, (int)st.n);
      e.col = st.col;
    }
  return tab;
}

// Fills the banded bf16 hi / lo tap blocks of the host-side plan and checks every phase's measured support against
// the band the plan assumes.
__global__ void resample_tc_plan_kernel(const float* __restrict__ kernel, const int2* __restrict__ support, int orig_r,
                                        int new_r, int width, int taps, const RsTcSteps plan, RsHeader* hdr,
                                        unsigned char* blocks) {
  __shared__ int s_bad;
  if (threadIdx.x == 0) s_bad = plan.ok ? 0 : 1;
  __syncthreads();
  if (plan.ok) {
    for (int j = threadIdx.x; j < new_r; j += blockDim.x) {
      const int2 sp = support[j];
      const int first = (int)(((int64_t)j * orig_r) / new_r);
      const int last = (int)(((int64_t)j * orig_r + new_r - 1) / new_r) + 2 * width;
      if (sp.y > 0 && (sp.x < first || sp.x + sp.y - 1 > last)) s_bad = 1;
    }
    for (int s = 0; s < plan.steps; ++s) {
      const RsTcStep st = plan.step[s];
      for (int i = threadIdx.x; i < (int)st.n * 16; i += blockDim.x) {
        const int nl = i >> 4, kk = i & 15;
        const int j = (int)st.col + nl, t = 16 * (int)st.kstep + kk;
        float v = 0.f;
        if (j < new_r && t < taps) {
          const int2 sp = support[j];
          if (t >= sp.x && t < sp.x + sp.y) v = kernel[(size_t)j * taps + t];
        }
        uint32_t h, l;
        rs_split_bf16x2(v, 0.f, h, l);
        const size_t o = st.b_off + (size_t)(kk >> 3) * st.n * 16 + (size_t)nl * 16 + (size_t)(kk & 7) * 2;
        *reinterpret_cast<uint16_t*>(blocks + o) = (uint16_t)(h & 0xffffu);
        *reinterpret_cast<uint16_t*>(blocks + o + (size_t)st.n * 32) = (uint16_t)(l & 0xffffu);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) hdr->tc_ok = s_bad ? 0 : 1;
}

struct RsTcParams {
  const float* wave;
  int64_t rows, length, row_stride;
  float* out;
  int64_t out_row_stride, out_len;
  const RsHeader* hdr;
  const unsigned char* blocks;
  int orig_r, new_r, width, taps;
  int64_t frames, tiles_per_row, total_tiles;
  int out_vec;
};
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
        "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
      : "r"(taddr)
      : "memory");
}
// after tcgen05.wait::ld: ties the registers to the wait so that no consumer is scheduled ahead of it
__device__ __forceinline__ void tmem_ld_pin(float (&v)[16]) {
  asm volatile(""
               : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]),
                 "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
               :
               : "memory");
}

__global__ void __launch_bounds__(kTcThreads, 1) resample_tc_kernel(const RsTcParams p, const __grid_constant__ RsTcIssueTab tab) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  if (p.hdr->tc_ok == 0) return;  // (uniform) the mma.sync kernel launched next does the work
  const RsTcSmem m = rs_tc_smem(p.orig_r, p.taps);
  unsigned char* s_a = smem_raw;                                              // [2][n_chunks][1024]
  unsigned char* s_zero = smem_raw + m.zero_off;                              // [2][1024]
  unsigned char* s_b = smem_raw + m.b_off;                                    // tap blocks
  float* s_x = reinterpret_cast<float*>(smem_raw + m.x_off);                  // [kTcSlots][slot_floats]
  uint4* s_issue = reinterpret_cast<uint4*>(smem_raw + m.issue_off);          // [2][2 kTcMaxKSteps + 2]
  uint64_t* s_full = reinterpret_cast<uint64_t*>(smem_raw + m.bar_off);       // [4] staged unit landed
  uint64_t* s_cdone = s_full + kTcSlots;                                      // [4] unit u converted by every warp (slot u free)
  uint64_t* s_aready = s_cdone + kTcSlots;                                    // [2] operand b complete (all convert warps)
  uint64_t* s_mma = s_aready + 2;                                             // [2] MMAs of buffer b complete: D[b] valid, A[b] free
  uint64_t* s_accfree = s_mma + 2;                                            // [2] accumulator b read out
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_accfree + 2);
  int* s_shift = reinterpret_cast<int*>(smem_raw + m.bar_off + 192);          // [4] slot index of the unit's sample T0

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int n_pad = tab.n_pad;
  const int n_chunks = m.n_chunks;
  {
    uint4* a4 = reinterpret_cast<uint4*>(s_a);
    for (int i = tid; i < m.b_off / 16; i += blockDim.x) a4[i] = make_uint4(0, 0, 0, 0);  // both operands + the zero k-step
    const uint4* src = reinterpret_cast<const uint4*>(p.blocks);
    uint4* b4 = reinterpret_cast<uint4*>(s_b);
    for (int i = tid; i < tab.b_bytes / 16; i += blockDim.x) b4[i] = src[i];
    uint4* x4 = reinterpret_cast<uint4*>(s_x);  // frames past the end of a row are converted from whatever the slot holds: keep it finite
    for (int i = tid; i < kTcSlots * m.slot_floats / 4; i += blockDim.x) x4[i] = make_uint4(0, 0, 0, 0);
  }
  // issue records {A descriptor low word, B descriptor low word, instruction descriptor, D column}, final for each
  // of the two (operand, accumulator) buffers: the issuing thread spends one 16-byte load + four moves per MMA
  if (tid <= tab.count) {
    const RsTcMma e = tid == 0 ? tab.clear : tab.m[tid - 1];
    const uint32_t b_base = smem_u32(s_b) >> 4;
    for (int b = 0; b < 2; ++b) {
      const uint32_t a_base = (tid == 0 ? smem_u32(s_zero) : smem_u32(s_a) + (uint32_t)(b * m.a_bytes)) >> 4;
      s_issue[b * (2 * kTcMaxKSteps + 2) + tid] =
          make_uint4(e.a_lo + a_base, e.b_lo + b_base, e.idesc, (uint32_t)(b * kTcAccStride) + e.col);
    }
  }
  if (tid == 0) {
    for (int i = 0; i < kTcSlots; ++i) {
      mbar_init(s_full + i, 1);
      mbar_init(s_cdone + i, kTcConvWarps);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(s_aready + i, kTcConvWarps);
      mbar_init(s_mma + i, 1);
      mbar_init(s_accfree + i, kTcEpiWarps);
    }
  }
  if (warp == 0) tmem_alloc(s_tmem, 512);  // two accumulators of <= 160 columns, kTcAccStride apart
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *reinterpret_cast<volatile uint32_t*>(s_tmem);

  // tiles of this CTA: t = blockIdx.x + n gridDim.x; unit u covers frames f0 + 8 u .. + 7
  auto tile_of = [&](int n, int64_t& row, int64_t& f0) {
    const int64_t t = blockIdx.x + (int64_t)n * gridDim.x;
    if (t >= p.total_tiles) return false;
    if (p.total_tiles < ((int64_t)1 << 31)) {
      const uint32_t r = (uint32_t)t / (uint32_t)p.tiles_per_row;
      row = r;
      f0 = (int64_t)((uint32_t)t - r * (uint32_t)p.tiles_per_row) * kTcFrames;
    } else {
      row = t / p.tiles_per_row;
      f0 = (t - row * p.tiles_per_row) * kTcFrames;
    }
    return true;
  };

  if (warp < kTcEpiWarps) {
    // ============ epilogue warps: TMEM lane quadrant = warp ==========================================================
    int64_t row, f0;
    for (int n = 0; tile_of(n, row, f0); ++n) {
      const int b = n & 1;
      mbar_wait(s_mma + b, (uint32_t)(n >> 1) & 1u);
      tc_fence_after();
      const uint32_t acc = tmem_d + ((uint32_t)(32 * warp) << 16) + (uint32_t)(b * kTcAccStride);
      const int64_t f = f0 + 8 * warp + (lane & 7);  // lanes 0-7: hi rows of frames 8 warp .. + 7, lanes 8-15: their lo rows
      const bool own = lane < 8 && f < p.frames;
      float* orow = p.out + row * p.out_row_stride + f * p.new_r;
      const int64_t n0 = f * p.new_r;
      auto store16 = [&](int j, const float (&y)[16]) {  // (j < n_pad follows from j < new'; ptxas uses 1 register less with it)
        if (p.out_vec && j + 16 <= n_pad && j + 16 <= p.new_r && n0 + j + 16 <= p.out_len) {
#pragma unroll
          for (int q = 0; q < 16; q += 4)
            *reinterpret_cast<float4*>(orow + j + q) = make_float4(y[q], y[q + 1], y[q + 2], y[q + 3]);
        } else {
#pragma unroll
          for (int q = 0; q < 16; ++q)
            if (j + q < n_pad && j + q < p.new_r && n0 + j + q < p.out_len) orow[j + q] = y[q];
        }
      };
      auto finish32 = [&](int j, float (&u)[16], float (&w)[16]) {
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          u[q] += __shfl_down_sync(0xffffffffu, u[q], 8);  // x_hi row + x_lo row
          w[q] += __shfl_down_sync(0xffffffffu, w[q], 8);
        }
        if (own) {
          store16(j, u);
          store16(j + 16, w);
        }
      };
      // two register sets: the tensor-memory load of the next 32 columns is in flight while these are summed and stored
      float ua[16], wa[16], ub[16], wb[16];
      tmem_ld16_nowait(acc, ua);
      tmem_ld16_nowait(acc + 16, wa);  // (columns past n_pad: allocated, never stored)
#pragma unroll 1
      for (int j0 = 0; j0 < n_pad; j0 += 64) {
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        tmem_ld_pin(ua);
        tmem_ld_pin(wa);
        if (j0 + 32 < n_pad) {
          tmem_ld16_nowait(acc + j0 + 32, ub);
          tmem_ld16_nowait(acc + j0 + 48, wb);
        }
        finish32(j0, ua, wa);
        if (j0 + 32 < n_pad) {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          tmem_ld_pin(ub);
          tmem_ld_pin(wb);
          if (j0 + 64 < n_pad) {
            tmem_ld16_nowait(acc + j0 + 64, ua);
            tmem_ld16_nowait(acc + j0 + 80, wa);
          }
          finish32(j0 + 32, ub, wb);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_accfree + b);
    }
    tc_fence_before();
    asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiWarps * 32) : "memory");
    if (warp == 0) tmem_dealloc(tmem_d, 512);
  } else if (warp == kTcIssuerWarp) {
    // ============ issuer warp ======================================================================================
    const bool leader = elect_one();  // ONE thread issues every instruction of the CTA
    auto desc = [](uint32_t lo) { return ((uint64_t)kTcDescHi << 32) | lo; };
    int64_t row, f0;
    for (int n = 0; tile_of(n, row, f0); ++n) {
      const int b = n & 1;
      const uint4* rec = s_issue + b * (2 * kTcMaxKSteps + 2);
      mbar_wait(s_aready + b, (uint32_t)(n >> 1) & 1u);  // every convert warp is through with the tile: operand complete
      if (n >= 2) mbar_wait(s_accfree + b, (uint32_t)((n >> 1) - 1) & 1u);  // tile n - 2 has left this accumulator
      tc_fence_after();
      if (leader) {
        {
          const uint4 e = rec[0];
          umma_bf16(tmem_d + e.w, desc(e.x), desc(e.y), e.z, 0u);  // clear: D = 0 x taps
        }
#pragma unroll 4
        for (int s = 1; s <= tab.count; ++s) {
          const uint4 e = rec[s];
          umma_bf16(tmem_d + e.w, desc(e.x), desc(e.y), e.z, 1u);
        }
        umma_commit(s_mma + b);
      }
      __syncwarp();
    }
  } else if (warp == kTcProducerWarp) {
    // ============ producer warp: unit u of tile n + 1 follows unit u of tile n into slot u ==========================
    // Everything a convert warp reads is put into the slot here: the 16-byte aligned middle by ONE bulk copy, and at
    // the ends of a row the few samples around it and the zeros beyond the signal by this warp (interior units: none).
    auto stage_unit = [&](int n, int u) {
      int64_t row, f0;
      if (!tile_of(n, row, f0)) return;
      const int slot = u;
      const float* x = p.wave + row * p.row_stride;
      const int64_t T0 = (f0 + kTcUnit * u) * p.orig_r - p.width;
      const int a0 = (int)((reinterpret_cast<uintptr_t>(x) >> 2) & 3);
      const int shift = (int)((a0 + (T0 & 3)) & 3);  // slot index of sample T0: the bulk copy keeps its 16-byte phase
      // frames of the unit that exist; the others are converted from stale (finite) slot contents and never stored
      int64_t nv = p.frames - (f0 + kTcUnit * u);
      nv = nv < 0 ? 0 : (nv > kTcUnit ? kTcUnit : nv);
      const int span_v = nv > 0 ? (int)(nv - 1) * p.orig_r + 8 * n_chunks : 0;
      int64_t lo = T0 < 0 ? 0 : T0, hi = T0 + span_v;
      if (hi > p.length) hi = p.length;
      if (lo > p.length) lo = p.length;
      if (hi < lo) hi = lo;
      // 16-byte boundaries OUTSIDE [lo, hi) where the signal has them, inside at the ends of a row
      const int back = (int)((a0 + lo) & 3), fwd = (int)((4 - ((a0 + hi) & 3)) & 3);
      int64_t lo_a = lo - back >= 0 ? lo - back : lo + ((4 - back) & 3);
      int64_t hi_a = hi + fwd <= p.length ? hi + fwd : hi - ((a0 + hi) & 3);
      if (hi_a < lo_a) hi_a = lo_a;
      float* xs = s_x + slot * m.slot_floats;
      const int first = (int)(lo_a - T0) + shift, end = (int)(hi_a - T0) + shift;  // staged by the bulk copy: [first, end)
      for (int i = shift + lane; i < first; i += 32) {
        const int64_t g = T0 + (i - shift);
        xs[i] = (g >= 0 && g < p.length) ? __ldg(x + g) : 0.f;
      }
      for (int i = (end > shift ? end : shift) + lane; i < shift + span_v; i += 32) {
        const int64_t g = T0 + (i - shift);
        xs[i] = (g >= 0 && g < p.length) ? __ldg(x + g) : 0.f;
      }
      if (lane == 0) s_shift[slot] = shift;
      __syncwarp();
      if (lane == 0) {
        uint64_t* bar = s_full + slot;
        if (hi_a > lo_a) {
          const uint32_t bytes = (uint32_t)(hi_a - lo_a) * 4u;
          mbar_expect_tx(bar, bytes);  // (release: the stores above are visible to whoever sees the phase complete)
          bulk_g2s(xs + first, x + lo_a, bytes, bar);
        } else {
          mbar_arrive(bar);
        }
      }
    };
    for (int u = 0; u < kTcUnits; ++u) stage_unit(0, u);
    int64_t row, f0;
    for (int n = 0; tile_of(n, row, f0); ++n) {
#pragma unroll 1
      for (int u = 0; u < kTcUnits; ++u) {
        mbar_wait(s_cdone + u, (uint32_t)n & 1u);
        stage_unit(n + 1, u);
      }
    }
  } else if ((warp & 3) != 3 && warp >= kTcEpiWarps) {
    // ============ convert warps: staged samples -> K-major bf16 hi / lo operand ====================================
    const int cv = ((warp - kTcEpiWarps) >> 2) * 3 + (warp & 3);  // the warps after the epilogue's with warp % 4 != 3 -> 0 .. 11
    const int fl = lane & 7, cq = lane >> 3;  // frame of the unit; this lane converts chunk 4 it + cq
    const int ipu = (n_chunks + 3) / 4;       // items per unit (an item = 8 frames x 4 consecutive chunks)
    const int lane_off = fl * p.orig_r;
    int64_t row, f0;
    for (int n = 0; tile_of(n, row, f0); ++n) {
      const int b = n & 1;
      if (n >= 2) mbar_wait(s_mma + b, (uint32_t)((n >> 1) - 1) & 1u);  // tile n - 2 has been multiplied: operand b is free
      unsigned char* abuf = s_a + b * m.a_bytes;
      int it = cv;  // items of the tile in unit order, dealt round robin: g = u ipu + it belongs to warp g % kTcConvWarps
#pragma unroll 1
      for (int u = 0; u < kTcUnits; ++u) {
        mbar_wait(s_full + u, (uint32_t)n & 1u);  // the unit's samples are staged (every warp waits, items or not)
        const float* xs = s_x + u * m.slot_floats + s_shift[u] + lane_off;  // this frame's tap 0
        // frame F = 8 u + fl: hi row in group 2 u, row fl; the lo row 128 bytes on
        unsigned char* arow = abuf + u * 256 + fl * 16;
        for (; it < ipu; it += kTcConvWarps) {
          const int c = 4 * it + cq;  // lanes 8 q .. 8 q + 7 read 8 q words on from lanes 0-7: conflict free for odd orig'
          if (c < n_chunks) {
            float v[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = xs[8 * c + t];
            uint4 hi, lo;
            rs_split_bf16x2(v[0], v[1], hi.x, lo.x);
            rs_split_bf16x2(v[2], v[3], hi.y, lo.y);
            rs_split_bf16x2(v[4], v[5], hi.z, lo.z);
            rs_split_bf16x2(v[6], v[7], hi.w, lo.w);
            unsigned char* d = arow + c * kTcAStride;
            *reinterpret_cast<uint4*>(d) = hi;
            *reinterpret_cast<uint4*>(d + 128) = lo;
          }
        }
        it -= ipu;  // position within the next unit
        __syncwarp();  // the unit's samples are in registers (or converted): the slot may be re-filled
        if (lane == 0) mbar_arrive(s_cdone + u);
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // my operand rows -> the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(s_aready + b);
    }
  }
}

// The kernel family of a ratio, from (orig', new', width) alone: resample_plan_info_impl reports it and
// resample_run_impl launches it (after the per-call conditions only a run can check).  Never chosen by the batch, so
// a row's result does not depend on what it is batched with.
enum RsFamily { kRsFamilyTc = 1, kRsFamilyMma = 2, kRsFamilyDirect = 3 };  // b200a_resample_plan_info info[0]
struct RsChoice {
  int family;
  RsTcSteps tc;       // the banded tcgen05 plan (tc.ok: it fits)
  int n_tiles;        // mma.sync kernel: groups of 8 phases,
  int xs_floats;      // floats per staging buffer,
  size_t smem_fixed;  // and its shared memory before the fragment copy
};
inline RsChoice rs_choose(int orig_r, int new_r, int width) {
  RsChoice c{};
  const int taps = 2 * width + orig_r;
  c.tc = rs_tc_steps(orig_r, new_r, width);
  c.n_tiles = rs_tiles(new_r);
  c.xs_floats = (kRsFrames * orig_r + taps + 16 + 4 + 3) & ~3;  // rs_fill's span + its alignment shift, whole float4
  c.smem_fixed = sizeof(float) * 2 * (size_t)c.xs_floats + 16 + sizeof(RsTile) * ((c.n_tiles + 3) & ~3);
  const bool mma = c.n_tiles <= kRsMaxTiles && c.smem_fixed + 1024 <= (size_t)kRsSmemBudget;
  // tcgen05 for odd orig' (conflict-free frame-per-lane reads) whenever its plan fits: 0.283 vs 0.391 ms at config 3,
  // bf16 x 3 arithmetic (~6e-6 of the output peak against ~1e-6 for TF32 x 3).  The mma.sync kernel runs behind it as
  // the device-side fallback, so it must fit too (within the tcgen05 limits it always does).
  const bool tc = (orig_r & 1) != 0 && c.tc.ok != 0;
  c.family = !mma ? kRsFamilyDirect : (tc ? kRsFamilyTc : kRsFamilyMma);
  return c;
}

}  // namespace

size_t resample_workspace_bytes_impl(int new_r, int taps) { return rs_layout(new_r, taps).total; }

// Host-only: what resample_run_impl will launch for this ratio (nothing touches the device).
//   info[0] kernel family: 1 tcgen05 (resample_tc_kernel), 2 mma.sync TF32 x 3, 3 direct
//   info[1] bytes of the banded bf16 tap blocks of the tcgen05 plan (0 if it does not apply)
//   info[2] dynamic shared memory of the tcgen05 kernel, info[3] its MMAs per 32-frame tile
int resample_plan_info_impl(int orig_r, int new_r, int width, int32_t* info) {
  if (orig_r < 1 || new_r < 1 || width < 0 || info == nullptr) return B200A_EINVAL;
  const RsChoice c = rs_choose(orig_r, new_r, width);
  info[0] = c.family;
  info[1] = c.tc.ok ? c.tc.b_bytes : 0;
  info[2] = c.tc.ok ? rs_tc_smem(orig_r, 2 * width + orig_r).total : 0;
  info[3] = c.tc.ok ? 2 * c.tc.steps + 1 : 0;
  return B200A_OK;
}

// Host-only: the live-tap band [first, last] the tcgen05 plan assumes for output phase `phase` (see rs_tc_band).
int resample_tc_band_impl(int orig_r, int new_r, int width, int phase, int32_t* first, int32_t* last) {
  if (orig_r < 1 || new_r < 1 || width < 0 || phase < 0 || phase >= new_r || first == nullptr || last == nullptr)
    return B200A_EINVAL;
  int f, l;
  rs_tc_band(phase, orig_r, new_r, width, f, l);
  const int taps = 2 * width + orig_r;
  *first = f;
  *last = l < taps - 1 ? l : taps - 1;
  return B200A_OK;
}

int resample_prepare_impl(const float* kernel, int orig_r, int new_r, int width, void* ws, size_t ws_bytes,
                          cudaStream_t stream) {
  if (kernel == nullptr || ws == nullptr || orig_r < 1 || new_r < 1 || width < 0) return B200A_EINVAL;
  const int taps = 2 * width + orig_r;
  const RsLayout l = rs_layout(new_r, taps);
  if (ws_bytes < l.total) return B200A_EWORKSPACE;
  unsigned char* base = static_cast<unsigned char*>(ws);
  if (cudaMemsetAsync(base + l.header, 0, sizeof(RsHeader), stream) != cudaSuccess) return B200A_ECUDA;
  RsHeader* hdr = reinterpret_cast<RsHeader*>(base + l.header);
  int2* support = reinterpret_cast<int2*>(base + l.support);
  resample_support_kernel<<<(new_r + 7) / 8, 256, 0, stream>>>(kernel, new_r, taps, orig_r, width, hdr, support);
  if (rs_tiles(new_r) <= kRsMaxTiles)
    resample_plan_kernel<<<1, 256, 0, stream>>>(kernel, support, new_r, taps, rs_tiles(new_r), hdr,
                                                reinterpret_cast<RsTile*>(base + l.tiles),
                                                reinterpret_cast<float4*>(base + l.frags));
  resample_tc_plan_kernel<<<1, 256, 0, stream>>>(kernel, support, orig_r, new_r, width, taps,
                                                 rs_tc_steps(orig_r, new_r, width), hdr, base + l.tcblocks);
  return launch_status();
}

int resample_run_impl(const void* ws, const float* kernel, int orig_r, int new_r, int width, const float* wave,
                      int64_t rows, int64_t length, int64_t row_stride, float* out, int64_t out_row_stride,
                      int64_t out_len, cudaStream_t stream) {
  if (orig_r < 1 || new_r < 1 || width < 0 || rows < 0 || length < 0 || out_len < 0) return B200A_EINVAL;
  if (rows == 0 || out_len == 0) return B200A_OK;  // empty batch: pointers may be null
  if (ws == nullptr || kernel == nullptr || wave == nullptr || out == nullptr) return B200A_EINVAL;
  const int taps = 2 * width + orig_r;
  const RsLayout l = rs_layout(new_r, taps);
  const unsigned char* base = static_cast<const unsigned char*>(ws);
  const RsChoice c = rs_choose(orig_r, new_r, width);
  // per call: the bulk copies of both tensor-core kernels need a 4-byte aligned input (rows may have any pitch), and
  // the tcgen05 kernel takes rows shorter than 2^31 samples (with a tile's margin); longer rows go to mma.sync
  const bool aligned = (reinterpret_cast<uintptr_t>(wave) & 3) == 0;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return B200A_ECUDA;

  // ---- tcgen05 path: banded bf16 x 3 product, operand built in shared memory per 32-frame tile --------------------
  bool tc_launched = false;
  if (c.family == kRsFamilyTc && aligned && length + (int64_t)taps + 64 * (int64_t)orig_r < ((int64_t)1 << 31)) {
    const RsTcSmem tcm = rs_tc_smem(orig_r, taps);
    RsTcParams p{};
    p.wave = wave;
    p.rows = rows;
    p.length = length;
    p.row_stride = row_stride;
    p.out = out;
    p.out_row_stride = out_row_stride;
    p.out_len = out_len;
    p.hdr = reinterpret_cast<const RsHeader*>(base + l.header);
    p.blocks = base + l.tcblocks;
    p.orig_r = orig_r;
    p.new_r = new_r;
    p.width = width;
    p.taps = taps;
    p.frames = (out_len + new_r - 1) / new_r;
    p.tiles_per_row = (p.frames + kTcFrames - 1) / kTcFrames;
    p.total_tiles = rows * p.tiles_per_row;
    p.out_vec = (new_r % 4 == 0 && out_row_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) ? 1 : 0;
    if (cudaFuncSetAttribute(resample_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return B200A_ECUDA;
    int64_t grid = p.total_tiles < sms ? p.total_tiles : sms;
    if (grid < 1) grid = 1;
    resample_tc_kernel<<<(unsigned)grid, kTcThreads, (size_t)tcm.total, stream>>>(p, rs_tc_issue_tab(c.tc, tcm.n_chunks));
    if (cudaPeekAtLastError() != cudaSuccess) return launch_status();
    tc_launched = true;  // the mma.sync kernel below runs only if the device-side plan did not fit
  }

  // ---- mma.sync path (also the device-side fallback behind the tcgen05 kernel) -------------------
  if (c.family != kRsFamilyDirect && aligned) {
    RsParams p{};
    p.wave = wave;
    p.rows = rows;
    p.length = length;
    p.row_stride = row_stride;
    p.out = out;
    p.out_row_stride = out_row_stride;
    p.out_len = out_len;
    p.hdr = reinterpret_cast<const RsHeader*>(base + l.header);
    p.tiles = reinterpret_cast<const RsTile*>(base + l.tiles);
    p.frags = reinterpret_cast<const float4*>(base + l.frags);
    p.orig_r = orig_r;
    p.new_r = new_r;
    p.width = width;
    p.taps = taps;
    p.n_tiles = c.n_tiles;
    p.frames = (out_len + new_r - 1) / new_r;
    p.blocks_per_row = (p.frames + kRsFrames - 1) / kRsFrames;
    p.total_blocks = rows * p.blocks_per_row;
    p.xs_floats = c.xs_floats;
    // fragments go to shared memory when they fit next to the staging buffers (the kernel compares the
    // device-side step count with the room granted here), otherwise they are read through L1
    p.frag_smem_bytes = (int)(((size_t)kRsSmemBudget - c.smem_fixed) & ~(size_t)511);  // everything that is left
    const size_t smem = c.smem_fixed + p.frag_smem_bytes;
    if (cudaFuncSetAttribute(resample_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return B200A_ECUDA;
    int64_t grid = p.total_blocks < sms ? p.total_blocks : sms;
    if (grid < 1) grid = 1;
    // row spread: the candidate with the fewest shared-memory bank conflicts for one A-fragment load
    // (8 rows x 4 consecutive words, rows spread*orig' words apart)
    int best_spread = 1, best_conf = 1 << 30;
    for (int spread = 1; spread <= 4; spread *= 2) {
      int banks[32] = {0};
      int worst = 0;
      for (int rr = 0; rr < 8; ++rr)
        for (int cc = 0; cc < 4; ++cc) {
          const int bnk = (int)(((int64_t)rr * spread * orig_r + cc) & 31);
          if (++banks[bnk] > worst) worst = banks[bnk];
        }
      if (worst < best_conf) { best_conf = worst; best_spread = spread; }
    }
    p.row_spread = best_spread;
    p.behind_tc = tc_launched ? 1 : 0;
    p.out_pair = (new_r % 2 == 0 && out_row_stride % 2 == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0) ? 1 : 0;
    // warps: n_tiles items (phase groups) per tile; prefer the largest count that divides them evenly
    const int items = c.n_tiles;
    int warps = 8;
    double best_idle = 2.0;
    for (int w = 8; w <= kRsMaxWarps; ++w) {
      const int rounds = (items + w - 1) / w;
      const double idle = 1.0 - (double)items / (double)(rounds * w);
      if (idle <= best_idle + 1e-9) { best_idle = idle; warps = w; }  // ties go to more warps
    }
    resample_mma_kernel<<<(unsigned)grid, warps * 32, smem, stream>>>(p);
    return launch_status();
  }

  // ---- direct path --------------------------------------------------------------------------------
  if (rows > 65535) return B200A_EUNSUPPORTED;
  unsigned bx = (unsigned)((out_len + 255) / 256);
  if (bx > 4096) bx = 4096;
  dim3 grid(bx, (unsigned)rows);
  resample_direct_kernel<<<grid, 256, 0, stream>>>(wave, length, row_stride, kernel,
                                                  reinterpret_cast<const int2*>(base + l.support), orig_r, new_r,
                                                  width, taps, out, out_row_stride, out_len);
  return launch_status();
}

}  // namespace b200a
