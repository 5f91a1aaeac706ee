// Entropy coder of JointAutoregressiveHierarchical (DESIGN.md section 9): quantised CDF tables, rANS encode, rANS decode.
//
//   codec_table_kernel    the ONE place where floats become integer frequencies (encoder and decoder both call it)
//   codec_encode_kernel   one thread per (image, lane): the lane's symbols in reverse decode order (wavefront, raster or
//                         checkerboard walk; the checkerboard walk over a channel window [c_off, c_off + m) of c_total channels
//                         for the channel slices of section 16) -> 16-bit words
//   codec_decode_kernel   one thread per (image, lane): one wavefront step of y, or all of z
//   codec_decode_step_kernel  one CTA per (image, lane): one wavefront step of y (section 11) or one checkerboard pass (section 14;
//                         of one channel slice, section 16), its tables built in shared memory
//   codec_checksum_kernel per-image 32-bit checksum of the y and z symbols
//
// rANS: 32-bit state in [2^16, 2^32), 16-bit renormalisation words, 16-bit probability precision.  A table row of one
// element is a window of n <= NIC_CODEC_WINDOW consecutive integers starting at `lo`, plus one escape bin (index n) that
// carries any other value; an escaped value follows the escape bin as two raw 16-bit words (zigzag value, low half first).
#include "codec_step.cuh"
#include "common.cuh"
#include "entropy_math.cuh"
#include "tc_host.cuh"

namespace nic {

constexpr int kProbBits = NIC_CODEC_PREC_BITS;
constexpr uint32_t kProbScale = 1u << kProbBits;
constexpr uint32_t kRansL = 1u << 16;                      // lower bound of the state
constexpr int kWin = NIC_CODEC_WINDOW;
constexpr int kRow = NIC_CODEC_WINDOW + 2;                 // cdf entries of one row: cdf[0] = 0 ... cdf[n + 1] = 2^16
constexpr float kTail = 6.0f;                              // window = [min mu_k - 6 sigma_k, max mu_k + 6 sigma_k]
constexpr float kSymLimit = 1048576.0f;                    // 2^20: compress() rejects larger magnitudes
constexpr int kNoSymbol = -2147483647 - 1;

__device__ __forceinline__ uint32_t zigzag(int v) { return v >= 0 ? 2u * static_cast<uint32_t>(v) : 2u * static_cast<uint32_t>(-v) - 1u; }
__device__ __forceinline__ float unzigzag(uint32_t z) {
  return (z & 1u) ? -static_cast<float>(static_cast<int64_t>(z >> 1) + 1) : static_cast<float>(z >> 1);
}

// The table of one element: window, frequencies, and either the cdf row (row != NULL) or the (start, freq, escape) code of
// `target`.  __noinline__ so that the float -> integer step exists as ONE compiled function: the encoder's call (row == NULL)
// and the decoder's (target == kNoSymbol) run the same instructions and cannot differ in FMA contraction.
//   kind GM:         p = [w_1..K | mu_1..K | s_1..K] raw entropy parameters (K = 1: [mu | s]), softmax / softplus + 1e-6 as
//                    gm_math (likelihood.cu), bin mass = sum_k w_k (Phi_k(upper edge) - Phi_k(lower edge)) with libdevice erff
//   kind FACTORIZED: p = the channel's 43 nic_pack_factorized parameters, bin mass as factorized_kernel; window of NIC_CODEC_WINDOW
//                    integers centred on the median (bisection of the logit)
// Frequencies: f_i = 1 + floor(mass_i * (2^16 - n - 1)), clamped so that every later bin and the escape bin keep >= 1; the
// escape bin gets the rest of 2^16.
__device__ __noinline__ uint64_t element_code(int kind, int K, const float* __restrict__ p, int target, uint32_t* __restrict__ row,
                                              int* __restrict__ lo_out, int* __restrict__ n_out) {
  float wk[5], mu[5], inv[5], prev[5];
  int lo, n;
  if (kind == NIC_CODEC_GM) {
    float sg[5];
    if (K == 1) {
      wk[0] = 1.f;
      mu[0] = p[0];
      sg[0] = softplus_torch(p[1]) + 1e-6f;
    } else {
      float mx = p[0];
      for (int k = 1; k < K; ++k) mx = fmaxf(mx, p[k]);
      float den = 0.f;
      for (int k = 0; k < K; ++k) { wk[k] = expf(p[k] - mx); den += wk[k]; }
      const float inv_den = 1.0f / den;
      for (int k = 0; k < K; ++k) {
        wk[k] *= inv_den;
        mu[k] = p[K + k];
        sg[k] = softplus_torch(p[2 * K + k]) + 1e-6f;
      }
    }
    float lo_f = kSymLimit, hi_f = -kSymLimit, centre = 0.f;
    for (int k = 0; k < K; ++k) {
      inv[k] = 1.0f / (sg[k] * 1.41421356237309515f);
      lo_f = fminf(lo_f, mu[k] - kTail * sg[k]);
      hi_f = fmaxf(hi_f, mu[k] + kTail * sg[k]);
      centre += wk[k] * mu[k];
    }
    lo_f = fmaxf(lo_f, -kSymLimit);                          // (fmaxf / fminf drop a NaN operand)
    hi_f = fminf(hi_f, kSymLimit);
    lo = static_cast<int>(floorf(lo_f));
    n = max(static_cast<int>(ceilf(hi_f)) - lo + 1, 1);
    if (n > kWin) {                                          // too wide: NIC_CODEC_WINDOW bins around the mixture mean
      lo = static_cast<int>(rintf(fminf(fmaxf(centre, -kSymLimit), kSymLimit))) - kWin / 2;
      n = kWin;
    }
    for (int k = 0; k < K; ++k) prev[k] = erff((static_cast<float>(lo) - 0.5f - mu[k]) * inv[k]);
  } else {
    float a = -kSymLimit, b = kSymLimit;
    for (int it = 0; it < 48; ++it) {
      const float m = 0.5f * (a + b);
      if (factorized_logit(m, p) < 0.f) a = m; else b = m;
    }
    lo = static_cast<int>(rintf(0.5f * (a + b))) - kWin / 2;
    n = kWin;
    prev[0] = factorized_logit(static_cast<float>(lo) - 0.5f, p);
  }
  const float R = static_cast<float>(kProbScale - static_cast<uint32_t>(n) - 1u);
  uint32_t cum = 0;
  uint64_t code = 0;
  bool found = false;
  if (row) row[0] = 0;
  for (int i = 0; i < n; ++i) {
    const float e = static_cast<float>(lo + i) + 0.5f;
    float mass;
    if (kind == NIC_CODEC_GM) {
      mass = 0.f;
      for (int k = 0; k < K; ++k) {
        const float eu = erff((e - mu[k]) * inv[k]);
        mass += wk[k] * (0.5f * (1.0f + eu) - 0.5f * (1.0f + prev[k]));
        prev[k] = eu;
      }
    } else {
      const float lower = prev[0], upper = factorized_logit(e, p);
      const float t = lower + upper;
      const float s = (t > 0.f) ? -1.f : ((t < 0.f) ? 1.f : 0.f);
      mass = fabsf(sigmoid_torch(s * upper) - sigmoid_torch(s * lower));
      prev[0] = upper;
    }
    uint32_t f = 1u + static_cast<uint32_t>(fminf(fmaxf(mass, 0.f), 1.f) * R);
    const uint32_t room = kProbScale - 1u - cum - static_cast<uint32_t>(n - 1 - i);
    f = min(f, room);
    if (lo + i == target) { code = cum | (static_cast<uint64_t>(f) << 16); found = true; }
    cum += f;
    if (row) row[i + 1] = cum;
  }
  if (row) row[n + 1] = kProbScale;
  if (!found) code = cum | (static_cast<uint64_t>(kProbScale - cum) << 16) | (1ull << 32);
  if (lo_out) *lo_out = lo;
  if (n_out) *n_out = n;
  return code;
}

// mode TABLES: kind GM = the elements of wavefront step t, e = (img * cnt + p) * m + c -> cdf row, lo, n;
//              kind FACTORIZED = one row per channel (e = c).
// mode SYMBOL: every element of the latent [b, m, h, w] (NCHW index e) with its symbol sym[e] -> code[e].
__global__ void __launch_bounds__(128)
codec_table_kernel(int kind, int mode, const float* __restrict__ params, const float* __restrict__ sym, int b, int m, int K,
                   int h, int w, int t, int i0, int cnt, uint32_t* __restrict__ cdf, int32_t* __restrict__ lo_out,
                   int32_t* __restrict__ n_out, uint64_t* __restrict__ code) {
  const long hw = static_cast<long>(h) * w;
  const long total = mode == NIC_CODEC_SYMBOL ? b * m * hw : (kind == NIC_CODEC_GM ? static_cast<long>(b) * cnt * m : m);
  const int np = kind == NIC_CODEC_GM ? (K == 1 ? 2 : 3 * K) : 43;
  for (long e = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += static_cast<long>(gridDim.x) * blockDim.x) {
    long img, c, pix;
    if (mode == NIC_CODEC_SYMBOL) {
      img = e / (m * hw); c = (e / hw) % m; pix = e % hw;
    } else if (kind == NIC_CODEC_GM) {
      img = e / (static_cast<long>(cnt) * m); c = e % m;
      const int i = i0 + static_cast<int>((e / m) % cnt);
      pix = static_cast<long>(i) * w + (t - 3 * i);
    } else {
      img = 0; c = e; pix = 0;
    }
    float q[43];
    if (kind == NIC_CODEC_GM) {
      const float* src = params + (img * np * m + c) * hw + pix;             // raw [b, np * m, h, w]: plane j * m + c
      for (int j = 0; j < np; ++j) q[j] = __ldg(src + static_cast<long>(j) * m * hw);
    } else {
      for (int j = 0; j < 43; ++j) q[j] = __ldg(params + c * 43 + j);
    }
    if (mode == NIC_CODEC_SYMBOL) {
      const float v = __ldg(sym + e);
      const int target = fabsf(v) < kSymLimit ? static_cast<int>(v) : kNoSymbol;
      code[e] = element_code(kind, K, q, target, nullptr, nullptr, nullptr);
    } else {
      element_code(kind, K, q, kNoSymbol, cdf + e * kRow, lo_out + e, n_out + e);
    }
  }
}

// The lane's symbols in DECODE order, as a sequence of steps, each a run of pixels with the lane's channels per pixel (c = c0,
// c0 + cl, ... ascending; c0 = lane % cl):
//   kind GM (y, wavefront)   steps t ascending, pixels of the step with i ascending; cl = lanes
//   kind FACTORIZED (z)      pixels in raster order, one per step; cl = lanes
//   kWalkCheckerboard (y)    lane = r * cl + l covers the rows [r band, r band + band): step t = pass s * nb + row i - r band
//                            (nb = the band's rows), pixels of row i with (i + j + s) even, j ascending - pass 0 the anchors, pass 1
//                            the non-anchors (DESIGN.md section 14)
// The encoder walks it backwards.
constexpr int kWalkCheckerboard = 2;

struct LaneWalk {
  int kind, m, h, w, lane, lanes, cl, band;
  __device__ int c0() const { return lane % cl; }
  __device__ int row0() const { return (lane / cl) * band; }
  __device__ int band_rows() const { return min(band, h - row0()); }
  __device__ int steps() const {
    return kind == NIC_CODEC_GM ? 3 * h + w - 3 : (kind == kWalkCheckerboard ? 2 * band_rows() : h * w);
  }
  __device__ void rows(int t, int& i0, int& cnt) const {
    if (kind == NIC_CODEC_GM) step_rows(t, h, w, i0, cnt);
    else if (kind == kWalkCheckerboard) {
      const int nb = band_rows(), s = t / nb;
      i0 = row0() + t - s * nb;
      cnt = (w - ((i0 + s) & 1) + 1) / 2;
    } else { i0 = t; cnt = 1; }
  }
  __device__ long pix(int t, int i0, int p) const {            // pixel index i * w + j of the p-th pixel of step t
    if (kind == NIC_CODEC_GM) { const int i = i0 + p; return static_cast<long>(i) * w + (t - 3 * i); }
    if (kind == kWalkCheckerboard) return static_cast<long>(i0) * w + ((i0 + t / band_rows()) & 1) + 2 * p;
    return t;
  }
  // the steps [t0, t1) as one run: its pixel count and its p-th pixel (<= 16 steps: a checkerboard pass of one band)
  __device__ int span_count(int t0, int t1) const {
    int n = 0;
    for (int t = t0; t < t1; ++t) { int i0, cnt; rows(t, i0, cnt); n += cnt; }
    return n;
  }
  __device__ long span_pix(int t0, int t1, int p) const {
    for (int t = t0; t < t1; ++t) {
      int i0, cnt;
      rows(t, i0, cnt);
      if (p < cnt) return pix(t, i0, p);
      p -= cnt;
    }
    return 0;                                                  // not reached: p < span_count(t0, t1)
  }
};

__device__ __forceinline__ void rans_put(uint32_t& x, uint32_t start, uint32_t freq, uint16_t* row, long& wp) {
  while (x >= (freq << 16)) { row[--wp] = static_cast<uint16_t>(x & 0xffffu); x >>= 16; }
  x = ((x / freq) << kProbBits) + (x % freq) + start;
}

__global__ void __launch_bounds__(64)
codec_encode_kernel(int kind, const uint64_t* __restrict__ code, const float* __restrict__ sym, int b, int c_total, int c_off, int m, int h,
                    int w, int lanes, int cl, int band, long cap, uint16_t* __restrict__ words, int32_t* __restrict__ count) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= b * lanes) return;
  const int img = g / lanes;
  const LaneWalk lw{kind, m, h, w, g % lanes, lanes, cl, band};
  const long hw = static_cast<long>(h) * w;
  uint16_t* row = words + g * cap;
  long wp = cap;
  uint32_t x = kRansL;
  const int c_last = lw.c0() + ((m - 1 - lw.c0()) / cl) * cl;
  for (int t = lw.steps() - 1; t >= 0; --t) {
    int i0, cnt;
    lw.rows(t, i0, cnt);
    for (int p = cnt - 1; p >= 0; --p) {
      const long pix = lw.pix(t, i0, p);
      for (int c = c_last; c >= 0; c -= cl) {
        const long e = (static_cast<long>(img) * c_total + c_off + c) * hw + pix;
        const uint64_t cd = code[e];
        if (cd >> 32) {                                        // escape: the raw value words first (they decode after the bin)
          const uint32_t z = zigzag(static_cast<int>(sym[e]));
          rans_put(x, z >> 16, 1u, row, wp);
          rans_put(x, z & 0xffffu, 1u, row, wp);
        }
        rans_put(x, static_cast<uint32_t>(cd & 0xffffu), static_cast<uint32_t>((cd >> 16) & 0xffffu), row, wp);
      }
    }
  }
  row[--wp] = static_cast<uint16_t>(x >> 16);
  row[--wp] = static_cast<uint16_t>(x & 0xffffu);              // the lane segment starts with the state, little-endian
  count[g] = static_cast<int32_t>(cap - wp);
}

struct LaneReader {
  const uint8_t* data;
  int words, pos;
  __device__ uint32_t next() {                                 // an exhausted lane reads zeros
    uint32_t v = 0;
    if (pos < words) v = data[2 * pos] | (static_cast<uint32_t>(data[2 * pos + 1]) << 8);
    ++pos;
    return v;
  }
};

__device__ __forceinline__ uint32_t rans_bypass(uint32_t& x, LaneReader& rd) {
  const uint32_t v = x & 0xffffu;
  x >>= 16;
  if (x < kRansL) x = (x << 16) | rd.next();
  return v;
}

// kind GM: step t of the wavefront, tables of the step's elements (e = (img * cnt + p) * m + c); kind FACTORIZED: every z symbol,
// one table per channel.  Writes the symbols into out (NHWC f32 [b, h, w, m]).  state / pos keep each lane's cursor between steps.
__global__ void __launch_bounds__(64)
codec_decode_kernel(int kind, const uint8_t* __restrict__ blob, const int64_t* __restrict__ lane_off, const int32_t* __restrict__ lane_words,
                    uint32_t* __restrict__ state, int32_t* __restrict__ pos, int init, const uint32_t* __restrict__ cdf,
                    const int32_t* __restrict__ lo_tab, const int32_t* __restrict__ n_tab, int b, int m, int h, int w, int lanes, int t,
                    float* __restrict__ out) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= b * lanes) return;
  const int img = g / lanes;
  const LaneWalk lw{kind, m, h, w, g % lanes, lanes, lanes, 0};
  const uint8_t* seg = blob + lane_off[g];
  LaneReader rd{seg + 4, lane_words[g], 0};
  uint32_t x;
  if (init) x = seg[0] | (seg[1] << 8) | (seg[2] << 16) | (static_cast<uint32_t>(seg[3]) << 24);
  else { x = state[g]; rd.pos = pos[g]; }
  const int t0 = kind == NIC_CODEC_GM ? t : 0, t1 = kind == NIC_CODEC_GM ? t + 1 : lw.steps();
  for (int s = t0; s < t1; ++s) {
    int i0, cnt;
    lw.rows(s, i0, cnt);
    for (int p = 0; p < cnt; ++p) {
      const long pix = lw.pix(s, i0, p);
      for (int c = lw.lane; c < m; c += lanes) {
        const long e = kind == NIC_CODEC_GM ? (static_cast<long>(img) * cnt + p) * m + c : c;
        const uint32_t* row = cdf + e * kRow;
        const int n = n_tab[e];
        const uint32_t slot = x & (kProbScale - 1u);
        int a = 0, z = n + 1;                                  // largest a with row[a] <= slot
        while (z - a > 1) {
          const int mid = (a + z) >> 1;
          if (row[mid] <= slot) a = mid; else z = mid;
        }
        const uint32_t start = row[a], freq = row[a + 1] - start;
        x = freq * (x >> kProbBits) + slot - start;
        if (x < kRansL) x = (x << 16) | rd.next();
        float v;
        if (a == n) {
          const uint32_t zlo = rans_bypass(x, rd);
          const uint32_t zhi = rans_bypass(x, rd);
          v = unzigzag(zlo | (zhi << 16));
        } else {
          v = static_cast<float>(lo_tab[e] + a);
        }
        out[(static_cast<long>(img) * h * w + pix) * m + c] = v;
      }
    }
  }
  state[g] = x;
  pos[g] = rd.pos;
}

// The steps [t0, t1) of the lane walk of y for one (image, lane) per CTA, tables in shared memory: one wavefront step (section 11)
// or one checkerboard pass (section 14; t0, t1 = pass * nb, (pass + 1) * nb with the lane's band of nb rows).  The lane's rows
// in its decode order are built by the builder warps with the same element_code as codec_table_kernel, kStepChunk rows at a time
// into one of two buffers; thread 0 decodes chunk k from one buffer while the builders fill the other with chunk k + 1.  The
// decode arithmetic is codec_decode_kernel's, so symbols, states and read positions are the same bits.  Every loop count is fixed
// by the shapes: a corrupted string only changes the values decoded.
constexpr int kStepChunk = 64;                                 // rows per chunk: one per builder thread
constexpr int kStepThreads = 32 + kStepChunk;                  // warp 0 decodes, warps 1 .. 2 build
constexpr size_t kStepSmem = 2ull * kStepChunk * (kRow * sizeof(uint32_t) + 3 * sizeof(int32_t));

__global__ void __launch_bounds__(kStepThreads)
codec_decode_step_kernel(const uint8_t* __restrict__ blob, const int64_t* __restrict__ lane_off, const int32_t* __restrict__ lane_words,
                         uint32_t* __restrict__ state, int32_t* __restrict__ pos, int init, const float* __restrict__ params, int m,
                         int K, int kind, int h, int w, int lanes, int cl, int band, int t, int c_total, int c_off,
                         float* __restrict__ out) {
  extern __shared__ __align__(16) uint32_t s_step[];
  uint32_t* s_cdf = s_step;                                    // [2][kStepChunk][kRow]
  int32_t* s_lo = reinterpret_cast<int32_t*>(s_step + 2 * kStepChunk * kRow);
  int32_t* s_n = s_lo + 2 * kStepChunk;
  int32_t* s_pix = s_n + 2 * kStepChunk;                       // the row's pixel i * w + j
  const int g = blockIdx.x, img = g / lanes;
  const LaneWalk lw{kind, m, h, w, g % lanes, lanes, cl, band};
  const int c0 = lw.c0();
  // t: the wavefront step, or the checkerboard pass
  const int t0 = kind == kWalkCheckerboard ? t * lw.band_rows() : t, t1 = kind == kWalkCheckerboard ? t0 + lw.band_rows() : t + 1;
  const int nc = (m - 1 - c0) / cl + 1;                        // channels of this lane
  const int rows = lw.span_count(t0, t1) * nc, chunks = (rows + kStepChunk - 1) / kStepChunk;
  const long hw = static_cast<long>(h) * w;
  const int np = K == 1 ? 2 : 3 * K;

  auto build = [&](int k) {                                    // builder thread: row k * kStepChunk + (tid - 32) into buffer k & 1
    const int b = threadIdx.x - 32, r = k * kStepChunk + b;
    if (r >= rows) return;
    const int p = r / nc, c = c0 + (r - p * nc) * cl;
    const long pix = lw.span_pix(t0, t1, p);
    const float* src = params + (static_cast<long>(img) * np * m + c) * hw + pix;
    float q[15];
    for (int j = 0; j < np; ++j) q[j] = __ldg(src + static_cast<long>(j) * m * hw);
    const int e = (k & 1) * kStepChunk + b;
    s_pix[e] = static_cast<int32_t>(pix);
    element_code(NIC_CODEC_GM, K, q, kNoSymbol, s_cdf + e * kRow, s_lo + e, s_n + e);
  };

  uint32_t x = 0;
  LaneReader rd{nullptr, 0, 0};
  if (threadIdx.x == 0) {
    const uint8_t* seg = blob + lane_off[g];
    rd = LaneReader{seg + 4, lane_words[g], 0};
    if (init) x = seg[0] | (seg[1] << 8) | (seg[2] << 16) | (static_cast<uint32_t>(seg[3]) << 24);
    else { x = state[g]; rd.pos = pos[g]; }
  }
  if (threadIdx.x >= 32) build(0);
  __syncthreads();
  for (int k = 0; k < chunks; ++k) {
    if (threadIdx.x >= 32) {
      if (k + 1 < chunks) build(k + 1);
    } else if (threadIdx.x == 0) {
      const int r1 = min(rows, (k + 1) * kStepChunk);
      for (int r = k * kStepChunk; r < r1; ++r) {
        const int e = (k & 1) * kStepChunk + (r - k * kStepChunk);
        const uint32_t* row = s_cdf + e * kRow;
        const int n = s_n[e];
        const uint32_t slot = x & (kProbScale - 1u);
        int a = 0, z = n + 1;                                  // largest a with row[a] <= slot
        while (z - a > 1) {
          const int mid = (a + z) >> 1;
          if (row[mid] <= slot) a = mid; else z = mid;
        }
        const uint32_t start = row[a], freq = row[a + 1] - start;
        x = freq * (x >> kProbBits) + slot - start;
        if (x < kRansL) x = (x << 16) | rd.next();
        float v;
        if (a == n) {
          const uint32_t zlo = rans_bypass(x, rd);
          const uint32_t zhi = rans_bypass(x, rd);
          v = unzigzag(zlo | (zhi << 16));
        } else {
          v = static_cast<float>(s_lo[e] + a);
        }
        const int p = r / nc, c = c0 + (r - p * nc) * cl;
        out[(static_cast<long>(img) * hw + s_pix[e]) * c_total + c_off + c] = v;
      }
    }
    __syncthreads();                                           // chunk k decoded, chunk k + 1 built
  }
  if (threadIdx.x == 0) {
    state[g] = x;
    pos[g] = rd.pos;
  }
}

__device__ __forceinline__ uint32_t mix32(uint32_t idx, uint32_t v) {
  uint32_t hsh = idx * 0x9E3779B1u ^ (v + 0x7F4A7C15u);
  hsh ^= hsh >> 16; hsh *= 0x85EBCA6Bu;
  hsh ^= hsh >> 13; hsh *= 0xC2B2AE35u;
  hsh ^= hsh >> 16;
  return hsh;
}

__global__ void __launch_bounds__(256)
codec_checksum_kernel(const float* __restrict__ y, long y_per, const float* __restrict__ z, long z_per, uint32_t* __restrict__ out) {
  const int img = blockIdx.y;
  uint32_t acc = 0;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < y_per + z_per; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float v = i < y_per ? y[img * y_per + i] : z[img * z_per + (i - y_per)];
    acc += mix32(static_cast<uint32_t>(i), static_cast<uint32_t>(__float2int_rn(v)));
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out + img, acc);      // integer sum: any order gives the same bits
}

}  // namespace nic

using namespace nic;

extern "C" {

int nic_codec_tables(int32_t kind, int32_t mode, const float* params, const float* sym, int32_t b, int32_t m, int32_t k, int32_t h,
                     int32_t w, int32_t t, uint32_t* cdf, int32_t* lo, int32_t* nbins, uint64_t* code, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if ((kind != NIC_CODEC_GM && kind != NIC_CODEC_FACTORIZED) || (mode != NIC_CODEC_TABLES && mode != NIC_CODEC_SYMBOL))
    return fail(NIC_E_BADSHAPE, "codec_tables: kind=%d mode=%d", kind, mode);
  if (b < 1 || m < 1 || k < 1 || k > 5 || h < 1 || w < (kind == NIC_CODEC_GM ? 3 : 1))
    return fail(NIC_E_BADSHAPE, "codec_tables: b=%d m=%d k=%d h=%d w=%d", b, m, k, h, w);
  if (!params || (mode == NIC_CODEC_SYMBOL && (!sym || !code)) || (mode == NIC_CODEC_TABLES && (!cdf || !lo || !nbins)))
    return fail(NIC_E_BADSHAPE, "codec_tables: null pointer");
  int i0 = 0, cnt = 1;
  if (kind == NIC_CODEC_GM && mode == NIC_CODEC_TABLES) {
    if (t < 0 || t >= 3 * h + w - 3) return fail(NIC_E_BADSHAPE, "codec_tables: step %d of %d", t, 3 * h + w - 3);
    step_rows(t, h, w, i0, cnt);
  }
  const long total = mode == NIC_CODEC_SYMBOL ? static_cast<long>(b) * m * h * w : (kind == NIC_CODEC_GM ? static_cast<long>(b) * cnt * m : m);
  long blocks = (total + 127) / 128;
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  codec_table_kernel<<<static_cast<unsigned>(blocks), 128, 0, as_stream(stream)>>>(kind, mode, params, sym, b, m, k, h, w, t, i0, cnt, cdf,
                                                                                  lo, nbins, code);
  return check_launch("codec_table_kernel");
}

int nic_codec_encode(int32_t kind, const uint64_t* code, const float* sym, int32_t b, int32_t m, int32_t h, int32_t w, int32_t lanes,
                     int64_t cap, uint16_t* words, int32_t* count, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 1 || m < 1 || h < 1 || w < (kind == NIC_CODEC_GM ? 3 : 1) || lanes < 1 || lanes > m)
    return fail(NIC_E_BADSHAPE, "codec_encode: b=%d m=%d h=%d w=%d lanes=%d", b, m, h, w, lanes);
  if (cap < 3L * ((m + lanes - 1) / lanes) * h * w + 2) return fail(NIC_E_WORKSPACE, "codec_encode: lane capacity %lld words", static_cast<long long>(cap));
  if (!code || !sym || !words || !count) return fail(NIC_E_BADSHAPE, "codec_encode: null pointer");
  codec_encode_kernel<<<(b * lanes + 63) / 64, 64, 0, as_stream(stream)>>>(kind, code, sym, b, m, 0, m, h, w, lanes, lanes, 0, cap, words,
                                                                           count);
  return check_launch("codec_encode_kernel");
}

int nic_codec_decode(int32_t kind, const uint8_t* blob, const int64_t* lane_off, const int32_t* lane_words, uint32_t* state, int32_t* pos,
                     int32_t init, const uint32_t* cdf, const int32_t* lo, const int32_t* nbins, int32_t b, int32_t m, int32_t h, int32_t w,
                     int32_t lanes, int32_t t, float* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 1 || m < 1 || h < 1 || w < (kind == NIC_CODEC_GM ? 3 : 1) || lanes < 1 || lanes > m)
    return fail(NIC_E_BADSHAPE, "codec_decode: b=%d m=%d h=%d w=%d lanes=%d", b, m, h, w, lanes);
  if (kind == NIC_CODEC_GM && (t < 0 || t >= 3 * h + w - 3)) return fail(NIC_E_BADSHAPE, "codec_decode: step %d", t);
  if (!blob || !lane_off || !lane_words || !state || !pos || !cdf || !lo || !nbins || !out) return fail(NIC_E_BADSHAPE, "codec_decode: null pointer");
  codec_decode_kernel<<<(b * lanes + 63) / 64, 64, 0, as_stream(stream)>>>(kind, blob, lane_off, lane_words, state, pos, init, cdf, lo, nbins,
                                                                           b, m, h, w, lanes, t, out);
  return check_launch("codec_decode_kernel");
}

int nic_codec_decode_step(const uint8_t* blob, const int64_t* lane_off, const int32_t* lane_words, uint32_t* state, int32_t* pos,
                          int32_t init, const float* params, int32_t b, int32_t m, int32_t k, int32_t h, int32_t w, int32_t lanes, int32_t t,
                          float* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 1 || m < 1 || k < 1 || k > 5 || h < 1 || w < 3 || lanes < 1 || lanes > m)
    return fail(NIC_E_BADSHAPE, "codec_decode_step: b=%d m=%d k=%d h=%d w=%d lanes=%d", b, m, k, h, w, lanes);
  if (t < 0 || t >= 3 * h + w - 3) return fail(NIC_E_BADSHAPE, "codec_decode_step: step %d of %d", t, 3 * h + w - 3);
  if (!blob || !lane_off || !lane_words || !state || !pos || !params || !out) return fail(NIC_E_BADSHAPE, "codec_decode_step: null pointer");
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(codec_decode_step_kernel), static_cast<int>(kStepSmem))) return rc;
  codec_decode_step_kernel<<<b * lanes, kStepThreads, kStepSmem, as_stream(stream)>>>(blob, lane_off, lane_words, state, pos, init, params,
                                                                                      m, k, NIC_CODEC_GM, h, w, lanes, lanes, 0, t, m, 0, out);
  return check_launch("codec_decode_step_kernel");
}

static int checkerboard_lanes(const char* what, int32_t b, int32_t m, int32_t h, int32_t w, int32_t lanes_c, int32_t band_rows, int* lanes) {
  if (b < 1 || m < 1 || h < 1 || w < 1 || lanes_c < 1 || lanes_c > m || band_rows < 1)
    return fail(NIC_E_BADSHAPE, "%s: b=%d m=%d h=%d w=%d lanes_c=%d band_rows=%d", what, b, m, h, w, lanes_c, band_rows);
  *lanes = lanes_c * ((h + band_rows - 1) / band_rows);
  return NIC_OK;
}

int nic_codec_encode_checkerboard_slice(const uint64_t* code, const float* sym, int32_t b, int32_t c_total, int32_t c_off, int32_t m,
                                        int32_t h, int32_t w, int32_t lanes_c, int32_t band_rows, int64_t cap, uint16_t* words, int32_t* count,
                                        void* stream) {
  if (int rc = nic_check_device()) return rc;
  int lanes;
  if (int rc = checkerboard_lanes("codec_encode_checkerboard", b, m, h, w, lanes_c, band_rows, &lanes)) return rc;
  if (c_off < 0 || c_total < c_off + m)
    return fail(NIC_E_BADSHAPE, "codec_encode_checkerboard: channels [%d, %d) of %d", c_off, c_off + m, c_total);
  if (cap < 3L * ((m + lanes_c - 1) / lanes_c) * band_rows * w + 2)
    return fail(NIC_E_WORKSPACE, "codec_encode_checkerboard: lane capacity %lld words", static_cast<long long>(cap));
  if (!code || !sym || !words || !count) return fail(NIC_E_BADSHAPE, "codec_encode_checkerboard: null pointer");
  codec_encode_kernel<<<(b * lanes + 63) / 64, 64, 0, as_stream(stream)>>>(kWalkCheckerboard, code, sym, b, c_total, c_off, m, h, w, lanes,
                                                                           lanes_c, band_rows, cap, words, count);
  return check_launch("codec_encode_kernel");
}

int nic_codec_encode_checkerboard(const uint64_t* code, const float* sym, int32_t b, int32_t m, int32_t h, int32_t w, int32_t lanes_c,
                                  int32_t band_rows, int64_t cap, uint16_t* words, int32_t* count, void* stream) {
  return nic_codec_encode_checkerboard_slice(code, sym, b, m, 0, m, h, w, lanes_c, band_rows, cap, words, count, stream);
}

int nic_codec_decode_pass_slice(const uint8_t* blob, const int64_t* lane_off, const int32_t* lane_words, uint32_t* state, int32_t* pos,
                                const float* params, int32_t b, int32_t c_total, int32_t c_off, int32_t m, int32_t k, int32_t h, int32_t w,
                                int32_t lanes_c, int32_t band_rows, int32_t pass, float* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  int lanes;
  if (int rc = checkerboard_lanes("codec_decode_pass", b, m, h, w, lanes_c, band_rows, &lanes)) return rc;
  if (k < 1 || k > 5 || (pass != 0 && pass != 1)) return fail(NIC_E_BADSHAPE, "codec_decode_pass: k=%d pass=%d", k, pass);
  if (c_off < 0 || c_total < c_off + m)
    return fail(NIC_E_BADSHAPE, "codec_decode_pass: channels [%d, %d) of %d", c_off, c_off + m, c_total);
  if (!blob || !lane_off || !lane_words || !state || !pos || !params || !out) return fail(NIC_E_BADSHAPE, "codec_decode_pass: null pointer");
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(codec_decode_step_kernel), static_cast<int>(kStepSmem))) return rc;
  codec_decode_step_kernel<<<b * lanes, kStepThreads, kStepSmem, as_stream(stream)>>>(blob, lane_off, lane_words, state, pos, pass == 0,
                                                                                      params, m, k, kWalkCheckerboard, h, w, lanes, lanes_c,
                                                                                      band_rows, pass, c_total, c_off, out);
  return check_launch("codec_decode_step_kernel");
}

int nic_codec_decode_pass(const uint8_t* blob, const int64_t* lane_off, const int32_t* lane_words, uint32_t* state, int32_t* pos,
                          const float* params, int32_t b, int32_t m, int32_t k, int32_t h, int32_t w, int32_t lanes_c, int32_t band_rows,
                          int32_t pass, float* out, void* stream) {
  return nic_codec_decode_pass_slice(blob, lane_off, lane_words, state, pos, params, b, m, 0, m, k, h, w, lanes_c, band_rows, pass, out,
                                     stream);
}

int nic_codec_checksum(const float* y, int64_t y_per_image, const float* z, int64_t z_per_image, int32_t b, uint32_t* out, void* stream) {
  if (int rc = nic_check_device()) return rc;
  if (b < 1 || y_per_image < 1 || z_per_image < 1 || !y || !z || !out) return fail(NIC_E_BADSHAPE, "codec_checksum: bad arguments");
  cudaStream_t st = as_stream(stream);
  if (int rc = check_cuda(cudaMemsetAsync(out, 0, sizeof(uint32_t) * b, st), "codec_checksum: memset")) return rc;
  long blocks = (y_per_image + z_per_image + 255) / 256;
  if (blocks > 64) blocks = 64;
  codec_checksum_kernel<<<dim3(static_cast<unsigned>(blocks), b), 256, 0, st>>>(y, y_per_image, z, z_per_image, out);
  return check_launch("codec_checksum_kernel");
}

}  // extern "C"
