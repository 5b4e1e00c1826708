/*
 * rx_chan.cu — polyphase channelizer (t41rx_chan_*, include/t41rx.h): one wideband complex capture at M x 96 kS/s
 * (M = 64, 320, 512 or 640 channels) cut into M channels of 192 kS/s, delivered in t41rx_process_device's iq layout.
 *
 * Transform (DESIGN §3.7): prototype h[0..N), N = K M, K = 10; decimation D = M / 2; channel k centred at
 * (k < M/2 ? k : k - M) x 96 kHz;
 *     z_k[m] = conj( sum_{i<N} h[i] x[mD - i] exp(-j 2 pi k (mD - i) / M) ).
 * With u_p[m] = sum_{q<K} h[p + qM] x[mD - p - qM] this is z_k[m] = (-1)^(k m) DFT_M(conj(u[m]))[k]: one M-point
 * forward FFT per output time, shared by all channels; for odd m the (-1)^k is a circular shift of the FFT input by M/2.
 * A call always produces a multiple of 2048 outputs (even), so m's parity is the same counted from the call or from
 * the channelizer's creation, and the only state between calls is the capture's last N - 1 samples (the tail).
 *
 * Kernel: one CTA per tile of kChanTile consecutive output times.  It stages the capture span of the tile in shared
 * memory (cp.async; samples before the call's first one come from the tail), each thread keeps the K taps of one branch
 * p in registers and forms u_p for its output times, the conj(u) rows are transformed in place (radix-8 passes of
 * rx_fft.h; half of the rows re-use the span's shared memory), and every mapped receiver gets its channel's kChanTile
 * samples, a 128-byte run.  Channels no receiver takes are computed but never written.  FP32 on the CUDA cores: a DFT
 * as a BF16 / TF32 matrix product keeps about 60 dB of dynamic range, the chain needs 90.
 *
 * Fine tuning (t41rx_chan_set_shift): receiver r's run is rotated on its way out,
 *     iq_r[m] = z_k[m] exp(+j 2 pi phi_r(m) / 192000),   phi_r(m) = (P_r + shift_r m_abs) mod 192000,
 * m_abs counting outputs since creation.  phi is exact integer arithmetic: the host keeps m_abs mod 192000 (passed per
 * call) and P_r, so the rotation of an output depends on the output alone, not on how the run was cut into calls.  The
 * factor comes from a two-level table, 192000 = 480 x 400: exp(j 2 pi a / 480) exp(j 2 pi b / 192000), phi = 400 a + b.
 * A receiver whose phase is identically 0 (shift 0, P 0) is stored unmultiplied, so its bits are those of an unshifted
 * channelizer ((x, y) (1, 0) would turn -0 into +0); a call in which no receiver is rotated runs the kernel instance
 * without fine tuning.
 *
 * Real captures (t41rx_chan_create_real, DESIGN §3.8): int16 s[n] at M x 96 kS/s, M = 128, 800, 1024 or 1280, x = s / 32768, the
 * same formula; channels k = 0 .. M/2 are distinct, channel k centred at +k x 96 kHz.  u_p[m] is real, so the M-point DFT
 * of a row is one M/2-point complex FFT of y[n] = u[2n] + j u[2n + 1] and a split,
 *     X[k] = (Y[k] + conj Y[-k]) / 2 - j e^(-j 2 pi k / M) (Y[k] - conj Y[-k]) / 2,   k = 0 .. M/2, indices mod M/2;
 * the odd-m shift of u by M/2 is a shift of y by M/4.  t41rx_chan_real_kernel is the complex kernel at M/2: thread n owns
 * branches 2n and 2n + 1 (20 taps), the span is staged as int16, the split runs in the store loop.
 *
 * Complex int16 captures (t41rx_chan_create_q15, DESIGN §3.9): (I, Q) int16 pairs, x = (I + jQ) / 32768, M as for float.
 * t41rx_chan_kernel<M, kRotate, short> converts the span once as it stages it; the rest of the kernel is the float
 * instance's, with the 1 / 32768 in the taps: the same FMAs on the same values, so the same bits as the float
 * channelizer on s / 32768.
 *
 * Digitizers' clocks (DESIGN §3.10): M = 320, 640 (complex) and 800, 1280 (real) give FFT lengths 320, 640 and 400, which
 * are 2^a 5^b.  Their rows are in natural order and run the mixed-radix DIF passes of ChanPlan (radix 5 beside 8, a
 * radix-2 pass where the factorisation needs it); X[k] ends at the mixed-radix digit reversal of k.  The power-of-two
 * instances never reach that code (if constexpr on kChanPow2), so their SASS is the same as before it was added.
 *
 * Diversity (t41rx_chan_create_diversity, DESIGN §3.11): 2 - 4 coherent captures of one kind, receiver r getting
 * rot_r(m) sum_a w[r][a] z^(a)_k[m].  A call runs the kind's kernel once per input on one stream, input 0's pass
 * storing v w f and the others adding it to iq (the kStore template parameter, behind if constexpr); each input keeps
 * its own tail.
 *
 * Image correction (t41rx_chan_set_image / _track_image, DESIGN §3.12), complex single-input channelizers: receiver r
 * on channel k gets rot_r(m) (z_k[m] + c_k conj(z_kbar[m])), kbar = (M - k) mod M.  The kChanImage / kChanImageTrack
 * instances correct the FFT rows in place, a mirror pair at a time, before the plain store loop; tracking also sums
 * each pair's products per tile, and t41rx_chan_image_update reduces them in a fixed order and moves the coefficients
 * the next call uses.  With every c_k 0 and tracking off a call runs the plain instances.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/t41rx.h"
#include "rx_design.h"
#include "rx_fft.h"
#include "rx_host.h"
#include "rx_launch.h"

namespace t41rx {

constexpr int kChanTaps = 10;             /* K: taps per branch */
constexpr int kChanTile = 16;             /* output times per CTA: one 128-byte run per receiver */
constexpr double kChanSpacing = 96000.0;  /* channel spacing = half the output rate (2x oversampled) */
constexpr double kChanBeta = 8.96;        /* Kaiser beta of a 90 dB design (the firmware's n_att) */
constexpr int kChanOutRate = 192000;      /* the phase of a fine-tuning rotation counts in 1 / 192000 of a turn */
constexpr int kRotCoarse = 480, kRotFine = 400;   /* kChanOutRate = kRotCoarse x kRotFine */
static_assert(kRotCoarse * kRotFine == kChanOutRate && kChanOutRate % 512 == 0, "rotation table shape");

/* FFT lengths that are not a power of two (320, 400, 640 = 2^a 5^b) run the mixed-radix passes of ChanPlan */
template <int L> constexpr bool kChanPow2 = (L & (L - 1)) == 0;

template <int M>
struct ChanShape {
  static constexpr int D = M / 2;
  static constexpr int N = kChanTaps * M;
  static constexpr int kThreads = M >= 256 ? M : 256;
  /* CTAs per SM (__launch_bounds__): shared memory allows 4 at M = 64, 3 at 320 (72 KiB each), 2 at 512, 1 at 640
     (137 KiB) */
  static constexpr int kMinBlocks = M == 512 ? 2 : M == 320 ? 3 : M == 640 ? 1 : 4;
  static constexpr int kGroups = kThreads / M;                  /* threads per branch */
  static constexpr int kTimes = kChanTile / kGroups;            /* output times per thread */
  static constexpr int kSpan = kChanTile * D + N;               /* capture samples a tile stages (one spare at the end) */
  static constexpr int kRow = M + 1;
  static constexpr int kHalf = kChanTile / 2;
  /* FFT rows: rows 0 .. kHalf - 1 after the span, rows kHalf .. in the span once it is dead.  Row r starts in bank
     column r (8-byte columns, 16 per 128 bytes), so a half-warp reading one channel of the 16 rows is conflict-free */
  static __device__ __forceinline__ int RowBase(int r) { return r < kHalf ? kSpan + r * kRow : (r - kHalf) * kRow + kHalf; }
  static constexpr int kSmemBytes = (kSpan + kHalf * kRow) * (int)sizeof(float2);
  /* with fine tuning the rotation table follows the rows (480 + 400 float2; two CTAs of 512 still fit an SM) */
  static constexpr int kRotBase = kSpan + kHalf * kRow;
  static constexpr int kSmemRotBytes = kSmemBytes + (kRotCoarse + kRotFine) * (int)sizeof(float2);
  static_assert(kChanTile % kGroups == 0 && T41RX_BLOCK_SAMPLES % kChanTile == 0 && kThreads % kChanTile == 0, "tile shape");
  static_assert(kSpan % 16 == 0 && (kHalf - 1) * kRow + kHalf + M <= kSpan, "row layout");
};

/* FFT row layout: element i (natural index) of a row lives at Phys(i); the DIF passes leave X[k] at OutPos(k) */
template <int M> __device__ __forceinline__ int ChanPhys(int i) { return M == 512 ? FftPhys(i) : i; }

/* mixed-radix DIF plans (DESIGN §3.10): the radices in pass order.  Rows of these lengths are in natural order */
template <int L> struct ChanPlan;
template <> struct ChanPlan<320> { static constexpr int kPasses = 3, kRadix[3] = {5, 8, 8}; };
template <> struct ChanPlan<400> { static constexpr int kPasses = 4, kRadix[4] = {5, 5, 8, 2}; };
template <> struct ChanPlan<640> { static constexpr int kPasses = 4, kRadix[4] = {5, 8, 8, 2}; };

/* where the DIF passes of ChanPlan<L> leave X[k]: the mixed-radix digit reversal.  The digits of k, least significant
   first, are in the radices r_0, r_1, ... of the passes, and digit s weighs L / (r_0 ... r_s) in the position */
template <int L, int kPass = 0, int Ls = L>
__device__ __forceinline__ int ChanMixedOutPos(int k) {
  constexpr int R = ChanPlan<L>::kRadix[kPass];
  if constexpr (kPass + 1 < ChanPlan<L>::kPasses) return (k % R) * (Ls / R) + ChanMixedOutPos<L, kPass + 1, Ls / R>(k / R);
  else return k * (Ls / R);
}

template <int M> __device__ __forceinline__ int ChanOutPos(int k) {
  if constexpr (!kChanPow2<M>) return ChanMixedOutPos<M>(k);
  else return M == 512 ? FftPhys((int)OctRev3((unsigned)k)) : (((k & 7) << 3) | (k >> 3));
}

/* (p + L/2) mod L for p in [0, L): the odd-m circular shift of a row's input */
template <int L> __device__ __forceinline__ int ChanHalfTurn(int p) {
  if constexpr (kChanPow2<L>) return p ^ (L / 2);
  else return p < L / 2 ? p + L / 2 : p - L / 2;
}

/* k mod L for k in [0, L] */
template <int L> __device__ __forceinline__ int ChanWrap(int k) {
  if constexpr (kChanPow2<L>) return k & (L - 1);
  else return k == L ? 0 : k;
}

/* one radix-8 DIF butterfly of the 64-point transform (two passes), twiddles from the 512-entry table */
__device__ __forceinline__ void Radix8Butterfly64(float2 *buf, const float2 *tw512, int pass, int b) {
  const int n2 = pass == 0 ? 8 : 1, j = pass == 0 ? b : 0, i0 = pass == 0 ? b : b * 8;
  float r[8], im[8];
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const float2 x = buf[i0 + m * n2];
    r[m] = x.x;
    im[m] = x.y;
  }
  Dft8(r, im);
  buf[i0] = float2{r[0], im[0]};
#pragma unroll
  for (int k = 1; k < 8; ++k) {
    float re = r[k], ie = im[k];
    if (j != 0) {
      const float2 w = tw512[j * k * 8];
      re = r[k] * w.x + im[k] * w.y;
      ie = im[k] * w.x - r[k] * w.y;
    }
    buf[i0 + k * n2] = float2{re, ie};
  }
}

__device__ __forceinline__ void CpAsync8(void *smem, const void *gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem) : "memory");
}

__device__ __forceinline__ void CpAsync16(void *smem, const void *gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
}

/* phi mod 192000 of x = shift m + P < 2^36: 192000 = 512 x 375, so x mod 192000 = ((x >> 9) mod 375) 512 + (x mod 512)
   with x >> 9 in 32 bits */
__device__ __forceinline__ unsigned ChanPhase(unsigned shift, unsigned m, unsigned p0) {
  const unsigned long long x = (unsigned long long)shift * m + p0;
  return (((unsigned)(x >> 9) % 375u) << 9) | ((unsigned)x & 511u);
}

/* exp(j 2 pi phi / 192000) for the entry (shift, P) = sp at output m_abs, from the staged two-level table */
__device__ __forceinline__ float2 ChanRotor(const float2 *tab, int2 sp, unsigned m_abs) {
  const unsigned phi = ChanPhase((unsigned)sp.x, m_abs, (unsigned)sp.y), a = phi / kRotFine;
  const float2 ca = tab[a], cb = tab[kRotCoarse + (phi - a * kRotFine)];
  return float2{ca.x * cb.x - ca.y * cb.y, ca.x * cb.y + ca.y * cb.x};
}

/* the store stage of a kernel instance (DESIGN §3.11): kChanPlain writes the (rotated) sample, as a single-input
   channelizer does; a diversity call runs the kernel once per input, kChanWeighted for input 0 (writes v w f) and
   kChanAccumulate for the others (adds v w f to iq).  Image correction (DESIGN §3.12, complex kinds only): kChanImage
   writes the (rotated) y_k = z_k + c_k conj(z_kbar), kChanImageTrack also writes each mirror pair's tile partials */
constexpr int kChanPlain = 0, kChanWeighted = 1, kChanAccumulate = 2, kChanImage = 3, kChanImageTrack = 4;

/* complex products with every rounding spelled out (__fmul_rn / __fmaf_rn are never contracted), so that the weighted
   instances round as the plain ones' SASS does whatever the compiler makes of their context:
   ChanMulRn(v, f) = (fma(v.x, f.x, -(v.y f.y)), fma(v.x, f.y, v.y f.x)), the plain store loop's v f;
   ChanRotorRn is ChanRotor's ca cb = (fma(ca.x, cb.x, -(ca.y cb.y)), fma(ca.y, cb.x, ca.x cb.y)) */
__device__ __forceinline__ float2 ChanMulRn(float2 v, float2 f) {
  return float2{__fmaf_rn(v.x, f.x, -__fmul_rn(v.y, f.y)), __fmaf_rn(v.x, f.y, __fmul_rn(v.y, f.x))};
}
__device__ __forceinline__ float2 ChanRotorRn(const float2 *tab, int2 sp, unsigned m_abs) {
  const unsigned phi = ChanPhase((unsigned)sp.x, m_abs, (unsigned)sp.y), a = phi / kRotFine;
  const float2 ca = tab[a], cb = tab[kRotCoarse + (phi - a * kRotFine)];
  return float2{__fmaf_rn(ca.x, cb.x, -__fmul_rn(ca.y, cb.y)), __fmaf_rn(ca.y, cb.x, __fmul_rn(ca.x, cb.y))};
}

/* a weighted instance's sample of one entry: v, its rotation factor f (from ChanRotorRn) and whether the entry is
   rotated (its phase is not identically 0) */
struct ChanSample {
  float2 v, f;
  bool rotated;
};

/* the store loop of the weighted instances: entry e = w / kChanTile, w = tid, tid + kThreads, ... < n_entries x
   kChanTile, four at a time; sample(e) is its ChanSample, iq the thread's sample of receiver 0's run (the thread
   always stores the same sample of the tile).  g = w f is formed once per sample; selects keep the default weights
   bit-exact: w = (1, 0) takes g = f, so v g is the plain instance's v f bit for bit, an entry with w = (1, 0) and no
   rotation stores v itself, and a zero weight leaves the accumulating pass's sample untouched rather than adding +0
   (-0 + 0 is +0).  The accumulating pass loads the four old samples before it stores any: with a store ahead of each
   next load (the compiler cannot tell the entries' addresses apart) every entry would wait for its own load */
template <int kStore, int kThreads, typename Sample>
__device__ __forceinline__ void ChanWeightedLoop(float2 *__restrict__ iq, const int32_t *__restrict__ recv,
                                                 const float2 *__restrict__ weight, int n_entries, int n_blocks, int tid,
                                                 Sample sample) {
  constexpr int kBatch = 4;
  const int n = n_entries * kChanTile;
  for (int w0 = tid; w0 < n; w0 += kBatch * kThreads) {
    float2 *dst[kBatch];
    float2 wt[kBatch], old[kBatch];
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      const int e = min(w0 + u * kThreads, n - 1) / kChanTile;
      dst[u] = iq + (long long)__ldg(recv + e) * n_blocks * T41RX_BLOCK_SAMPLES;
      wt[u] = __ldg(weight + e);
      if (kStore == kChanAccumulate && w0 + u * kThreads < n && (wt[u].x != 0.f || wt[u].y != 0.f)) old[u] = *dst[u];
    }
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      if (w0 + u * kThreads >= n) break;
      const float2 w = wt[u];
      const bool unit = w.x == 1.f && w.y == 0.f;
      if (kStore == kChanAccumulate && w.x == 0.f && w.y == 0.f) continue;
      const ChanSample s = sample((w0 + u * kThreads) / kChanTile);
      const float2 g = !s.rotated ? w : unit ? s.f : ChanMulRn(w, s.f);
      const float2 p = ChanMulRn(s.v, g);
      if constexpr (kStore == kChanWeighted)
        *dst[u] = !s.rotated && unit ? s.v : p;
      else
        *dst[u] = float2{__fadd_rn(old[u].x, p.x), __fadd_rn(old[u].y, p.y)};
    }
  }
}

/* z + c conj(zm), every rounding spelled out */
__device__ __forceinline__ float2 ChanImageRn(float2 z, float2 zm, float2 c) {
  return float2{__fmaf_rn(c.x, zm.x, __fmaf_rn(c.y, zm.y, z.x)), __fmaf_rn(c.y, zm.x, __fmaf_rn(-c.x, zm.y, z.y))};
}

/* the store stage of the kChanImage / kChanImageTrack instances.  image: the channelizer's image table, the M
   coefficients c_k and after them the tracking partials, float4 (Re A, Im A, P_k, P_kbar) [M/2 + 1][gridDim.x] (pair
   k, tile).
   First the FFT rows are corrected in place, a mirror pair (k, kbar = (M - k) mod M) at a time: y_k = z_k + c_k
   conj(z_kbar) and y_kbar = z_kbar + c_kbar conj(z_k) from the same z, each, when its c is 0, the z itself, selected.
   The rows hold every z_k with its (-1)^(k m) applied, and (-1)^((M - k) m) = (-1)^(k m) as M is even, so the mirror
   sample is used as it stands.  Half-warp h takes pairs h, h + kThreads / 16, ..., lane mm row mm (conflict-free: row
   r starts in bank column r); the tracking instance also sums the pair's three products over the 16 rows by a fixed
   shuffle tree.  Then the store loop is the plain one on the corrected rows, the rotation rounded as the plain
   instance's SASS rounds it (the Rn forms), so a channel whose c_k is 0 gets the plain instance's bits. */
template <int M, bool kRotate, bool kTrack, typename S>
__device__ __forceinline__ void ChanImageStore(float2 *smem, const int32_t *__restrict__ recv,
                                               const int32_t *__restrict__ chan, const int2 *__restrict__ phase,
                                               int m_base, long long m0, int n_entries, float2 *__restrict__ iq,
                                               int n_blocks, const float2 *__restrict__ image) {
  /* tid read again here: kept live from the span stage it spills a register in the q15 M = 512 tracking instance */
  int tid;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
  constexpr int kPairs = M / 2 + 1, kHalfWarps = S::kThreads / kChanTile;
  const int mm = tid % kChanTile;
  float2 *row = smem + S::RowBase(mm);
  float4 *part = reinterpret_cast<float4 *>(const_cast<float2 *>(image + M)) + blockIdx.x;
  /* unrolled 3 times without tracking, not with it (measured: about 0.5 % faster without, 1 - 2 % slower with) */
#pragma unroll (kTrack ? 1 : 3)
  for (int k0 = 0; k0 < kPairs; k0 += kHalfWarps) {    /* uniform over the warp: the shuffles need all 32 lanes */
    const int k = k0 + tid / kChanTile;
    if (!kTrack && k >= kPairs) break;
    const int kk = k < kPairs ? k : 0, kb = ChanWrap<M>(M - kk);
    const int pk = ChanOutPos<M>(kk), pb = ChanOutPos<M>(kb);
    const float2 zk = row[pk], zb = row[pb], ck = __ldg(image + kk), cb = __ldg(image + kb);
    const float2 yk = ck.x == 0.f && ck.y == 0.f ? zk : ChanImageRn(zk, zb, ck);
    const float2 yb = cb.x == 0.f && cb.y == 0.f ? zb : ChanImageRn(zb, zk, cb);
    if (k < kPairs) {
      row[pk] = yk;
      row[pb] = yb;    /* the same value as yk for the pairs 0 and M/2, their own mirrors */
    }
    if constexpr (kTrack) {
      float s[4] = {yk.x * yb.x - yk.y * yb.y, yk.x * yb.y + yk.y * yb.x, yk.x * yk.x + yk.y * yk.y,
                    yb.x * yb.x + yb.y * yb.y};
#pragma unroll
      for (int d = kChanTile / 2; d > 0; d >>= 1)
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] += __shfl_xor_sync(0xffffffffu, s[i], d);
      if (mm == 0 && k < kPairs) part[(long long)k * gridDim.x] = float4{s[0], s[1], s[2], s[3]};
    }
  }
  __syncthreads();
  const long long blk = m0 / T41RX_BLOCK_SAMPLES;
  const int s0 = (int)(m0 % T41RX_BLOCK_SAMPLES);
  const unsigned m_abs = (unsigned)((m_base + m0) % kChanOutRate) + mm;
#pragma unroll 4
  for (int w = tid; w < n_entries * kChanTile; w += S::kThreads) {
    const int e = w / kChanTile;
    const int k = __ldg(chan + e), r = __ldg(recv + e);
    const float2 y = row[ChanOutPos<M>(k)];
    float2 out = y;
    if constexpr (kRotate) {
      const int2 sp = __ldg(phase + e);
      out = (sp.x | sp.y) ? ChanMulRn(y, ChanRotorRn(smem + S::kRotBase, sp, m_abs)) : y;
    }
    iq[((long long)r * n_blocks + blk) * T41RX_BLOCK_SAMPLES + s0 + mm] = out;
  }
}

constexpr float kC51 = 0.309016994374947f, kC52 = -0.809016994374947f;   /* cos(2 pi / 5), cos(4 pi / 5) */
constexpr float kS51 = 0.951056516295154f, kS52 = 0.587785252292473f;    /* sin(2 pi / 5), sin(4 pi / 5) */

/* R-point DFTs (R = 2, 5, 8: the radices of ChanPlan), forward, natural-order output; r[], i[] are overwritten */
template <int R> __device__ __forceinline__ void ChanDft(float *r, float *i);
template <> __device__ __forceinline__ void ChanDft<8>(float *r, float *i) { Dft8(r, i); }
template <> __device__ __forceinline__ void ChanDft<5>(float *r, float *i) {
  const float t1r = r[1] + r[4], t1i = i[1] + i[4], t3r = r[1] - r[4], t3i = i[1] - i[4];
  const float t2r = r[2] + r[3], t2i = i[2] + i[3], t4r = r[2] - r[3], t4i = i[2] - i[3];
  const float a1r = r[0] + kC51 * t1r + kC52 * t2r, a1i = i[0] + kC51 * t1i + kC52 * t2i;
  const float a2r = r[0] + kC52 * t1r + kC51 * t2r, a2i = i[0] + kC52 * t1i + kC51 * t2i;
  const float b1r = kS51 * t3r + kS52 * t4r, b1i = kS51 * t3i + kS52 * t4i;   /* X1, X4 = a1 -/+ j b1 */
  const float b2r = kS52 * t3r - kS51 * t4r, b2i = kS52 * t3i - kS51 * t4i;   /* X2, X3 = a2 -/+ j b2 */
  r[0] = r[0] + t1r + t2r; i[0] = i[0] + t1i + t2i;
  r[1] = a1r + b1i; i[1] = a1i - b1r;
  r[4] = a1r - b1i; i[4] = a1i + b1r;
  r[2] = a2r + b2i; i[2] = a2i - b2r;
  r[3] = a2r - b2i; i[3] = a2i + b2r;
}
template <> __device__ __forceinline__ void ChanDft<2>(float *r, float *i) {
  const float sr = r[0] + r[1], si = i[0] + i[1];
  r[1] = r[0] - r[1]; i[1] = i[0] - i[1];
  r[0] = sr; i[0] = si;
}

/* butterfly b of a radix-R DIF pass that splits sub-transforms of length Ls of an L-point row (natural order):
   inputs i0 + m Ls / R, outputs k times exp(-j 2 pi j k / Ls) from tw, the L (cos, sin) of 2 pi t / L */
template <int L, int Ls, int R>
__device__ __forceinline__ void ChanMixedButterfly(float2 *row, const float2 *tw, int b) {
  constexpr int n2 = Ls / R;
  const int j = b % n2, i0 = (b / n2) * Ls + j;
  float r[R], im[R];
#pragma unroll
  for (int m = 0; m < R; ++m) {
    const float2 x = row[i0 + m * n2];
    r[m] = x.x;
    im[m] = x.y;
  }
  ChanDft<R>(r, im);
  row[i0] = float2{r[0], im[0]};
#pragma unroll
  for (int k = 1; k < R; ++k) {
    float re = r[k], ie = im[k];
    if (n2 > 1 && j != 0) {
      const float2 w = tw[j * k * (L / Ls)];
      re = r[k] * w.x + im[k] * w.y;
      ie = im[k] * w.x - r[k] * w.y;
    }
    row[i0 + k * n2] = float2{re, ie};
  }
}

/* pass kPass and the ones after it of the kChanTile rows' L-point FFTs; Ls: the sub-transform length it splits */
template <int L, typename S, int kPass, int Ls>
__device__ __forceinline__ void ChanMixedPasses(float2 *smem, const float2 *tw, int tid) {
  constexpr int R = ChanPlan<L>::kRadix[kPass], kBflyPerRow = L / R, kBfly = kChanTile * kBflyPerRow;
  for (int b = tid; b < kBfly; b += S::kThreads)
    ChanMixedButterfly<L, Ls, R>(smem + S::RowBase(b / kBflyPerRow), tw, b % kBflyPerRow);
  __syncthreads();
  if constexpr (kPass + 1 < ChanPlan<L>::kPasses) ChanMixedPasses<L, S, kPass + 1, Ls / R>(smem, tw, tid);
}

/* the in-place FFTs of the kChanTile rows of a tile (M-point; S::RowBase places the rows).  tw512: the 512 (cos, sin)
   of 2 pi k / 512, or for a mixed-radix M the M of 2 pi k / M */
template <int M, typename S>
__device__ __forceinline__ void ChanRowsFft(float2 *smem, const float2 *tw512, int tid) {
  if constexpr (!kChanPow2<M>) {
    ChanMixedPasses<M, S, 0, M>(smem, tw512, tid);
  } else {
    constexpr int kBflyPerRow = M / 8, kBfly = kChanTile * kBflyPerRow;
#pragma unroll
    for (int pass = 0; pass < (M == 512 ? 3 : 2); ++pass) {
      for (int b = tid; b < kBfly; b += S::kThreads) {
        float2 *row = smem + S::RowBase(b / kBflyPerRow);
        if (M == 512) Radix8Butterfly<true>(row, tw512, pass, b % kBflyPerRow);
        else Radix8Butterfly64(row, tw512, pass, b % kBflyPerRow);
      }
      __syncthreads();
    }
  }
}

/* int16 -> float, exactly: 0x4B400000 + v are the bits of 1.5 x 2^23 + v (|v| < 2^22 keeps the exponent), one integer
   add and one float subtract where a conversion instruction issues at an eighth of the FMA rate */
__device__ __forceinline__ float ChanS16(short v) { return __int_as_float(0x4B400000 + (int)v) - 12582912.0f; }

/* t41rx_chan_kernel's dynamic shared memory.  The q15 instances have their own name for it: their float4 stores would
   otherwise change what the compiler infers about the float instances' smem, and with it their code; 16-byte aligned
   for those stores */
template <typename T> __device__ __forceinline__ float2 *ChanSmem();
template <> __device__ __forceinline__ float2 *ChanSmem<float2>() {
  extern __shared__ float2 smem[];
  return smem;
}
template <> __device__ __forceinline__ float2 *ChanSmem<short>() {
  extern __shared__ __align__(16) float2 smem_q15[];
  return smem_q15;
}

/* capture: the call's samples; tail: the N samples before them; T = float2 (complex float) or short (int16 (I, Q)
   pairs, 16-byte aligned, with h / 32768 in taps: the input scale, exact); recv / chan: the mapped receivers grouped by
   channel (CSR order) and the channel of each; phase: each entry's (shift, P) in [0, 192000), or null when no entry is
   rotated; rot: the 480 + 400 factors of the rotation table; m_base: outputs before this call, mod 192000;
   iq: [n_receivers][n_blocks][2048].  kRotate = false (no entry rotated) is the kernel without fine tuning.
   kStore: the store stage (ChanWeightedLoop, ChanImageStore); weight: each entry's weight for this pass's input, in
   the order of recv (read by the weighted instances only), or for the image instances the channelizer's image table
   (ChanImageStore).
   The int16 span goes through registers (16-byte loads of four pairs) and lands converted, (I, Q) as integer-valued
   floats, where the float span is staged: each sample is converted once, not at each of the ~9 branch loads that read
   it, and the rest of the kernel is the same for both.  h / 32768 times I is h times I / 32768 exactly, so every FMA,
   and every output bit, is that of the float instance on x = s / 32768. */
template <int M, bool kRotate, typename T, int kStore>
__global__ void __launch_bounds__(ChanShape<M>::kThreads, ChanShape<M>::kMinBlocks)
t41rx_chan_kernel(const T *__restrict__ capture, const T *__restrict__ tail, const float *__restrict__ taps,
                  const float2 *__restrict__ tw512, const int32_t *__restrict__ recv, const int32_t *__restrict__ chan,
                  const int2 *__restrict__ phase, const float2 *__restrict__ rot, int m_base, int n_entries,
                  float2 *__restrict__ iq, int n_blocks, const float2 *__restrict__ weight) {
  using S = ChanShape<M>;
  float2 *smem = ChanSmem<T>();
  const int tid = threadIdx.x;
  const long long m0 = (long long)blockIdx.x * kChanTile;
  const long long n_base = m0 * S::D - S::N;    /* capture index of smem[0]; a multiple of 4, as N is */

  if constexpr (std::is_same_v<T, float2>) {
    for (int l = tid; l < S::kSpan; l += S::kThreads) {
      const long long n = n_base + l;
      CpAsync8(smem + l, n < 0 ? tail + (n + S::N) : capture + n);
    }
    if (kRotate)
      for (int l = tid; l < kRotCoarse + kRotFine; l += S::kThreads) CpAsync8(smem + S::kRotBase + l, rot + l);
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
  } else {
    constexpr int kQuads = S::kSpan / 4;                                  /* 16 bytes of int16 pairs each */
    constexpr int kPerThread = (kQuads + S::kThreads - 1) / S::kThreads;
    if (kRotate)
      for (int l = tid; l < kRotCoarse + kRotFine; l += S::kThreads) CpAsync8(smem + S::kRotBase + l, rot + l);
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    uint4 quad[kPerThread];
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      const int l = tid + i * S::kThreads;
      const long long n = n_base + 4 * l;
      if (l < kQuads) quad[i] = __ldg(reinterpret_cast<const uint4 *>(n < 0 ? tail + 2 * (n + S::N) : capture + 2 * n));
    }
    auto pair = [](unsigned v) { return float2{ChanS16((short)(v & 0xFFFFu)), ChanS16((short)(v >> 16))}; };
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      const int l = tid + i * S::kThreads;
      if (l < kQuads) {
        float4 *dst = reinterpret_cast<float4 *>(smem + 4 * l);
        const float2 a = pair(quad[i].x), b = pair(quad[i].y), c = pair(quad[i].z), d = pair(quad[i].w);
        dst[0] = float4{a.x, a.y, b.x, b.y};
        dst[1] = float4{c.x, c.y, d.x, d.y};
      }
    }
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  }

  const int p = tid % M, g = tid / M;
  float h[kChanTaps];
#pragma unroll
  for (int q = 0; q < kChanTaps; ++q) h[q] = __ldg(taps + p + q * M);
  __syncthreads();

  /* u_p[m] for this thread's output times m = g + kGroups t (smem index of x[mD - p - qM]: mD + N - p - qM), conj(u)
     stored at index p of row m, or p + M/2 (mod M) for odd m (m0 is even: m and the tile's row have the same parity).
     The first half of the rows lies outside the span and is written at once; the second half waits for the barrier
     that ends the span's life.  Half the accumulators live at a time: 512 threads x 2 CTAs per SM leave 64 registers. */
  auto branch = [&](int t) {
    const float2 *x = smem + (g + S::kGroups * t) * S::D + S::N - p;
    float ar = 0.f, ai = 0.f;
#pragma unroll
    for (int q = 0; q < kChanTaps; ++q) {
      const float2 v = x[-q * M];
      ar = fmaf(h[q], v.x, ar);
      ai = fmaf(h[q], v.y, ai);
    }
    return float2{ar, -ai};
  };
  auto slot = [&](int t) {
    const int mm = g + S::kGroups * t;
    return S::RowBase(mm) + ChanPhys<M>((mm & 1) ? ChanHalfTurn<M>(p) : p);
  };
  constexpr int kLate = S::kTimes / 2;
#pragma unroll
  for (int t = 0; t < kLate; ++t) smem[slot(t)] = branch(t);
  float2 u[kLate];
#pragma unroll
  for (int t = 0; t < kLate; ++t) u[t] = branch(kLate + t);
  __syncthreads();
#pragma unroll
  for (int t = 0; t < kLate; ++t) smem[slot(kLate + t)] = u[t];
  __syncthreads();

  ChanRowsFft<M, S>(smem, tw512, tid);

  /* each receiver's run: kChanTile consecutive samples inside one block (the tile size divides 2048).  The store loops
     are written out here and again in t41rx_chan_real_kernel: as one __device__ function taking the sample as a lambda
     they compile to different (longer) code in every instance of this kernel. */
  if constexpr (kStore == kChanImage || kStore == kChanImageTrack) {
    ChanImageStore<M, kRotate, kStore == kChanImageTrack, S>(smem, recv, chan, phase, m_base, m0, n_entries, iq, n_blocks,
                                                             weight);
    return;
  }
  const long long blk = m0 / T41RX_BLOCK_SAMPLES;
  const int s0 = (int)(m0 % T41RX_BLOCK_SAMPLES);
  if constexpr (kStore == kChanWeighted || kStore == kChanAccumulate) {
    const int mm = tid % kChanTile;
    const unsigned m_abs = (unsigned)((m_base + m0) % kChanOutRate) + mm;
    ChanWeightedLoop<kStore, S::kThreads>(iq + (blk * T41RX_BLOCK_SAMPLES + s0 + mm), recv, weight, n_entries, n_blocks,
                                          tid, [&](int e) {
      const float2 v = smem[S::RowBase(mm) + ChanOutPos<M>(__ldg(chan + e))];
      if constexpr (!kRotate) {
        return ChanSample{v, float2{1.f, 0.f}, false};
      } else {
        const int2 sp = __ldg(phase + e);
        return ChanSample{v, ChanRotorRn(smem + S::kRotBase, sp, m_abs), (sp.x | sp.y) != 0};
      }
    });
    return;
  }
  if (!kRotate) {
    for (int w = tid; w < n_entries * kChanTile; w += S::kThreads) {
      const int e = w / kChanTile, mm = w % kChanTile;
      const int k = __ldg(chan + e), r = __ldg(recv + e);
      iq[((long long)r * n_blocks + blk) * T41RX_BLOCK_SAMPLES + s0 + mm] = smem[S::RowBase(mm) + ChanOutPos<M>(k)];
    }
    return;
  }
  /* a thread always stores the same sample mm of the tile (kThreads is a multiple of kChanTile): its m_abs mod 192000.
     The body has no branch (an entry with phase 0 selects the sample unmultiplied), so unrolled iterations overlap. */
  const int mm = tid % kChanTile;
  const unsigned m_abs = (unsigned)((m_base + m0) % kChanOutRate) + mm;
  const float2 *tab = smem + S::kRotBase;
#pragma unroll 4
  for (int w = tid; w < n_entries * kChanTile; w += S::kThreads) {
    const int e = w / kChanTile;
    const int k = __ldg(chan + e), r = __ldg(recv + e);
    const int2 sp = __ldg(phase + e);
    const float2 v = smem[S::RowBase(mm) + ChanOutPos<M>(k)];
    const float2 f = ChanRotor(tab, sp, m_abs);
    const float2 vr = float2{v.x * f.x - v.y * f.y, v.x * f.y + v.y * f.x};
    iq[((long long)r * n_blocks + blk) * T41RX_BLOCK_SAMPLES + s0 + mm] = (sp.x | sp.y) ? vr : v;
  }
}

template <int M>
struct ChanRealShape {
  static constexpr int Mc = M / 2;                              /* length of the complex FFT */
  static constexpr int D = M / 2;
  static constexpr int N = kChanTaps * M;
  static constexpr int kThreads = Mc >= 256 ? Mc : 256;
  /* CTAs per SM (__launch_bounds__): 4 at M = 128, 2 at 800 (76 KiB each) and 1024, 1 at 1280 (117 KiB) */
  static constexpr int kMinBlocks = M == 1024 || M == 800 ? 2 : M == 1280 ? 1 : 4;
  static constexpr int kGroups = kThreads / Mc;                 /* threads per branch pair */
  static constexpr int kTimes = kChanTile / kGroups;
  static constexpr int kSpan = kChanTile * D + N;               /* int16 capture samples a tile stages */
  static constexpr int kSpanF2 = kSpan * 2 / (int)sizeof(float2);
  static constexpr int kRow = Mc + 1;
  /* the int16 span is half the size of the complex kernel's, so only a quarter of the rows wait for it to die: the
     thread holds 4 accumulators beside its 20 taps (8 spill at the 64 registers two CTAs of 512 allow) */
  static constexpr int kLateTimes = kTimes / 4;
  static constexpr int kEarly = kChanTile - kGroups * kLateTimes;   /* rows outside the span */
  /* row r starts in bank column r, as in t41rx_chan_kernel */
  static __device__ __forceinline__ int RowBase(int r) { return r < kEarly ? kSpanF2 + r * kRow : (r - kEarly) * kRow + kEarly; }
  static constexpr int kSplitBase = kSpanF2 + kEarly * kRow;    /* Mc + 1 (cos, sin) of 2 pi k / M */
  static constexpr int kRotBase = kSplitBase + Mc + 1;
  static constexpr int kSmemBytes = kRotBase * (int)sizeof(float2);
  static constexpr int kSmemRotBytes = kSmemBytes + (kRotCoarse + kRotFine) * (int)sizeof(float2);
  static_assert(kChanTile % kGroups == 0 && kThreads % kChanTile == 0, "tile shape");
  static_assert(kSpan % 8 == 0 && N % 8 == 0 && kSpanF2 % 16 == 0 && kTimes % 4 == 0, "span shape");
  static_assert((kChanTile - 1 - kEarly) * kRow + kEarly + Mc <= kSpanF2, "late rows inside the span");
};

/* capture / tail: int16, 16-byte aligned; taps: h / 65536 (the 1 / 32768 of the input scale and the split's 1 / 2,
   both exact); split: (cos, sin) of 2 pi k / M, k <= M / 2; the rest as t41rx_chan_kernel.  Channel k in [0, M/2]. */
template <int M, bool kRotate, int kStore>
__global__ void __launch_bounds__(ChanRealShape<M>::kThreads, ChanRealShape<M>::kMinBlocks)
t41rx_chan_real_kernel(const short *__restrict__ capture, const short *__restrict__ tail, const float *__restrict__ taps,
                       const float2 *__restrict__ tw512, const float2 *__restrict__ split, const int32_t *__restrict__ recv,
                       const int32_t *__restrict__ chan, const int2 *__restrict__ phase, const float2 *__restrict__ rot,
                       int m_base, int n_entries, float2 *__restrict__ iq, int n_blocks, const float2 *__restrict__ weight) {
  using S = ChanRealShape<M>;
  constexpr int Mc = S::Mc;
  extern __shared__ float2 smem[];
  const short *span = reinterpret_cast<const short *>(smem);
  const int tid = threadIdx.x;
  const long long m0 = (long long)blockIdx.x * kChanTile;
  const long long n_base = m0 * S::D - S::N;    /* capture index of span[0]; a multiple of 8, as N is */

  for (int l = tid; l < S::kSpan / 8; l += S::kThreads) {
    const long long n = n_base + 8 * l;
    CpAsync16(smem + 2 * l, n < 0 ? tail + (n + S::N) : capture + n);
  }
  for (int l = tid; l <= Mc; l += S::kThreads) CpAsync8(smem + S::kSplitBase + l, split + l);
  if (kRotate)
    for (int l = tid; l < kRotCoarse + kRotFine; l += S::kThreads) CpAsync8(smem + S::kRotBase + l, rot + l);
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");

  const int p = tid % Mc, g = tid / Mc;
  float he[kChanTaps], ho[kChanTaps];
#pragma unroll
  for (int q = 0; q < kChanTaps; ++q) {
    he[q] = __ldg(taps + 2 * p + q * M);
    ho[q] = __ldg(taps + 2 * p + 1 + q * M);
  }
  __syncthreads();

  /* y_p[m] = u_2p[m] + j u_2p+1[m] (span index of x[mD - 2p - qM]: mD + N - 2p - qM), stored at index p of row m, or
     p + Mc/2 (mod Mc) for odd m; the late rows wait for the barrier that ends the span's life, as in t41rx_chan_kernel */
  auto branch = [&](int t) {
    const short *x = span + (g + S::kGroups * t) * S::D + S::N - 2 * p;
    float ar = 0.f, ai = 0.f;
#pragma unroll
    for (int q = 0; q < kChanTaps; ++q) {
      ar = fmaf(he[q], ChanS16(x[-q * M]), ar);
      ai = fmaf(ho[q], ChanS16(x[-q * M - 1]), ai);
    }
    return float2{ar, ai};
  };
  auto slot = [&](int t) {
    const int mm = g + S::kGroups * t;
    return S::RowBase(mm) + ChanPhys<Mc>((mm & 1) ? ChanHalfTurn<Mc>(p) : p);
  };
  constexpr int kEarlyTimes = S::kTimes - S::kLateTimes;
  /* not unrolled: interleaving the output times' loads pushes two taps out of the 64 registers at M = 1024 */
#pragma unroll 1
  for (int t = 0; t < kEarlyTimes; ++t) smem[slot(t)] = branch(t);
  float2 u[S::kLateTimes];
#pragma unroll
  for (int t = 0; t < S::kLateTimes; ++t) u[t] = branch(kEarlyTimes + t);
  __syncthreads();
#pragma unroll
  for (int t = 0; t < S::kLateTimes; ++t) smem[slot(kEarlyTimes + t)] = u[t];
  __syncthreads();

  ChanRowsFft<Mc, S>(smem, tw512, tid);

  /* X[k] of row mm from Y[k] and Y[Mc - k] (the 1 / 2 is in the taps) */
  const float2 *w_tab = smem + S::kSplitBase;
  auto sample = [&](int mm, int k) {
    const float2 a = smem[S::RowBase(mm) + ChanOutPos<Mc>(ChanWrap<Mc>(k))];
    const float2 b = smem[S::RowBase(mm) + ChanOutPos<Mc>(ChanWrap<Mc>(Mc - k))];
    const float2 w = w_tab[k];
    const float sr = a.x + b.x, si = a.y - b.y, dr = a.x - b.x, di = a.y + b.y;
    return float2{sr + w.x * di - w.y * dr, si - w.y * di - w.x * dr};
  };
  const long long blk = m0 / T41RX_BLOCK_SAMPLES;
  const int s0 = (int)(m0 % T41RX_BLOCK_SAMPLES);
  const int mm = tid % kChanTile;    /* w % kChanTile below: kThreads is a multiple of kChanTile */
  if constexpr (kStore != kChanPlain) {
    const unsigned m_abs = (unsigned)((m_base + m0) % kChanOutRate) + mm;
    ChanWeightedLoop<kStore, S::kThreads>(iq + (blk * T41RX_BLOCK_SAMPLES + s0 + mm), recv, weight, n_entries, n_blocks,
                                          tid, [&](int e) {
      const float2 v = sample(mm, __ldg(chan + e));
      if constexpr (!kRotate) {
        return ChanSample{v, float2{1.f, 0.f}, false};
      } else {
        const int2 sp = __ldg(phase + e);
        return ChanSample{v, ChanRotorRn(smem + S::kRotBase, sp, m_abs), (sp.x | sp.y) != 0};
      }
    });
    return;
  }
  if (!kRotate) {
    for (int w = tid; w < n_entries * kChanTile; w += S::kThreads) {
      const int e = w / kChanTile;
      const int k = __ldg(chan + e), r = __ldg(recv + e);
      iq[((long long)r * n_blocks + blk) * T41RX_BLOCK_SAMPLES + s0 + mm] = sample(mm, k);
    }
    return;
  }
  const unsigned m_abs = (unsigned)((m_base + m0) % kChanOutRate) + mm;
  const float2 *tab = smem + S::kRotBase;
#pragma unroll 4
  for (int w = tid; w < n_entries * kChanTile; w += S::kThreads) {
    const int e = w / kChanTile;
    const int k = __ldg(chan + e), r = __ldg(recv + e);
    const int2 sp = __ldg(phase + e);
    const float2 v = sample(mm, k);
    const float2 f = ChanRotor(tab, sp, m_abs);
    const float2 vr = float2{v.x * f.x - v.y * f.y, v.x * f.y + v.y * f.x};
    iq[((long long)r * n_blocks + blk) * T41RX_BLOCK_SAMPLES + s0 + mm] = (sp.x | sp.y) ? vr : v;
  }
}

/* image tracking, after a kChanImageTrack pass on the same stream: CTA k sums pair k's `tiles` partials in double, in
   a fixed order (thread t takes tiles t, t + 256, ..., then a shared-memory tree), so the sums do not depend on how
   the tiles were scheduled.  It writes stats[k] = (Re A, Im A, P_k, P_kbar) and, for k = 1 .. M/2 - 1, applies the
   dominant-side rule: c_kbar -= A / P_k if P_k >= T P_kbar, else c_k -= A / P_kbar if P_kbar >= T P_k (T = dominance
   >= 1, both P > 0), in double, rounded to float.  Channels 0 and M/2 are never updated. */
constexpr int kChanImageThreads = 256;
__global__ void __launch_bounds__(kChanImageThreads)
t41rx_chan_image_update(float2 *__restrict__ image, int M, int tiles, double dominance, double *__restrict__ stats) {
  __shared__ double red[4][kChanImageThreads];
  const int k = blockIdx.x, tid = threadIdx.x;
  const float4 *part = reinterpret_cast<const float4 *>(image + M) + (long long)k * tiles;
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  for (int t = tid; t < tiles; t += kChanImageThreads) {
    const float4 v = part[t];
    s[0] = __dadd_rn(s[0], (double)v.x);
    s[1] = __dadd_rn(s[1], (double)v.y);
    s[2] = __dadd_rn(s[2], (double)v.z);
    s[3] = __dadd_rn(s[3], (double)v.w);
  }
  for (int i = 0; i < 4; ++i) red[i][tid] = s[i];
  for (int h = kChanImageThreads / 2; h > 0; h >>= 1) {
    __syncthreads();
    if (tid < h)
      for (int i = 0; i < 4; ++i) red[i][tid] = __dadd_rn(red[i][tid], red[i][tid + h]);
  }
  if (tid != 0) return;
  const double ar = red[0][0], ai = red[1][0], pk = red[2][0], pb = red[3][0];
  stats[4 * k] = ar;
  stats[4 * k + 1] = ai;
  stats[4 * k + 2] = pk;
  stats[4 * k + 3] = pb;
  if (k < 1 || k >= M / 2) return;
  int j = -1;
  double p = 0.0;
  if (pk > 0.0 && pk >= __dmul_rn(dominance, pb)) j = M - k, p = pk;
  else if (pb > 0.0 && pb >= __dmul_rn(dominance, pk)) j = k, p = pb;
  if (j < 0) return;
  const float2 c = image[j];
  image[j] = float2{(float)__dsub_rn((double)c.x, __ddiv_rn(ar, p)), (float)__dsub_rn((double)c.y, __ddiv_rn(ai, p))};
}

/* modified Bessel function I0 (power series; terms fall below 1e-17 of the sum well before k = 60 for beta <= 9) */
static double BesselI0(double x) {
  double sum = 1.0, term = 1.0;
  const double q = 0.25 * x * x;
  for (int k = 1; k < 60; ++k) {
    term *= q / ((double)k * k);
    sum += term;
    if (term < 1e-17 * sum) break;
  }
  return sum;
}

/* the prototype: Kaiser-windowed sinc, cutoff 96 kHz at M x 96 kS/s (2 / M of Nyquist), designed in FP64, unit DC gain,
   mirrored so that it is symmetric to the bit, rounded to float */
static void DesignChanTaps(int M, float *out) {
  const int N = kChanTaps * M;
  const double fc = 2.0 / M, half = 0.5 * (N - 1);
  std::vector<double> h(N);
  double sum = 0.0;
  for (int n = 0; n < N / 2; ++n) {
    const double t = n - half;                       /* never 0: N is even */
    const double sinc = sin(M_PI * fc * t) / (M_PI * fc * t);
    const double r = (n - half) / half;
    const double w = BesselI0(kChanBeta * sqrt(std::max(0.0, 1.0 - r * r))) / BesselI0(kChanBeta);
    h[n] = h[N - 1 - n] = fc * sinc * w;
    sum += 2.0 * h[n];
  }
  for (int n = 0; n < N; ++n) out[n] = (float)(h[n] / sum);
}

/* complex: 6.144, 30.72, 49.152, 61.44 MS/s; real: 12.288, 76.8, 98.304, 122.88 MS/s */
static bool ChanCountOk(int n_channels) {
  return n_channels == 64 || n_channels == 320 || n_channels == 512 || n_channels == 640;
}
static bool ChanRealCountOk(int n_channels) {
  return n_channels == 128 || n_channels == 800 || n_channels == 1024 || n_channels == 1280;
}

template <typename K>
static cudaError_t ChanSmemAttr(K plain, int plain_bytes, K rotating, int rotating_bytes) {
  const cudaError_t e = cudaFuncSetAttribute(plain, cudaFuncAttributeMaxDynamicSharedMemorySize, plain_bytes);
  return e != cudaSuccess ? e : cudaFuncSetAttribute(rotating, cudaFuncAttributeMaxDynamicSharedMemorySize, rotating_bytes);
}

/* the channel centre j x 96 kHz nearest to offset_hz (j in [-M/2, M/2]; j = M/2 is channel M/2, centre -Fs/2, the same
   frequency as +Fs/2), the offset from it, and whether the mode's front end mirrors the stream.  real: a real
   channelizer's M, offset_hz is the absolute frequency in [0, Fs/2] and the channel is j itself, in [0, M/2]. */
static int ChanNearest(const char *fn, bool real, int n_channels, int32_t mode, double offset_hz, int32_t *channel,
                       double *f_rel, bool *mirrored) {
  if (!channel || !(real ? ChanRealCountOk(n_channels) : ChanCountOk(n_channels)))
    return SetApiError(T41RX_EINVAL, (std::string(fn) + ": bad arguments").c_str());
  t41rx_params p;
  DefaultParams(&p);
  p.mode = mode;
  t41rx_mode_default_cuts(mode, &p.f_lo_cut, &p.f_hi_cut);
  if (!ValidateParams(p)) return SetApiError(T41RX_EINVAL, (std::string(fn) + ": invalid mode").c_str());
  const double half = 0.5 * n_channels * kChanSpacing;
  if (real ? !(offset_hz >= 0.0 && offset_hz <= half) : !(offset_hz >= -half && offset_hz < half))
    return SetApiError(T41RX_EINVAL, (std::string(fn) + (real ? ": frequency outside the capture's band [0, Fs/2]"
                                                               : ": offset outside the capture's band [-Fs/2, Fs/2)")).c_str());
  const int j = (int)floor(offset_hz / kChanSpacing + 0.5);
  *f_rel = offset_hz - j * kChanSpacing;
  *mirrored = mode == T41RX_DEMOD_USB || mode == T41RX_DEMOD_LSB || mode == T41RX_DEMOD_AM || mode == T41RX_DEMOD_SAM;
  *channel = real ? j : (j + n_channels) % n_channels;
  return T41RX_OK;
}

/* t41rx_chan_tune / _tune_real */
static int ChanTune(const char *fn, bool real, int n_channels, int32_t mode, double offset_hz, int32_t *channel,
                    int32_t *nco_freq) {
  if (!nco_freq) return SetApiError(T41RX_EINVAL, (std::string(fn) + ": bad arguments").c_str());
  double f_rel = 0.0;
  bool mirrored = false;
  const int rc = ChanNearest(fn, real, n_channels, mode, offset_hz, channel, &f_rel, &mirrored);
  if (rc) return rc;
  *nco_freq = (int32_t)llrint(mirrored ? 48000.0 + f_rel : 48000.0 - f_rel);
  return T41RX_OK;
}

/* t41rx_chan_place / _place_real */
static int ChanPlace(const char *fn, bool real, int n_channels, int32_t mode, double offset_hz, int32_t *channel,
                     int32_t *shift_hz, int32_t *nco_freq) {
  if (!shift_hz || !nco_freq) return SetApiError(T41RX_EINVAL, (std::string(fn) + ": bad arguments").c_str());
  double f_rel = 0.0;
  bool mirrored = false;
  const int rc = ChanNearest(fn, real, n_channels, mode, offset_hz, channel, &f_rel, &mirrored);
  if (rc) return rc;
  /* the signal moved from where t41rx_chan_tune's NCOFreq picks it up to NCOFreq 0: the mirrored modes see the stream
     conjugated, so their shift has the opposite sign */
  *shift_hz = (int32_t)llrint(mirrored ? 48000.0 + f_rel : f_rel - 48000.0);
  *nco_freq = 0;
  return T41RX_OK;
}

/* what a channelizer takes: complex float (t41rx_chan_create), real int16 (t41rx_chan_create_real, channels
   0 .. n_channels / 2), complex int16 pairs (t41rx_chan_create_q15) */
enum class ChanKind { kFloat, kReal, kQ15 };

/* bytes of one capture sample of a kind (the tail keeps N of them) */
static size_t ChanSampleBytes(ChanKind kind) {
  return kind == ChanKind::kFloat ? sizeof(float2) : kind == ChanKind::kReal ? sizeof(int16_t) : 2 * sizeof(int16_t);
}

/* a channelizer's kernels (without and with fine tuning, in each store mode), chosen by kind and M at creation: prepare
   raises their dynamic shared memory limits, launch enqueues one pass over one input: capture and tail are that
   input's, store its kChanPlain / kChanWeighted / kChanAccumulate, weight its entries' weights */
struct ChanKernels {
  cudaError_t (*prepare)();
  cudaError_t (*launch)(const t41rx_chan *c, const void *capture, const void *tail, int store, const float2 *weight,
                        float2 *iq, int n_blocks, cudaStream_t st);
};

}  // namespace t41rx

using namespace t41rx;

struct t41rx_chan {
  int device = 0;
  int n_channels = 0;
  int n_receivers = 0;
  ChanKind kind = ChanKind::kFloat;
  int n_inputs = 1;              /* 2 .. 4: a diversity channelizer (t41rx_chan_create_diversity) */
  cudaStream_t stream = nullptr;
  /* t41rx_chan_process_device may enqueue on a caller-supplied stream: its end is recorded here, and set_map /
     synchronize / destroy wait for it (the ordering contract of t41rx_process_device) */
  cudaEvent_t ev_ext = nullptr;
  bool ext_pending = false;
  float *d_taps = nullptr;       /* N (real: h / 65536, q15: h / 32768) */
  float2 *d_tw = nullptr;        /* 512 (cos, sin) of 2 pi k / 512, or L of 2 pi k / L (mixed-radix FFT length L) */
  float2 *d_split = nullptr;     /* real: n_channels / 2 + 1 (cos, sin) of 2 pi k / n_channels */
  void *d_tail = nullptr;        /* per input, the last N capture samples of the previous calls (zeros at creation) */
  int32_t *d_recv = nullptr, *d_chan = nullptr;   /* mapped receivers grouped by channel, and their channel */
  int2 *d_phase = nullptr;       /* each entry's (shift, P), in the order of d_recv */
  float2 *d_weight = nullptr;    /* diversity: [n_inputs][n_receivers], input a's weight of each entry, in the order of d_recv */
  float2 *d_rot = nullptr;       /* 480 + 400: exp(j 2 pi a / 480), exp(j 2 pi b / 192000) */
  int n_entries = 0;
  bool any_rotated = false;      /* some entry's phase is not identically 0 */
  std::vector<int32_t> map;      /* receiver -> channel or -1 */
  std::vector<int32_t> shift, p0;   /* receiver -> shift and phase offset P, both in [0, 192000) */
  std::vector<float2> weight;    /* diversity: [n_receivers][n_inputs], (1, 0) for input 0 and 0 for the others at creation */
  int m_done = 0;                /* outputs produced since creation, mod 192000 */
  ChanKernels kernels{};
  /* image correction (complex single-input channelizers, DESIGN §3.12) */
  ChanKernels image_kernels{};
  float2 *d_image = nullptr;     /* the image table: n_channels c_k, then the tracking partials of image_tiles tiles */
  double *d_image_stats = nullptr;   /* [n_channels / 2 + 1][4] of the last call with tracking on */
  long long image_tiles = 0;
  bool any_image = false;        /* some c_k is not 0 (as of the last set_image or tracking switch-off) */
  bool track = false, has_stats = false;
  double dominance = 100.0;      /* tracking's T, linear (20 dB) */
};

/* fn was called on a channelizer of another kind, or with a diversity channelizer's call on a single-input one or the
   other way round: EINVAL, naming the entry point this one takes */
static int ChanWrongKind(const char *fn, const t41rx_chan *c) {
  const char *takes = c->n_inputs > 1 ? ": a diversity channelizer takes t41rx_chan_process_device_diversity"
                      : c->kind == ChanKind::kFloat ? ": a complex float channelizer takes t41rx_chan_process_device"
                      : c->kind == ChanKind::kReal  ? ": a real channelizer takes t41rx_chan_process_device_real"
                                                    : ": a q15 channelizer takes t41rx_chan_process_device_q15";
  return SetApiError(T41RX_EINVAL, (std::string(fn) + takes).c_str());
}

/* K::Pass<kStore> launches the kernel of one store mode, the one without or with fine tuning by c->any_rotated.  A
   channelizer's kernels come in sets: a single-input channelizer's are the plain ones (kChanSetPlain), a diversity
   channelizer's the two weighted modes (kChanSetDiversity), and a complex single-input channelizer also has the two
   image modes (kChanSetImage).  The sets are kept apart so that the plain instances are instantiated first and in the
   order they always were, then the weighted ones, then the image ones: the compiler's code for the M = 320 and 512
   instances depends on where the other instances fall in the module */
constexpr int kChanSetPlain = 0, kChanSetDiversity = 1, kChanSetImage = 2;
template <typename K, int kSet>
static cudaError_t ChanPrepare() {
  if constexpr (kSet == kChanSetPlain) {
    return K::template PrepareStore<kChanPlain>();
  } else if constexpr (kSet == kChanSetDiversity) {
    const cudaError_t e = K::template PrepareStore<kChanWeighted>();
    return e == cudaSuccess ? K::template PrepareStore<kChanAccumulate>() : e;
  } else {
    const cudaError_t e = K::template PrepareStore<kChanImage>();
    return e == cudaSuccess ? K::template PrepareStore<kChanImageTrack>() : e;
  }
}
template <typename K, int kSet>
static cudaError_t ChanLaunch(const t41rx_chan *c, const void *capture, const void *tail, int store,
                              const float2 *weight, float2 *iq, int n_blocks, cudaStream_t st) {
  if constexpr (kSet == kChanSetPlain) {
    K::template Pass<kChanPlain>(c, capture, tail, weight, iq, n_blocks, st);
  } else if constexpr (kSet == kChanSetDiversity) {
    if (store == kChanWeighted) K::template Pass<kChanWeighted>(c, capture, tail, weight, iq, n_blocks, st);
    else K::template Pass<kChanAccumulate>(c, capture, tail, weight, iq, n_blocks, st);
  } else {
    if (store == kChanImage) K::template Pass<kChanImage>(c, capture, tail, weight, iq, n_blocks, st);
    else K::template Pass<kChanImageTrack>(c, capture, tail, weight, iq, n_blocks, st);
  }
  return cudaGetLastError();
}

/* T = float2 (t41rx_chan_create) or short (t41rx_chan_create_q15) */
template <int M, typename T>
struct ChanComplex {
  using S = ChanShape<M>;
  template <int kStore>
  static cudaError_t PrepareStore() {
    return ChanSmemAttr(t41rx_chan_kernel<M, false, T, kStore>, S::kSmemBytes, t41rx_chan_kernel<M, true, T, kStore>,
                        S::kSmemRotBytes);
  }
  template <int kStore>
  static void Pass(const t41rx_chan *c, const void *capture, const void *tail, const float2 *weight, float2 *iq,
                   int n_blocks, cudaStream_t st) {
    const int tiles = n_blocks * (T41RX_BLOCK_SAMPLES / kChanTile);
    const T *cap = (const T *)capture, *tl = (const T *)tail;
    if (c->any_rotated)
      t41rx_chan_kernel<M, true, T, kStore><<<tiles, S::kThreads, S::kSmemRotBytes, st>>>(
          cap, tl, c->d_taps, c->d_tw, c->d_recv, c->d_chan, c->d_phase, c->d_rot, c->m_done, c->n_entries, iq, n_blocks,
          weight);
    else
      t41rx_chan_kernel<M, false, T, kStore><<<tiles, S::kThreads, S::kSmemBytes, st>>>(
          cap, tl, c->d_taps, c->d_tw, c->d_recv, c->d_chan, nullptr, c->d_rot, c->m_done, c->n_entries, iq, n_blocks,
          weight);
  }
};

template <int M>
struct ChanReal {
  using S = ChanRealShape<M>;
  template <int kStore>
  static cudaError_t PrepareStore() {
    return ChanSmemAttr(t41rx_chan_real_kernel<M, false, kStore>, S::kSmemBytes, t41rx_chan_real_kernel<M, true, kStore>,
                        S::kSmemRotBytes);
  }
  template <int kStore>
  static void Pass(const t41rx_chan *c, const void *capture, const void *tail, const float2 *weight, float2 *iq,
                   int n_blocks, cudaStream_t st) {
    const int tiles = n_blocks * (T41RX_BLOCK_SAMPLES / kChanTile);
    const short *cap = (const short *)capture, *tl = (const short *)tail;
    if (c->any_rotated)
      t41rx_chan_real_kernel<M, true, kStore><<<tiles, S::kThreads, S::kSmemRotBytes, st>>>(
          cap, tl, c->d_taps, c->d_tw, c->d_split, c->d_recv, c->d_chan, c->d_phase, c->d_rot, c->m_done, c->n_entries,
          iq, n_blocks, weight);
    else
      t41rx_chan_real_kernel<M, false, kStore><<<tiles, S::kThreads, S::kSmemBytes, st>>>(
          cap, tl, c->d_taps, c->d_tw, c->d_split, c->d_recv, c->d_chan, nullptr, c->d_rot, c->m_done, c->n_entries, iq,
          n_blocks, weight);
  }
};

template <typename K, int kSet>
constexpr ChanKernels kChanKernels{ChanPrepare<K, kSet>, ChanLaunch<K, kSet>};

/* the kernels of a kind at a channel count its Chan*CountOk accepts */
template <int M, int kSet>
static ChanKernels ChanComplexKernels(ChanKind kind) {
  return kind == ChanKind::kQ15 ? kChanKernels<ChanComplex<M, short>, kSet> : kChanKernels<ChanComplex<M, float2>, kSet>;
}
template <int kSet>
static ChanKernels ChanKernelsOf(ChanKind kind, int n_channels) {
  if (kind == ChanKind::kReal)
    switch (n_channels) {
      case 128: return kChanKernels<ChanReal<128>, kSet>;
      case 800: return kChanKernels<ChanReal<800>, kSet>;
      case 1024: return kChanKernels<ChanReal<1024>, kSet>;
      default: return kChanKernels<ChanReal<1280>, kSet>;
    }
  switch (n_channels) {
    case 64: return ChanComplexKernels<64, kSet>(kind);
    case 320: return ChanComplexKernels<320, kSet>(kind);
    case 512: return ChanComplexKernels<512, kSet>(kind);
    default: return ChanComplexKernels<640, kSet>(kind);
  }
}
static ChanKernels ChanKernelsFor(ChanKind kind, int n_channels, int n_inputs) {
  if (n_inputs == 1) return ChanKernelsOf<kChanSetPlain>(kind, n_channels);
  return ChanKernelsOf<kChanSetDiversity>(kind, n_channels);
}
/* a complex single-input channelizer's image-correcting kernels (DESIGN §3.12) */
static ChanKernels ChanImageKernelsFor(ChanKind kind, int n_channels) {
  switch (n_channels) {
    case 64: return ChanComplexKernels<64, kChanSetImage>(kind);
    case 320: return ChanComplexKernels<320, kChanSetImage>(kind);
    case 512: return ChanComplexKernels<512, kChanSetImage>(kind);
    default: return ChanComplexKernels<640, kChanSetImage>(kind);
  }
}

static int ChanQuiesce(t41rx_chan *c) {
  if (c->ext_pending) {
    if (cudaEventSynchronize(c->ev_ext) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan: synchronisation failed");
    c->ext_pending = false;
  }
  if (cudaStreamSynchronize(c->stream) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan: synchronisation failed");
  return T41RX_OK;
}

extern "C" {

void t41rx_chan_destroy(t41rx_chan *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->ext_pending && c->ev_ext) cudaEventSynchronize(c->ev_ext);
  if (c->stream) cudaStreamSynchronize(c->stream);
  void *bufs[] = {c->d_taps, c->d_tw, c->d_split, c->d_tail, c->d_recv, c->d_chan, c->d_phase, c->d_weight, c->d_rot,
                  c->d_image, c->d_image_stats};
  for (void *b : bufs)
    if (b) cudaFree(b);
  if (c->ev_ext) cudaEventDestroy(c->ev_ext);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

}  // extern "C"

/* t41rx_chan_create / _create_real / _create_q15 (n_inputs 1) and _create_diversity; fn names the entry point in
   error messages */
static int ChanCreate(const char *fn, ChanKind kind, t41rx_chan **out, int n_channels, int n_inputs, int n_receivers,
                      int device) {
  const std::string f(fn);
  const bool real = kind == ChanKind::kReal;
  if (!out || !(real ? ChanRealCountOk(n_channels) : ChanCountOk(n_channels)) || n_receivers <= 0)
    return SetApiError(T41RX_EINVAL, (f + (real ? ": bad arguments (n_channels must be 128, 800, 1024 or 1280)"
                                               : ": bad arguments (n_channels must be 64, 320, 512 or 640)")).c_str());
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0)
    return SetApiError(T41RX_ENODEV, (f + ": no CUDA device (this library has no CPU path)").c_str());
  if (device < 0 || device >= n_dev) return SetApiError(T41RX_EINVAL, (f + ": device index out of range").c_str());
  if (cudaSetDevice(device) != cudaSuccess) return SetApiError(T41RX_ECUDA, (f + ": cudaSetDevice failed").c_str());
  t41rx_chan *c = new (std::nothrow) t41rx_chan();
  if (!c) return SetApiError(T41RX_ENOMEM, (f + ": out of memory").c_str());
  c->device = device;
  c->n_channels = n_channels;
  c->n_receivers = n_receivers;
  c->kind = kind;
  c->n_inputs = n_inputs;
  c->map.assign(n_receivers, -1);
  c->shift.assign(n_receivers, 0);
  c->p0.assign(n_receivers, 0);
  if (n_inputs > 1) {
    c->weight.assign((size_t)n_receivers * n_inputs, float2{0.f, 0.f});
    for (int r = 0; r < n_receivers; ++r) c->weight[(size_t)r * n_inputs] = float2{1.f, 0.f};
  }
  auto bail = [&](int code) {
    t41rx_chan_destroy(c);
    return code;
  };
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_ext, cudaEventDisableTiming) != cudaSuccess)
    return bail(SetApiError(T41RX_ECUDA, (f + ": stream/event creation failed").c_str()));
  const bool image = !real && n_inputs == 1;
  c->kernels = ChanKernelsFor(kind, n_channels, n_inputs);
  if (image) c->image_kernels = ChanImageKernelsFor(kind, n_channels);
  if (c->kernels.prepare() != cudaSuccess || (image && c->image_kernels.prepare() != cudaSuccess))
    return bail(SetApiError(T41RX_ECUDA, (f + ": kernel image for this GPU missing (built for sm_100a)").c_str()));
  const int N = kChanTaps * n_channels;
  std::vector<float> taps(N);
  DesignChanTaps(n_channels, taps.data());
  if (real)
    for (float &h : taps) h = ldexpf(h, -16);   /* x = s / 32768 and the split's 1 / 2, exact */
  if (kind == ChanKind::kQ15)
    for (float &h : taps) h = ldexpf(h, -15);   /* x = s / 32768, exact */
  /* the row FFTs' twiddles: 2 pi k / 512 for the radix-8 lengths 64 and 512, 2 pi k / L for a mixed-radix length L */
  const int fft_len = real ? n_channels / 2 : n_channels;
  const int tw_len = (fft_len & (fft_len - 1)) == 0 ? 512 : fft_len;
  std::vector<float2> tw(tw_len);
  for (int k = 0; k < tw_len; ++k)
    tw[k] = float2{(float)cos(2.0 * M_PI * k / tw_len), (float)sin(2.0 * M_PI * k / tw_len)};
  std::vector<float2> split(real ? n_channels / 2 + 1 : 0);
  for (size_t k = 0; k < split.size(); ++k)
    split[k] = float2{(float)cos(2.0 * M_PI * k / n_channels), (float)sin(2.0 * M_PI * k / n_channels)};
  std::vector<float2> rot(kRotCoarse + kRotFine);
  for (int a = 0; a < kRotCoarse; ++a) rot[a] = float2{(float)cos(2.0 * M_PI * a / kRotCoarse), (float)sin(2.0 * M_PI * a / kRotCoarse)};
  for (int b = 0; b < kRotFine; ++b)
    rot[kRotCoarse + b] = float2{(float)cos(2.0 * M_PI * b / kChanOutRate), (float)sin(2.0 * M_PI * b / kChanOutRate)};
  const size_t tail_bytes = ChanSampleBytes(kind) * N * n_inputs;
  if (cudaMalloc(&c->d_taps, sizeof(float) * N) != cudaSuccess || cudaMalloc(&c->d_tw, sizeof(float2) * tw_len) != cudaSuccess ||
      (real && cudaMalloc(&c->d_split, sizeof(float2) * split.size()) != cudaSuccess) ||
      cudaMalloc(&c->d_tail, tail_bytes) != cudaSuccess ||
      cudaMalloc(&c->d_recv, sizeof(int32_t) * n_receivers) != cudaSuccess ||
      cudaMalloc(&c->d_chan, sizeof(int32_t) * n_receivers) != cudaSuccess ||
      cudaMalloc(&c->d_phase, sizeof(int2) * n_receivers) != cudaSuccess ||
      (n_inputs > 1 && cudaMalloc(&c->d_weight, sizeof(float2) * n_receivers * n_inputs) != cudaSuccess) ||
      cudaMalloc(&c->d_rot, sizeof(float2) * rot.size()) != cudaSuccess ||
      (image && (cudaMalloc(&c->d_image, sizeof(float2) * n_channels) != cudaSuccess ||
                 cudaMalloc(&c->d_image_stats, sizeof(double) * 4 * (n_channels / 2 + 1)) != cudaSuccess)))
    return bail(SetApiError(T41RX_ENOMEM, (f + ": device allocation failed").c_str()));
  if (cudaMemcpy(c->d_taps, taps.data(), sizeof(float) * N, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(c->d_tw, tw.data(), sizeof(float2) * tw_len, cudaMemcpyHostToDevice) != cudaSuccess ||
      (real && cudaMemcpy(c->d_split, split.data(), sizeof(float2) * split.size(), cudaMemcpyHostToDevice) != cudaSuccess) ||
      cudaMemcpy(c->d_rot, rot.data(), sizeof(float2) * rot.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemset(c->d_tail, 0, tail_bytes) != cudaSuccess ||
      (image && cudaMemset(c->d_image, 0, sizeof(float2) * n_channels) != cudaSuccess))
    return bail(SetApiError(T41RX_ECUDA, (f + ": table upload failed").c_str()));
  *out = c;
  return T41RX_OK;
}

extern "C" {

int t41rx_chan_create(t41rx_chan **out, int n_channels, int n_receivers, int device) {
  return ChanCreate("t41rx_chan_create", ChanKind::kFloat, out, n_channels, 1, n_receivers, device);
}

int t41rx_chan_create_real(t41rx_chan **out, int n_channels, int n_receivers, int device) {
  return ChanCreate("t41rx_chan_create_real", ChanKind::kReal, out, n_channels, 1, n_receivers, device);
}

int t41rx_chan_create_q15(t41rx_chan **out, int n_channels, int n_receivers, int device) {
  return ChanCreate("t41rx_chan_create_q15", ChanKind::kQ15, out, n_channels, 1, n_receivers, device);
}

int t41rx_chan_create_diversity(t41rx_chan **out, int kind, int n_channels, int n_inputs, int n_receivers, int device) {
  const char *fn = "t41rx_chan_create_diversity";
  if (kind != T41RX_CHAN_FLOAT && kind != T41RX_CHAN_Q15 && kind != T41RX_CHAN_REAL)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_create_diversity: bad arguments (kind must be T41RX_CHAN_FLOAT, "
                                     "T41RX_CHAN_Q15 or T41RX_CHAN_REAL)");
  if (n_inputs < 2 || n_inputs > 4)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_create_diversity: bad arguments (n_inputs must be 2, 3 or 4)");
  const ChanKind k = kind == T41RX_CHAN_FLOAT ? ChanKind::kFloat : kind == T41RX_CHAN_Q15 ? ChanKind::kQ15 : ChanKind::kReal;
  return ChanCreate(fn, k, out, n_channels, n_inputs, n_receivers, device);
}

}  // extern "C"

/* the map, shifts, phase offsets and weights as the kernel reads them (after ChanQuiesce): CSR order, receivers grouped
   by channel, ascending within a channel, each entry with its channel and (shift, P); a diversity channelizer's
   weights input by input, input a's n_entries from d_weight + a * n_entries */
static int ChanUpload(t41rx_chan *c, const char *what) {
  std::vector<int32_t> start(c->n_channels + 1, 0);
  for (int32_t k : c->map)
    if (k >= 0) ++start[k + 1];
  for (int k = 0; k < c->n_channels; ++k) start[k + 1] += start[k];
  const int n = start[c->n_channels];
  std::vector<int32_t> recv(std::max(n, 1)), chan(std::max(n, 1)), fill(start.begin(), start.end() - 1);
  std::vector<int2> phase(std::max(n, 1));
  std::vector<float2> weight((size_t)std::max(n, 1) * (c->n_inputs > 1 ? c->n_inputs : 0));
  bool any = false;
  for (int r = 0; r < c->n_receivers; ++r)
    if (c->map[r] >= 0) {
      const int e = fill[c->map[r]]++;
      recv[e] = r;
      chan[e] = c->map[r];
      phase[e] = int2{c->shift[r], c->p0[r]};
      if (c->n_inputs > 1)
        for (int a = 0; a < c->n_inputs; ++a) weight[(size_t)a * n + e] = c->weight[(size_t)r * c->n_inputs + a];
      any = any || c->shift[r] != 0 || c->p0[r] != 0;
    }
  if (n > 0 && (cudaMemcpy(c->d_recv, recv.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMemcpy(c->d_chan, chan.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMemcpy(c->d_phase, phase.data(), sizeof(int2) * n, cudaMemcpyHostToDevice) != cudaSuccess ||
                (c->n_inputs > 1 && cudaMemcpy(c->d_weight, weight.data(), sizeof(float2) * n * c->n_inputs,
                                               cudaMemcpyHostToDevice) != cudaSuccess))) {
    c->n_entries = 0;    /* a partial upload must not be used */
    return SetApiError(T41RX_ECUDA, what);
  }
  c->n_entries = n;
  c->any_rotated = any;
  return T41RX_OK;
}

extern "C" {

int t41rx_chan_set_map(t41rx_chan *c, int first, int count, const int32_t *channel) {
  if (!c || !channel || first < 0 || count <= 0 || first + count > c->n_receivers)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_set_map: bad range");
  const int last = c->kind == ChanKind::kReal ? c->n_channels / 2 : c->n_channels - 1;
  for (int i = 0; i < count; ++i)
    if (channel[i] < -1 || channel[i] > last)
      return SetApiError(T41RX_EINVAL, "t41rx_chan_set_map: channel out of range");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_set_map: cudaSetDevice failed");
  int rc = ChanQuiesce(c);
  if (rc) return rc;
  std::copy(channel, channel + count, c->map.begin() + first);
  return ChanUpload(c, "t41rx_chan_set_map: upload failed");
}

int t41rx_chan_set_shift(t41rx_chan *c, int first, int count, const int32_t *shift_hz) {
  if (!c || !shift_hz || first < 0 || count <= 0 || first + count > c->n_receivers)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_set_shift: bad range");
  for (int i = 0; i < count; ++i)
    if (shift_hz[i] <= -kChanOutRate || shift_hz[i] >= kChanOutRate)
      return SetApiError(T41RX_EINVAL, "t41rx_chan_set_shift: |shift| must be below 192000 Hz");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_set_shift: cudaSetDevice failed");
  int rc = ChanQuiesce(c);
  if (rc) return rc;
  /* continuous phase: the next output, m_abs = m_done, keeps the phase the old shift gives it */
  for (int i = 0; i < count; ++i) {
    const int r = first + i;
    const int32_t s_new = (shift_hz[i] + kChanOutRate) % kChanOutRate;
    const long long p = c->p0[r] + (long long)(c->shift[r] - s_new) * c->m_done;
    c->p0[r] = (int32_t)(((p % kChanOutRate) + kChanOutRate) % kChanOutRate);
    c->shift[r] = s_new;
  }
  return ChanUpload(c, "t41rx_chan_set_shift: upload failed");
}

int t41rx_chan_set_weights(t41rx_chan *c, int first, int count, const float *w) {
  if (!c || !w || first < 0 || count <= 0 || first + count > c->n_receivers)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_set_weights: bad range");
  if (c->n_inputs < 2)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_set_weights: a single-input channelizer has no weights (create it with "
                                     "t41rx_chan_create_diversity)");
  const size_t n = (size_t)count * c->n_inputs;
  for (size_t i = 0; i < 2 * n; ++i)
    if (!std::isfinite(w[i])) return SetApiError(T41RX_EINVAL, "t41rx_chan_set_weights: weights must be finite");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_set_weights: cudaSetDevice failed");
  int rc = ChanQuiesce(c);
  if (rc) return rc;
  for (size_t i = 0; i < n; ++i) c->weight[(size_t)first * c->n_inputs + i] = float2{w[2 * i], w[2 * i + 1]};
  return ChanUpload(c, "t41rx_chan_set_weights: upload failed");
}

}  // extern "C"

/* the image entry points (DESIGN §3.12) take a complex single-input channelizer; EINVAL on the others, saying why */
static int ChanImageKind(const std::string &fn, const t41rx_chan *c) {
  if (!c) return SetApiError(T41RX_EINVAL, (fn + ": null channelizer").c_str());
  if (c->kind == ChanKind::kReal)
    return SetApiError(T41RX_EINVAL, (fn + ": a real channelizer has no image correction (a real capture has no I/Q "
                                           "imbalance, and channel M - k is not a channel it delivers)").c_str());
  if (c->n_inputs > 1)
    return SetApiError(T41RX_EINVAL, (fn + ": a diversity channelizer has no image correction (it acts on one "
                                           "capture's mirror channels; use a single-input channelizer per capture)").c_str());
  return T41RX_OK;
}

/* the image table's M coefficients as the next call will read them (after ChanQuiesce) */
static int ChanImageDownload(t41rx_chan *c, float2 *coef, const std::string &fn) {
  if (cudaMemcpy(coef, c->d_image, sizeof(float2) * c->n_channels, cudaMemcpyDeviceToHost) != cudaSuccess)
    return SetApiError(T41RX_ECUDA, (fn + ": download failed").c_str());
  return T41RX_OK;
}

static bool ChanImageAny(const std::vector<float2> &tab) {
  return std::any_of(tab.begin(), tab.end(), [](float2 v) { return v.x != 0.f || v.y != 0.f; });
}

/* room for the tracking partials of `tiles` tiles: a larger image table, the coefficients copied over.  It waits for
   the channelizer's calls (and the call's stream st) before it frees the old table */
static int ChanImageReserve(t41rx_chan *c, long long tiles, cudaStream_t st, const std::string &fn) {
  if (cudaStreamSynchronize(st) != cudaSuccess) return SetApiError(T41RX_ECUDA, (fn + ": synchronisation failed").c_str());
  const int rc = ChanQuiesce(c);
  if (rc) return rc;
  const size_t pairs = c->n_channels / 2 + 1;
  float2 *buf = nullptr;
  if (cudaMalloc(&buf, sizeof(float2) * c->n_channels + sizeof(float4) * pairs * tiles) != cudaSuccess)
    return SetApiError(T41RX_ENOMEM, (fn + ": device allocation failed (image tracking partials)").c_str());
  if (cudaMemcpy(buf, c->d_image, sizeof(float2) * c->n_channels, cudaMemcpyDeviceToDevice) != cudaSuccess) {
    cudaFree(buf);
    return SetApiError(T41RX_ECUDA, (fn + ": image table copy failed").c_str());
  }
  cudaFree(c->d_image);
  c->d_image = buf;
  c->image_tiles = tiles;
  return T41RX_OK;
}

extern "C" {

int t41rx_chan_set_image(t41rx_chan *c, int first, int count, const float *coef) {
  const std::string fn = "t41rx_chan_set_image";
  if (const int rc = ChanImageKind(fn, c)) return rc;
  if (!coef || first < 0 || count <= 0 || count > c->n_channels - first)
    return SetApiError(T41RX_EINVAL, "t41rx_chan_set_image: bad range");
  for (int i = 0; i < 2 * count; ++i)
    if (!std::isfinite(coef[i])) return SetApiError(T41RX_EINVAL, "t41rx_chan_set_image: coefficients must be finite");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_set_image: cudaSetDevice failed");
  int rc = ChanQuiesce(c);
  if (rc) return rc;
  std::vector<float2> tab(c->n_channels);
  if ((rc = ChanImageDownload(c, tab.data(), fn))) return rc;    /* tracking may have moved the others */
  for (int i = 0; i < count; ++i) tab[first + i] = float2{coef[2 * i], coef[2 * i + 1]};
  if (cudaMemcpy(c->d_image, tab.data(), sizeof(float2) * c->n_channels, cudaMemcpyHostToDevice) != cudaSuccess)
    return SetApiError(T41RX_ECUDA, "t41rx_chan_set_image: upload failed");
  c->any_image = ChanImageAny(tab);
  return T41RX_OK;
}

int t41rx_chan_get_image(t41rx_chan *c, float *coef) {
  const std::string fn = "t41rx_chan_get_image";
  if (const int rc = ChanImageKind(fn, c)) return rc;
  if (!coef) return SetApiError(T41RX_EINVAL, "t41rx_chan_get_image: null coef");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_get_image: cudaSetDevice failed");
  const int rc = ChanQuiesce(c);
  return rc ? rc : ChanImageDownload(c, reinterpret_cast<float2 *>(coef), fn);
}

int t41rx_chan_track_image(t41rx_chan *c, int on, float dominance_db) {
  const std::string fn = "t41rx_chan_track_image";
  if (const int rc = ChanImageKind(fn, c)) return rc;
  if (on && !(dominance_db >= T41RX_CHAN_DOMINANCE_MIN_DB && dominance_db <= T41RX_CHAN_DOMINANCE_MAX_DB))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_track_image: dominance_db must be in [3, 60]");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_track_image: cudaSetDevice failed");
  int rc = ChanQuiesce(c);
  if (rc) return rc;
  if (on) {
    c->track = true;
    c->dominance = pow(10.0, (double)dominance_db / 10.0);
    return T41RX_OK;
  }
  c->track = false;
  std::vector<float2> tab(c->n_channels);
  if ((rc = ChanImageDownload(c, tab.data(), fn))) return rc;
  c->any_image = ChanImageAny(tab);
  return T41RX_OK;
}

int t41rx_chan_image_stats(t41rx_chan *c, double *stats) {
  const std::string fn = "t41rx_chan_image_stats";
  if (const int rc = ChanImageKind(fn, c)) return rc;
  if (!stats) return SetApiError(T41RX_EINVAL, "t41rx_chan_image_stats: null stats");
  if (!c->has_stats) return SetApiError(T41RX_EINVAL, "t41rx_chan_image_stats: no call has run with tracking on");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_image_stats: cudaSetDevice failed");
  const int rc = ChanQuiesce(c);
  if (rc) return rc;
  if (cudaMemcpy(stats, c->d_image_stats, sizeof(double) * 4 * (c->n_channels / 2 + 1), cudaMemcpyDeviceToHost) != cudaSuccess)
    return SetApiError(T41RX_ECUDA, "t41rx_chan_image_stats: download failed");
  return T41RX_OK;
}

}  // extern "C"

/* one call of any kind (the caller has checked the pointers and the kind): captures[a], a < n_inputs, holds
   n_blocks x 2048 x D samples of ChanSampleBytes(c->kind) each.  A diversity call runs one pass per input on the same
   stream, input 0 storing and the others accumulating, always in this order, so cutting a run into calls gives the
   same bits */
static int ChanProcess(const char *fn, t41rx_chan *c, const void *const *captures, float *iq, int n_blocks,
                       void *cuda_stream) {
  const std::string f(fn);
  if (n_blocks > INT_MAX / (T41RX_BLOCK_SAMPLES / kChanTile))
    return SetApiError(T41RX_EINVAL, (f + ": n_blocks too large for one call").c_str());
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, (f + ": cudaSetDevice failed").c_str());
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
  const size_t N = (size_t)kChanTaps * c->n_channels;
  const size_t total = (size_t)n_blocks * T41RX_BLOCK_SAMPLES * (c->n_channels / 2);
  const size_t sample_bytes = ChanSampleBytes(c->kind);
  char *tails = (char *)c->d_tail;
  cudaError_t e = cudaSuccess;
  if (c->track || c->any_image) {
    /* image correction (DESIGN §3.12): one pass of an image instance; with tracking, it runs whether or not a receiver
       is mapped (every pair is measured), and the update follows it on the same stream */
    const long long tiles = (long long)n_blocks * (T41RX_BLOCK_SAMPLES / kChanTile);
    if (c->track && tiles > c->image_tiles) {
      const int rc = ChanImageReserve(c, tiles, st, f);
      if (rc) return rc;
    }
    if (c->n_entries > 0 || c->track)
      e = c->image_kernels.launch(c, captures[0], tails, c->track ? kChanImageTrack : kChanImage, c->d_image,
                                  (float2 *)iq, n_blocks, st);
    if (c->track && e == cudaSuccess) {
      t41rx_chan_image_update<<<c->n_channels / 2 + 1, kChanImageThreads, 0, st>>>(c->d_image, c->n_channels, (int)tiles,
                                                                                     c->dominance, c->d_image_stats);
      e = cudaGetLastError();
      c->has_stats = c->has_stats || e == cudaSuccess;
    }
  } else {
    for (int a = 0; a < c->n_inputs && c->n_entries > 0 && e == cudaSuccess; ++a) {
      const int store = c->n_inputs == 1 ? kChanPlain : a == 0 ? kChanWeighted : kChanAccumulate;
      e = c->kernels.launch(c, captures[a], tails + a * N * sample_bytes, store,
                            c->d_weight ? c->d_weight + (size_t)a * c->n_entries : nullptr, (float2 *)iq, n_blocks, st);
    }
  }
  /* the new tails: each input's last N samples, copied after the last pass on the same stream so no tile reads them
     early */
  for (int a = 0; a < c->n_inputs && e == cudaSuccess; ++a)
    e = cudaMemcpyAsync(tails + a * N * sample_bytes, (const char *)captures[a] + (total - N) * sample_bytes,
                        sample_bytes * N, cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess)
    c->m_done = (int)((c->m_done + (long long)n_blocks * T41RX_BLOCK_SAMPLES) % kChanOutRate);
  if (st != c->stream) {
    cudaEventRecord(c->ev_ext, st);
    c->ext_pending = true;
  }
  if (e != cudaSuccess) return SetApiError(T41RX_ECUDA, (f + ": launch failed").c_str());
  return T41RX_OK;
}

extern "C" {

int t41rx_chan_process_device(t41rx_chan *c, const float *capture, float *iq, int n_blocks, void *cuda_stream) {
  if (!c || !capture || !iq || n_blocks <= 0 || ((uintptr_t)capture & 7) || ((uintptr_t)iq & 7))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_process_device: bad arguments (null or not 8-byte aligned pointer, n_blocks <= 0)");
  if (c->kind != ChanKind::kFloat || c->n_inputs > 1) return ChanWrongKind("t41rx_chan_process_device", c);
  const void *captures[] = {capture};
  return ChanProcess("t41rx_chan_process_device", c, captures, iq, n_blocks, cuda_stream);
}

int t41rx_chan_process_device_real(t41rx_chan *c, const int16_t *capture, float *iq, int n_blocks, void *cuda_stream) {
  if (!c || !capture || !iq || n_blocks <= 0 || ((uintptr_t)capture & 15) || ((uintptr_t)iq & 7))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_process_device_real: bad arguments (null pointer, capture not 16-byte or "
                                     "iq not 8-byte aligned, n_blocks <= 0)");
  if (c->kind != ChanKind::kReal || c->n_inputs > 1) return ChanWrongKind("t41rx_chan_process_device_real", c);
  const void *captures[] = {capture};
  return ChanProcess("t41rx_chan_process_device_real", c, captures, iq, n_blocks, cuda_stream);
}

int t41rx_chan_process_device_q15(t41rx_chan *c, const int16_t *capture, float *iq, int n_blocks, void *cuda_stream) {
  if (!c || !capture || !iq || n_blocks <= 0 || ((uintptr_t)capture & 15) || ((uintptr_t)iq & 7))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_process_device_q15: bad arguments (null pointer, capture not 16-byte or "
                                     "iq not 8-byte aligned, n_blocks <= 0)");
  if (c->kind != ChanKind::kQ15 || c->n_inputs > 1) return ChanWrongKind("t41rx_chan_process_device_q15", c);
  const void *captures[] = {capture};
  return ChanProcess("t41rx_chan_process_device_q15", c, captures, iq, n_blocks, cuda_stream);
}

int t41rx_chan_process_device_diversity(t41rx_chan *c, const void *const *captures, float *iq, int n_blocks,
                                        void *cuda_stream) {
  if (!c || !captures || !iq || n_blocks <= 0 || ((uintptr_t)iq & 7))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_process_device_diversity: bad arguments (null pointer, iq not 8-byte "
                                     "aligned, n_blocks <= 0)");
  if (c->n_inputs < 2) return ChanWrongKind("t41rx_chan_process_device_diversity", c);
  const uintptr_t align = c->kind == ChanKind::kFloat ? 7 : 15;
  for (int a = 0; a < c->n_inputs; ++a)
    if (!captures[a] || ((uintptr_t)captures[a] & align))
      return SetApiError(T41RX_EINVAL, (std::string("t41rx_chan_process_device_diversity: capture ") + std::to_string(a) +
                                        (align == 7 ? " null or not 8-byte aligned" : " null or not 16-byte aligned")).c_str());
  return ChanProcess("t41rx_chan_process_device_diversity", c, captures, iq, n_blocks, cuda_stream);
}

int t41rx_chan_synchronize(t41rx_chan *c) {
  if (!c) return SetApiError(T41RX_EINVAL, "t41rx_chan_synchronize: null channelizer");
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, "t41rx_chan_synchronize: cudaSetDevice failed");
  return ChanQuiesce(c);
}

int t41rx_chan_taps(int n_channels, float *taps) {
  if (!taps || !(ChanCountOk(n_channels) || ChanRealCountOk(n_channels)))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_taps: bad arguments (n_channels must be 64, 128, 320, 512, 640, 800, 1024 or 1280)");
  DesignChanTaps(n_channels, taps);
  return T41RX_OK;
}

int t41rx_chan_tune(int n_channels, int32_t mode, double offset_hz, int32_t *channel, int32_t *nco_freq) {
  return ChanTune("t41rx_chan_tune", false, n_channels, mode, offset_hz, channel, nco_freq);
}

int t41rx_chan_place(int n_channels, int32_t mode, double offset_hz, int32_t *channel, int32_t *shift_hz,
                     int32_t *nco_freq) {
  return ChanPlace("t41rx_chan_place", false, n_channels, mode, offset_hz, channel, shift_hz, nco_freq);
}

int t41rx_chan_tune_real(int n_channels, int32_t mode, double freq_hz, int32_t *channel, int32_t *nco_freq) {
  return ChanTune("t41rx_chan_tune_real", true, n_channels, mode, freq_hz, channel, nco_freq);
}

int t41rx_chan_place_real(int n_channels, int32_t mode, double freq_hz, int32_t *channel, int32_t *shift_hz,
                          int32_t *nco_freq) {
  return ChanPlace("t41rx_chan_place_real", true, n_channels, mode, freq_hz, channel, shift_hz, nco_freq);
}

}  // extern "C"
