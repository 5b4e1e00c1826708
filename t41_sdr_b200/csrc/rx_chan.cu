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
   The int16 span goes through registers (16-byte loads of four pairs) and lands converted, (I, Q) as integer-valued
   floats, where the float span is staged: each sample is converted once, not at each of the ~9 branch loads that read
   it, and the rest of the kernel is the same for both.  h / 32768 times I is h times I / 32768 exactly, so every FMA,
   and every output bit, is that of the float instance on x = s / 32768. */
template <int M, bool kRotate, typename T>
__global__ void __launch_bounds__(ChanShape<M>::kThreads, ChanShape<M>::kMinBlocks)
t41rx_chan_kernel(const T *__restrict__ capture, const T *__restrict__ tail, const float *__restrict__ taps,
                  const float2 *__restrict__ tw512, const int32_t *__restrict__ recv, const int32_t *__restrict__ chan,
                  const int2 *__restrict__ phase, const float2 *__restrict__ rot, int m_base, int n_entries,
                  float2 *__restrict__ iq, int n_blocks) {
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
  const long long blk = m0 / T41RX_BLOCK_SAMPLES;
  const int s0 = (int)(m0 % T41RX_BLOCK_SAMPLES);
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
template <int M, bool kRotate>
__global__ void __launch_bounds__(ChanRealShape<M>::kThreads, ChanRealShape<M>::kMinBlocks)
t41rx_chan_real_kernel(const short *__restrict__ capture, const short *__restrict__ tail, const float *__restrict__ taps,
                       const float2 *__restrict__ tw512, const float2 *__restrict__ split, const int32_t *__restrict__ recv,
                       const int32_t *__restrict__ chan, const int2 *__restrict__ phase, const float2 *__restrict__ rot,
                       int m_base, int n_entries, float2 *__restrict__ iq, int n_blocks) {
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

/* fn was called on a channelizer of another kind: EINVAL, naming the entry point this one takes */
static int ChanWrongKind(const char *fn, ChanKind kind) {
  const char *takes = kind == ChanKind::kFloat ? ": a complex float channelizer takes t41rx_chan_process_device"
                      : kind == ChanKind::kReal ? ": a real channelizer takes t41rx_chan_process_device_real"
                                                : ": a q15 channelizer takes t41rx_chan_process_device_q15";
  return SetApiError(T41RX_EINVAL, (std::string(fn) + takes).c_str());
}

/* a channelizer's kernel pair (without and with fine tuning), chosen by kind and M at creation: prepare raises the
   pair's dynamic shared memory limits, launch enqueues one call */
struct ChanKernels {
  cudaError_t (*prepare)();
  cudaError_t (*launch)(const t41rx_chan *c, const void *capture, float2 *iq, int n_blocks, cudaStream_t st);
};

}  // namespace t41rx

using namespace t41rx;

struct t41rx_chan {
  int device = 0;
  int n_channels = 0;
  int n_receivers = 0;
  ChanKind kind = ChanKind::kFloat;
  cudaStream_t stream = nullptr;
  /* t41rx_chan_process_device may enqueue on a caller-supplied stream: its end is recorded here, and set_map /
     synchronize / destroy wait for it (the ordering contract of t41rx_process_device) */
  cudaEvent_t ev_ext = nullptr;
  bool ext_pending = false;
  float *d_taps = nullptr;       /* N (real: h / 65536, q15: h / 32768) */
  float2 *d_tw = nullptr;        /* 512 (cos, sin) of 2 pi k / 512, or L of 2 pi k / L (mixed-radix FFT length L) */
  float2 *d_split = nullptr;     /* real: n_channels / 2 + 1 (cos, sin) of 2 pi k / n_channels */
  void *d_tail = nullptr;        /* the last N capture samples of the previous calls (zeros at creation) */
  int32_t *d_recv = nullptr, *d_chan = nullptr;   /* mapped receivers grouped by channel, and their channel */
  int2 *d_phase = nullptr;       /* each entry's (shift, P), in the order of d_recv */
  float2 *d_rot = nullptr;       /* 480 + 400: exp(j 2 pi a / 480), exp(j 2 pi b / 192000) */
  int n_entries = 0;
  bool any_rotated = false;      /* some entry's phase is not identically 0 */
  std::vector<int32_t> map;      /* receiver -> channel or -1 */
  std::vector<int32_t> shift, p0;   /* receiver -> shift and phase offset P, both in [0, 192000) */
  int m_done = 0;                /* outputs produced since creation, mod 192000 */
  ChanKernels kernels{};
};

/* T = float2 (t41rx_chan_create) or short (t41rx_chan_create_q15) */
template <int M, typename T>
struct ChanComplex {
  using S = ChanShape<M>;
  static cudaError_t Prepare() {
    return ChanSmemAttr(t41rx_chan_kernel<M, false, T>, S::kSmemBytes, t41rx_chan_kernel<M, true, T>, S::kSmemRotBytes);
  }
  static cudaError_t Launch(const t41rx_chan *c, const void *capture, float2 *iq, int n_blocks, cudaStream_t st) {
    const int tiles = n_blocks * (T41RX_BLOCK_SAMPLES / kChanTile);
    const T *cap = (const T *)capture, *tail = (const T *)c->d_tail;
    if (c->any_rotated)
      t41rx_chan_kernel<M, true, T><<<tiles, S::kThreads, S::kSmemRotBytes, st>>>(
          cap, tail, c->d_taps, c->d_tw, c->d_recv, c->d_chan, c->d_phase, c->d_rot, c->m_done, c->n_entries, iq, n_blocks);
    else
      t41rx_chan_kernel<M, false, T><<<tiles, S::kThreads, S::kSmemBytes, st>>>(
          cap, tail, c->d_taps, c->d_tw, c->d_recv, c->d_chan, nullptr, c->d_rot, c->m_done, c->n_entries, iq, n_blocks);
    return cudaGetLastError();
  }
};

template <int M>
struct ChanReal {
  using S = ChanRealShape<M>;
  static cudaError_t Prepare() {
    return ChanSmemAttr(t41rx_chan_real_kernel<M, false>, S::kSmemBytes, t41rx_chan_real_kernel<M, true>, S::kSmemRotBytes);
  }
  static cudaError_t Launch(const t41rx_chan *c, const void *capture, float2 *iq, int n_blocks, cudaStream_t st) {
    const int tiles = n_blocks * (T41RX_BLOCK_SAMPLES / kChanTile);
    const short *cap = (const short *)capture, *tail = (const short *)c->d_tail;
    if (c->any_rotated)
      t41rx_chan_real_kernel<M, true><<<tiles, S::kThreads, S::kSmemRotBytes, st>>>(
          cap, tail, c->d_taps, c->d_tw, c->d_split, c->d_recv, c->d_chan, c->d_phase, c->d_rot, c->m_done, c->n_entries,
          iq, n_blocks);
    else
      t41rx_chan_real_kernel<M, false><<<tiles, S::kThreads, S::kSmemBytes, st>>>(
          cap, tail, c->d_taps, c->d_tw, c->d_split, c->d_recv, c->d_chan, nullptr, c->d_rot, c->m_done, c->n_entries, iq,
          n_blocks);
    return cudaGetLastError();
  }
};

template <typename K>
constexpr ChanKernels kChanKernels{K::Prepare, K::Launch};

/* the kernel pair of a kind at a channel count its Chan*CountOk accepts */
template <int M>
static ChanKernels ChanComplexKernels(ChanKind kind) {
  return kind == ChanKind::kQ15 ? kChanKernels<ChanComplex<M, short>> : kChanKernels<ChanComplex<M, float2>>;
}
static ChanKernels ChanKernelsFor(ChanKind kind, int n_channels) {
  if (kind == ChanKind::kReal)
    switch (n_channels) {
      case 128: return kChanKernels<ChanReal<128>>;
      case 800: return kChanKernels<ChanReal<800>>;
      case 1024: return kChanKernels<ChanReal<1024>>;
      default: return kChanKernels<ChanReal<1280>>;
    }
  switch (n_channels) {
    case 64: return ChanComplexKernels<64>(kind);
    case 320: return ChanComplexKernels<320>(kind);
    case 512: return ChanComplexKernels<512>(kind);
    default: return ChanComplexKernels<640>(kind);
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
  void *bufs[] = {c->d_taps, c->d_tw, c->d_split, c->d_tail, c->d_recv, c->d_chan, c->d_phase, c->d_rot};
  for (void *b : bufs)
    if (b) cudaFree(b);
  if (c->ev_ext) cudaEventDestroy(c->ev_ext);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

}  // extern "C"

/* t41rx_chan_create / _create_real / _create_q15; fn names the entry point in error messages */
static int ChanCreate(const char *fn, ChanKind kind, t41rx_chan **out, int n_channels, int n_receivers, int device) {
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
  c->map.assign(n_receivers, -1);
  c->shift.assign(n_receivers, 0);
  c->p0.assign(n_receivers, 0);
  auto bail = [&](int code) {
    t41rx_chan_destroy(c);
    return code;
  };
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_ext, cudaEventDisableTiming) != cudaSuccess)
    return bail(SetApiError(T41RX_ECUDA, (f + ": stream/event creation failed").c_str()));
  c->kernels = ChanKernelsFor(kind, n_channels);
  if (c->kernels.prepare() != cudaSuccess)
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
  const size_t tail_bytes = ChanSampleBytes(kind) * N;
  if (cudaMalloc(&c->d_taps, sizeof(float) * N) != cudaSuccess || cudaMalloc(&c->d_tw, sizeof(float2) * tw_len) != cudaSuccess ||
      (real && cudaMalloc(&c->d_split, sizeof(float2) * split.size()) != cudaSuccess) ||
      cudaMalloc(&c->d_tail, tail_bytes) != cudaSuccess ||
      cudaMalloc(&c->d_recv, sizeof(int32_t) * n_receivers) != cudaSuccess ||
      cudaMalloc(&c->d_chan, sizeof(int32_t) * n_receivers) != cudaSuccess ||
      cudaMalloc(&c->d_phase, sizeof(int2) * n_receivers) != cudaSuccess ||
      cudaMalloc(&c->d_rot, sizeof(float2) * rot.size()) != cudaSuccess)
    return bail(SetApiError(T41RX_ENOMEM, (f + ": device allocation failed").c_str()));
  if (cudaMemcpy(c->d_taps, taps.data(), sizeof(float) * N, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(c->d_tw, tw.data(), sizeof(float2) * tw_len, cudaMemcpyHostToDevice) != cudaSuccess ||
      (real && cudaMemcpy(c->d_split, split.data(), sizeof(float2) * split.size(), cudaMemcpyHostToDevice) != cudaSuccess) ||
      cudaMemcpy(c->d_rot, rot.data(), sizeof(float2) * rot.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemset(c->d_tail, 0, tail_bytes) != cudaSuccess)
    return bail(SetApiError(T41RX_ECUDA, (f + ": table upload failed").c_str()));
  *out = c;
  return T41RX_OK;
}

extern "C" {

int t41rx_chan_create(t41rx_chan **out, int n_channels, int n_receivers, int device) {
  return ChanCreate("t41rx_chan_create", ChanKind::kFloat, out, n_channels, n_receivers, device);
}

int t41rx_chan_create_real(t41rx_chan **out, int n_channels, int n_receivers, int device) {
  return ChanCreate("t41rx_chan_create_real", ChanKind::kReal, out, n_channels, n_receivers, device);
}

int t41rx_chan_create_q15(t41rx_chan **out, int n_channels, int n_receivers, int device) {
  return ChanCreate("t41rx_chan_create_q15", ChanKind::kQ15, out, n_channels, n_receivers, device);
}

}  // extern "C"

/* the map, shifts and phase offsets as the kernel reads them (after ChanQuiesce): CSR order, receivers grouped by
   channel, ascending within a channel, each entry with its channel and (shift, P) */
static int ChanUpload(t41rx_chan *c, const char *what) {
  std::vector<int32_t> start(c->n_channels + 1, 0);
  for (int32_t k : c->map)
    if (k >= 0) ++start[k + 1];
  for (int k = 0; k < c->n_channels; ++k) start[k + 1] += start[k];
  const int n = start[c->n_channels];
  std::vector<int32_t> recv(std::max(n, 1)), chan(std::max(n, 1)), fill(start.begin(), start.end() - 1);
  std::vector<int2> phase(std::max(n, 1));
  bool any = false;
  for (int r = 0; r < c->n_receivers; ++r)
    if (c->map[r] >= 0) {
      const int e = fill[c->map[r]]++;
      recv[e] = r;
      chan[e] = c->map[r];
      phase[e] = int2{c->shift[r], c->p0[r]};
      any = any || c->shift[r] != 0 || c->p0[r] != 0;
    }
  if (n > 0 && (cudaMemcpy(c->d_recv, recv.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMemcpy(c->d_chan, chan.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMemcpy(c->d_phase, phase.data(), sizeof(int2) * n, cudaMemcpyHostToDevice) != cudaSuccess)) {
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

}  // extern "C"

/* one call of any kind (the caller has checked the pointers and the kind): capture holds n_blocks x 2048 x D samples
   of ChanSampleBytes(c->kind) each */
static int ChanProcess(const char *fn, t41rx_chan *c, const void *capture, float *iq, int n_blocks, void *cuda_stream) {
  const std::string f(fn);
  if (n_blocks > INT_MAX / (T41RX_BLOCK_SAMPLES / kChanTile))
    return SetApiError(T41RX_EINVAL, (f + ": n_blocks too large for one call").c_str());
  if (cudaSetDevice(c->device) != cudaSuccess) return SetApiError(T41RX_ECUDA, (f + ": cudaSetDevice failed").c_str());
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
  cudaError_t e = c->n_entries > 0 ? c->kernels.launch(c, capture, (float2 *)iq, n_blocks, st) : cudaSuccess;
  /* the new tail: the call's last N samples, copied after the kernel on the same stream so no tile reads it early */
  const size_t N = (size_t)kChanTaps * c->n_channels;
  const size_t total = (size_t)n_blocks * T41RX_BLOCK_SAMPLES * (c->n_channels / 2);
  const size_t sample_bytes = ChanSampleBytes(c->kind);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(c->d_tail, (const char *)capture + (total - N) * sample_bytes, sample_bytes * N,
                        cudaMemcpyDeviceToDevice, st);
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
  if (c->kind != ChanKind::kFloat) return ChanWrongKind("t41rx_chan_process_device", c->kind);
  return ChanProcess("t41rx_chan_process_device", c, capture, iq, n_blocks, cuda_stream);
}

int t41rx_chan_process_device_real(t41rx_chan *c, const int16_t *capture, float *iq, int n_blocks, void *cuda_stream) {
  if (!c || !capture || !iq || n_blocks <= 0 || ((uintptr_t)capture & 15) || ((uintptr_t)iq & 7))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_process_device_real: bad arguments (null pointer, capture not 16-byte or "
                                     "iq not 8-byte aligned, n_blocks <= 0)");
  if (c->kind != ChanKind::kReal) return ChanWrongKind("t41rx_chan_process_device_real", c->kind);
  return ChanProcess("t41rx_chan_process_device_real", c, capture, iq, n_blocks, cuda_stream);
}

int t41rx_chan_process_device_q15(t41rx_chan *c, const int16_t *capture, float *iq, int n_blocks, void *cuda_stream) {
  if (!c || !capture || !iq || n_blocks <= 0 || ((uintptr_t)capture & 15) || ((uintptr_t)iq & 7))
    return SetApiError(T41RX_EINVAL, "t41rx_chan_process_device_q15: bad arguments (null pointer, capture not 16-byte or "
                                     "iq not 8-byte aligned, n_blocks <= 0)");
  if (c->kind != ChanKind::kQ15) return ChanWrongKind("t41rx_chan_process_device_q15", c->kind);
  return ChanProcess("t41rx_chan_process_device_q15", c, capture, iq, n_blocks, cuda_stream);
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
