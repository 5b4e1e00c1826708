/*
 * rx_fast.cuh — t41rx_stream_rx_kernel: the throughput form of the fused T41 receive chain.
 *
 * Same chain as rx_phases.cuh (ProcessIQData(), reference Process.cpp:70-944), same HBM state
 * (StreamState) and tables, different mapping (DESIGN.md 3.2):
 *   - one CTA owns G <= kFastMaxG receivers for all n_blocks blocks of a launch;
 *   - TWO WARPS PER RECEIVER run every sample-parallel stage (64-thread named barriers between stages);
 *   - one extra warp runs the AGC envelope state machine with lane = receiver;
 *   - blocks are software-pipelined through mbarriers (no block-wide barrier in the steady state): in superstep k a receiver's
 *     warp pair does back end(k-2) then front end(k), the AGC warp does AGC(k-1).
 * Linear recurrences (DC block, AM detector filters) are blocked scans, the NCO is a closed-form
 * FP32 phasor driven by an FP64 block phasor, the fast-convolution filter fuses the last forward
 * FFT pass, the mask multiply and the first inverse pass in registers.  FP32 with FMA contraction:
 * results agree with the oracle to the stated tolerance (audio SNR >= 90 dB; in practice > 110 dB),
 * not bit for bit; the bit-exact kernel is t41rx_fused_rx_kernel.
 *
 * Row-producing blocks (display spectrum) and amplitude-transient blocks of the oscillator take
 * slower side paths inside the same kernel.
 */
#ifndef T41RX_FAST_CUH
#define T41RX_FAST_CUH

#include "rx_phases.cuh"

namespace t41rx {
namespace fast {

constexpr int kFastMaxG = 7;          /* receivers per CTA (shared memory: 7 x 31.7 KB) */
constexpr unsigned kFull = 0xffffffffu;

/* ---- per-receiver shared-memory slot, in 4-byte words ---- */
constexpr int kRawChunkWords = 20;                    /* 8 samples (16 words) + 4 pad: conflict-free LDS.128 */
constexpr int kRawBufWords = 64 * kRawChunkWords;     /* one 512-sample quarter: 1280 */
constexpr int oRaw = 0;                               /* 2 quarter buffers */
constexpr int oMix = oRaw + 2 * kRawBufWords;         /* 2304: mixed samples, 8 planes (ch, phase) x 136; FFT buffer overlay */
constexpr int kMixPlane = 136;                        /* 8 history + 128 */
constexpr int kMixWords = 1152;                       /* >= 8 * 136 = 1088 and >= 2 * 576 (padded FFT buffer) */
constexpr int oD1 = oMix + kMixWords;                 /* 3456: dec1 output, 4 planes (ch, parity) x 280; overlays below */
constexpr int kD1Plane = 280;                         /* 24 history + 256 */
constexpr int kD1Words = 1152;
constexpr int oOlaF = oD1 + kD1Words;                 /* 4608: previous 256 complex filter inputs (interleaved) */
constexpr int oStA = oOlaF + 512;                     /* 5120: 2 x (|z| delayed [256], window max -> volts [256]) */
constexpr int kStABuf = 576;                          /* |z| delayed [256] | window max -> volts [256] | (PF, PH)[32] */
constexpr int oStZ = oStA + 2 * kStABuf;                     /* 6144: 2 x 256 complex: delayed filter output */
constexpr int kStZBuf = 576;                          /* 256 complex, 2 pad words after every 8 (ZPos) */
constexpr int oZH = oStZ + 2 * kStZBuf;                      /* 7168: last 97 complex filter outputs */
constexpr int oTapsF = oZH + 196;                     /* 7464: dec1 28 | dec2 46 | int1 48 | int2 32 (+2) */
constexpr int oNcoW = oTapsF + 156;                   /* 7620: W[8] float2, Q[4] float2 */
constexpr int oXtra = oNcoW + 24;                     /* 7644: 16 words of once-per-block scalars (enum x*) */
constexpr int oIH = oNcoW + 40;                       /* 7660: int1 history 23 (24) | int2 history 7 (8) */
constexpr int oMH = oIH + 32;                         /* 7692: dec1 history, 8 planes x 8 */
constexpr int oDH = oMH + 64;                         /* 7756: dec2 history, 4 planes x 24 */
constexpr int oMiscF = oDH + 96;                      /* 7852 */
constexpr int kSlotF = oMiscF + 36;                   /* == 4 (mod 8): the AGC warp's LDS.128 hit distinct banks */
enum { mEndI = 0, mEndQ = 1, mSettled = 2, mMidI = 3, mMidQ = 11, mPhasor = 4 /* 2 doubles */, mInvIn = 8, mTarget = 9, mSlope = 10,
       mOmF = 12, mOmH = 13, mFbm = 14, mHbm = 15,
       mAmWold = 16, mAmX1 = 17, mAmX2 = 18, mAmY1 = 19, mAmY2 = 20, mNfmI = 21, mNfmQ = 22, mAmLp = 23 /* 5 */,
       mBlkRot = 28 /* 2 doubles: rotation of the block phasor over 2048 samples */, mVolScale = 32, mVolume = 33,
       mFixedGain = 34, mIqPhase = 35 };
enum { xInGain = 0 /* rfGainValue * b0 * 1.1 (DC-block numerator and freqAdjFactor folded) */, xRfGain = 1 /* int */,
       xCodecTimer = 2 /* unsigned */, xNegIqAmp = 3, xFilterId = 4 /* int */ };
static_assert((oMiscF % 2) == 0 && (oTapsF % 4) == 0, "alignment");
static_assert(kSlotF % 8 == 4, "slot stride");
static_assert((oStA % 4) == 0 && (oStZ % 4) == 0 && (oRaw % 4) == 0 && (oMix % 4) == 0 && (oD1 % 4) == 0, "16-byte alignment");

/* overlays on the dec1 region once dec2 has consumed it (front end) */
constexpr int vE = oD1;                               /* |z| extended: 97 history + 256 new (360) */
constexpr int vSfx = vE + 360;                        /* suffix maxima inside chunks of 8 */
constexpr int vPfx = vSfx + 360;                      /* prefix maxima */
constexpr int vCM = vPfx + 360;                       /* chunk maxima (45 -> 48) */
constexpr int vF = vE;                                /* 11-chunk window maxima (36), over |z| once it is consumed */
static_assert(vCM + 48 <= oD1 + kD1Words, "sliding max scratch");
/* overlays on the dec1 region in the back end */
constexpr int vAudF = oD1;                            /* 24 (1 pad + 23 history) + 256 demodulated samples */
constexpr int vI1 = oD1 + 288;                        /* 8 (1 pad + 7 history) + 512 */
static_assert(vI1 + 520 <= oD1 + kD1Words, "back-end scratch");

/* the 512-point FFT buffer: element i lives at float2 index i ^ ((i >> 3) & 15): an XOR swizzle under which
   every access pattern of the radix-8 passes (stride 64, stride 8, 8 contiguous) and of the code around them
   is bank-conflict-free without padding (searched exhaustively, tools/fft_swizzle_search.py) */
__device__ __forceinline__ int FPos(int i) { return i ^ ((i >> 3) & 15); }
/* dec1 output planes: word w of a plane lives at D1W(w): adjacent float4 are swapped in every other group of 8,
   which makes dec2's window loads (8 consecutive float4 per lane, lanes 2 float4 apart) conflict-free */
__device__ __forceinline__ int D1W(int w) { return (((w >> 2) ^ ((w >> 5) & 1)) << 2) | (w & 3); }
/* staged filter output: complex sample i lives at float2 index i + (i >> 3) (8 contiguous samples per lane
   and stride-1 lanes are both conflict-free) */
__device__ __forceinline__ int ZPos(int i) { return i + (i >> 3); }
/* overlap-save history of channel ch: sample i at word (i & 7) * 32 + (i >> 3): lane L owns samples 8 L .. 8 L + 7 */
__device__ __forceinline__ int OlaW(int ch, int i) { return oOlaF + ch * 256 + (i & 7) * 32 + (i >> 3); }

constexpr float kDcA1 = 0.854352383886757938f;        /* FIR.cpp:87-89 */
constexpr float kDcB0 = 0.927176191943378969f;

__device__ __forceinline__ float PowA1(int n) {       /* a1^n, n >= 0, by squaring (set-up only) */
  float r = 1.0f, b = kDcA1;
  while (n) {
    if (n & 1) r *= b;
    b *= b;
    n >>= 1;
  }
  return r;
}

#ifdef T41RX_FAST_TIMING
/* developer build: cycles per section, CTA 0, receiver warp 0 (slots 0..15) and the AGC warp (16..19) */
__device__ unsigned long long g_fast_cycles[32];
struct SectionTimer {
  long long mark;
  bool on;
  int base;
  __device__ __forceinline__ void Start(bool enable, int b) { on = enable; base = b; mark = clock64(); }
  __device__ __forceinline__ void Lap(int slot) {
    if (on) {
      const long long now = clock64();
      g_fast_cycles[base + slot] += (unsigned long long)(now - mark);
      mark = now;
    }
  }
};
#define T41RX_LAP(tm, slot) (tm).Lap(slot)
#else
struct SectionTimer {
  __device__ __forceinline__ void Start(bool, int) {}
};
#define T41RX_LAP(tm, slot) ((void)0)
#endif

/* sqrt.approx.f32: maximum relative error 2^-23 (the envelope detector's input; SNR budget 90 dB) */
__device__ __forceinline__ float SqrtFast(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

/* arm_float_to_q15 (Process.cpp:936): saturate(trunc(x * 32768)) to 16 bits; cvt.rzi.s16.f32 truncates toward zero,
   saturates, and converts NaN to 0 like the target's VCVT */
__device__ __forceinline__ unsigned PackQ15(float lo, float hi) {
  short a, b;
  asm("cvt.rzi.s16.f32 %0, %1;" : "=h"(a) : "f"(lo * 32768.0f));
  asm("cvt.rzi.s16.f32 %0, %1;" : "=h"(b) : "f"(hi * 32768.0f));
  return (unsigned)(unsigned short)a | ((unsigned)(unsigned short)b << 16);
}

struct F2 { float x, y; };

/* packed FP32 pairs (sm_100 FFMA2: two FMAs per issue slot) */
typedef unsigned long long P2;
__device__ __forceinline__ P2 Pack2(float lo, float hi) {
  P2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void Unpack2(P2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ float Lo(P2 v) { float a, b; Unpack2(v, a, b); return a; }
__device__ __forceinline__ float Hi(P2 v) { float a, b; Unpack2(v, a, b); return b; }
__device__ __forceinline__ P2 Dup(float x) { return Pack2(x, x); }     /* ptxas folds it into FFMA2's scalar operand */
__device__ __forceinline__ P2 Fma2(P2 a, P2 b, P2 c) {
  P2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ F2 CMul(F2 a, F2 b) { return F2{a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }

__device__ __forceinline__ void CpAsync16(void *smem_dst, const void *gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void CpAsyncCommit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void CpAsyncWaitAll() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

/* ---- mbarriers (shared::cta): the hand-shake between the receiver pairs and the AGC warp ---- */
__device__ __forceinline__ void MbarInit(uint64_t *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void MbarArrive(uint64_t *bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
/* upper bound of the time a waiting thread may stay suspended before try_wait returns false and the loop retries: the
   hardware wakes the thread when the phase completes, so a long hint costs nothing, while the default (short) one makes
   the waiting warp spin through issue slots its scheduler's other warps could use */
#ifndef T41RX_MBAR_HINT
#define T41RX_MBAR_HINT 0x989680u
#endif
constexpr unsigned kMbarSuspendHint = T41RX_MBAR_HINT;
__device__ __forceinline__ void MbarWait(uint64_t *bar, unsigned parity) {
  const unsigned addr = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(addr), "r"(parity), "r"(kMbarSuspendHint) : "memory");
}

/* everything a receiver warp keeps in registers across blocks (uniform over the lanes unless noted) */
struct RxRegs {
  /* configuration */
  /* small integers share one register (the kernel sits at its 128-register cap; spills go to L2 here) */
  unsigned mode : 4, agc_mode : 3, mirrored : 1, first_block : 1, nco_closed : 1, psk_enable : 1, eq_on : 1, nr_lms : 1,
      anr_notch : 1, cw_filter : 1;
  F2 tw_a, tw_b;         /* this thread's base twiddles of the stride-64 and stride-8 radix-8 passes */
  const char *cp_src;    /* this thread's first 16-byte piece of quarter 0 of block 0 */
  unsigned cp_dst;       /* its shared-memory address in raw buffer 0 */
  /* lane constants */
  F2 lane_rot;           /* nco_amp * exp(-j * delta * (8 * tau + 1)) */
  float pow8;            /* a1^(8 * lane): decay of the carry entering the warp's half quarter up to this lane */
};

/* ------------------------------------------------------------------ */
/* radix-8 passes on the padded buffer                                  */
/* ------------------------------------------------------------------ */
/* w[k] = (cos, sin)(2 pi k e / 512), k = 1..7, from one table entry and six complex products (shared
   memory and L1 bandwidth is the scarce resource of this kernel, FMAs are not) */
__device__ __forceinline__ void TwiddlePowers(F2 t, F2 (&w)[8]) {
  w[1] = t;
  w[2] = CMul(w[1], w[1]);
  w[3] = CMul(w[2], w[1]);
  w[4] = CMul(w[2], w[2]);
  w[5] = CMul(w[4], w[1]);
  w[6] = CMul(w[3], w[3]);
  w[7] = CMul(w[4], w[3]);
}

template <int PASS>
__device__ __forceinline__ void FwdPass(float2 *buf, F2 tw1, int b) {
  int n2, i0;
  if (PASS == 0) { n2 = 64; i0 = b; }
  else { n2 = 8; i0 = (b >> 3) * 64 + (b & 7); }
  float r[8], im[8];
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const float2 x = buf[FPos(i0 + m * n2)];
    r[m] = x.x;
    im[m] = x.y;
  }
  Dft8(r, im);
  buf[FPos(i0)] = float2{r[0], im[0]};
  F2 w[8];
  TwiddlePowers(tw1, w);
#pragma unroll
  for (int k = 1; k < 8; ++k)
    buf[FPos(i0 + k * n2)] = float2{r[k] * w[k].x + im[k] * w[k].y, im[k] * w[k].x - r[k] * w[k].y};
}

/* inverse of FwdPass<PASS> without the 1/8: conjugate twiddles on the inputs, inverse 8-point DFT.
 * kUpperHalf: store only outputs 256..511 (the valid half of the overlap-save result). */
template <int PASS, bool kUpperHalf>
__device__ __forceinline__ void InvPass(float2 *buf, F2 tw1, int b) {
  int n2, i0;
  if (PASS == 0) { n2 = 64; i0 = b; }
  else { n2 = 8; i0 = (b >> 3) * 64 + (b & 7); }
  float r[8], im[8];
  {
    const float2 x = buf[FPos(i0)];
    r[0] = x.x;
    im[0] = x.y;
  }
  F2 w[8];
  TwiddlePowers(tw1, w);
#pragma unroll
  for (int k = 1; k < 8; ++k) {
    const float2 x = buf[FPos(i0 + k * n2)];
    r[k] = x.x * w[k].x - x.y * w[k].y;
    im[k] = x.y * w[k].x + x.x * w[k].y;
  }
  Dft8(im, r);   /* swapping the roles of re and im turns the forward DFT into the inverse */
#pragma unroll
  for (int m = (kUpperHalf ? 4 : 0); m < 8; ++m) buf[FPos(i0 + m * n2)] = float2{r[m], im[m]};
}

/* forward pass 2 (8 contiguous elements, no twiddles), multiply by the filter mask (bins sit in
 * octal-digit-reversed positions), inverse pass 2: all in registers */
/* arow: where a row-producing block leaves the masked spectrum for the audio-spectrum by-product, or NULL */
__device__ __forceinline__ void MidPass(float2 *buf, const float2 (&hm)[8], int b, float2 *arow) {
  float r[8], im[8];
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const float2 x = buf[FPos(8 * b + m)];
    r[m] = x.x;
    im[m] = x.y;
  }
  Dft8(r, im);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float2 h = hm[k];
    const float xr = r[k], xi = im[k];
    r[k] = xr * h.x - xi * h.y;
    im[k] = xr * h.y + xi * h.x;
  }
  if (arow) {
#pragma unroll
    for (int k = 0; k < 8; ++k) arow[OctRev3((unsigned)(8 * b + k))] = float2{r[k], im[k]};
  }
  Dft8(im, r);
#pragma unroll
  for (int m = 0; m < 8; ++m) buf[FPos(8 * b + m)] = float2{r[m], im[m]};
}

/* ------------------------------------------------------------------ */
/* SAM (AMDecodeSAM, Demod.cpp:40-139) on ONE lane: the PLL is a serial  */
/* chain over the 256 samples.  Only under T41RX_FLAG_FAST_SAM: the loop */
/* is chaotic while it pulls in (ApproxAtan2's 2 pi quirk), so a 1e-7    */
/* difference at its input gives a different acquisition transient; once */
/* locked, the two trajectories agree again.                             */
/* ------------------------------------------------------------------ */
/* Atan2Approx (rx_phases.cuh, Demod.cpp:148-197, 2 pi quirk included) with the approximate division: the PLL lane is
   one long dependent chain and an IEEE division is a third of it */
__device__ __forceinline__ float Atan2Quick(float y, float x) {
  const float pi = 3.1415926535897932384626433832795f;
  const float tpi = 6.283185307179586476925286766559f;
  const bool wide = fabsf(x) > fabsf(y);
  const float p = AtanPoly(__fdividef(wide ? y : x, wide ? x : y));
  const float r_wide = (x > 0.0f) ? p : ((y >= 0.0f) ? p + pi : p - pi);
  const float r_tall = (y > 0.0f) ? tpi - p : -p - tpi;
  const float r_axis = (y > 0.0f) ? tpi : ((y < 0.0f) ? -tpi : 0.0f);
  return (x != 0.0f) ? (wide ? r_wide : r_tall) : r_axis;
}

__device__ __noinline__ void SamPllLane(const float *tab, const float *sam_consts, StreamState &st, const float2 *z,
                                        float *audio) {
  const float tpi = 6.283185307179586476925286766559f;
  const float omega_min = __ldg(sam_consts + 0), omega_max = __ldg(sam_consts + 1);
  const float g1 = __ldg(sam_consts + 2), g2 = __ldg(sam_consts + 3);
  float phz = st.sam_phzerror, fil = st.sam_fil_out, om2 = st.sam_omega2;
  /* arm_sin_f32 / arm_cos_f32 (table + linear interpolation) with one index computation: phz is in [0, 2 pi), the
     cosine reads a quarter of the table further on */
  auto sincos_tab = [&](float ph, float &sn_, float &cs_) {
    const float fidx = ph * (512.0f * 0.159154943092f);
    const int idx = (int)fidx;
    const float fr = fidx - (float)idx;
    const int is = idx & 511, ic = (idx + 128) & 511;
    const float s0 = tab[is], s1 = tab[is + 1], c0 = tab[ic], c1 = tab[ic + 1];
    sn_ = fmaf(fr, s1 - s0, s0);
    cs_ = fmaf(fr, c1 - c0, c0);
  };
  /* the phase of sample i + 1 is phz + the loop filter's output of sample i - 1: its sine / cosine are formed beside
     sample i's arctangent, two dependent chains side by side */
  float sn, cs;
  sincos_tab(phz, sn, cs);
  float2 v = z[0];
#pragma unroll 1
  for (int i = 0; i < kDec; ++i) {
    const float2 vn = z[min(i + 1, kDec - 1)];     /* off the chain */
    float phz_n = phz + fil;
    phz_n = (phz_n >= tpi) ? phz_n - tpi : phz_n;  /* |fil_out| is far below 2 pi: one wrap at most */
    phz_n = (phz_n < 0.0f) ? phz_n + tpi : phz_n;
    float sn_n, cs_n;
    sincos_tab(phz_n, sn_n, cs_n);
    const float ai = cs * v.x, bi = sn * v.x, aq = cs * v.y, bq = sn * v.y;
    const float corr0 = ai + bq;
    const float corr1 = aq - bi;
    audio[i] = (ai - bi) + (aq + bq);              /* the fade leveller is a no-op (SURVEY B3) */
    const float det = Atan2Quick(corr1, corr0);
    om2 = fminf(fmaxf(fmaf(g2, det, om2), omega_min), omega_max);
    fil = fmaf(g1, det, om2);
    phz = phz_n;
    sn = sn_n;
    cs = cs_n;
    v = vn;
  }
  st.sam_phzerror = phz;
  st.sam_fil_out = fil;
  st.sam_omega2 = om2;
}

/* CW audio low-pass, 6 transposed-direct-form-II biquads over 256 samples in place (CwFilterLane of rx_phases.cuh with
   FMA contraction) */
__device__ __noinline__ void CwFilterFast(float *aud, const float *coef, float *st) {
  float b0[6], b1[6], b2[6], a1[6], a2[6], d1[6], d2[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    b0[j] = __ldg(coef + 5 * j); b1[j] = __ldg(coef + 5 * j + 1); b2[j] = __ldg(coef + 5 * j + 2);
    a1[j] = __ldg(coef + 5 * j + 3); a2[j] = __ldg(coef + 5 * j + 4);
    d1[j] = st[2 * j]; d2[j] = st[2 * j + 1];
  }
  float v = aud[0];
#pragma unroll 2
  for (int n = 0; n < kDec; ++n) {
    const float vn = aud[min(n + 1, kDec - 1)];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const float y = fmaf(b0[j], v, d1[j]);
      d1[j] = fmaf(a1[j], y, fmaf(b1[j], v, d2[j]));
      d2[j] = fmaf(a2[j], y, b2[j] * v);
      v = y;
    }
    aud[n] = v;
    v = vn;
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) { st[2 * j] = d1[j]; st[2 * j + 1] = d2[j]; }
}

/* ------------------------------------------------------------------ */
/* optional audio stages between the demodulator and the interpolators */
/* (free functions, not inlined: the default path's code and register  */
/* allocation stay what they are without them)                         */
/* ------------------------------------------------------------------ */
/* Xanr (Noise.cpp:322-369): variable-leak LMS, 64 taps behind a delay of 16, one pass over the 256 samples at x,
   run by ONE warp (the adaptation is a serial chain over the samples; two taps per lane, j = lane and lane + 32,
   keep both dot products inside the warp: butterfly shuffles, no barrier).  The samples sit in a linear window
   (79 of history + 256) so that tap j of sample i is a plain offset.  State in StreamState in the reference's
   layout (delay line as a 512-deep ring with the write index running down), crossing to and from HBM once per
   pass.  FP32 throughout (the reference's FP64 sub-expressions included): its branch on two nearly equal error
   estimates can fall the other way once in a while, which moves the leak by one step of ~1e-6. */
__device__ __noinline__ void XanrWarp(float *s, StreamState &st, float *x, int lane, bool notch) {
  constexpr int kHist = 79, kMask = 511;
  constexpr float den_mult = 6.25e-10f, gamma = 0.1f, lidx_min = 120.0f, lidx_max = 200.0f, lincr = 1.0f, ldecr = 3.0f,
                  two_mu = 0.0001f;
  float *W = s + oMix;                            /* [79 + 256]: free between two front ends */
  const int i0 = st.anr_in_idx;
  float lidx = st.anr_lidx, ngamma = st.anr_ngamma;
  float w0 = st.anr_w[lane], w1 = st.anr_w[lane + 32];
  for (int k = lane + 1; k <= kHist; k += 32) W[kHist - k] = st.anr_d[(i0 + k) & kMask];
  for (int i = lane; i < kDec; i += 32) W[kHist + i] = x[i];
  __syncwarp();
  float mine = 0.0f;
#pragma unroll 1
  for (int i = 0; i < kDec; ++i) {
    const float a = W[kHist - 16 + i - lane], b = W[kHist - 48 + i - lane], xi = W[kHist + i];
    float y = fmaf(w0, a, w1 * b), sigma = fmaf(a, a, b * b);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
      y += __shfl_xor_sync(kFull, y, d);
      sigma += __shfl_xor_sync(kFull, sigma, d);
    }
    const float inv_sigp = 1.0f / (sigma + 1e-10f);
    const float error = xi - y;
    if ((i & 31) == lane) mine = error;
    const float se = two_mu * sigma * inv_sigp;
    const float nel = fabsf(error * (1.0f - se));
    const float nev = fabsf(xi - (1.0f - two_mu * ngamma) * y - error * se);
    if (nev < nel) {
      if ((lidx += lincr) > lidx_max) lidx = lidx_max;
      else if ((lidx -= ldecr) < lidx_min) lidx = lidx_min;
    }
    ngamma = gamma * (lidx * lidx) * (lidx * lidx) * den_mult;
    const float c0 = 1.0f - two_mu * ngamma;
    const float c1 = two_mu * error * inv_sigp;
    w0 = fmaf(c0, w0, c1 * a);
    w1 = fmaf(c0, w1, c1 * b);
    if (notch && (i & 31) == 31) x[i - 31 + lane] = mine;      /* the window, not x, feeds the taps */
  }
  st.anr_w[lane] = w0;
  st.anr_w[lane + 32] = w1;
  for (int i = lane; i < kDec; i += 32) st.anr_d[(i0 - i) & kMask] = W[kHist + i];
  if (lane == 0) {
    st.anr_in_idx = (i0 - kDec) & kMask;
    st.anr_lidx = lidx;
    st.anr_ngamma = ngamma;
  }
  __syncwarp();
}

/* Receive equaliser (DoReceiveEQ, Filter.cpp:117-165; hook Process.cpp:827-831) on the 256 demodulated samples,
   in place: 14 band-passes of 4 transposed-direct-form-II biquads (FIR.cpp:279-371), scaled by -/+ level and added
   in band order.  Thread (band, stage) = (tau >> 2, tau & 3): the 56 biquads run as a software pipeline over the
   samples, stage j one sample behind stage j - 1, whose output it receives by shuffle (the four stages of a band
   are four adjacent lanes); the last stages write their scaled outputs for 64 samples, which the pair then adds
   up.  Band states live in StreamState in the layout the bit-exact kernel uses (they cross to and from HBM once
   per block: only receivers with the equaliser on pay for it). */
__device__ __noinline__ void ReceiveEqPair(float *s, const float *eq_coeffs, const StreamCfg &cf, StreamState &st, float *aud,
                                         int tau, int bar_id) {
  constexpr int kEqStride = 65;                    /* band stride of the chunk buffer: the writers hit 8 banks */
  const int band = tau >> 2, j = tau & 3;
  const bool live = band < 14;
  float b0 = 0.0f, b1 = 0.0f, b2 = 0.0f, a1 = 0.0f, a2 = 0.0f, d1 = 0.0f, d2 = 0.0f, scale = 0.0f;
  if (live) {
    const float *k = eq_coeffs + 20 * band + 5 * j;
    b0 = __ldg(k); b1 = __ldg(k + 1); b2 = __ldg(k + 2); a1 = __ldg(k + 3); a2 = __ldg(k + 4);
    d1 = st.eq_state[band][2 * j];
    d2 = st.eq_state[band][2 * j + 1];
    scale = cf.eq_scale[band];
  }
  float *E = s + oMix;                             /* [14][65]: free between two front ends */
  const float *x = aud + 24;
  float ylast = 0.0f, xnext = x[0];
  float *eout = E + (live ? band : 0) * kEqStride;
  const bool writer = live && j == 3;
  /* one pipeline step; kEdge: some stages are outside the block (the first and the last three steps) */
#define T41RX_EQ_STEP(kEdge, k_, slot_)                                    \
{                                                                        \
  const float up = __shfl_up_sync(kFull, ylast, 1);                      \
  const float xin = (j == 0) ? xnext : up;                               \
  xnext = x[(k_) + 1];                 /* x[256] at the end: in the scratch, unused */ \
  const float y = fmaf(b0, xin, d1);                                     \
  const float nd1 = fmaf(a1, y, fmaf(b1, xin, d2));                      \
  const float nd2 = fmaf(a2, y, b2 * xin);                               \
  bool valid = true;                                                     \
  if (kEdge) {                                                           \
    const int n = (k_) - j;                                              \
    valid = n >= 0 && n < kDec;                                          \
  }                                                                      \
  if (valid) {                                                           \
    d1 = nd1;                                                            \
    d2 = nd2;                                                            \
    ylast = y;                                                           \
    if (writer) eout[slot_] = y * scale;                                 \
  }                                                                      \
}
  for (int k = 0; k < 3; ++k) T41RX_EQ_STEP(true, k, 0)            /* no writer is valid yet */
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    const int k0 = 64 * c + 3;                     /* the steps whose outputs are samples 64 c .. 64 c + 63 */
    if (c < 3) {
#pragma unroll 4
      for (int i = 0; i < 64; ++i) T41RX_EQ_STEP(false, k0 + i, i)
    } else {
#pragma unroll 1
      for (int i = 0; i < 61; ++i) T41RX_EQ_STEP(false, k0 + i, i)
      for (int i = 61; i < 64; ++i) T41RX_EQ_STEP(true, k0 + i, i)
    }
    asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
    float acc = E[tau] + E[kEqStride + tau];
#pragma unroll
    for (int b = 2; b < 14; ++b) acc += E[b * kEqStride + tau];
    aud[24 + 64 * c + tau] = acc;                  /* stage 0 is past these inputs */
    asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
  }
#undef T41RX_EQ_STEP
  if (live) {
    st.eq_state[band][2 * j] = d1;
    st.eq_state[band][2 * j + 1] = d2;
  }
  asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
}


/* ------------------------------------------------------------------ */
/* receiver pair: two warps (64 threads) per receiver                   */
/* ------------------------------------------------------------------ */
/* kQ15: the call's blocks are the firmware's q15 format (a.iq16 / a.audio16: arm_q15_to_float on the way in,
   Process.cpp:107-108, arm_float_to_q15 on the way out, :936): 8 KiB in + 4 KiB out per stream-block instead of 16 + 8 */
constexpr int kRawChunkWordsQ = 12;                   /* q15: 8 samples (8 words) + 4 pad: conflict-free LDS.128 */
template <bool kQ15>
struct RxPair {
  const LaunchArgs &a;
  float *s;          /* this receiver's slot */
  int sid;           /* receiver index */
  int lane;          /* lane in the warp */
  int w2;            /* warp in the pair: 0 / 1 (also: the channel I / Q it owns in the FIR stages) */
  int tau;           /* thread in the pair: 0..63 */
  int bar_id;        /* named barrier of the pair */
  RxRegs r;
  SectionTimer tm;

  __device__ __forceinline__ RxPair(const LaunchArgs &a_, float *s_, int sid_, int lane_, int w2_, int bar_)
      : a(a_), s(s_), sid(sid_), lane(lane_), w2(w2_), tau(32 * w2_ + lane_), bar_id(bar_) {}

  /* Make the thread indices opaque at a stage boundary: address arithmetic derived from them is then
     recomputed inside the stage instead of being kept live (and spilled) across the whole block loop. */
  __device__ __forceinline__ void Launder() {
    asm volatile("" : "+r"(lane), "+r"(tau));
  }

  __device__ __forceinline__ void PairSync() const {
    asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
  }

  __device__ __forceinline__ const float *BlockIq(int t) const {
    return a.iq + ((size_t)sid * a.t_stride + t) * (2 * kBlock);
  }
  __device__ __forceinline__ const int16_t *BlockIq16(int t) const {
    return a.iq16 + ((size_t)sid * a.t_stride + t) * (2 * kBlock);
  }

  /* issue this thread's share of the asynchronous copy of quarter q of block t into raw buffer (q & 1) */
  __device__ __forceinline__ void IssueQuarter(int t, int q) {
    /* one warp instruction copies 8 chunks (512 contiguous bytes); the 8 lanes of a quarter-warp write the
       same 16-byte piece of 8 different chunks: distinct banks (chunk stride 20 words).  Thread (w2, lane)
       copies piece (lane >> 3) of chunks 16 i + 8 w2 + (lane & 7), i = 0..3 */
    const unsigned dst = r.cp_dst + (q & 1) * (kRawBufWords * 4);
    if (kQ15) {
      /* q15: a chunk is 32 bytes = 2 pieces; thread (w2, lane) copies piece (lane >> 4) of chunks 32 i + 16 w2 + (lane & 15),
         i = 0, 1: one warp instruction reads 512 contiguous bytes, 8 lanes write 8 different chunks (stride 12 words) */
      const char *src = r.cp_src + ((size_t)t * 4 + q) * 2048;
#pragma unroll
      for (int i = 0; i < 2; ++i)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + i * 32 * (kRawChunkWordsQ * 4)), "l"(src + i * 1024) : "memory");
    } else {
      const char *src = r.cp_src + ((size_t)t * 4 + q) * 4096;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + i * 16 * (kRawChunkWords * 4)), "l"(src + i * 1024) : "memory");
    }
    CpAsyncCommit();
  }

  /* ---------------- launch prologue ---------------- */
  __device__ void LoadState() {
    const StreamState &st = a.st[sid];
    const StreamCfg &cf = a.cfg[sid];
    const FilterSet &fs = a.fsets[cf.filter_id];
    r.mode = cf.mode;
    r.agc_mode = cf.agc_mode;
    r.mirrored = cf.mirrored != 0;
    if (tau == 4) {
      s[oXtra + xInGain] = cf.rf_gain_value * kDcB0 * 1.1f;
      s[oXtra + xNegIqAmp] = cf.neg_iq_amp;
      reinterpret_cast<int *>(s)[oXtra + xRfGain] = st.rf_gain;
      reinterpret_cast<int *>(s)[oXtra + xFilterId] = cf.filter_id;
      reinterpret_cast<unsigned *>(s)[oXtra + xCodecTimer] = st.codec_timer;
    }
    r.first_block = st.first_block != 0;
    r.nco_closed = (st.nco_closed && st.nco_epoch_seen == cf.nco_epoch) ? 1 : 0;
    {
      double sn, cs;
      sincos(st.nco_phase, &sn, &cs);
      if (st.fast_native && r.nco_closed) {
        cs = st.fast_ph_re;
        sn = st.fast_ph_im;
      }
      if (tau == 0) {               /* unit block phasor exp(j * phase) of the oscillator: shared memory, FP64 */
        double *md = reinterpret_cast<double *>(s + oMiscF + mPhasor);
        md[0] = cs;
        md[1] = sn;
      }
      /* Osc_Vect of a still-settling oscillator lives in the HBM state (rare path, one thread) */
      if (st.nco_closed && !r.nco_closed && tau == 0) {   /* leaving closed form (retune): rebuild it at the settled radius */
        const double rr = sqrt(st.osc_q * st.osc_q + st.osc_i * st.osc_i);
        a.st[sid].osc_q = rr * cs;
        a.st[sid].osc_i = rr * sn;
      }
    }
    {
      double sn, cs;
      sincos(-cf.nco_delta * (double)(8 * tau + 1), &sn, &cs);
      r.lane_rot = F2{(float)(cf.nco_amp * cs), (float)(cf.nco_amp * sn)};
    }
    r.pow8 = PowA1(8 * lane);
    {
      const float2 ta = __ldg(a.twiddle + tau), tb = __ldg(a.twiddle + 8 * (tau & 7));
      r.tw_a = F2{ta.x, ta.y};
      r.tw_b = F2{tb.x, tb.y};
    }
    r.psk_enable = cf.psk31_enable != 0;
    r.eq_on = cf.eq_on != 0;
    r.nr_lms = cf.nr_lms != 0;
    r.anr_notch = cf.anr_notch != 0;
    r.cw_filter = cf.cw_filter >= 0;
    if (tau == 2) {
      s[oMiscF + mAmWold] = st.am_wold;
      s[oMiscF + mAmX1] = st.am_lp_state[0];
      s[oMiscF + mAmX2] = st.am_lp_state[1];
      s[oMiscF + mAmY1] = st.am_lp_state[2];
      s[oMiscF + mAmY2] = st.am_lp_state[3];
      s[oMiscF + mNfmI] = st.nfm_last_i;
      s[oMiscF + mNfmQ] = st.nfm_last_q;
      for (int i = 0; i < 5; ++i) s[oMiscF + mAmLp + i] = cf.am_lp[i];
    }
    if (tau == 3) {
      double bs, bc;
      sincos(cf.nco_block_delta, &bs, &bc);
      double *rot = reinterpret_cast<double *>(s + oMiscF + mBlkRot);
      rot[0] = bc;
      rot[1] = bs;
      s[oMiscF + mVolScale] = cf.vol_scale;
      s[oMiscF + mVolume] = cf.volume;
      s[oMiscF + mFixedGain] = cf.agc.fixed_gain;
      s[oMiscF + mIqPhase] = cf.iq_phase;
    }
    if (kQ15) {
      const int chunk0 = 16 * w2 + (lane & 15), piece = lane >> 4;
      r.cp_src = reinterpret_cast<const char *>(BlockIq16(0)) + chunk0 * 32 + piece * 16;
      r.cp_dst = (unsigned)__cvta_generic_to_shared(s + oRaw) + chunk0 * (kRawChunkWordsQ * 4) + piece * 16;
    } else {
      const int chunk0 = 8 * w2 + (lane & 7), piece = lane >> 3;
      r.cp_src = reinterpret_cast<const char *>(BlockIq(0)) + chunk0 * 64 + piece * 16;
      r.cp_dst = (unsigned)__cvta_generic_to_shared(s + oRaw) + chunk0 * (kRawChunkWords * 4) + piece * 16;
    }
    if (tau == 1) {
      s[oMiscF + mInvIn] = cf.agc.inv_max_input;
      s[oMiscF + mTarget] = cf.agc.out_target;
      s[oMiscF + mSlope] = cf.agc.slope_constant;
      s[oMiscF + mOmF] = cf.agc.onemfast_backmult;
      s[oMiscF + mOmH] = cf.agc.onemhang_backmult;
      s[oMiscF + mFbm] = cf.agc.fast_backmult;
      s[oMiscF + mHbm] = cf.agc.hang_backmult;
    }
    /* DC-block recurrence value after the previous block's last Q sample (feeds this block's I chain, B6) */
    if (tau == 0) {
      s[oMiscF + mEndQ] = st.fast_native ? st.fast_dc_w : st.dc_d1 / (kDcB0 * (kDcA1 - 1.0f) * cf.rf_gain_value);
      s[oMiscF + mEndI] = 0.0f;
    }
    for (int i = tau; i < 154; i += 64) {
      float v;
      if (i < 28) v = fs.dec1[i];
      else if (i < 74) v = fs.dec2[i - 28];
      else if (i < 122) v = fs.int1[i - 74];
      else v = fs.int2[i - 122];
      s[oTapsF + i] = v;
    }
    /* oscillator tables: W[j] = j^j * exp(-j delta j), j < 8 (Fs/4 shift folded); Q[q] = exp(-j delta 512 q) */
    if (tau < 12) {
      const int n = tau < 8 ? tau : 512 * (tau - 8);
      double sn, cs;
      sincos(-cf.nco_delta * (double)n, &sn, &cs);
      float wr = (float)cs, wi = (float)sn;
      if (tau < 8) {
        const int k = tau & 3;               /* multiply by j^k */
        const float a0 = wr, b0 = wi;
        if (k == 1) { wr = -b0; wi = a0; }
        else if (k == 2) { wr = -a0; wi = -b0; }
        else if (k == 3) { wr = b0; wi = -a0; }
      }
      s[oNcoW + 2 * tau] = wr;
      s[oNcoW + 2 * tau + 1] = wi;
    }
    /* histories */
    {                                            /* dec1: plane (ch, p) entry e = -8..-1 holds sample 4 e + p */
      const int i = tau;
      const int pl = i >> 3, e = (i & 7) - 8;
      const int ch = pl >> 2, p = pl & 3;
      const int n = 4 * e + p;                   /* -32 .. -1 */
      s[oMH + i] = (n >= -(kDec1Taps - 1)) ? st.dec1_hist[ch][n + (kDec1Taps - 1)] : 0.0f;
    }
    for (int i = tau; i < 96; i += 64) {         /* dec2: plane (ch, par) entry e = -24..-1 holds sample 2 e + par */
      const int pl = i / 24, e = (i % 24) - 24;
      const int ch = pl >> 1, par = pl & 1;
      const int n = 2 * e + par;
      s[oDH + i] = (n >= -(kDec2Taps - 1)) ? st.dec2_hist[ch][n + (kDec2Taps - 1)] : 0.0f;
    }
    for (int i = tau; i < 256; i += 64) {
      s[OlaW(0, i)] = st.ola_prev[0][i];
      s[OlaW(1, i)] = st.ola_prev[1][i];
    }
    for (int i = tau; i < kAgcDelay; i += 64) {  /* sample -(97 - i) sits at ring index 31 + i */
      s[oZH + 2 * i] = st.agc_re[31 + i];
      s[oZH + 2 * i + 1] = st.agc_im[31 + i];
    }
    if (tau < 23) s[oIH + tau] = st.int1_hist[tau];
    if (tau < 7) s[oIH + 24 + tau] = st.int2_hist[tau];
    PairSync();
  }

  __device__ void StoreState() {
    StreamState &st = a.st[sid];
    const StreamCfg &cf = a.cfg[sid];
    PairSync();
    for (int i = tau; i < 2 * (kDec1Taps - 1); i += 64) {
      const int ch = i / (kDec1Taps - 1), n = (i % (kDec1Taps - 1)) - (kDec1Taps - 1);   /* -27..-1 */
      const int p = n & 3, e = (n - p) / 4;                                              /* e = -7..-1 */
      st.dec1_hist[ch][n + (kDec1Taps - 1)] = s[oMH + (ch * 4 + p) * 8 + (e + 8)];
    }
    for (int i = tau; i < 2 * (kDec2Taps - 1); i += 64) {
      const int ch = i / (kDec2Taps - 1), n = (i % (kDec2Taps - 1)) - (kDec2Taps - 1);   /* -45..-1 */
      const int par = n & 1, e = (n - par) / 2;                                          /* e = -23..-1 */
      st.dec2_hist[ch][n + (kDec2Taps - 1)] = s[oDH + (ch * 2 + par) * 24 + (e + 24)];
    }
    for (int i = tau; i < 256; i += 64) {
      st.ola_prev[0][i] = s[OlaW(0, i)];
      st.ola_prev[1][i] = s[OlaW(1, i)];
    }
    for (int i = tau; i < kAgcDelay; i += 64) {
      st.agc_re[31 + i] = s[oZH + 2 * i];
      st.agc_im[31 + i] = s[oZH + 2 * i + 1];
      st.agc_abs[31 + i] = __fsqrt_rn(s[oZH + 2 * i] * s[oZH + 2 * i] + s[oZH + 2 * i + 1] * s[oZH + 2 * i + 1]);
    }
    if (tau < 23) st.int1_hist[tau] = s[oIH + tau];
    if (tau < 7) st.int2_hist[tau] = s[oIH + 24 + tau];
    if (tau == 1) {
      st.am_wold = s[oMiscF + mAmWold];
      st.am_lp_state[0] = s[oMiscF + mAmX1];
      st.am_lp_state[1] = s[oMiscF + mAmX2];
      st.am_lp_state[2] = s[oMiscF + mAmY1];
      st.am_lp_state[3] = s[oMiscF + mAmY2];
      st.nfm_last_i = s[oMiscF + mNfmI];
      st.nfm_last_q = s[oMiscF + mNfmQ];
    }
    if (tau == 0) {
      st.dc_d1 = s[oMiscF + mEndQ] * (kDcB0 * (kDcA1 - 1.0f) * cf.rf_gain_value);
      st.dc_d2 = 0.0f;
      st.fast_native = 1;
      st.fast_dc_w = s[oMiscF + mEndQ];
      const double *md = reinterpret_cast<const double *>(s + oMiscF + mPhasor);
      const double ph_re = md[0], ph_im = md[1];
      st.fast_ph_re = ph_re;
      st.fast_ph_im = ph_im;
      st.rf_gain = reinterpret_cast<const int *>(s)[oXtra + xRfGain];
      st.codec_timer = reinterpret_cast<const unsigned *>(s)[oXtra + xCodecTimer];
      st.first_block = r.first_block;
      if (r.nco_closed) {
        double ph = atan2(ph_im, ph_re);
        if (ph < 0) ph += 6.283185307179586476925286766559;
        st.nco_phase = ph;
        st.nco_closed = 1;
        st.nco_epoch_seen = cf.nco_epoch;
        /* keep (osc_q, osc_i) at the settled radius so that a later exact block restarts correctly */
        const double rr = sqrt(cf.nco_r2_fix);
        st.osc_q = rr * ph_re;
        st.osc_i = rr * ph_im;
      } else {
        st.nco_closed = 0;
        st.nco_epoch_seen = cf.nco_epoch;
      }
    }
  }

  /* ---------------- front end ---------------- */
  /* blocked inclusive scan over the lanes of a warp of chunk-end values of the recurrence w <- a1 w + x
     (8 samples per lane): after it, lane L holds the true w at the end of its chunk */
  /* the same scan on an (I, Q) pair */
  __device__ __forceinline__ P2 ScanDc2(P2 e) const {
    float m = kDcA1;
    m *= m; m *= m; m *= m;            /* a1^8 */
    P2 v = e;
#pragma unroll
    for (int d = 1; d <= 8; d <<= 1) {
      const P2 t = Pack2(__shfl_up_sync(kFull, Lo(v), d), __shfl_up_sync(kFull, Hi(v), d));
      if (lane >= d) v = Fma2(Dup(m), t, v);
      m *= m;
    }
    /* a1^128 ~ 2e-9: the 16-lane step is below a float's resolution */
    return v;
  }
  __device__ __forceinline__ float ScanDc(float e) const {
    float m = kDcA1;
    m *= m; m *= m; m *= m;            /* a1^8 */
    float v = e, t;
    t = __shfl_up_sync(kFull, v, 1); if (lane >= 1) v = fmaf(m, t, v);
    m *= m;
    t = __shfl_up_sync(kFull, v, 2); if (lane >= 2) v = fmaf(m, t, v);
    m *= m;
    t = __shfl_up_sync(kFull, v, 4); if (lane >= 4) v = fmaf(m, t, v);
    m *= m;
    t = __shfl_up_sync(kFull, v, 8); if (lane >= 8) v = fmaf(m, t, v);
    /* a1^128 ~ 2e-9: the 16-lane step is below a float's resolution */
    return v;
  }

  /* one 512-sample quarter, 8 samples per thread: DC block + IQ correction + Fs/4 + NCO mix -> phase planes.
     cI / cQ: recurrence values entering the quarter (used by warp 0).  base: conj(block phasor) * Q[q] * gain. */
  template <bool kTable>
  __device__ __forceinline__ void QuarterMix(int q, float cI, float cQ, F2 base, const float2 *osc) {
    /* the I and the Q chain run the same recurrence with the same constants: packed FP32 on (I, Q) pairs, which
       is how the samples sit in memory */
    P2 x[8];
    if (kQ15) {
      /* arm_q15_to_float: x / 32768, exact.  A word holds (I, Q) as two int16: flip the sign bits (offset binary), drop
         each half into the mantissa of 256.0f (whose last place weighs 2^-15) and take 257 away again */
      const float *raw = s + oRaw + (q & 1) * kRawBufWords + tau * kRawChunkWordsQ;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const uint4 v = *reinterpret_cast<const uint4 *>(raw + 4 * k);
        const unsigned w[4] = {v.x ^ 0x80008000u, v.y ^ 0x80008000u, v.z ^ 0x80008000u, v.w ^ 0x80008000u};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float fi = __uint_as_float(__byte_perm(w[j], 0x43800000u, 0x7610));
          const float fq = __uint_as_float(__byte_perm(w[j], 0x43800000u, 0x7632));
          x[4 * k + j] = Fma2(Pack2(fi, fq), Dup(1.0f), Dup(-257.0f));
        }
      }
    } else {
      const float *raw = s + oRaw + (q & 1) * kRawBufWords + tau * kRawChunkWords;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(raw + 4 * k);
        x[2 * k] = v.x;
        x[2 * k + 1] = v.y;
      }
    }
    /* zero-state recurrences */
    P2 w[8];
    {
      P2 acc = 0ull;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc = Fma2(Dup(kDcA1), acc, x[j]);
        w[j] = acc;
      }
    }
    float p8 = kDcA1;
    p8 *= p8; p8 *= p8; p8 *= p8;
    /* warp 0 knows the value entering its half (cI, cQ) and folds it into lane 0's chunk end; warp 1 scans from
       zero and adds the decayed end value of warp 0's half once that is known (the recurrence is linear) */
    P2 e = w[7];
    if (tau == 0) e = Fma2(Dup(p8), Pack2(cI, cQ), e);
    const P2 sc = ScanDc2(e);
    P2 c = Pack2(__shfl_up_sync(kFull, Lo(sc), 1), __shfl_up_sync(kFull, Hi(sc), 1));
    if (tau == 31) {
      s[oMiscF + mMidI] = Lo(sc);
      s[oMiscF + mMidQ] = Hi(sc);
    }
    PairSync();
    if (w2 == 0) {
      if (lane == 0) c = Pack2(cI, cQ);
    } else {
      const P2 mid = Pack2(s[oMiscF + mMidI], s[oMiscF + mMidQ]);
      if (lane == 0) c = mid;
      else c = Fma2(Dup(r.pow8), mid, c);
      if (lane == 31) {              /* recurrence values leaving the quarter (a1^256 of warp 0's end is below resolution) */
        s[oMiscF + mEndI] = Lo(sc);
        s[oMiscF + mEndQ] = Hi(sc);
      }
    }
    /* true recurrence values, first difference (DC-block numerator 1 - z^-1) */
    float yi[8], yq[8];
    {
      float pw = kDcA1;
      P2 prev = c;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const P2 t = Fma2(Dup(pw), c, w[j]);
        const P2 y = Fma2(Dup(-1.0f), prev, t);
        Unpack2(y, yi[j], yq[j]);
        prev = t;
        pw *= kDcA1;    /* compile-time constant after unrolling */
      }
    }
    /* I *= -IQAmp, phase correction (Process.cpp:165-174, Utility.cpp:178-187) */
    if (r.mirrored) {
      const float iq_phase_ = s[oMiscF + mIqPhase];
      const float neg_iq_amp = s[oXtra + xNegIqAmp];
      if (neg_iq_amp == -1.0f) {
#pragma unroll
        for (int j = 0; j < 8; ++j) yi[j] = -yi[j];      /* folds into the consumers' operand modifiers */
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) yi[j] *= neg_iq_amp;
      }
      if (iq_phase_ != 0.0f) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (iq_phase_ < 0.0f) yq[j] = fmaf(yi[j], iq_phase_, yq[j]);
          else yi[j] = fmaf(yq[j], iq_phase_, yi[j]);
        }
      }
    }
    /* mix: multiplier of sample j = base * lane_rot * W[j] */
    const F2 m = CMul(base, r.lane_rot);
    const float4 *wt = reinterpret_cast<const float4 *>(s + oNcoW);
    float oi[8], oq[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      F2 m0, m1;
      if (kTable) {
        /* settling oscillator: multiplier = gain * conj(osc[n]) * j^n, osc from the step-by-step table */
        const float4 o2 = *reinterpret_cast<const float4 *>(osc + 8 * tau + 2 * k);
        const F2 c0 = F2{o2.x * base.x, -o2.y * base.x}, c1 = F2{o2.z * base.x, -o2.w * base.x};
        m0 = (k & 1) ? F2{-c0.x, -c0.y} : c0;                    /* sample 2k:   j^(2k)   = (-1)^k   */
        m1 = (k & 1) ? F2{c1.y, -c1.x} : F2{-c1.y, c1.x};        /* sample 2k+1: j^(2k+1) = j (-1)^k */
      } else {
        const float4 w2_ = wt[k];
        m0 = CMul(m, F2{w2_.x, w2_.y});
        m1 = CMul(m, F2{w2_.z, w2_.w});
      }
      oi[2 * k] = yi[2 * k] * m0.x - yq[2 * k] * m0.y;
      oq[2 * k] = yi[2 * k] * m0.y + yq[2 * k] * m0.x;
      oi[2 * k + 1] = yi[2 * k + 1] * m1.x - yq[2 * k + 1] * m1.y;
      oq[2 * k + 1] = yi[2 * k + 1] * m1.y + yq[2 * k + 1] * m1.x;
    }
    /* phase planes: sample 8 tau + j -> plane (j & 3), entry 2 tau + (j >> 2) */
    float *mix = s + oMix;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      *reinterpret_cast<float2 *>(mix + p * kMixPlane + 8 + 2 * tau) = float2{oi[p], oi[4 + p]};
      *reinterpret_cast<float2 *>(mix + (4 + p) * kMixPlane + 8 + 2 * tau) = float2{oq[p], oq[4 + p]};
    }
  }

  /* arm_fir_decimate_f32, M = 4, 28 taps (Process.cpp:474-475): warp w2 filters channel w2, 4 outputs per
     lane per quarter.  Output m (quarter-local) = sum_t h[t] x[4 m - 27 + t]; sample 4 m - 27 + t = plane
     (1 + t) & 3, entry m - 7 + ((1 + t) >> 2). */
  __device__ __forceinline__ void Dec1Quarter(int q) {
    const int ch = w2;
    const float *mix = s + oMix;
    float *d1 = s + oD1;
    float tap[kDec1Taps];
#pragma unroll
    for (int k = 0; k < kDec1Taps / 4; ++k) {
      const float4 v = *reinterpret_cast<const float4 *>(s + oTapsF + 4 * k);
      tap[4 * k] = v.x; tap[4 * k + 1] = v.y; tap[4 * k + 2] = v.z; tap[4 * k + 3] = v.w;
    }
    /* packed FP32 as in Dec2: even window offsets feed the output pairs (0,1)(2,3), odd ones the pair (1,2) plus
       outputs 0 and 3 alone */
    P2 w[4][6];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(mix + (ch * 4 + p) * kMixPlane + 4 * lane);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const ulonglong2 v = src[k];
        w[p][2 * k] = v.x;
        w[p][2 * k + 1] = v.y;
      }
    }
    P2 e0 = 0ull, e1 = 0ull, od = 0ull;
    float s0 = 0.0f, s3 = 0.0f;
#pragma unroll
    for (int t = 0; t < kDec1Taps; ++t) {
      const int p = (1 + t) & 3, off = 1 + ((1 + t) >> 2);        /* output o reads window word o + off */
      if ((off & 1) == 0) {
        e0 = Fma2(w[p][off >> 1], Dup(tap[t]), e0);
        e1 = Fma2(w[p][(off >> 1) + 1], Dup(tap[t]), e1);
      } else {
        s0 = fmaf(Hi(w[p][(off - 1) >> 1]), tap[t], s0);
        od = Fma2(w[p][(off + 1) >> 1], Dup(tap[t]), od);
        s3 = fmaf(Lo(w[p][(off + 3) >> 1]), tap[t], s3);
      }
    }
    const float acc[4] = {Lo(e0) + s0, Hi(e0) + Lo(od), Lo(e1) + Hi(od), Hi(e1) + s3};
    /* d1 sample n = 128 q + 4 L + o -> plane (n & 1), entry n >> 1 */
    const int e = 64 * q + 2 * lane;
    *reinterpret_cast<float2 *>(d1 + (ch * 2 + 0) * kD1Plane + D1W(24 + e)) = float2{acc[0], acc[2]};
    *reinterpret_cast<float2 *>(d1 + (ch * 2 + 1) * kD1Plane + D1W(24 + e)) = float2{acc[1], acc[3]};
    __syncwarp();
    /* slide this channel's plane histories: entries 120..127 become -8..-1 (one value per lane) */
    {
      const int pl = ch * 4 + (lane >> 3), e8 = lane & 7;
      const float v = s[oMix + pl * kMixPlane + 8 + 120 + e8];
      __syncwarp();
      s[oMix + pl * kMixPlane + e8] = v;
    }
  }

  /* arm_fir_decimate_f32, M = 2, 46 taps (Process.cpp:478-479): warp w2 filters channel w2, 8 outputs per lane.
     Output o = sum_t h[t] d[2 o - 45 + t]; sample 2 o - 45 + t = plane (1 + t) & 1, entry o - 23 + ((1 + t) >> 1).
     Packed FP32 (FFMA2, scalar tap x pair of window entries): the window sits in registers as aligned pairs
     (w[2m], w[2m+1]); a tap whose window offset is even feeds the output pairs (0,1)(2,3)(4,5)(6,7), one whose
     offset is odd feeds the pairs (1,2)(3,4)(5,6) plus outputs 0 and 7 alone; the two sets are added at the end. */
  __device__ __forceinline__ void Dec2(float (&out)[8]) {
    const int ch = w2;
    const float *d1 = s + oD1;
    const float *tp = s + oTapsF + 28;
    P2 w[2][16];
#pragma unroll
    for (int par = 0; par < 2; ++par) {
      const float *pl = d1 + (ch * 2 + par) * kD1Plane;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(pl + D1W(8 * lane + 4 * k));
        w[par][2 * k] = v.x;
        w[par][2 * k + 1] = v.y;
      }
    }
    P2 e[4] = {0ull, 0ull, 0ull, 0ull}, od[3] = {0ull, 0ull, 0ull};
    float s0 = 0.0f, s7 = 0.0f;
#pragma unroll
    for (int t2 = 0; t2 < kDec2Taps; t2 += 2) {
      const float2 h2 = *reinterpret_cast<const float2 *>(tp + t2);
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int t = t2 + u;
        const int par = (1 + t) & 1, off = 1 + ((1 + t) >> 1);     /* output o reads window word o + off */
        const float h = u ? h2.y : h2.x;
        if ((off & 1) == 0) {
#pragma unroll
          for (int m = 0; m < 4; ++m) e[m] = Fma2(w[par][(2 * m + off) >> 1], Dup(h), e[m]);
        } else {
          s0 = fmaf(Hi(w[par][(off - 1) >> 1]), h, s0);                       /* output 0: word off (odd) */
#pragma unroll
          for (int m = 0; m < 3; ++m) od[m] = Fma2(w[par][(2 * m + 1 + off) >> 1], Dup(h), od[m]);
          s7 = fmaf(Lo(w[par][(7 + off) >> 1]), h, s7);                        /* output 7: word 7 + off (even) */
        }
      }
    }
    out[0] = Lo(e[0]) + s0;
    out[1] = Hi(e[0]) + Lo(od[0]);
    out[2] = Lo(e[1]) + Hi(od[0]);
    out[3] = Hi(e[1]) + Lo(od[1]);
    out[4] = Lo(e[2]) + Hi(od[1]);
    out[5] = Hi(e[2]) + Lo(od[2]);
    out[6] = Lo(e[3]) + Hi(od[2]);
    out[7] = Hi(e[3]) + s7;
  }

  /* FE for block t */
  __device__ void FrontEnd(int t, int buf, float4 tail_u, float4 tail_v) {
    const StreamCfg &cf = a.cfg[sid];
    /* the recurrence value entering the Q chain is the one leaving the I chain (B6): pre-read the last
       128 I samples of the block (a1^128 ~ 2e-9); only warp 0's lane 0 consumes it */
    float tail = 0.0f;
    if (w2 == 0) {
      const float4 u = tail_u, v = tail_v;            /* samples n0 .. n0+3, n0 = 2044 - 4 lane */
      float acc = u.x;                                 /* oldest first */
      acc = fmaf(kDcA1, acc, u.z);
      acc = fmaf(kDcA1, acc, v.x);
      acc = fmaf(kDcA1, acc, v.z);
      tail = acc * PowA1(4 * lane);      /* weight of this lane's partial sum */
#pragma unroll
      for (int d = 16; d >= 1; d >>= 1) tail += __shfl_xor_sync(kFull, tail, d);
    }
    /* restore the decimator histories in front of the planes (each warp: its own channel) */
    {
      const int i = 32 * w2 + lane;                  /* 64 dec1 history values: planes 4 w2 .. 4 w2 + 3 */
      s[oMix + (i >> 3) * kMixPlane + (i & 7)] = s[oMH + i];
      for (int j = lane; j < 48; j += 32) {          /* 96 dec2 history values: planes 2 w2, 2 w2 + 1 */
        const int k = 48 * w2 + j;
        s[oD1 + (k / 24) * kD1Plane + (k % 24)] = s[oDH + k];          /* D1W is the identity on words 0..31 */
      }
    }
    /* gains of this block (Process.cpp:117,133): rfGainValue and RFgain are folded into the phasor */
    const float gain = s[oXtra + xInGain] * (float)reinterpret_cast<const int *>(s)[oXtra + xRfGain];
    F2 pb;
    {
      const double *md = reinterpret_cast<const double *>(s + oMiscF + mPhasor);
      pb = F2{(float)md[0] * gain, -(float)md[1] * gain};
    }
    T41RX_LAP(tm, 0);
    const bool closed = r.nco_closed != 0;
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {
      /* recurrence values entering the quarter (written by thread 63 before the previous quarter's
         second barrier; read before this quarter's first barrier: no race with this quarter's writes) */
      float cI, cQ;
      if (q == 0) { cI = s[oMiscF + mEndQ]; cQ = tail; }
      else { cI = s[oMiscF + mEndI]; cQ = s[oMiscF + mEndQ]; }
      CpAsyncWaitAll();
      PairSync();                     /* raw quarter visible; planes free (previous dec1 done) */
      T41RX_LAP(tm, 1);
      if (closed) {
        if (q < 3) IssueQuarter(t, q + 1);
        else if (t + 1 < a.n_blocks) IssueQuarter(t + 1, 0);
        const F2 qq = F2{s[oNcoW + 16 + 2 * q], s[oNcoW + 16 + 2 * q + 1]};
        __syncwarp();
        QuarterMix<false>(q, cI, cQ, CMul(pb, qq), nullptr);
      } else {
        /* the oscillator's amplitude loop has not settled (first block of a receiver, block after a
           retune): FreqShift2's FP64 recurrence step by step (Freq_Shift.cpp:126-140) on one thread, one
           quarter at a time into the idle raw buffer (so no copy is in flight during such a block) */
        float2 *tab = reinterpret_cast<float2 *>(s + oRaw + ((q + 1) & 1) * kRawBufWords);
        if (tau == 0) {
          StreamState &stt = a.st[sid];
          double vq = stt.osc_q, vi = stt.osc_i;
          const double oc = cf.osc_cos, os = cf.osc_sin;
          for (int n = 0; n < 512; ++n) {
            const double oq = (vq * oc) - (vi * os);
            const double oi = (vi * oc) + (vq * os);
            const double gn = 1.95 - ((vq * vq) + (vi * vi));
            vq = gn * oq;
            vi = gn * oi;
            tab[n] = float2{(float)oq, (float)oi};
          }
          stt.osc_q = vq;
          stt.osc_i = vi;
          if (q == 3) {               /* settled?  then continue in closed form from the vector's angle */
            const double r2 = vq * vq + vi * vi;
            const double inv = rsqrt(r2);
            double *md = reinterpret_cast<double *>(s + oMiscF + mPhasor);
            md[0] = vq * inv;
            md[1] = vi * inv;
            s[oMiscF + mSettled] = (fabs(r2 - cf.nco_r2_fix) < 4.0e-15) ? 1.0f : 0.0f;
          }
        }
        PairSync();
        QuarterMix<true>(q, cI, cQ, F2{gain, 0.0f}, tab);
      }
      PairSync();                     /* planes visible */
      if (!closed) {
        if (q < 3) IssueQuarter(t, q + 1);
        else if (t + 1 < a.n_blocks) IssueQuarter(t + 1, 0);
      }
      T41RX_LAP(tm, 2);
      Dec1Quarter(q);
      T41RX_LAP(tm, 3);
    }
    if (closed) {
      /* advance the block phasor by 2048 samples */
      const double *rot = reinterpret_cast<const double *>(s + oMiscF + mBlkRot);
      const double bc = rot[0], bs = rot[1];
      if (tau == 0) {               /* every reader is past the quarter loop's barriers; next read is a block away */
        double *md = reinterpret_cast<double *>(s + oMiscF + mPhasor);
        const double pr = md[0], pi = md[1];
        md[0] = pr * bc - pi * bs;
        md[1] = pr * bs + pi * bc;
      }
    } else if (s[oMiscF + mSettled] != 0.0f) {      /* written (with the phasor) before the last PairSync of quarter 3 */
      r.nco_closed = 1;
    }
    /* save this channel's dec1 plane histories (the FFT buffer overlays the planes) */
    __syncwarp();
    {
      const int i = 32 * w2 + lane;
      s[oMH + i] = s[oMix + (i >> 3) * kMixPlane + (i & 7)];
    }
    T41RX_LAP(tm, 4);
    float dq[8];
    Dec2(dq);
    __syncwarp();
    /* this channel's dec2 history for the next block: entries 232..255 of each plane */
    for (int j = lane; j < 48; j += 32) {
      const int k = 48 * w2 + j;
      s[oDH + k] = s[oD1 + (k / 24) * kD1Plane + 24 + 232 + (k % 24)];   /* words 256..279: D1W is the identity */
    }
    T41RX_LAP(tm, 5);
    AfterDec2(dq, buf, t);
    /* Codec_gain (Process.cpp:979-1016 with the clip flags never set) */
    if (tau == 0) {                   /* the gain was read at the top of this block, behind many barriers */
      int *rg = reinterpret_cast<int *>(s) + oXtra + xRfGain;
      unsigned *ct = reinterpret_cast<unsigned *>(s) + oXtra + xCodecTimer;
      unsigned timer = *ct + 1;
      if (timer > 10000) timer = 10000;
      if (timer >= 50) {
        *rg = min(*rg + 1, 15);
        timer = 0;
      }
      *ct = timer;
    }
  }

  /* level adjust + overlap-save + fast convolution + |z| + window maximum -> staging.
     dq: this warp's channel (w2) of the 8 decimated samples 8 lane .. 8 lane + 7 */
  __device__ void AfterDec2(float (&dq)[8], int buf, int t) {
    Launder();
    float *fbw = s + oMix;                                   /* FFT buffer as words */
    float2 *fb = reinterpret_cast<float2 *>(s + oMix);
    float2 *stz = reinterpret_cast<float2 *>(s + oStZ + buf * kStZBuf);
    const int o0 = 8 * lane;
    if (r.mode == kModePsk31) {           /* Process.cpp:376-387,745: raw decimated I, no filter, no AGC */
      if (w2 == 0) {
#pragma unroll
        for (int o = 0; o < 8; ++o) stz[ZPos(o0 + o)] = float2{dq[o], 0.0f};
      }
      return;
    }
    PairSync();                           /* both warps are done with the planes the FFT buffer overlays */
    if (r.mode == kModeNfm) {
      NfmDiscriminator(dq, fb);
    } else {
      /* component w2 of: first half = previous block, second half = this block (Process.cpp:498-522) */
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        const float cur = dq[o] * s[oMiscF + mVolScale];                                       /* Process.cpp:482-492 */
        float prev = s[OlaW(w2, o0 + o)];
        if (r.first_block) prev = 0.0f;                                              /* Process.cpp:498-504 */
        fbw[2 * FPos(o0 + o) + w2] = prev;
        fbw[2 * FPos(256 + o0 + o) + w2] = cur;
        s[OlaW(w2, o0 + o)] = cur;
      }
      r.first_block = 0;
    }
    PairSync();
    /* frequency-domain filter mask of the receiver's filter set */
    const float2 *mask = reinterpret_cast<const float2 *>(a.fsets[reinterpret_cast<const int *>(s)[oXtra + xFilterId]].mask);
    /* this thread's 8 mask bins (they sit at octal-digit-reversed positions after the forward passes): fetched
       now, used two passes later -- there is next to no L1 beside 227 KB of shared memory, so these come from L2 */
    float2 hm[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) hm[k] = __ldg(mask + OctRev3((unsigned)(8 * tau + k)));
    FwdPass<0>(fb, r.tw_a, tau);
    PairSync();
    FwdPass<1>(fb, r.tw_b, tau);
    PairSync();
    float2 *arow = nullptr;
    if (a.aspec && a.row_every > 0 && ((a.t0 + t) % a.row_every) == 0)
      arow = a.aspec + ((size_t)sid * a.n_rows + (a.t0 + t) / a.row_every) * kFft;
    MidPass(fb, hm, tau, arow);
    PairSync();
    InvPass<1, false>(fb, r.tw_b, tau);
    PairSync();
    InvPass<0, true>(fb, r.tw_a, tau);
    PairSync();
    T41RX_LAP(tm, 6);
    /* valid outputs 256..511, scaled by 1/512: thread tau takes i = tau + 64 o (stride-1 lanes) */
    float2 z[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const float2 v = fb[FPos(256 + tau + 64 * o)];
      z[o] = float2{v.x * (1.0f / 512.0f), v.y * (1.0f / 512.0f)};
    }
    if (r.agc_mode == 0) {                /* DSP_Fn.cpp:494-502: fixed gain, no delay line */
#pragma unroll
      for (int o = 0; o < 4; ++o) stz[ZPos(tau + 64 * o)] = z[o];
      return;
    }
    /* delayed output: zd[i] = z[i - 97]; keep the last 97 for the next block */
    float2 *zh = reinterpret_cast<float2 *>(s + oZH);
    float *E = s + vE;
    float *sta = s + oStA + buf * kStABuf;
    for (int i = tau; i < kAgcDelay; i += 64) {
      const float2 h = zh[i];
      stz[ZPos(i)] = h;
      E[i] = SqrtFast(h.x * h.x + h.y * h.y);
    }
    PairSync();
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const int i = tau + 64 * o;
      if (i + kAgcDelay < kDec) stz[ZPos(i + kAgcDelay)] = z[o];
      else zh[i + kAgcDelay - kDec] = z[o];
      E[kAgcDelay + i] = SqrtFast(z[o].x * z[o].x + z[o].y * z[o].y);
    }
    if (tau < 7) E[353 + tau] = 0.0f;
    PairSync();
    /* chunk pass: prefix / suffix maxima inside chunks of 8 (NaN magnitudes count as 0); the |z| history
       moves on and the delayed |z| goes to the AGC staging while E is complete */
    if (tau < 45) {
      const int c = tau;
      float v[8];
      const float4 u0 = *reinterpret_cast<const float4 *>(E + 8 * c), u1 = *reinterpret_cast<const float4 *>(E + 8 * c + 4);
      v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w; v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
      float p[8], sf[8];
      p[0] = fmaxf(v[0], 0.0f);
#pragma unroll
      for (int k = 1; k < 8; ++k) p[k] = fmaxf(p[k - 1], v[k]);
      sf[7] = fmaxf(v[7], 0.0f);
#pragma unroll
      for (int k = 6; k >= 0; --k) sf[k] = fmaxf(sf[k + 1], v[k]);
      *reinterpret_cast<float4 *>(s + vPfx + 8 * c) = float4{p[0], p[1], p[2], p[3]};
      *reinterpret_cast<float4 *>(s + vPfx + 8 * c + 4) = float4{p[4], p[5], p[6], p[7]};
      *reinterpret_cast<float4 *>(s + vSfx + 8 * c) = float4{sf[0], sf[1], sf[2], sf[3]};
      *reinterpret_cast<float4 *>(s + vSfx + 8 * c + 4) = float4{sf[4], sf[5], sf[6], sf[7]};
      s[vCM + c] = p[7];
      if (c < 32) {
        /* zero-state advance of the AGC's two back-averages over this chunk of 8 delayed magnitudes
           (DSP_Fn.cpp:521-522 are linear recurrences: the AGC warp applies them once per chunk) */
        const float of = s[oMiscF + mOmF], oh = s[oMiscF + mOmH];
        float pf = 0.0f, ph = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          pf = fmaf(of, pf, v[k]);
          ph = fmaf(oh, ph, v[k]);
        }
        *reinterpret_cast<float2 *>(sta + 512 + 2 * c) = float2{pf * s[oMiscF + mFbm], ph * s[oMiscF + mHbm]};
      }
    }
#pragma unroll
    for (int o = 0; o < 4; ++o) sta[tau + 64 * o] = E[tau + 64 * o];
    PairSync();
    /* F[c] = max(CM[c .. c+10]), c = 0 .. 34, written over the (consumed) |z| array */
    if (tau < 35) {
      float f = 0.0f;
#pragma unroll
      for (int k = 0; k < 11; ++k) f = fmaxf(f, s[vCM + min(tau + k, 44)]);
      s[vF + tau] = f;
    }
    PairSync();
    /* rm[i] = max(E[i+1 .. i+97]) = max(Sfx[i+1], F[((i+1) >> 3) + 1], Pfx[i+97]) */
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const int i = tau + 64 * o;
      sta[256 + i] = fmaxf(fmaxf(s[vSfx + i + 1], s[vF + ((i + 1) >> 3) + 1]), s[vPfx + i + 97]);
    }
    T41RX_LAP(tm, 7);
  }

  /* NFM: discriminator on the decimated samples, then the audio goes through the filter as a real
     signal (Demod.cpp:220-235, Process.cpp:716-727,765-779).  The two warps hold I and Q: exchange through
     the second half of the FFT buffer. */
  __device__ __forceinline__ void NfmDiscriminator(float (&dq)[8], float2 *fb) {
    float *fbw = reinterpret_cast<float *>(fb);
    const float kq = 0.340447550238101026565118445432744920253753662109375f;
    const int o0 = 8 * lane;
#pragma unroll
    for (int o = 0; o < 8; ++o) fbw[2 * FPos(256 + o0 + o) + w2] = dq[o];
    PairSync();
    const int i0 = 4 * tau;
    float2 cur[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) cur[o] = fb[FPos(256 + i0 + o)];
    float2 prev = float2{s[oMiscF + mNfmI], s[oMiscF + mNfmQ]};
    if (tau > 0) prev = fb[FPos(256 + i0 - 1)];
    float outv[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const float I = cur[o].x, Q = cur[o].y;
      const float den = I * I + Q * Q;
      float out;
      if (i0 + o == 0) {
        const float num = I * (Q - prev.y) - Q * (I - prev.x);
        out = kq * num / den;
      } else {
        const float num = Q * prev.x - I * prev.y;
        out = kq * num / den;
        out = (1.0f < out) ? 1.0f : out;          /* limiter skips index 0 (B5) */
        out = (-1.0f > out) ? -1.0f : out;
      }
      outv[o] = out;
      prev = cur[o];
    }
    PairSync();
    if (tau == 31) {                               /* "last sample" = complex sample 127 (B4) */
      s[oMiscF + mNfmI] = cur[3].x;
      s[oMiscF + mNfmQ] = cur[3].y;
    }
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      fb[FPos(i0 + o)] = float2{s[OlaW(0, i0 + o)], 0.0f};
      fb[FPos(256 + i0 + o)] = float2{outv[o], 0.0f};
      s[OlaW(0, i0 + o)] = outv[o];
    }
  }

  /* ---------------- back end ---------------- */
  __device__ void BackEnd(int t, int buf) {
    Launder();
    const StreamCfg &cf = a.cfg[sid];
    StreamState &st = a.st[sid];
    const float2 *stz = reinterpret_cast<const float2 *>(s + oStZ + buf * kStZBuf);
    const float *volts = s + oStA + buf * kStABuf + 256;
    float *aud = s + vAudF;
    /* gain and the sample-parallel part of the demodulators: thread tau takes i = tau + 64 o */
    {
      float2 dem[4];
      GainedSamples(cf, stz, volts, dem);
      if (a.psk_bits || a.psk_chars || r.psk_enable) PskTap(t, dem[0], cf, st);
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        /* AM: alpha-beta magnitude (Process.cpp:697-699); USB / LSB / NFM / PSK31: real part (:616-624,688-695) */
        aud[24 + tau + 64 * o] = (r.mode == kModeAm) ? AlphaBetaMag(dem[o].x, dem[o].y) : dem[o].x;
      }
      if (r.mode == kModeSam) {
        /* the PLL lane needs the 256 gained samples in order, and arm_sin_f32's table within reach */
        float2 *zs = reinterpret_cast<float2 *>(s + oMix);
#pragma unroll
        for (int o = 0; o < 4; ++o) zs[tau + 64 * o] = dem[o];
        for (int i = tau; i < 513; i += 64) s[oMix + 2 * kDec + i] = __ldg(a.sin_table + i);
      }
    }
    if (tau < 23) aud[1 + tau] = s[oIH + tau];
    if (tau >= 32 && tau < 39) s[vI1 + 1 + (tau - 32)] = s[oIH + 24 + (tau - 32)];
    PairSync();
    if (r.mode == kModeSam) {
      if (tau == 0) SamPllLane(s + oMix + 2 * kDec, a.sam_consts, st, reinterpret_cast<const float2 *>(s + oMix), aud + 24);
      PairSync();
    }
    if (r.mode == kModeAm) {
      /* the detector's recurrences are blocked scans over one warp (8 samples per lane), in place */
      if (w2 == 0) {
        float m[8], au[8];
        const float4 m0 = *reinterpret_cast<const float4 *>(aud + 24 + 8 * lane), m1 = *reinterpret_cast<const float4 *>(aud + 24 + 8 * lane + 4);
        m[0] = m0.x; m[1] = m0.y; m[2] = m0.z; m[3] = m0.w; m[4] = m1.x; m[5] = m1.y; m[6] = m1.z; m[7] = m1.w;
        AmDetect(m, au, st);
        *reinterpret_cast<float4 *>(aud + 24 + 8 * lane) = float4{au[0], au[1], au[2], au[3]};
        *reinterpret_cast<float4 *>(aud + 24 + 8 * lane + 4) = float4{au[4], au[5], au[6], au[7]};
      }
      PairSync();
    }
    if (r.eq_on) ReceiveEqPair(s, a.eq_coeffs, cf, st, aud, tau, bar_id);
    if (r.nr_lms || r.anr_notch) {
      /* Process.cpp:841-865: LMS noise reduction (Xanr's output is dropped: the audio is float_buffer_L x 1.5, the
         adaptive state still advances), then the automatic notch (the error signal replaces the audio) */
      if (w2 == 0) {
        if (r.nr_lms) {
          XanrWarp(s, st, aud + 24, lane, false);
          for (int i = lane; i < kDec; i += 32) aud[24 + i] *= 1.5f;
          __syncwarp();
        }
        if (r.anr_notch) XanrWarp(s, st, aud + 24, lane, true);
      }
      PairSync();
    }
    if (r.cw_filter) {
      /* Process.cpp:878-914: the CW receive state's audio low-pass; one lane (6 chained biquads per sample) */
      if (tau == 0) CwFilterFast(aud + 24, a.cw_coeffs + 30 * cf.cw_filter, st.cw_state[cf.cw_filter]);
      PairSync();
    }
    T41RX_LAP(tm, 8);
    Interp1();
    PairSync();
    T41RX_LAP(tm, 9);
    if (tau < 23) s[oIH + tau] = aud[24 + 233 + tau];
    Interp2(t);
    PairSync();
    if (tau < 7) s[oIH + 24 + tau] = s[vI1 + 8 + 505 + tau];
    T41RX_LAP(tm, 10);
  }

  /* AGC gain from volts (DSP_Fn.cpp:628) or the fixed gain (DSP_Fn.cpp:494-502) applied to the delayed
     samples i = tau + 64 o */
  __device__ __forceinline__ void GainedSamples(const StreamCfg &cf, const float2 *stz, const float *volts,
                                                float2 (&dem)[4]) const {
#pragma unroll
    for (int o = 0; o < 4; ++o) dem[o] = stz[ZPos(tau + 64 * o)];
    if (r.mode == kModePsk31) return;
    if (r.agc_mode == 0) {
#pragma unroll
      for (int o = 0; o < 4; ++o) dem[o] = float2{dem[o].x * s[oMiscF + mFixedGain], dem[o].y * s[oMiscF + mFixedGain]};
      return;
    }
    const float inv_in = s[oMiscF + mInvIn], tgt = s[oMiscF + mTarget], slope = s[oMiscF + mSlope];
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const float v = volts[tau + 64 * o];
      const float lg = Log10Fast(inv_in * v);
      const float clipped = (0.0f < lg) ? 0.0f : lg;
      const float mult = __fdividef(tgt - slope * clipped, v);    /* 2 ulp: far inside the tolerance, a fifth of the instructions */
      dem[o] = float2{dem[o].x * mult, dem[o].y * mult};
    }
  }

  /* arm_fir_interpolate_f32, L = 2, 48 taps (Process.cpp:917): 4 inputs per thread */
  __device__ __forceinline__ void Interp1() {
    const float *aud = s + vAudF;
    const float *tp = s + oTapsF + 74;
    float w[28];
    const float4 *src = reinterpret_cast<const float4 *>(aud + 4 * tau);
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      const float4 v = src[k];
      w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
    }
    /* packed FP32: (phase 0, phase 1) of an input = x * (c[2k+1], c[2k]) summed over k */
    P2 acc[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
    for (int k = 0; k < 24; ++k) {
      const float2 c = *reinterpret_cast<const float2 *>(tp + 2 * k);
      const P2 cc = Pack2(c.y, c.x);           /* phase 0: c[(L-1) + k L], phase 1: c[0 + k L] */
#pragma unroll
      for (int o = 0; o < 4; ++o)
        acc[o] = Fma2(Dup(w[o + 1 + k]), cc, acc[o]);   /* input n - 23 + k, n = 4 tau + o, lives at word 4 tau + o + 1 + k */
    }
    ulonglong2 *i1 = reinterpret_cast<ulonglong2 *>(s + vI1 + 8 + 8 * tau);
    i1[0] = ulonglong2{acc[0], acc[1]};
    i1[1] = ulonglong2{acc[2], acc[3]};
  }

  /* arm_fir_interpolate_f32, L = 4, 32 taps + volume (Process.cpp:919-931): 2 x 4 inputs per thread.
     Packed FP32: the four phases of an input are two (phase 0, phase 1) / (phase 2, phase 3) pairs; out[4 n + p] =
     sum_k x[n - 7 + k] c[(3 - p) + 4 k], volume folded into the taps. */
  __device__ __forceinline__ void Interp2(int t) {
    const float *tp = s + oTapsF + 122;
    const float vol = s[oMiscF + mVolume];
    P2 c01[8], c23[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float2 lo = *reinterpret_cast<const float2 *>(tp + 4 * k), hi = *reinterpret_cast<const float2 *>(tp + 4 * k + 2);
      c01[k] = Pack2(hi.y * vol, hi.x * vol);                              /* phases 0, 1: c[4k+3], c[4k+2] */
      c23[k] = Pack2(lo.y * vol, lo.x * vol);                              /* phases 2, 3: c[4k+1], c[4k]   */
    }
    float4 *dst = reinterpret_cast<float4 *>(a.audio + ((size_t)sid * a.t_stride + t) * kBlock);
    uint2 *dst16 = reinterpret_cast<uint2 *>(a.audio16 + ((size_t)sid * a.t_stride + t) * kBlock);
#pragma unroll 1
    for (int rr = 0; rr < 2; ++rr) {
      const int n0 = 4 * tau + 256 * rr;
      P2 w[12];
      const float4 *src = reinterpret_cast<const float4 *>(s + vI1 + n0);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float4 v = src[k];
        w[4 * k] = Pack2(v.x, v.x); w[4 * k + 1] = Pack2(v.y, v.y); w[4 * k + 2] = Pack2(v.z, v.z); w[4 * k + 3] = Pack2(v.w, v.w);
      }
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        P2 a01 = 0ull, a23 = 0ull;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          a01 = Fma2(w[o + 1 + k], c01[k], a01);     /* input n - 7 + k at word n + 1 + k */
          a23 = Fma2(w[o + 1 + k], c23[k], a23);
        }
        float4 o4;
        Unpack2(a01, o4.x, o4.y);
        Unpack2(a23, o4.z, o4.w);
        if (kQ15) dst16[n0 + o] = uint2{PackQ15(o4.x, o4.y), PackQ15(o4.z, o4.w)};
        else dst[n0 + o] = o4;
      }
    }
  }

  /* AM: alpha-beta magnitude, 1-pole DC removal, 1-stage DF1 low-pass (Process.cpp:697-707) as blocked
     linear scans over the lanes (8 samples per lane) */
  __device__ __forceinline__ void AmDetect(const float (&m)[8], float (&au)[8], StreamState &st) {
    /* w[i] = m[i] + 0.99 w[i-1] */
    const float g = 0.99f;
    float w[8];
    {
      float acc = 0.0f;
#pragma unroll
      for (int o = 0; o < 8; ++o) { acc = fmaf(g, acc, m[o]); w[o] = acc; }
    }
    const float wold = s[oMiscF + mAmWold];
    float g8 = g * g; g8 *= g8; g8 *= g8;       /* 0.99^8 */
    float e = w[7];
    if (lane == 0) e = fmaf(g8, wold, e);
    {
      float mult = g8, v = e, tt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        tt = __shfl_up_sync(kFull, v, d);
        if (lane >= d) v = fmaf(mult, tt, v);
        mult *= mult;
      }
      e = v;
    }
    float cin = __shfl_up_sync(kFull, e, 1);
    if (lane == 0) cin = wold;
    const float wend = __shfl_sync(kFull, e, 31);
    float x[8];
    {
      float pw = g, prev = cin;
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        const float tw_ = fmaf(pw, cin, w[o]);
        x[o] = tw_ - prev;
        prev = tw_;
        pw *= g;
      }
    }
    /* biquad: y[i] = b0 x[i] + b1 x[i-1] + b2 x[i-2] + a1 y[i-1] + a2 y[i-2] */
    const float b0 = s[oMiscF + mAmLp], b1 = s[oMiscF + mAmLp + 1], b2 = s[oMiscF + mAmLp + 2], a1 = s[oMiscF + mAmLp + 3],
                a2 = s[oMiscF + mAmLp + 4];
    float xm1 = __shfl_up_sync(kFull, x[7], 1), xm2 = __shfl_up_sync(kFull, x[6], 1);
    if (lane == 0) { xm1 = s[oMiscF + mAmX1]; xm2 = s[oMiscF + mAmX2]; }
    float y[8];
    {
      float p1 = 0.0f, p2 = 0.0f, q1 = xm1, q2 = xm2;
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        float f = b0 * x[o];
        f = fmaf(b1, q1, f);
        f = fmaf(b2, q2, f);
        const float yy = fmaf(a1, p1, fmaf(a2, p2, f));
        y[o] = yy;
        p2 = p1; p1 = yy;
        q2 = q1; q1 = x[o];
      }
    }
    /* homogeneous responses h1 (y[-1] = 1, y[-2] = 0) and h2 (y[-1] = 0, y[-2] = 1) over 8 steps */
    float h1[8], h2[8];
    {
      float u1 = 1.0f, u2 = 0.0f, v1 = 0.0f, v2 = 1.0f;
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        const float un = a1 * u1 + a2 * u2, vn = a1 * v1 + a2 * v2;
        h1[o] = un; h2[o] = vn;
        u2 = u1; u1 = un;
        v2 = v1; v1 = vn;
      }
    }
    /* chunk transfer matrix M = [[h1[7], h2[7]], [h1[6], h2[6]]]; scan of (y[7], y[6]) */
    float m00 = h1[7], m01 = h2[7], m10 = h1[6], m11 = h2[6];
    float s1 = y[7], s2 = y[6];
    if (lane == 0) {
      const float y1 = s[oMiscF + mAmY1], y2 = s[oMiscF + mAmY2];
      s1 += m00 * y1 + m01 * y2;
      s2 += m10 * y1 + m11 * y2;
    }
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const float t1 = __shfl_up_sync(kFull, s1, d), t2 = __shfl_up_sync(kFull, s2, d);
      if (lane >= d) {
        s1 += m00 * t1 + m01 * t2;
        s2 += m10 * t1 + m11 * t2;
      }
      const float n00 = m00 * m00 + m01 * m10, n01 = m00 * m01 + m01 * m11;
      const float n10 = m10 * m00 + m11 * m10, n11 = m10 * m01 + m11 * m11;
      m00 = n00; m01 = n01; m10 = n10; m11 = n11;
    }
    float c1 = __shfl_up_sync(kFull, s1, 1), c2 = __shfl_up_sync(kFull, s2, 1);
    if (lane == 0) { c1 = s[oMiscF + mAmY1]; c2 = s[oMiscF + mAmY2]; }
#pragma unroll
    for (int o = 0; o < 8; ++o) au[o] = y[o] + h1[o] * c1 + h2[o] * c2;
    __syncwarp();
    if (lane == 31) {
      s[oMiscF + mAmWold] = wend;
      s[oMiscF + mAmX1] = x[7];
      s[oMiscF + mAmX2] = x[6];
      s[oMiscF + mAmY1] = au[7];
      s[oMiscF + mAmY2] = au[6];
    }
  }


  __device__ void PskTap(int t, float2 d0, const StreamCfg &cf, StreamState &st) {
    if (tau != 0) return;
    int8_t bit_out = -1;
    uint8_t char_out = 0;
    if (cf.psk31_enable && r.mode != kModeNfm && r.mode != kModePsk31) {
      if (st.psk_block_count % 3u == 0u) {
        const double pi_d = 3.1415926535897932384626433832795;
        const float phase = Atan2Approx(d0.y, d0.x);
        float dphase = phase - st.psk_last_phase;
        while ((double)dphase < -pi_d) dphase = (float)((double)dphase + 2 * pi_d);
        while ((double)dphase >= pi_d) dphase = (float)((double)dphase - 2 * pi_d);
        const uint8_t bit = (((double)dphase > (pi_d / 2)) || ((double)dphase < (-pi_d / 2))) ? 0 : 1;
        st.psk_last_phase = phase;
        bit_out = (int8_t)bit;
        unsigned long long shr = (st.psk_shr << 1) | (unsigned long long)bit;
        if ((shr & 0xFFFull) != 0) {
          for (int i = 0; i < 128; ++i) {
            const uint32_t e = __ldg(a.varicode + i);
            const unsigned long long want = ((unsigned long long)(e & 0xFFFFu)) << 2;
            const unsigned nbits = (((e >> 16) & 0xFFu) + 4u) & 63u;
            const unsigned long long keep = (nbits == 0) ? 0ull : (~0ull >> (64u - nbits));
            if (want == (shr & keep)) {
              shr = 0;
              char_out = (uint8_t)(e >> 24);
              break;
            }
          }
        }
        st.psk_shr = shr;
      }
      st.psk_block_count++;
    }
    const size_t o = (size_t)sid * a.t_stride + t;
    if (a.psk_bits) a.psk_bits[o] = bit_out;
    if (a.psk_chars) a.psk_chars[o] = char_out;
  }
};

/* ------------------------------------------------------------------ */
/* AGC warp: lane = receiver (DSP_Fn.cpp:504-631)                       */
/* ------------------------------------------------------------------ */
struct AgcLane {
  /* constants */
  float fbm, omfbm, hbm, omhbm, attack, decay, fdecay, hdecay, pop, hlevel, minv;
  float om8f, om8h;      /* onemfast_backmult^8, onemhang_backmult^8 */
  int hload, henable;
  /* state */
  float fast, hang, v, save, rm;
  int hc, state, dtype, action;

  __device__ void Load(const StreamCfg &cf, const StreamState &st) {
    fbm = cf.agc.fast_backmult; omfbm = cf.agc.onemfast_backmult;
    hbm = cf.agc.hang_backmult; omhbm = cf.agc.onemhang_backmult;
    attack = cf.agc.attack_mult; decay = cf.agc.decay_mult; fdecay = cf.agc.fast_decay_mult;
    hdecay = cf.agc.hang_decay_mult; pop = cf.agc.pop_ratio; hlevel = cf.agc.hang_level;
    minv = cf.agc.min_volts;
    om8f = omfbm * omfbm; om8f *= om8f; om8f *= om8f;
    om8h = omhbm * omhbm; om8h *= om8h; om8h *= om8h;
    hload = cf.agc.hang_counter_load; henable = cf.agc.hang_enable;
    fast = st.agc_fast_back; hang = st.agc_hang_back; v = st.agc_volts; save = st.agc_save_volts;
    rm = st.agc_ring_max;
    hc = st.agc_hang_counter; state = st.agc_state; dtype = st.agc_decay_type; action = st.agc_action;
  }
  __device__ void Store(StreamState &st) const {
    st.agc_fast_back = fast; st.agc_hang_back = hang; st.agc_volts = v; st.agc_save_volts = save;
    st.agc_ring_max = rm;
    st.agc_hang_counter = hc; st.agc_state = state; st.agc_decay_type = dtype; st.agc_action = action;
  }

  /* one sample of the envelope state machine; returns volts */
  __device__ __forceinline__ float Step(float abs_out, float r) {
    fast = fbm * abs_out + omfbm * fast;
    hang = hbm * abs_out + omhbm * hang;
    rm = r;
    if (hc > 0) --hc;
    const float d = r - v;
    if (r >= v) {
      if (state >= 2) save = v;
      state = 0;
      v += d * attack;
    } else if (state == 3) {
      v = fmaf(d * decay, 0.05f, v);      /* reference: double product and sum, then float */
    } else if (state == 0) {
      if (v > pop * fast) {
        state = 1;
        v += d * fdecay;
      } else if (henable && (hang > hlevel)) {
        state = 2;
        hc = hload;
        dtype = 1;
      } else {
        state = 3;
        v += d * decay;
        dtype = 0;
      }
    } else if (state == 1) {
      if (v > save) {
        v += d * fdecay;
      } else if (hc > 0) {
        state = 2;
      } else if (dtype == 0) {
        state = 3;
        v += d * decay;
      } else {
        state = 4;
        v += d * hdecay;
      }
    } else if (state == 2) {
      if (hc == 0) {
        state = 4;
        v += d * hdecay;
      }
    } else {
      v += d * hdecay;
    }
    action = (v < minv) ? 0 : 1;
    v = (v < minv) ? minv : v;
    return v;
  }
};

/* one block of one receiver per lane.  sta: |z| delayed [256] | window max [256] (overwritten by volts) |
 * per-chunk zero-state advances (PF, PH)[32] of the two back-averages.
 *
 * Almost every sample CONTINUES the state the envelope detector is in (attack, fast decay, hang, slow decay, hang
 * decay), where the update is v <- max(v + (r - v) c, min_volts) with a per-state constant and no branch.  The
 * warp runs 8 samples at a time speculatively on that form (all lanes), and a lane re-runs the chunk through the
 * exact per-sample state machine (Step) only when it saw a transition between states. */
__device__ __forceinline__ void AgcBlock(AgcLane &g, float *sta, bool active) {
  constexpr int kC = 8;
  /* window maxima and back-average advances of the chunk being processed; the next chunk's are fetched
     while this one runs (the recurrence below is pure latency: nothing else can hide the loads) */
  float4 r0 = float4{0, 0, 0, 0}, r1 = r0;
  float2 pfh = float2{0.0f, 0.0f};
  if (active) {
    r0 = *reinterpret_cast<const float4 *>(sta + 256);
    r1 = *reinterpret_cast<const float4 *>(sta + 256 + 4);
    pfh = *reinterpret_cast<const float2 *>(sta + 512);
  }
#pragma unroll 1
  for (int i0 = 0; i0 < kDec; i0 += kC) {
    const float rm[kC] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
    const float2 pf = pfh;
    if (active && i0 + kC < kDec) {
      r0 = *reinterpret_cast<const float4 *>(sta + 256 + i0 + kC);
      r1 = *reinterpret_cast<const float4 *>(sta + 256 + i0 + kC + 4);
      pfh = *reinterpret_cast<const float2 *>(sta + 512 + 2 * (i0 / kC + 1));
    }
    /* speculative quiet path: state 3: v + ((r - v) decay) 0.05 -> one rounded constant (the step is ~1e-6 v,
       so the difference from the reference's rounding is ~1e-13 v); state 4: v + (r - v) hang_decay; state 2
       with the hang counter not expiring inside the chunk: v unchanged */
    const int st = g.state;
    /* continuation steps of every state: 0 = attack while the window maximum stays at or above volts; 1 = fast
       decay while volts stays above the saved level; 2 = hang; 3 / 4 = slow / hang decay; all have the form
       v <- max(v + (r - v) c, min_volts).  Only the transitions between them need the full state machine. */
    const bool att = (st == 0);
    const float c = att ? g.attack : ((st == 1) ? g.fdecay : ((st == 3) ? g.decay * 0.05f : ((st == 4) ? g.hdecay : 0.0f)));
    const float floor1 = (st == 1) ? g.save : -3.0e38f;       /* state 1 continues only while v > save */
    bool ok = (st != 2) || (g.hc > kC);
    float v = g.v, last = g.v;
    float vo[kC];
#pragma unroll
    for (int k = 0; k < kC; ++k) {
      ok = ok && ((rm[k] >= v) == att) && (v > floor1);
      last = fmaf(rm[k] - v, c, v);
      v = fmaxf(last, g.minv);
      vo[k] = v;
    }
    /* per lane, not per warp: a receiver's result must not depend on whether a neighbour in its CTA took a
       transition in this chunk (the quiet form and Step round differently) */
    if (ok || !active) {
      g.v = v;
      g.fast = fmaf(g.om8f, g.fast, pf.x);
      g.hang = fmaf(g.om8h, g.hang, pf.y);
      g.rm = rm[kC - 1];
      g.hc = max(g.hc - kC, 0);
      g.action = (last < g.minv) ? 0 : 1;
    } else if (active) {
#ifdef T41RX_FAST_TIMING
      if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) g_fast_cycles[20] += 1;
#endif
      float ab[kC];
#pragma unroll
      for (int k = 0; k < kC; k += 4) {
        const float4 a4 = *reinterpret_cast<const float4 *>(sta + i0 + k);
        ab[k] = a4.x; ab[k + 1] = a4.y; ab[k + 2] = a4.z; ab[k + 3] = a4.w;
      }
#pragma unroll 1
      for (int k = 0; k < kC; ++k) {
        /* select ab[k], rm[k] without dynamic register indexing */
        float a_ = ab[0], r_ = rm[0];
#pragma unroll
        for (int j = 1; j < kC; ++j) { if (k == j) { a_ = ab[j]; r_ = rm[j]; } }
        const float vv = g.Step(a_, r_);
#pragma unroll
        for (int j = 0; j < kC; ++j) { if (k == j) vo[j] = vv; }
      }
    }
    if (active) {
      *reinterpret_cast<float4 *>(sta + 256 + i0) = float4{vo[0], vo[1], vo[2], vo[3]};
      *reinterpret_cast<float4 *>(sta + 256 + i0 + 4) = float4{vo[4], vo[5], vo[6], vo[7]};
    }
  }
}

/* ------------------------------------------------------------------ */
/* kernel body                                                          */
/* ------------------------------------------------------------------ */
template <bool kQ15>
__device__ __forceinline__ void StreamKernelBody(const LaunchArgs &a, int G, float *smem) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s0 = blockIdx.x * G;
  const int ng = min(G, a.n_streams - s0);
  const int T = a.n_blocks;
  /* block j's front ends -> AGC: full[j & 1] (every thread of every live pair arrives);
     AGC -> block j's back ends: done[j & 1] (the AGC warp's 32 lanes arrive).  A receiver pair may run up
     to one block ahead of the others; the double-buffered hand-off areas allow exactly that. */
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + G * kSlotF);
  uint64_t *done = full + 2;
  if (threadIdx.x == 0) {
    MbarInit(full + 0, 64u * ng);
    MbarInit(full + 1, 64u * ng);
    MbarInit(done + 0, 32u);
    MbarInit(done + 1, 32u);
  }
  __syncthreads();
  /* warp 0 = the AGC warp (measured: the latency-critical warp does better with the lowest warp id),
     warps 1 + 2 p, 2 + 2 p = receiver pair p */
  const int pw = warp - 1;
  if (warp != 0) {
    /* ---- receiver pair ---- */
    const int pair = pw >> 1;
    const bool live = pair < ng;
    if (!live) return;
    const int sid = a.stream_ids ? __ldg(a.stream_ids + s0 + pair) : a.stream_base + s0 + pair;
    RxPair<kQ15> w(a, smem + pair * kSlotF, sid, lane, pw & 1, 1 + pair);
    w.LoadState();
    w.IssueQuarter(0, 0);
    w.tm.Start(blockIdx.x == 0 && pw == 0 && lane == 0, 0);
    for (int k = 0; k < T + 2; ++k) {
      /* the last 128 I samples of block k (see FrontEnd) are fetched before the back end: their HBM
         latency hides behind it */
      float4 tu = float4{0, 0, 0, 0}, tv = tu;
      if (k < T && (pw & 1) == 0) {
        if (kQ15) {                    /* only the I components (.x, .z) are used */
          const uint4 v = __ldg(reinterpret_cast<const uint4 *>(w.BlockIq16(k) + 2 * (kBlock - 4 * (lane + 1))));
          tu = float4{(float)(short)(v.x & 0xffffu) * (1.0f / 32768.0f), 0.0f, (float)(short)(v.y & 0xffffu) * (1.0f / 32768.0f), 0.0f};
          tv = float4{(float)(short)(v.z & 0xffffu) * (1.0f / 32768.0f), 0.0f, (float)(short)(v.w & 0xffffu) * (1.0f / 32768.0f), 0.0f};
        } else {
          const float4 *p = reinterpret_cast<const float4 *>(w.BlockIq(k) + 2 * (kBlock - 4 * (lane + 1)));
          tu = __ldg(p);
          tv = __ldg(p + 1);
        }
      }
      if (k >= 2) {
        MbarWait(done + (k & 1), (unsigned)(((k - 2) >> 1) & 1));
        T41RX_LAP(w.tm, 12);
        w.BackEnd(k - 2, k & 1);
      }
      if (k < T) {
        w.FrontEnd(k, k & 1, tu, tv);
        MbarArrive(full + (k & 1));
      }
      T41RX_LAP(w.tm, 11);
    }
    w.StoreState();
  } else {
    /* ---- AGC warp ---- */
    AgcLane g;
    const bool mine = lane < ng;
    bool active = false;
    const int sid = mine ? (a.stream_ids ? __ldg(a.stream_ids + s0 + lane) : a.stream_base + s0 + lane) : 0;
    if (mine) {
      const StreamCfg &cf = a.cfg[sid];
      g.Load(cf, a.st[sid]);
      active = (cf.mode != kModePsk31) && (cf.agc_mode != 0);
    }
    float *slot = smem + (mine ? lane : 0) * kSlotF;
    SectionTimer tm;
    tm.Start(blockIdx.x == 0 && lane == 0, 16);
    for (int j = 0; j < T; ++j) {
      MbarWait(full + (j & 1), (unsigned)((j >> 1) & 1));
      T41RX_LAP(tm, 1);
      AgcBlock(g, slot + oStA + (j & 1) * kStABuf, active);
      MbarArrive(done + (j & 1));
      T41RX_LAP(tm, 0);
    }
    if (mine && active) g.Store(a.st[sid]);
  }
}

}  // namespace fast
}  // namespace t41rx
#endif
