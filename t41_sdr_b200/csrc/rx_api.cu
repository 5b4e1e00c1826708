/*
 * rx_api.cu — libt41rx.so: the fused sm_100a receive-chain kernel and the C-ABI around it
 * (include/t41rx.h).  Host side = parameter cache + control-path design (rx_design.cpp) +
 * device memory / stream plumbing.  There is no CPU processing path in this library.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <new>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/t41rx.h"
#include "rx_design.h"
#include "rx_host.h"
#include "rx_launch.h"
#include "rx_phases.cuh"
#include "rx_tables_data.h"

namespace t41rx {

/* ------------------------------------------------------------------ */
/* the kernel                                                          */
/* ------------------------------------------------------------------ */
#ifdef T41RX_PHASE_TIMING
__device__ unsigned long long g_phase_cycles[128];
#endif

__global__ void __launch_bounds__(kNT, 8 / kG) t41rx_fused_rx_kernel(const LaunchArgs a) {
  extern __shared__ __align__(16) float smem[];
  Cta c;
  c.a = a;
  c.smem = smem;
  c.s0 = blockIdx.x * kG;
  c.ng = min(kG, a.n_streams - c.s0);
  c.t = 0;
  c.row = 0;
  c.row_idx = 0;
  c.rows_only = 0;
  c.casc_warp = 0;
  c.dc_carried = 0;
  const int tid = threadIdx.x;
  PhCtaInit(c, tid);
  __syncthreads();
  PhStateIn(c, tid);
  __syncthreads();
  for (int t = 0; t < a.n_blocks; ++t) {
    c.t = t;
    c.row = (a.row_every > 0) && ((a.t0 + t) % a.row_every == 0);
    c.row_idx = c.row ? (a.t0 + t) / a.row_every : 0;
#ifdef T41RX_PHASE_TIMING
    /* developer build only: cycles per phase of CTA 0 (work and the wait at the barrier) */
    int phase_no = 0;
#define T41RX_KPHASE(stmt)                                                                   \
  do {                                                                                       \
    const long long t0_ = clock64();                                                         \
    stmt;                                                                                    \
    const long long t1_ = clock64();                                                         \
    __syncthreads();                                                                         \
    const long long t2_ = clock64();                                                         \
    if (blockIdx.x == 0 && tid == 0) {                                                       \
      g_phase_cycles[2 * phase_no] += (unsigned long long)(t2_ - t0_);                       \
      g_phase_cycles[2 * phase_no + 1] += (unsigned long long)(t1_ - t0_);                   \
    }                                                                                        \
    ++phase_no;                                                                              \
  } while (0)
#else
#define T41RX_KPHASE(stmt) \
  do {                     \
    stmt;                  \
    __syncthreads();       \
  } while (0)
#endif
    T41RX_BLOCK_SCHEDULE(T41RX_KPHASE)
#undef T41RX_KPHASE
  }
  PhStateOut(c, tid);
}

/* The same chain as three kernels (rx_phases.cuh, "Split form of the chain"): the sample-parallel phases up to the AGC
   look-ahead, the serial stages with THREAD = RECEIVER, the sample-parallel phases behind the demodulator.  Bit-identical
   to t41rx_fused_rx_kernel; the default route of every receiver that needs the bit-exact chain. */
#define T41RX_KPHASE(stmt) \
  do {                     \
    stmt;                  \
    __syncthreads();       \
  } while (0)
__global__ void __launch_bounds__(kNT, 8 / kG) t41rx_exact_front_kernel(const LaunchArgs a) {
  extern __shared__ __align__(16) float smem[];
  Cta c;
  c.a = a;
  c.smem = smem;
  c.s0 = blockIdx.x * kG;
  c.ng = min(kG, a.n_streams - c.s0);
  c.t = 0;
  c.row = 0;
  c.row_idx = 0;
  c.rows_only = 0;
  c.casc_warp = 0;
  c.dc_carried = 0;
  const int tid = threadIdx.x;
  PhCtaInit(c, tid);
  __syncthreads();
  PhStateIn(c, tid);
  __syncthreads();
  for (int t = 0; t < a.n_blocks; ++t) {
    c.t = t;
    c.row = (a.row_every > 0) && ((a.t0 + t) % a.row_every == 0);
    c.row_idx = c.row ? (a.t0 + t) / a.row_every : 0;
#ifdef T41RX_PHASE_TIMING
    /* developer build only: cycles per phase of CTA 0, the slots the fused kernel uses (it does not run beside this one) */
    int phase_no = 0;
#define T41RX_KPHASE_T(stmt)                                                                 \
  do {                                                                                       \
    const long long t0_ = clock64();                                                         \
    stmt;                                                                                    \
    const long long t1_ = clock64();                                                         \
    __syncthreads();                                                                         \
    const long long t2_ = clock64();                                                         \
    if (blockIdx.x == 0 && tid == 0) {                                                       \
      g_phase_cycles[2 * phase_no] += (unsigned long long)(t2_ - t0_);                       \
      g_phase_cycles[2 * phase_no + 1] += (unsigned long long)(t1_ - t0_);                   \
    }                                                                                        \
    ++phase_no;                                                                              \
  } while (0)
    T41RX_FRONT_SCHEDULE(T41RX_KPHASE_T)
#undef T41RX_KPHASE_T
#else
    T41RX_FRONT_SCHEDULE(T41RX_KPHASE)
#endif
  }
  PhFrontStateOut(c, tid);
}

/* The serial stages as a pipeline of three warps over chunks of kSerU samples, LANE = RECEIVER (32 receivers per CTA):
   warp 0 the AGC envelope state machine, warp 1 the gain from volts (its FP64 division and logarithm are off every
   recurrence), warp 2 the demodulator (SAM PLL / AM detector) and the PSK31 tap.  Each stage is one long dependent
   chain per receiver, so a warp issues an instruction every few clocks at best: three warps on three schedulers run
   the chains side by side.  Hand-over through double-buffered shared memory with named barriers (producer arrives on
   "full", consumer arrives on "empty").  The arithmetic is SerAgc / SerGain / SerDemod of rx_phases.cuh, the same
   objects the host emulation steps sample by sample. */
constexpr int kSerialThreads = 96;
constexpr int kSerialLanes = 32;
constexpr int kSerU = 8;
__device__ __forceinline__ void NamedSync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void NamedArrive(int id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }

#ifndef T41RX_SER_UNROLL
#define T41RX_SER_UNROLL 4
#endif
#define T41RX_SER_PRAGMA_(x) _Pragma(#x)
#define T41RX_SER_PRAGMA(x) T41RX_SER_PRAGMA_(x)
#define T41RX_SER_LOOP T41RX_SER_PRAGMA(unroll T41RX_SER_UNROLL)
__global__ void __launch_bounds__(kSerialThreads) t41rx_exact_serial_kernel(const LaunchArgs a) {
  __shared__ float sin_tab[513];
  __shared__ float2 inbuf[2][kSerU][kSerialLanes];     /* each loading stage's own staging of its global inputs */
  __shared__ float vbuf[2][kSerU][kSerialLanes];
  __shared__ float2 dbuf[2][kSerU][kSerialLanes];
  for (int i = threadIdx.x; i < 513; i += kSerialThreads) sin_tab[i] = __ldg(a.sin_table + i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * kSerialLanes + lane;
  const bool live = r < a.n_streams;
  const int sid = live ? (a.stream_ids ? __ldg(a.stream_ids + r) : a.stream_base + r) : 0;
  const StreamCfg &cf = a.cfg[sid];
  StreamState &st = a.st[sid];
  const bool agc_on = live && UsesFilter(cf.mode) && cf.agc_mode != 0;
  const size_t n = (size_t)a.n_streams;
  const int n_chunks = a.n_blocks * (kDec / kSerU);
  /* named barriers 1..8: full_v[b] = 1 + b, empty_v[b] = 3 + b, full_d[b] = 5 + b, empty_d[b] = 7 + b.
     The per-sample loops stay rolled (T41RX_SER_UNROLL): with one warp per stage nothing hides an instruction-cache
     miss, and the unrolled bodies of the three stages do not fit the cache together. */
  const float2 *in2 = reinterpret_cast<const float2 *>(a.ser_in) + 2 * (size_t)(live ? r : 0);   /* + 2 n per sample */
  if (warp == 0) {
    SerAgc agc;
    agc.Load(cf, st);
    float2 nx[kSerU];
#pragma unroll
    for (int k = 0; k < kSerU; ++k) nx[k] = agc_on ? __ldg(in2 + 2 * n * k + 1) : float2{0.0f, 0.0f};
    for (int c = 0; c < n_chunks; ++c) {
      const int b = c & 1;
#pragma unroll
      for (int k = 0; k < kSerU; ++k) inbuf[0][k][lane] = nx[k];
      if (agc_on && c + 1 < n_chunks) {
#pragma unroll
        for (int k = 0; k < kSerU; ++k) nx[k] = __ldg(in2 + 2 * n * ((size_t)(c + 1) * kSerU + k) + 1);
      }
      if (c >= 2) NamedSync(3 + b);
      __syncwarp();
      T41RX_SER_LOOP
      for (int k = 0; k < kSerU; ++k) {
        const float2 x = inbuf[0][k][lane];
#ifdef T41RX_SER_NO_AGC
        vbuf[b][k][lane] = x.y + 1.0f;
#else
        vbuf[b][k][lane] = agc_on ? agc.Step(x.x, x.y) : 0.0f;
#endif
      }
      NamedArrive(1 + b);
    }
    if (agc_on) agc.Store(st);
  } else if (warp == 1) {
    SerGain gain;
    gain.Load(cf);
    float2 nx[kSerU];
#pragma unroll
    for (int k = 0; k < kSerU; ++k) nx[k] = live ? __ldg(in2 + 2 * n * k) : float2{0.0f, 0.0f};
    for (int c = 0; c < n_chunks; ++c) {
      const int b = c & 1;
#pragma unroll
      for (int k = 0; k < kSerU; ++k) inbuf[1][k][lane] = nx[k];
      if (live && c + 1 < n_chunks) {
#pragma unroll
        for (int k = 0; k < kSerU; ++k) nx[k] = __ldg(in2 + 2 * n * ((size_t)(c + 1) * kSerU + k));
      }
      NamedSync(1 + b);
      if (c >= 2) NamedSync(7 + b);
      __syncwarp();
      T41RX_SER_LOOP
      for (int k = 0; k < kSerU; ++k) {
        float2 z = inbuf[1][k][lane];
        if (agc_on) {
#ifdef T41RX_SER_NO_GAIN
          const float m = vbuf[b][k][lane];
#else
          const float m = gain.Mult(vbuf[b][k][lane]);
#endif
          z.x = z.x * m;
          z.y = z.y * m;
        }
        dbuf[b][k][lane] = z;
      }
      if (c + 2 < n_chunks) NamedArrive(3 + b);
      NamedArrive(5 + b);
    }
  } else {
    SerDemod dem;
    dem.Load(a, cf, st, sin_tab);
    float *dst = a.ser_out + (live ? r : 0);
    float2 dem0 = float2{0.0f, 0.0f};
    for (int c = 0; c < n_chunks; ++c) {
      const int b = c & 1;
      NamedSync(5 + b);
      const int i0 = (c % (kDec / kSerU)) * kSerU;
      if (i0 == 0) {
        dem.BlockStart();
        dem0 = dbuf[b][0][lane];
      }
      T41RX_SER_LOOP
      for (int k = 0; k < kSerU; ++k) {
        const float2 z = dbuf[b][k][lane];
#ifdef T41RX_SER_NO_DEMOD
        const float au = z.x;
#else
        const float au = dem.Step(z.x, z.y);
#endif
        if (live) dst[((size_t)c * kSerU + k) * n] = au;
      }
      if (c + 2 < n_chunks) NamedArrive(7 + b);
      if (live && i0 == kDec - kSerU) SerPskTap(a, cf, st, sid, c / (kDec / kSerU), dem0);
    }
    if (live) dem.Store(st);
  }
}

__global__ void __launch_bounds__(kNT, 8 / kG) t41rx_exact_back_kernel(const LaunchArgs a) {
  extern __shared__ __align__(16) float smem[];
  Cta c;
  c.a = a;
  c.smem = smem;
  c.s0 = blockIdx.x * kG;
  c.ng = min(kG, a.n_streams - c.s0);
  c.t = 0;
  c.row = 0;
  c.row_idx = 0;
  c.rows_only = 0;
  c.casc_warp = 0;
  c.dc_carried = 0;
  const int tid = threadIdx.x;
  PhCtaInit(c, tid);
  __syncthreads();
  PhBackStateIn(c, tid);
  __syncthreads();
  for (int t = 0; t < a.n_blocks; ++t) {
    c.t = t;
    T41RX_BACK_SCHEDULE(T41RX_KPHASE)
  }
  PhBackStateOut(c, tid);
}
#undef T41RX_KPHASE

/* by-products of the row-producing blocks, launched after the chain (and rows) kernels on the same stream:
   audio spectrum + S-meter average (Process.cpp:550-570,791-805) from the masked spectra the chain kernels left in
   a.aspec, and the two frames for the control app's serial port (FFT.cpp:142-194 from the pixelnew rows,
   Process.cpp:818-825).  The running average makes the rows of one receiver a serial chain; receivers are
   independent. */
__global__ void __launch_bounds__(kNT) t41rx_row_byproducts_kernel(const LaunchArgs a) {
  extern __shared__ __align__(16) float smem[];
  Cta c;
  c.a = a;
  c.smem = smem;
  c.s0 = blockIdx.x * kG;
  c.ng = min(kG, a.n_streams - c.s0);
  c.row = 1;
  c.rows_only = 1;
  c.casc_warp = 0;
  c.dc_carried = 0;
  const int tid = threadIdx.x;
  PhCtaInit(c, tid);
  __syncthreads();
  /* the rows of this launch's blocks t0 .. t0 + n_blocks - 1 */
  for (int r = (a.t0 + a.row_every - 1) / a.row_every; r < a.n_rows && r * a.row_every < a.t0 + a.n_blocks; ++r) {
    c.t = r * a.row_every - a.t0;
    c.row_idx = r;
#define T41RX_KPHASE(stmt) \
  do {                     \
    stmt;                  \
    __syncthreads();       \
  } while (0)
    if (a.aspec) {
      T41RX_AUDIO_SPEC_SCHEDULE(T41RX_KPHASE)
    }
    if (a.spec_frames) {
      T41RX_SPEC_FRAME_SCHEDULE(T41RX_KPHASE)
    }
#undef T41RX_KPHASE
  }
}

}  // namespace t41rx

using namespace t41rx;

/* ------------------------------------------------------------------ */
/* error plumbing                                                      */
/* ------------------------------------------------------------------ */
static thread_local std::string g_last_error;

static int Fail(int code, const char *fmt, const char *detail = "") {
  char buf[512];
  snprintf(buf, sizeof(buf), fmt, detail);
  g_last_error = buf;
  return code;
}

int t41rx::SetApiError(int code, const char *text) {
  g_last_error = text;
  return code;
}

#define CUDA_TRY(expr)                                                              \
  do {                                                                              \
    cudaError_t e_ = (expr);                                                        \
    if (e_ != cudaSuccess) return Fail(T41RX_ECUDA, #expr ": %s", cudaGetErrorString(e_)); \
  } while (0)

/* ------------------------------------------------------------------ */
/* context                                                             */
/* ------------------------------------------------------------------ */
constexpr int kKernelEventRing = 32;
constexpr int kProcessChunks = 16;  /* most chunks of the host-buffer entry point's copy / compute pipeline (cut over time) */
constexpr int kReceiverChunks = 8;  /* chunks when a short call is cut over receivers */
constexpr size_t kSerialScratchBytes = (size_t)2048 << 20;  /* most hand-over scratch of the split bit-exact chain */
#ifndef T41RX_PIPE_CHUNKS
#define T41RX_PIPE_CHUNKS 2
#endif
constexpr int kPipeChunks = T41RX_PIPE_CHUNKS;   /* chunks a long launch is cut into (not below kPipeMinBlocks / 2 blocks each) */
constexpr int kPipeMinBlocks = 16;          /* launches this long run their bit-exact chain as a pipeline of chunks (LaunchExact) */

struct t41rx_ctx {
  int device = 0;
  int n_streams = 0;
  int n_sms = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_in = nullptr, copy_out = nullptr;   /* t41rx_process: copies overlap the kernels */
  /* the serial kernel of the split bit-exact chain is a bundle of latency-bound chains (one warp trio per 32
     receivers): in a mixed bank it runs on this stream beside the throughput kernel of the other receivers */
  cudaStream_t aux = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join_b = nullptr;   /* front done -> serial; serial done -> back (alternating) */
  cudaEvent_t ev_in[kProcessChunks] = {}, ev_done[kProcessChunks] = {};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool ev_valid = false;
  /* t41rx_process_device may enqueue on a caller-supplied stream: the end of its work is recorded here and every
     entry point that touches the context's device tables, state or scratch waits for it first */
  cudaEvent_t ev_ext = nullptr;
  bool ext_pending = false;
  /* CUDA events around the most recent launches of the dominant kernel (ring), for bench.py's roofline */
  cudaEvent_t kev[kKernelEventRing][2] = {};
  int64_t kev_count = 0;
  int64_t launches = 0;

  HostModel host;          /* parameter cache + host copies of every table */
  int fset_capacity = 0;

  StreamCfg *d_cfg = nullptr;
  StreamState *d_state = nullptr;
  FilterSet *d_fsets = nullptr;
  double *d_nco_tab = nullptr;
  float2 *d_twiddle = nullptr;
  double *d_hann = nullptr;
  float *d_sin = nullptr;
  float *d_zoom_iir = nullptr;
  float *d_eq_coeffs = nullptr;
  float *d_cw_coeffs = nullptr;
  float *d_sam = nullptr;
  float *d_nr_tab = nullptr;
  NrState *d_nr = nullptr;      /* allocated (zeroed) when the first receiver switches a spectral NR stage / the blanker on */
  uint16_t *d_gradient = nullptr;
  uint32_t *d_varicode = nullptr;

  /* receivers by kernel: the SAM PLL is chaotic while it acquires lock, and the LMS notch cancels most of its
     input, which amplifies any FP32 re-ordering beyond the stated tolerance: those receivers stay on the bit-exact
     kernel; everything else runs on the throughput kernel.  The variants of the lists are the splits under
     T41RX_FLAG_FAST_LMS (bit 0 of the index: LMS / notch receivers on the throughput kernel too) and
     T41RX_FLAG_FAST_SAM (bit 1: SAM receivers too). */
  std::vector<int32_t> h_fast_ids[4], h_phased_ids[4];
  int32_t *d_fast_ids[4] = {nullptr, nullptr, nullptr, nullptr}, *d_phased_ids[4] = {nullptr, nullptr, nullptr, nullptr};
  /* the throughput kernel's receivers once more, those with a slow serial stage (SAM PLL, equaliser, LMS, CW filter)
     first: the pairs of a CTA advance in lock-step, so slow receivers share CTAs among themselves when a launch
     covers the whole bank; empty when there is nothing to group */
  std::vector<int32_t> h_fast_grouped[4];
  int32_t *d_fast_grouped[4] = {nullptr, nullptr, nullptr, nullptr};
  bool ids_dirty = true;

  /* hand-over buffers of the split bit-exact chain (front | serial | back kernels): 5 KiB per stream-block; calls
     whose exact receivers need more than kSerialScratchBytes are cut over time */
  void *d_ser_in = nullptr, *d_ser_out = nullptr;
  size_t cap_ser_in = 0, cap_ser_out = 0;

  /* device staging for the host-buffer entry point */
  void *d_iq = nullptr, *d_audio = nullptr, *d_spec = nullptr, *d_wf = nullptr, *d_bits = nullptr, *d_chars = nullptr;
  void *d_iq16 = nullptr, *d_audio16 = nullptr;   /* q15 staging of t41rx_process_q15 */
  size_t cap_iq = 0, cap_audio = 0, cap_spec = 0, cap_wf = 0, cap_bits = 0, cap_chars = 0, cap_iq16 = 0, cap_audio16 = 0;

  /* audio-spectrum by-product: where the caller wants it (t41rx_bind_audio_spectrum; host pointers for the
     host-buffer entry points, device pointers for t41rx_process_device), the masked-spectrum scratch the
     chain kernels fill on row-producing blocks, and device staging for the host-buffer entry points */
  int32_t *bind_ypixel = nullptr;
  float *bind_max_ave = nullptr;
  uint8_t *bind_spec_frames = nullptr, *bind_audio_frames = nullptr;   /* t41rx_bind_control_frames */
  void *d_aspec = nullptr, *d_ypixel = nullptr, *d_max_ave = nullptr, *d_sframes = nullptr, *d_aframes = nullptr;
  size_t cap_aspec = 0, cap_ypixel = 0, cap_max_ave = 0, cap_sframes = 0, cap_aframes = 0;
  bool WantAudioSpec() const { return bind_ypixel || bind_max_ave || bind_audio_frames; }
};

/* wait for everything the context has enqueued: its own streams and the last caller-supplied stream */
static int Quiesce(t41rx_ctx *ctx) {
  if (ctx->ext_pending) {
    CUDA_TRY(cudaEventSynchronize(ctx->ev_ext));
    ctx->ext_pending = false;
  }
  CUDA_TRY(cudaStreamSynchronize(ctx->copy_in));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->aux));
  CUDA_TRY(cudaStreamSynchronize(ctx->copy_out));
  return 0;
}

static int EnsureFsetCapacity(t41rx_ctx *ctx, int need) {
  if (need <= ctx->fset_capacity) return 0;
  int cap = ctx->fset_capacity ? ctx->fset_capacity : 16;
  while (cap < need) cap *= 2;
  FilterSet *d = nullptr;
  CUDA_TRY(cudaMalloc(&d, sizeof(FilterSet) * cap));
  if (ctx->d_fsets) {
    CUDA_TRY(cudaMemcpy(d, ctx->d_fsets, sizeof(FilterSet) * ctx->fset_capacity, cudaMemcpyDeviceToDevice));
    CUDA_TRY(cudaFree(ctx->d_fsets));
  }
  ctx->d_fsets = d;
  ctx->fset_capacity = cap;
  return 0;
}

static int UploadFset(t41rx_ctx *ctx, int id) {
  int rc = EnsureFsetCapacity(ctx, id + 1);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpy(ctx->d_fsets + id, &ctx->host.fsets[id], sizeof(FilterSet), cudaMemcpyHostToDevice));
  return 0;
}

template <class T, class U>
static int UploadConst(T **dst, const std::vector<U> &src) {
  static_assert(sizeof(T) % sizeof(U) == 0, "element size");
  CUDA_TRY(cudaMalloc(dst, src.size() * sizeof(U)));
  CUDA_TRY(cudaMemcpy(*dst, src.data(), src.size() * sizeof(U), cudaMemcpyHostToDevice));
  return 0;
}

static int UploadConstTables(t41rx_ctx *ctx) {
  int rc;
  const HostModel &h = ctx->host;
  if ((rc = UploadConst(&ctx->d_twiddle, h.twiddle))) return rc;
  if ((rc = UploadConst(&ctx->d_hann, h.hann))) return rc;
  if ((rc = UploadConst(&ctx->d_sin, h.sin_table))) return rc;
  if ((rc = UploadConst(&ctx->d_zoom_iir, h.zoom_iir))) return rc;
  if ((rc = UploadConst(&ctx->d_eq_coeffs, h.eq_coeffs))) return rc;
  if ((rc = UploadConst(&ctx->d_cw_coeffs, h.cw_coeffs))) return rc;
  if ((rc = UploadConst(&ctx->d_sam, h.sam_consts))) return rc;
  if ((rc = UploadConst(&ctx->d_nr_tab, h.nr_tab))) return rc;
  if ((rc = UploadConst(&ctx->d_gradient, h.gradient))) return rc;
  if ((rc = UploadConst(&ctx->d_varicode, h.varicode))) return rc;
  return 0;
}

static int Grow(void **buf, size_t *cap, size_t need) {
  if (need <= *cap) return 0;
  if (*buf) CUDA_TRY(cudaFree(*buf));
  *buf = nullptr;
  *cap = 0;
  CUDA_TRY(cudaMalloc(buf, need));
  *cap = need;
  return 0;
}

/* ------------------------------------------------------------------ */
/* C-ABI                                                               */
/* ------------------------------------------------------------------ */
extern "C" {

const char *t41rx_last_error(void) { return g_last_error.c_str(); }
const char *t41rx_version(void) { return "t41rx-b200 0.1 (sm_100a)"; }

void t41rx_default_params(t41rx_params *p) { DefaultParams(p); }

void t41rx_mode_default_cuts(int32_t mode, int32_t *f_lo_cut, int32_t *f_hi_cut) {
  switch (mode) {
    case T41RX_DEMOD_LSB: *f_hi_cut = -200; *f_lo_cut = -3000; break;
    case T41RX_DEMOD_AM:
    case T41RX_DEMOD_SAM: *f_hi_cut = 3000; *f_lo_cut = -3000; break;
    default: *f_hi_cut = 3000; *f_lo_cut = 200; break;
  }
}

void t41rx_destroy(t41rx_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->ext_pending && ctx->ev_ext) cudaEventSynchronize(ctx->ev_ext);
  if (ctx->copy_in) cudaStreamSynchronize(ctx->copy_in);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->aux) cudaStreamSynchronize(ctx->aux);
  if (ctx->copy_out) cudaStreamSynchronize(ctx->copy_out);
  void *bufs[] = {ctx->d_cfg, ctx->d_state, ctx->d_fsets, ctx->d_nco_tab, ctx->d_twiddle, ctx->d_hann, ctx->d_sin,
                  ctx->d_zoom_iir, ctx->d_eq_coeffs, ctx->d_cw_coeffs, ctx->d_sam, ctx->d_nr_tab, ctx->d_nr, ctx->d_gradient, ctx->d_varicode, ctx->d_iq, ctx->d_audio,
                  ctx->d_spec, ctx->d_wf, ctx->d_bits, ctx->d_chars, ctx->d_fast_ids[0], ctx->d_phased_ids[0], ctx->d_fast_ids[1],
                  ctx->d_phased_ids[1], ctx->d_fast_ids[2], ctx->d_phased_ids[2], ctx->d_fast_ids[3], ctx->d_phased_ids[3],
                  ctx->d_fast_grouped[0], ctx->d_fast_grouped[1], ctx->d_fast_grouped[2], ctx->d_fast_grouped[3],
                  ctx->d_iq16, ctx->d_audio16, ctx->d_ser_in, ctx->d_ser_out, ctx->d_aspec, ctx->d_ypixel, ctx->d_max_ave,
                  ctx->d_sframes, ctx->d_aframes};
  for (void *b : bufs)
    if (b) cudaFree(b);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->ev_ext) cudaEventDestroy(ctx->ev_ext);
  for (int i = 0; i < kKernelEventRing; ++i)
    for (int j = 0; j < 2; ++j)
      if (ctx->kev[i][j]) cudaEventDestroy(ctx->kev[i][j]);
  for (int i = 0; i < kProcessChunks; ++i) {
    if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
    if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]);
  }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_join_b) cudaEventDestroy(ctx->ev_join_b);
  if (ctx->aux) cudaStreamDestroy(ctx->aux);
  if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
  if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int t41rx_create(t41rx_ctx **out, int n_streams, int device) {
  if (!out || n_streams <= 0) return Fail(T41RX_EINVAL, "t41rx_create: bad arguments%s");
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0)
    return Fail(T41RX_ENODEV, "t41rx_create: no CUDA device (this library has no CPU path)%s");
  if (device < 0 || device >= n_dev) return Fail(T41RX_EINVAL, "t41rx_create: device index out of range%s");
  CUDA_TRY(cudaSetDevice(device));
  t41rx_ctx *ctx = new (std::nothrow) t41rx_ctx();
  if (!ctx) return Fail(T41RX_ENOMEM, "t41rx_create: out of memory%s");
  ctx->device = device;
  ctx->n_streams = n_streams;
  int rc = 0;
  auto bail = [&](int code) {
    t41rx_destroy(ctx);
    return code;
  };
  for (int i = 0; i < kKernelEventRing; ++i)
    if (cudaEventCreate(&ctx->kev[i][0]) != cudaSuccess || cudaEventCreate(&ctx->kev[i][1]) != cudaSuccess)
      return bail(Fail(T41RX_ECUDA, "t41rx_create: event creation failed%s"));
  for (int i = 0; i < kProcessChunks; ++i)
    if (cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming) != cudaSuccess)
      return bail(Fail(T41RX_ECUDA, "t41rx_create: event creation failed%s"));
  if (cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->aux, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_join_b, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_ext, cudaEventDisableTiming) != cudaSuccess)
    return bail(Fail(T41RX_ECUDA, "t41rx_create: stream/event creation failed%s"));
  if (cudaFuncSetAttribute(t41rx_fused_rx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (int)(kSmemFloats * sizeof(float))) != cudaSuccess ||
      cudaFuncSetAttribute(t41rx_exact_front_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (int)(kSmemFloats * sizeof(float))) != cudaSuccess ||
      cudaFuncSetAttribute(t41rx_exact_back_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (int)(kSmemFloats * sizeof(float))) != cudaSuccess ||
      ConfigureRowsKernel() != cudaSuccess ||
      cudaFuncSetAttribute(t41rx_row_byproducts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (int)(kSmemFloats * sizeof(float))) != cudaSuccess)
    return bail(Fail(T41RX_ECUDA, "t41rx_create: kernel image for this GPU missing (built for sm_100a)%s"));
  if (ConfigureStreamKernel() != cudaSuccess ||
      cudaDeviceGetAttribute(&ctx->n_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->n_sms <= 0)
    return bail(Fail(T41RX_ECUDA, "t41rx_create: throughput kernel unavailable on this GPU (built for sm_100a)%s"));
  ctx->host.Init(n_streams);
  if ((rc = UploadConstTables(ctx))) return bail(rc);
  if (cudaMalloc(&ctx->d_cfg, sizeof(StreamCfg) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_state, sizeof(StreamState) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_nco_tab, sizeof(double) * 192 * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_grouped[0], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_grouped[1], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_grouped[2], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_grouped[3], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_ids[0], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_phased_ids[0], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_ids[1], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_phased_ids[1], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_ids[2], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_phased_ids[2], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_fast_ids[3], sizeof(int32_t) * n_streams) != cudaSuccess ||
      cudaMalloc(&ctx->d_phased_ids[3], sizeof(int32_t) * n_streams) != cudaSuccess)
    return bail(Fail(T41RX_ENOMEM, "t41rx_create: device allocation failed%s"));
  {
    std::vector<StreamState> init(n_streams);
    for (int s = 0; s < n_streams; ++s) HostStateInit(&init[s]);
    if (cudaMemcpy(ctx->d_state, init.data(), sizeof(StreamState) * n_streams, cudaMemcpyHostToDevice) != cudaSuccess)
      return bail(Fail(T41RX_ECUDA, "t41rx_create: state upload failed%s"));
  }
  if ((rc = UploadFset(ctx, 0))) return bail(rc);
  if (cudaMemcpy(ctx->d_nco_tab, ctx->host.nco_tab.data(), sizeof(double) * ctx->host.nco_tab.size(),
                 cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(ctx->d_cfg, ctx->host.cfg.data(), sizeof(StreamCfg) * n_streams, cudaMemcpyHostToDevice) != cudaSuccess)
    return bail(Fail(T41RX_ECUDA, "t41rx_create: table upload failed%s"));
  *out = ctx;
  return T41RX_OK;
}

int t41rx_num_streams(const t41rx_ctx *ctx) { return ctx ? ctx->n_streams : 0; }

static int SetParamsImpl(t41rx_ctx *ctx, int first, int count, const t41rx_params *p, bool each) {
  if (!ctx || !p || first < 0 || count <= 0 || first + count > ctx->n_streams)
    return Fail(T41RX_EINVAL, "t41rx_set_params: bad range%s");
  for (int i = 0; i < count; ++i)
    if (!ValidateParams(each ? p[i] : p[0])) return Fail(T41RX_EINVAL, "t41rx_set_params: parameter out of range%s");
  CUDA_TRY(cudaSetDevice(ctx->device));
  {                                               /* changes apply at a block boundary: nothing may be in flight */
    const int rc = Quiesce(ctx);
    if (rc) return rc;
  }
  /* room for every filter set this call can add BEFORE the host model changes: the device allocation is the step that
     can fail, and a failure after HostModel::Apply would leave host and device out of step */
  {
    const int rc = EnsureFsetCapacity(ctx, (int)ctx->host.fsets.size() + count);
    if (rc) return rc;
  }
  for (int i = 0; i < count; ++i) {
    const int s = first + i;
    StatePatch patch;
    int new_fset = -1;
    if (ctx->host.Apply(s, each ? p[i] : p[0], &patch, &new_fset)) return Fail(T41RX_EINVAL, "t41rx_set_params: rejected%s");
    if (new_fset >= 0) {
      int rc = UploadFset(ctx, new_fset);
      if (rc) return rc;
    }
    const StreamCfg &ncf = ctx->host.cfg[s];
    if ((ncf.nr_kim || ncf.nr_spectral || ncf.nb_on) && !ctx->d_nr) {
      CUDA_TRY(cudaMalloc(&ctx->d_nr, sizeof(NrState) * (size_t)ctx->n_streams));
      CUDA_TRY(cudaMemset(ctx->d_nr, 0, sizeof(NrState) * (size_t)ctx->n_streams));
    }
    if (patch.set_rf_gain)
      CUDA_TRY(cudaMemcpy(&ctx->d_state[s].rf_gain, &patch.rf_gain, sizeof(int32_t), cudaMemcpyHostToDevice));
    if (patch.reset_zoom_ptr) {
      const int32_t z = 0;
      CUDA_TRY(cudaMemcpy(&ctx->d_state[s].zoom_ptr, &z, sizeof(z), cudaMemcpyHostToDevice));
    }
    if (patch.clear_fast_native) {
      const int32_t z = 0;
      CUDA_TRY(cudaMemcpy(&ctx->d_state[s].fast_native, &z, sizeof(z), cudaMemcpyHostToDevice));
    }
  }
  ctx->ids_dirty = true;
  CUDA_TRY(cudaMemcpy(ctx->d_cfg + first, ctx->host.cfg.data() + first, sizeof(StreamCfg) * count, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(ctx->d_nco_tab + (size_t)192 * first, ctx->host.nco_tab.data() + (size_t)192 * first,
                      sizeof(double) * 192 * count, cudaMemcpyHostToDevice));
  return T41RX_OK;
}

int t41rx_set_params(t41rx_ctx *ctx, int first, int count, const t41rx_params *p) {
  return SetParamsImpl(ctx, first, count, p, false);
}
int t41rx_set_params_each(t41rx_ctx *ctx, int first, int count, const t41rx_params *p) {
  return SetParamsImpl(ctx, first, count, p, true);
}

int t41rx_get_params(const t41rx_ctx *ctx, int stream, t41rx_params *p) {
  if (!ctx || !p || stream < 0 || stream >= ctx->n_streams) return Fail(T41RX_EINVAL, "t41rx_get_params: bad arguments%s");
  *p = ctx->host.params[stream];
  return T41RX_OK;
}

static void FillTables(const HostModel &h, int stream, t41rx_tables *t) {
  memset(t, 0, sizeof(*t));
  const StreamCfg &c = h.cfg[stream];
  const FilterSet &fs = h.fsets[c.filter_id];
  memcpy(t->dec1, fs.dec1, sizeof(t->dec1));
  memcpy(t->dec2, fs.dec2, sizeof(t->dec2));
  memcpy(t->int1, fs.int1, sizeof(t->int1));
  memcpy(t->int2, fs.int2, sizeof(t->int2));
  memcpy(t->mask, fs.mask, sizeof(t->mask));
  memcpy(t->am_lp, c.am_lp, sizeof(t->am_lp));
  memcpy(t->zoom_fir, c.zoom_fir, sizeof(t->zoom_fir));
  const AgcConsts &a = c.agc;
  const float v[16] = {a.max_gain, a.attack_mult, a.decay_mult, a.fast_decay_mult, a.fast_backmult,
                       a.onemfast_backmult, a.out_target, a.min_volts, a.slope_constant, a.inv_max_input,
                       a.hang_level, a.hang_backmult, a.onemhang_backmult, a.hang_decay_mult, a.hangtime,
                       a.fixed_gain};
  memcpy(t->agc, v, sizeof(v));
  t->attack_buffsize = h.attack_buffsize[stream];
  t->hang_counter_load = a.hang_counter_load;
}

int t41rx_get_tables(const t41rx_ctx *ctx, int stream, t41rx_tables *t) {
  if (!ctx || !t || stream < 0 || stream >= ctx->n_streams) return Fail(T41RX_EINVAL, "t41rx_get_tables: bad arguments%s");
  FillTables(ctx->host, stream, t);
  return T41RX_OK;
}

int t41rx_design_tables(const t41rx_params *seq, int n_seq, t41rx_tables *t) {
  if (!t || n_seq < 0 || (n_seq > 0 && !seq)) return Fail(T41RX_EINVAL, "t41rx_design_tables: bad arguments%s");
  HostModel h;
  h.Init(1);
  for (int i = 0; i < n_seq; ++i) {
    StatePatch patch;
    int new_fset = -1;
    if (h.Apply(0, seq[i], &patch, &new_fset)) return Fail(T41RX_EINVAL, "t41rx_design_tables: parameter out of range%s");
  }
  FillTables(h, 0, t);
  return T41RX_OK;
}

int t41rx_get_debug(t41rx_ctx *ctx, int stream, t41rx_debug *d) {
  if (!ctx || !d || stream < 0 || stream >= ctx->n_streams) return Fail(T41RX_EINVAL, "t41rx_get_debug: bad arguments%s");
  CUDA_TRY(cudaSetDevice(ctx->device));
  {
    const int rc = Quiesce(ctx);
    if (rc) return rc;
  }
  StreamState st;
  CUDA_TRY(cudaMemcpy(&st, ctx->d_state + stream, sizeof(st), cudaMemcpyDeviceToHost));
  memset(d, 0, sizeof(*d));
  d->agc_state = st.agc_state;
  d->agc_decay_type = st.agc_decay_type;
  d->agc_hang_counter = st.agc_hang_counter;
  d->agc_action = st.agc_action;
  d->rf_gain = st.rf_gain;
  d->codec_timer = (int32_t)st.codec_timer;
  d->zoom_sample_ptr = st.zoom_ptr;
  d->first_block = st.first_block;
  d->agc_volts = st.agc_volts;
  d->agc_ring_max = st.agc_ring_max;
  d->agc_save_volts = st.agc_save_volts;
  d->agc_fast_backaverage = st.agc_fast_back;
  d->agc_hang_backaverage = st.agc_hang_back;
  d->sam_phzerror = st.sam_phzerror;
  d->sam_omega2 = st.sam_omega2;
  d->sam_fil_out = st.sam_fil_out;
  d->dc_state[0] = st.dc_d1;
  d->dc_state[1] = st.dc_d2;
  d->am_wold = st.am_wold;
  if (st.nco_closed) {
    const double r = sqrt(st.osc_q * st.osc_q + st.osc_i * st.osc_i);
    d->osc_vect_q = r * cos(st.nco_phase);
    d->osc_vect_i = r * sin(st.nco_phase);
  } else {
    d->osc_vect_q = st.osc_q;
    d->osc_vect_i = st.osc_i;
  }
  return T41RX_OK;
}

/* which part of a call a group of launches covers: receivers [first, first + count), blocks [t0, t0 + nt) of the
   n_blocks the call's buffers hold per receiver */
struct Span {
  int first, count, t0, nt;
};

/* the bit-exact chain for the receivers of `p` (p.n_streams of them, p.stream_ids / p.stream_base) on stream st:
   front | serial | back kernels with the hand-over in HBM, cut over time so that the scratch stays bounded;
   T41RX_FLAG_FUSED_EXACT: the single fused kernel (one lane per receiver in the serial phases) instead */
static int LaunchExact(t41rx_ctx *ctx, const LaunchArgs &p, cudaStream_t st, const std::function<int()> &overlap) {
  const int n = p.n_streams;
  const int grid = (n + kG - 1) / kG;
  if (p.flags & T41RX_FLAG_FUSED_EXACT) {
    t41rx_fused_rx_kernel<<<grid, kNT, kSmemFloats * sizeof(float), st>>>(p);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
    return overlap();
  }
  /* The launch is cut over time into chunks (scratch bounded; a launch of kPipeMinBlocks blocks or more into at least
     two) and the chunks are pipelined over two scratch halves:
         st :  F0  F1  [the other receivers' kernels]  B0  F2  B1  F3  B2 ...
         aux:      S0  S1 .........................        S2      S3 ...
     S(c) waits for F(c) and follows S(c - 1); B(c) waits for S(c).  The serial kernel is three latency-bound warps per 32
     receivers: beside a front kernel, the throughput kernel or a back kernel it costs them little, alone it leaves the
     GPU idle.  Hazards: F, S and B own disjoint parts of the receiver state; F(c + 2) re-uses the scratch half of chunk c,
     and B(c), which has waited for S(c), precedes it on st. */
  const size_t per_block = (size_t)n * kDec * (sizeof(float4) + sizeof(float));
  const bool pipe = p.n_blocks >= kPipeMinBlocks;
  const size_t budget = pipe ? kSerialScratchBytes / 2 : kSerialScratchBytes;
  int chunk = (int)std::min<size_t>((size_t)p.n_blocks, std::max<size_t>(1, budget / per_block));
  if (pipe) chunk = std::min(chunk, std::max(kPipeMinBlocks / 2, (p.n_blocks + kPipeChunks - 1) / kPipeChunks));
  const int n_chunks = (p.n_blocks + chunk - 1) / chunk;
  const int halves = n_chunks > 1 ? 2 : 1;
  const size_t in_elems = (size_t)n * chunk * kDec, out_elems = (size_t)n * chunk * kDec;
  int rc;
  if ((rc = Grow(&ctx->d_ser_in, &ctx->cap_ser_in, halves * in_elems * sizeof(float4)))) return rc;
  if ((rc = Grow(&ctx->d_ser_out, &ctx->cap_ser_out, halves * out_elems * sizeof(float)))) return rc;
  auto args_of = [&](int c) {
    const int c0 = c * chunk;
    LaunchArgs q = p;
    q.iq = p.iq ? p.iq + (size_t)c0 * 2 * kBlock : nullptr;
    q.audio = p.audio ? p.audio + (size_t)c0 * kBlock : nullptr;
    q.iq16 = p.iq16 ? p.iq16 + (size_t)c0 * 2 * kBlock : nullptr;
    q.audio16 = p.audio16 ? p.audio16 + (size_t)c0 * kBlock : nullptr;
    q.psk_bits = p.psk_bits ? p.psk_bits + c0 : nullptr;
    q.psk_chars = p.psk_chars ? p.psk_chars + c0 : nullptr;
    q.t0 = p.t0 + c0;
    q.n_blocks = std::min(chunk, p.n_blocks - c0);
    q.ser_in = (float4 *)ctx->d_ser_in + (size_t)(c & (halves - 1)) * in_elems;
    q.ser_out = (float *)ctx->d_ser_out + (size_t)(c & (halves - 1)) * out_elems;
    return q;
  };
  auto front_and_serial = [&](int c) -> int {
    const LaunchArgs q = args_of(c);
    t41rx_exact_front_kernel<<<grid, kNT, kSmemFloats * sizeof(float), st>>>(q);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev_fork, st));
    CUDA_TRY(cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
    t41rx_exact_serial_kernel<<<(n + kSerialLanes - 1) / kSerialLanes, kSerialThreads, 0, ctx->aux>>>(q);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord((c & 1) ? ctx->ev_join_b : ctx->ev_join, ctx->aux));
    ctx->launches += 2;
    return T41RX_OK;
  };
  auto back = [&](int c) -> int {
    const LaunchArgs q = args_of(c);
    CUDA_TRY(cudaStreamWaitEvent(st, (c & 1) ? ctx->ev_join_b : ctx->ev_join, 0));
    t41rx_exact_back_kernel<<<grid, kNT, kSmemFloats * sizeof(float), st>>>(q);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
    return T41RX_OK;
  };
  if ((rc = front_and_serial(0))) return rc;
  for (int c = 1; c < n_chunks; ++c) {
    if ((rc = front_and_serial(c))) return rc;
    if (c == 1 && (rc = overlap())) return rc;
    if ((rc = back(c - 1))) return rc;
  }
  if (n_chunks == 1 && (rc = overlap())) return rc;
  return back(n_chunks - 1);
}

/* enqueue the kernels for a span of the call on stream st (buffer pointers are those of the whole call) */
static int LaunchRange(t41rx_ctx *ctx, const void *iq_any, void *audio_any, bool q15, int n_blocks, int row_every,
                       int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                       uint32_t flags, cudaStream_t st, Span sp, int32_t *d_ypixel = nullptr,
                       float *d_max_ave = nullptr, uint8_t *d_sframes = nullptr, uint8_t *d_aframes = nullptr) {
  const int first = sp.first, count = sp.count;
  LaunchArgs a;
  memset(&a, 0, sizeof(a));
  if (q15) {
    a.iq16 = (const int16_t *)iq_any + (size_t)sp.t0 * 2 * kBlock;
    a.audio16 = (int16_t *)audio_any + (size_t)sp.t0 * kBlock;
  } else {
    a.iq = (const float *)iq_any + (size_t)sp.t0 * 2 * kBlock;
    a.audio = (float *)audio_any + (size_t)sp.t0 * kBlock;
  }
  a.spec_rows = row_every > 0 ? spec_rows : nullptr;
  a.wf_rows = row_every > 0 ? wf_rows : nullptr;
  a.psk_bits = psk_bits ? psk_bits + sp.t0 : nullptr;
  a.psk_chars = psk_chars ? psk_chars + sp.t0 : nullptr;
  a.cfg = ctx->d_cfg;
  a.st = ctx->d_state;
  a.fsets = ctx->d_fsets;
  a.nco_tab = ctx->d_nco_tab;
  a.twiddle = ctx->d_twiddle;
  a.hann = ctx->d_hann;
  a.sin_table = ctx->d_sin;
  a.zoom_iir = ctx->d_zoom_iir;
  a.eq_coeffs = ctx->d_eq_coeffs;
  a.cw_coeffs = ctx->d_cw_coeffs;
  a.sam_consts = ctx->d_sam;
  a.nr = ctx->d_nr;
  a.nr_tab = ctx->d_nr_tab;
  a.gradient = ctx->d_gradient;
  a.varicode = ctx->d_varicode;
  a.n_streams = count;
  a.stream_base = first;
  a.n_blocks = sp.nt;
  a.t0 = sp.t0;
  a.t_stride = n_blocks;
  a.row_every = row_every;
  a.n_rows = row_every > 0 ? (n_blocks + row_every - 1) / row_every : 0;
  a.flags = flags;
  /* does this block range hold a row-producing block (absolute index a multiple of row_every)? */
  const bool has_row = row_every > 0 && ((sp.t0 + row_every - 1) / row_every) * row_every < sp.t0 + sp.nt;
  if (a.n_rows > 0 && (d_ypixel || d_max_ave || d_aframes)) {
    a.aspec = (float2 *)ctx->d_aspec;         /* sized by the caller (EnsureAudioSpecScratch) */
    a.audio_ypixel = d_ypixel;
    a.audio_max_ave = d_max_ave;
    a.audio_frames = d_aframes;
  }
  if (a.n_rows > 0 && d_sframes) {
    if (!a.spec_rows) return Fail(T41RX_EINVAL, "t41rx_process: the spectrum frames are built from spec_rows, which is NULL%s");
    a.spec_frames = d_sframes;
  }
  /* the by-product kernel runs after the chain kernels of the range, on the whole (contiguous) range */
  auto audio_spectrum = [&]() -> int {
    if ((!a.aspec && !a.spec_frames) || !has_row) return T41RX_OK;
    t41rx_row_byproducts_kernel<<<(count + kG - 1) / kG, kNT, kSmemFloats * sizeof(float), st>>>(a);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
    return T41RX_OK;
  };
  /* kernel choice: the throughput kernel unless the caller asks for the bit-exact oscillator or the
     phase-structured kernel; SAM receivers always take the phase-structured kernel (see t41rx_ctx) */
  const bool all_phased = (flags & (T41RX_FLAG_EXACT_NCO | T41RX_FLAG_PHASED_KERNEL)) != 0;
  if (all_phased) {
    const int rc = LaunchExact(ctx, a, st, []() { return (int)T41RX_OK; });
    if (rc) return rc;
    return audio_spectrum();
  }
  /* the slices of the (sorted) per-kernel receiver lists that fall into the range */
  auto slice = [&](const std::vector<int32_t> &ids, int *off, int *len) {
    const auto lo = std::lower_bound(ids.begin(), ids.end(), first), hi = std::lower_bound(ids.begin(), ids.end(), first + count);
    *off = (int)(lo - ids.begin());
    *len = (int)(hi - lo);
  };
  int p_off, p_len, f_off, f_len;
  const int v = ((flags & T41RX_FLAG_FAST_LMS) ? 1 : 0) | ((flags & T41RX_FLAG_FAST_SAM) ? 2 : 0);
  slice(ctx->h_phased_ids[v], &p_off, &p_len);
  slice(ctx->h_fast_ids[v], &f_off, &f_len);
  /* the throughput kernel's receivers (rows kernel first: it reads the launch-start state) */
  auto fast_kernels = [&]() -> int {
    if (f_len <= 0) return T41RX_OK;
    LaunchArgs f = a;
    f.n_streams = f_len;
    f.stream_ids = (p_len > 0) ? ctx->d_fast_ids[v] + f_off : nullptr;     /* nothing for the other kernel in range: contiguous */
    if (first == 0 && count == ctx->n_streams && !ctx->h_fast_grouped[v].empty()) f.stream_ids = ctx->d_fast_grouped[v];
    if (has_row && (a.spec_rows || a.wf_rows)) {
      CUDA_TRY(LaunchRowsKernel(f, ctx->n_sms, st));
      ctx->launches += 1;
    }
    cudaEvent_t *kev = ctx->kev[ctx->kev_count % kKernelEventRing];
    CUDA_TRY(cudaEventRecord(kev[0], st));
    CUDA_TRY(LaunchStreamKernel(f, ctx->n_sms, st));
    CUDA_TRY(cudaEventRecord(kev[1], st));
    ctx->kev_count += 1;
    ctx->launches += 1;
    return T41RX_OK;
  };
  if (p_len > 0) {
    /* the bit-exact chain's receivers; the throughput kernel of the others runs beside its serial kernel */
    LaunchArgs p = a;
    p.n_streams = p_len;
    p.stream_ids = ctx->d_phased_ids[v] + p_off;
    const int rc = LaunchExact(ctx, p, st, fast_kernels);
    if (rc) return rc;
  } else {
    const int rc = fast_kernels();
    if (rc) return rc;
  }
  return audio_spectrum();
}

/* scratch for the masked spectra of the row-producing blocks: [n_streams][n_rows][512] float2 */
static int EnsureAudioSpecScratch(t41rx_ctx *ctx, size_t n_rows) {
  if (!ctx->WantAudioSpec() || n_rows == 0) return T41RX_OK;
  return Grow(&ctx->d_aspec, &ctx->cap_aspec, (size_t)ctx->n_streams * n_rows * kFft * sizeof(float2));
}

/* (re)build the per-kernel receiver lists after a parameter change */
static int RefreshKernelLists(t41rx_ctx *ctx) {
  if (!ctx->ids_dirty) return T41RX_OK;
  CUDA_TRY(cudaDeviceSynchronize());
  for (int v = 0; v < 4; ++v) {
    ctx->h_fast_ids[v].clear();
    ctx->h_phased_ids[v].clear();
    for (int s = 0; s < ctx->n_streams; ++s) {
      const StreamCfg &cf = ctx->host.cfg[s];
      /* the 256-point spectral NR stages and the noise blanker only exist on the bit-exact chain */
      const bool phased = (cf.mode == kModeSam && !(v & 2)) || (!(v & 1) && (cf.nr_lms || cf.anr_notch)) || cf.nr_kim ||
                          cf.nr_spectral || cf.nb_on;
      (phased ? ctx->h_phased_ids[v] : ctx->h_fast_ids[v]).push_back(s);
    }
    if (!ctx->h_fast_ids[v].empty())
      CUDA_TRY(cudaMemcpy(ctx->d_fast_ids[v], ctx->h_fast_ids[v].data(), sizeof(int32_t) * ctx->h_fast_ids[v].size(), cudaMemcpyHostToDevice));
    {
      auto slow = [&](int32_t s) {
        const StreamCfg &cf = ctx->host.cfg[s];
        return cf.mode == kModeSam || cf.eq_on || cf.nr_lms || cf.anr_notch || cf.cw_filter >= 0;
      };
      std::vector<int32_t> &g = ctx->h_fast_grouped[v];
      g = ctx->h_fast_ids[v];
      const auto mid = std::stable_partition(g.begin(), g.end(), slow);
      if (mid == g.begin() || mid == g.end()) g.clear();         /* all alike: the plain list (or no list) does */
      else CUDA_TRY(cudaMemcpy(ctx->d_fast_grouped[v], g.data(), sizeof(int32_t) * g.size(), cudaMemcpyHostToDevice));
    }
    if (!ctx->h_phased_ids[v].empty())
      CUDA_TRY(cudaMemcpy(ctx->d_phased_ids[v], ctx->h_phased_ids[v].data(), sizeof(int32_t) * ctx->h_phased_ids[v].size(), cudaMemcpyHostToDevice));
  }
  ctx->ids_dirty = false;
  return T41RX_OK;
}

static int ProcessDevice(t41rx_ctx *ctx, const void *iq, void *audio, bool q15, int n_blocks, int row_every,
                         int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                         uint32_t flags, void *cuda_stream) {
  if (!ctx || !iq || !audio || n_blocks <= 0 || row_every < 0)
    return Fail(T41RX_EINVAL, "t41rx_process_device: bad arguments%s");
  CUDA_TRY(cudaSetDevice(ctx->device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  int rc = RefreshKernelLists(ctx);
  if (rc) return rc;
  if ((rc = EnsureAudioSpecScratch(ctx, row_every > 0 ? (size_t)(n_blocks + row_every - 1) / row_every : 0))) return rc;
  CUDA_TRY(cudaEventRecord(ctx->ev0, st));
  rc = LaunchRange(ctx, iq, audio, q15, n_blocks, row_every, spec_rows, wf_rows, psk_bits, psk_chars, flags, st,
                   Span{0, ctx->n_streams, 0, n_blocks}, ctx->bind_ypixel, ctx->bind_max_ave, ctx->bind_spec_frames,
                   ctx->bind_audio_frames);
  if (st != ctx->stream) {                        /* ordering contract (t41rx.h): remember the caller's stream */
    cudaEventRecord(ctx->ev_ext, st);
    ctx->ext_pending = true;
  }
  if (rc) return rc;
  CUDA_TRY(cudaEventRecord(ctx->ev1, st));
  ctx->ev_valid = true;
  return T41RX_OK;
}

int t41rx_process_device(t41rx_ctx *ctx, const float *iq, float *audio, int n_blocks, int row_every,
                         int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                         uint32_t flags, void *cuda_stream) {
  return ProcessDevice(ctx, iq, audio, false, n_blocks, row_every, spec_rows, wf_rows, psk_bits, psk_chars, flags, cuda_stream);
}

int t41rx_process_device_q15(t41rx_ctx *ctx, const int16_t *iq_q15, int16_t *audio_q15, int n_blocks, int row_every,
                             int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                             uint32_t flags, void *cuda_stream) {
  return ProcessDevice(ctx, iq_q15, audio_q15, true, n_blocks, row_every, spec_rows, wf_rows, psk_bits, psk_chars, flags, cuda_stream);
}

/* log10f_fast (Utility.cpp:245-258) on the host, for the S-meter helper */
static float HostLog10Fast(float x) {
  int e;
  const float f = frexpf(fabsf(x), &e);
  volatile float y = 1.23149591368684f;     /* volatile: one rounding per operation whatever the host flags */
  y = y * f;
  y = y + -4.11852516267426f;
  y = y * f;
  y = y + 6.02197014179219f;
  y = y * f;
  y = y + -3.13396450166353f;
  y = y + (float)e;
  return y * 0.3010299956639812f;
}

int t41rx_bind_audio_spectrum(t41rx_ctx *ctx, int32_t *audio_ypixel, float *audio_max_sq_ave) {
  if (!ctx) return Fail(T41RX_EINVAL, "t41rx_bind_audio_spectrum: null context%s");
  ctx->bind_ypixel = audio_ypixel;
  ctx->bind_max_ave = audio_max_sq_ave;
  return T41RX_OK;
}

int t41rx_bind_control_frames(t41rx_ctx *ctx, uint8_t *spec_frames, uint8_t *audio_frames) {
  if (!ctx) return Fail(T41RX_EINVAL, "t41rx_bind_control_frames: null context%s");
  ctx->bind_spec_frames = spec_frames;
  ctx->bind_audio_frames = audio_frames;
  return T41RX_OK;
}

/* Display.cpp:959-981 (TCVSDR_SMETER build): float sum up to the constant, then the FP64 tail the double literal
   1.5 forces; log10f_fast is Utility.cpp:245-258 */
float t41rx_smeter_dbm(float audio_max_sq_ave, float gain_correction, int32_t rf_gain, int32_t rf_gain_all_bands) {
  const float dbm_calibration = 22.0f, slope = 10.0f, cons = -92.0f;
  const int attenuator = 0;                 /* Display.cpp:146 */
  const float head = dbm_calibration + gain_correction + (float)attenuator + slope * HostLog10Fast(audio_max_sq_ave) + cons;
  return (float)((double)head - (double)(float)rf_gain * 1.5 - (double)rf_gain_all_bands);
}

/* Display.cpp:942,995-998 (TCVSDR_SMETER: pixels_per_s = 12) */
int32_t t41rx_smeter_bar(float dbm) {
  const float pixels_per_s = 12;
  const float in_min = (float)(-73.0 - 9 * 6.0), in_max = (float)-73.0, out_min = (float)0, out_max = (float)(9 * pixels_per_s);
  const volatile float num = (dbm - in_min) * (out_max - out_min);
  const float v = num / (in_max - in_min) + out_min;
  int pad;
  if (!(v > -32769.0f)) pad = -32768;        /* the int16 conversion of what does not fit saturates on the target */
  else if (v > 32767.0f) pad = 32767;
  else pad = (int16_t)v;
  pad = pad < 0 ? 0 : pad;
  pad = pad > 180 ? 180 : pad;
  return pad;
}

int t41rx_synchronize(t41rx_ctx *ctx) {
  if (!ctx) return Fail(T41RX_EINVAL, "t41rx_synchronize: null context%s");
  CUDA_TRY(cudaSetDevice(ctx->device));
  return Quiesce(ctx) ? T41RX_ECUDA : T41RX_OK;
}

/* host-buffer entry points: float (iq / audio) or q15 (iq16 / audio16) blocks */
static int ProcessHost(t41rx_ctx *ctx, const float *iq, float *audio, const int16_t *iq16, int16_t *audio16,
                       int n_blocks, int row_every, int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits,
                       uint8_t *psk_chars, uint32_t flags) {
  const bool q15 = iq16 != nullptr;
  if (!ctx || (!q15 && (!iq || !audio)) || (q15 && !audio16) || n_blocks <= 0 || row_every < 0)
    return Fail(T41RX_EINVAL, "t41rx_process: bad arguments%s");
  const bool want_rows_out = ctx && (ctx->WantAudioSpec() || ctx->bind_spec_frames);
  if (row_every > 0 && !spec_rows && !wf_rows && !want_rows_out) row_every = 0;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const size_t S = (size_t)ctx->n_streams, T = (size_t)n_blocks;
  const size_t n_rows = row_every > 0 ? (T + row_every - 1) / row_every : 0;
  const size_t b_iq = S * T * 2 * kBlock * sizeof(float), b_audio = S * T * kBlock * sizeof(float);
  const size_t b_spec = S * n_rows * kSpecRes * sizeof(int16_t), b_wf = S * n_rows * kSpecRes * sizeof(uint16_t);
  const size_t b_psk = S * T;
  int rc;
  if (!q15 && (rc = Grow(&ctx->d_iq, &ctx->cap_iq, b_iq))) return rc;
  if (!q15 && (rc = Grow(&ctx->d_audio, &ctx->cap_audio, b_audio))) return rc;
  const bool need_spec = n_rows && (spec_rows || ctx->bind_spec_frames);     /* the frames are built from the rows */
  if (need_spec && (rc = Grow(&ctx->d_spec, &ctx->cap_spec, b_spec))) return rc;
  if (n_rows && wf_rows && (rc = Grow(&ctx->d_wf, &ctx->cap_wf, b_wf))) return rc;
  if (psk_bits && (rc = Grow(&ctx->d_bits, &ctx->cap_bits, b_psk))) return rc;
  if (psk_chars && (rc = Grow(&ctx->d_chars, &ctx->cap_chars, b_psk))) return rc;
  if (q15 && (rc = Grow(&ctx->d_iq16, &ctx->cap_iq16, b_iq / 2))) return rc;
  if (q15 && (rc = Grow(&ctx->d_audio16, &ctx->cap_audio16, b_audio / 2))) return rc;
  const size_t b_ypix = S * n_rows * kAudioSpecPixels * sizeof(int32_t), b_max = S * n_rows * sizeof(float);
  if (n_rows && ctx->bind_ypixel && (rc = Grow(&ctx->d_ypixel, &ctx->cap_ypixel, b_ypix))) return rc;
  if (n_rows && ctx->bind_max_ave && (rc = Grow(&ctx->d_max_ave, &ctx->cap_max_ave, b_max))) return rc;
  if ((rc = EnsureAudioSpecScratch(ctx, n_rows))) return rc;
  if (n_rows && ctx->bind_spec_frames && (rc = Grow(&ctx->d_sframes, &ctx->cap_sframes, S * n_rows * kSpecFrameBytes))) return rc;
  if (n_rows && ctx->bind_audio_frames && (rc = Grow(&ctx->d_aframes, &ctx->cap_aframes, S * n_rows * kAudioSpecPixels))) return rc;
  uint8_t *d_sfr = (n_rows && ctx->bind_spec_frames) ? (uint8_t *)ctx->d_sframes : nullptr;
  uint8_t *d_afr = (n_rows && ctx->bind_audio_frames) ? (uint8_t *)ctx->d_aframes : nullptr;
  int32_t *d_ypix = (n_rows && ctx->bind_ypixel) ? (int32_t *)ctx->d_ypixel : nullptr;
  float *d_maxave = (n_rows && ctx->bind_max_ave) ? (float *)ctx->d_max_ave : nullptr;
  if ((rc = RefreshKernelLists(ctx))) return rc;
  /* Cut the call into chunks and overlap the copy-in of chunk i+1, the kernels of chunk i and the copy-out of
     chunk i-1 on three streams (full-duplex host link).  Long calls are cut over TIME (every receiver, a range of
     blocks: each launch keeps the whole GPU busy and the last chunk, which nothing overlaps, is short; the state
     travels between the launches through HBM exactly as between two calls); short calls of a large bank are cut
     over RECEIVERS (they are independent). */
  const bool big = S * T >= 2048;                          /* >= 32 MiB of I/Q: below that one chunk, one launch */
  const bool by_time = big && T >= 16;
  const int n_chunks = !big ? 1
                       : by_time ? (int)std::min<size_t>(kProcessChunks, T / 4)
                                 : ((ctx->n_streams >= 8 * kReceiverChunks) ? kReceiverChunks : 1);
  int16_t *d_spec = need_spec ? (int16_t *)ctx->d_spec : nullptr;
  uint16_t *d_wf = (n_rows && wf_rows) ? (uint16_t *)ctx->d_wf : nullptr;
  int8_t *d_bits = psk_bits ? (int8_t *)ctx->d_bits : nullptr;
  uint8_t *d_chars = psk_chars ? (uint8_t *)ctx->d_chars : nullptr;
  /* everything enqueued below reads or writes the caller's host buffers asynchronously: whatever fails, no copy may
     still be in flight when the call returns */
  auto enqueue = [&]() -> int {
  CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
  const size_t blk_iq = 2 * kBlock, blk_audio = kBlock;       /* elements per block */
  for (int ch = 0; ch < n_chunks; ++ch) {
    /* the chunk: receivers [s0, s0 + n) x blocks [t0, t0 + nt) */
    const size_t s0 = by_time ? 0 : S * ch / n_chunks, n = by_time ? S : S * (ch + 1) / n_chunks - s0;
    const size_t t0 = by_time ? T * ch / n_chunks : 0, nt = by_time ? T * (ch + 1) / n_chunks - t0 : T;
    const size_t off_iq = (s0 * T + t0) * blk_iq, off_audio = (s0 * T + t0) * blk_audio;
    const size_t in_esz = q15 ? sizeof(int16_t) : sizeof(float);
    const char *h_in = q15 ? (const char *)(iq16 + off_iq) : (const char *)(iq + off_iq);
    char *d_in = q15 ? (char *)((int16_t *)ctx->d_iq16 + off_iq) : (char *)((float *)ctx->d_iq + off_iq);
    CUDA_TRY(cudaMemcpy2DAsync(d_in, T * blk_iq * in_esz, h_in, T * blk_iq * in_esz, nt * blk_iq * in_esz, n,
                               cudaMemcpyHostToDevice, ctx->copy_in));
    CUDA_TRY(cudaEventRecord(ctx->ev_in[ch], ctx->copy_in));
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[ch], 0));
    /* q15 blocks go through the kernels as they are: each converts at its own load / store */
    rc = LaunchRange(ctx, q15 ? ctx->d_iq16 : ctx->d_iq, q15 ? ctx->d_audio16 : ctx->d_audio, q15, n_blocks, row_every, d_spec,
                     d_wf, d_bits, d_chars, flags, ctx->stream, Span{(int)s0, (int)n, (int)t0, (int)nt}, d_ypix, d_maxave,
                     d_sfr, d_afr);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev_done[ch], ctx->stream));
    CUDA_TRY(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_done[ch], 0));
    const size_t out_esz = q15 ? sizeof(int16_t) : sizeof(float);
    char *h_out = q15 ? (char *)(audio16 + off_audio) : (char *)(audio + off_audio);
    const char *d_out = q15 ? (const char *)((int16_t *)ctx->d_audio16 + off_audio) : (const char *)((float *)ctx->d_audio + off_audio);
    CUDA_TRY(cudaMemcpy2DAsync(h_out, T * blk_audio * out_esz, d_out, T * blk_audio * out_esz, nt * blk_audio * out_esz, n,
                               cudaMemcpyDeviceToHost, ctx->copy_out));
    /* the small per-row / per-block outputs of receivers [r0, r0 + rn): with the chunk when cutting over receivers,
       after the last chunk when cutting over time */
    if (by_time && ch + 1 < n_chunks) continue;
    const size_t r0 = by_time ? 0 : s0, rn = by_time ? S : n;
    const size_t per_row = n_rows * kSpecRes;
    if (d_sfr) CUDA_TRY(cudaMemcpyAsync(ctx->bind_spec_frames + r0 * n_rows * kSpecFrameBytes, d_sfr + r0 * n_rows * kSpecFrameBytes, rn * n_rows * kSpecFrameBytes, cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_afr) CUDA_TRY(cudaMemcpyAsync(ctx->bind_audio_frames + r0 * n_rows * kAudioSpecPixels, d_afr + r0 * n_rows * kAudioSpecPixels, rn * n_rows * kAudioSpecPixels, cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_spec && spec_rows) CUDA_TRY(cudaMemcpyAsync(spec_rows + r0 * per_row, d_spec + r0 * per_row, rn * per_row * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_wf) CUDA_TRY(cudaMemcpyAsync(wf_rows + r0 * per_row, d_wf + r0 * per_row, rn * per_row * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_ypix) CUDA_TRY(cudaMemcpyAsync(ctx->bind_ypixel + r0 * n_rows * kAudioSpecPixels, d_ypix + r0 * n_rows * kAudioSpecPixels, rn * n_rows * kAudioSpecPixels * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_maxave) CUDA_TRY(cudaMemcpyAsync(ctx->bind_max_ave + r0 * n_rows, d_maxave + r0 * n_rows, rn * n_rows * sizeof(float), cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_bits) CUDA_TRY(cudaMemcpyAsync(psk_bits + r0 * T, d_bits + r0 * T, rn * T, cudaMemcpyDeviceToHost, ctx->copy_out));
    if (d_chars) CUDA_TRY(cudaMemcpyAsync(psk_chars + r0 * T, d_chars + r0 * T, rn * T, cudaMemcpyDeviceToHost, ctx->copy_out));
  }
  CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->ev_valid = true;
  CUDA_TRY(cudaStreamSynchronize(ctx->copy_out));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return T41RX_OK;
  };
  rc = enqueue();
  if (rc) {                                        /* keep the first error's text */
    cudaStreamSynchronize(ctx->copy_in);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->aux);
    cudaStreamSynchronize(ctx->copy_out);
  }
  return rc;
}

int t41rx_process(t41rx_ctx *ctx, const float *iq, float *audio, int n_blocks, int row_every,
                  int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars, uint32_t flags) {
  return ProcessHost(ctx, iq, audio, nullptr, nullptr, n_blocks, row_every, spec_rows, wf_rows, psk_bits, psk_chars, flags);
}

int t41rx_process_q15(t41rx_ctx *ctx, const int16_t *iq_q15, int16_t *audio_q15, int n_blocks, int row_every,
                      int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars, uint32_t flags) {
  if (!iq_q15) return Fail(T41RX_EINVAL, "t41rx_process_q15: bad arguments%s");
  return ProcessHost(ctx, nullptr, nullptr, iq_q15, audio_q15, n_blocks, row_every, spec_rows, wf_rows, psk_bits, psk_chars, flags);
}

#ifdef T41RX_PHASE_TIMING
int t41rx_debug_phase_cycles(unsigned long long *out128, int reset) {
  if (cudaMemcpyFromSymbol(out128, g_phase_cycles, sizeof(unsigned long long) * 128) != cudaSuccess) return -1;
  if (RowsPhaseCycles(out128 + 64, reset) != cudaSuccess) return -1;       /* slots 32.. : the rows-only kernel (rx_rows.cu) */
  if (reset) {
    unsigned long long z[128] = {0};
    cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z));
  }
  return 0;
}
#endif

int64_t t41rx_kernel_launches(const t41rx_ctx *ctx) { return ctx ? ctx->launches : 0; }

int64_t t41rx_dc_refilter_count(void) {
  unsigned long long v = 0;
  if (cudaMemcpyFromSymbol(&v, g_dc_refilter_count, sizeof(v)) != cudaSuccess) return -1;
  const long long rows = RowsDcRefilterCount();                              /* the rows-only kernel counts in its own unit */
  if (rows < 0) return -1;
  return (int64_t)v + rows;
}

int t41rx_stream_kernel_times(t41rx_ctx *ctx, float *ms, int max_n) {
  if (!ctx || !ms || max_n <= 0) return Fail(T41RX_EINVAL, "t41rx_stream_kernel_times: bad arguments%s");
  CUDA_TRY(cudaSetDevice(ctx->device));
  int n = (int)std::min<int64_t>(std::min<int64_t>(ctx->kev_count, kKernelEventRing), max_n);
  for (int i = 0; i < n; ++i) {
    cudaEvent_t *kev = ctx->kev[(ctx->kev_count - n + i) % kKernelEventRing];
    CUDA_TRY(cudaEventSynchronize(kev[1]));
    CUDA_TRY(cudaEventElapsedTime(ms + i, kev[0], kev[1]));
  }
  return n;
}

int t41rx_last_kernel_ms(t41rx_ctx *ctx, float *ms) {
  if (!ctx || !ms) return Fail(T41RX_EINVAL, "t41rx_last_kernel_ms: bad arguments%s");
  if (!ctx->ev_valid) return Fail(T41RX_EINVAL, "t41rx_last_kernel_ms: no launch yet%s");
  CUDA_TRY(cudaSetDevice(ctx->device));
  CUDA_TRY(cudaEventSynchronize(ctx->ev1));
  CUDA_TRY(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return T41RX_OK;
}

}  // extern "C"
