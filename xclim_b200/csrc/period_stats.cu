// Streaming per-period statistics: threshold counts, run-length statistics, reductions.
//
// Replaces (reference paths relative to /root/reference/src/xclim):
//   indices/generic.py:301-361      compare, threshold_count
//   indices/generic.py:543-585      _spell_length_statistics (window == 1)
//   indices/run_length.py:87-132    resample_and_rl
//   indices/run_length.py:143-335   _cumsum_reset_np, rle, rle_statistics
//   indices/run_length.py:381-488   windowed_run_events / windowed_run_count
//   indices/generic.py:83-125       select_resample_op ; 1514-1552 cumulative_difference
//   core/missing.py:296-322         MissingAny's valid-step count (fused as `valid_count`)
//
// Design (B200): the (time, lat, lon) buffer is coalesced along cells, so a THREAD owns VEC=4
// adjacent cells (one 128-bit load per time step; a warp reads 512 contiguous bytes per step) and
// marches through the time steps of ONE period keeping the run-length state machine in
// registers -- no shuffles, no shared memory, no intermediate arrays.  The grid is
// (cell-vectors, periods): every (period, cell) unit is independent when runs are cut at period
// edges; with resample_before_rl == 0 a unit additionally looks one step back (to skip a run
// that started earlier) and reads past the period end until its open runs close.  UNROLL
// independent 16-byte loads are issued before any use so that each thread keeps >= 128 B in
// flight; data is read exactly once (ld.global.nc.L1::no_allocate).
#include <type_traits>

#include "common.cuh"

namespace xc {
namespace {

constexpr int kThreads = 128;
constexpr int kUnroll = 8;

template <int VEC>
struct Vec;
template <>
struct Vec<1> {
  float v[1];
  __device__ __forceinline__ void load(const float* p) { v[0] = ld_stream(p); }
};
template <>
struct Vec<4> {
  float v[4];
  __device__ __forceinline__ void load(const float* p) {
    float4 q = ld_stream4(p);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
};

template <int VEC, typename T>
__device__ __forceinline__ void store_vec(T* dst, const T (&v)[VEC]) {
  if constexpr (VEC == 4 && sizeof(T) == 4) {
    uint4 q;
    q.x = *reinterpret_cast<const uint32_t*>(&v[0]);
    q.y = *reinterpret_cast<const uint32_t*>(&v[1]);
    q.z = *reinterpret_cast<const uint32_t*>(&v[2]);
    q.w = *reinterpret_cast<const uint32_t*>(&v[3]);
    *reinterpret_cast<uint4*>(dst) = q;
  } else {
#pragma unroll
    for (int i = 0; i < VEC; ++i) dst[i] = v[i];
  }
}

// Iterate f(t, Vec) over t in [t0, t1) with UNROLL loads in flight.
template <int VEC, int UNROLL = kUnroll, typename F>
__device__ __forceinline__ void stream_rows(const float* __restrict__ col, int64_t ldx, int t0, int t1,
                                            F&& f) {
  int t = t0;
  const float* p = col + (int64_t)t0 * ldx;
  for (; t + UNROLL <= t1; t += UNROLL) {
    Vec<VEC> r[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) r[u].load(p + (int64_t)u * ldx);
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) f(r[u]);
    p += (int64_t)UNROLL * ldx;
  }
  for (; t < t1; ++t) {
    Vec<VEC> r;
    r.load(p);
    f(r);
    p += ldx;
  }
}

// ------------------------------------------------------------------------------------------------
// threshold count (+ valid count)
// ------------------------------------------------------------------------------------------------
template <int OP, int VEC, bool VALID>
__global__ void __launch_bounds__(kThreads)
period_count_kernel(const float* __restrict__ x, int64_t C, int64_t ldx,
                    const int32_t* __restrict__ poff, float thr,
                    int32_t* __restrict__ out, int32_t* __restrict__ valid) {
  const int64_t c0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  if (c0 >= C) return;
  const int p = blockIdx.y;
  const int t0 = poff[p], t1 = poff[p + 1];
  int32_t cnt[VEC], nv[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { cnt[i] = 0; nv[i] = 0; }
  stream_rows<VEC>(x + c0, ldx, t0, t1, [&](const Vec<VEC>& r) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      cnt[i] += cmp<OP>(r.v[i], thr) ? 1 : 0;
      if constexpr (VALID) nv[i] += (r.v[i] == r.v[i]) ? 1 : 0;
    }
  });
  store_vec<VEC>(out + (int64_t)p * C + c0, cnt);
  if constexpr (VALID) store_vec<VEC>(valid + (int64_t)p * C + c0, nv);
}

// ------------------------------------------------------------------------------------------------
// run-length statistics
// ------------------------------------------------------------------------------------------------
// Per-cell accumulator over the run lengths L >= window attributed to the period.
template <int RED>
struct RunAcc {
  int32_t a;        // MAX: max L ; MIN: min L ; SUM: sum L ; COUNT/MEAN/STD: n runs
  int32_t s;        // MEAN/STD: sum L
  unsigned long long q;  // STD: sum L^2
  __device__ __forceinline__ void init() {
    a = (RED == XC_RL_MIN) ? 0x7fffffff : 0;
    s = 0;
    q = 0ull;
  }
  __device__ __forceinline__ void add(int32_t L, bool take) {
    if constexpr (RED == XC_RL_MAX) a = take ? max(a, L) : a;
    if constexpr (RED == XC_RL_MIN) a = take ? min(a, L) : a;
    if constexpr (RED == XC_RL_SUM) a += take ? L : 0;
    if constexpr (RED == XC_RL_COUNT) a += take ? 1 : 0;
    if constexpr (RED == XC_RL_MEAN || RED == XC_RL_STD) {
      a += take ? 1 : 0;
      s += take ? L : 0;
    }
    if constexpr (RED == XC_RL_STD) q += take ? (unsigned long long)L * (unsigned long long)L : 0ull;
  }
  __device__ __forceinline__ float result() const {
    if constexpr (RED == XC_RL_MAX || RED == XC_RL_SUM || RED == XC_RL_COUNT) return (float)a;
    if constexpr (RED == XC_RL_MIN) return a == 0x7fffffff ? 0.f : (float)a;
    if constexpr (RED == XC_RL_MEAN) return a == 0 ? 0.f : (float)((double)s / (double)a);
    if constexpr (RED == XC_RL_STD) {
      if (a == 0) return 0.f;
      double n = (double)a, m = (double)s / n;
      double var = (double)q / n - m * m;
      return (float)sqrt(var > 0.0 ? var : 0.0);
    }
    return 0.f;
  }
};

// FASTMAX: reducer == max and window == 1 needs no run-end detection: max over t of the running
// length (this is the maximum_consecutive_dry_days configuration).
template <int OP, int RED, int VEC, bool VALID, bool AFTER, bool FASTMAX>
__global__ void __launch_bounds__(kThreads)
period_runstat_kernel(const float* __restrict__ x, int64_t T, int64_t C, int64_t ldx,
                      const int32_t* __restrict__ poff, float thr, int32_t window,
                      float* __restrict__ out, int32_t* __restrict__ valid) {
  const int64_t c0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  if (c0 >= C) return;
  const int p = blockIdx.y;
  const int t0 = poff[p], t1 = poff[p + 1];
  const float* col = x + c0;

  int32_t cur[VEC], nv[VEC];
  bool skip[VEC];
  RunAcc<RED> acc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { cur[i] = 0; nv[i] = 0; skip[i] = false; acc[i].init(); }

  if constexpr (AFTER) {
    // A run already under way at the period start belongs to an earlier period
    // (indices/run_length.py:329-334: run lengths sit on the run's FIRST element).
    if (t0 > 0) {
      Vec<VEC> r;
      r.load(col + (int64_t)(t0 - 1) * ldx);
#pragma unroll
      for (int i = 0; i < VEC; ++i) skip[i] = cmp<OP>(r.v[i], thr);
    }
  }

  auto step = [&](const Vec<VEC>& r) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      bool c = cmp<OP>(r.v[i], thr);
      if constexpr (VALID) nv[i] += (r.v[i] == r.v[i]) ? 1 : 0;
      if constexpr (AFTER) {
        skip[i] = skip[i] && c;
        c = c && !skip[i];
      }
      if constexpr (FASTMAX) {
        cur[i] = c ? cur[i] + 1 : 0;
        acc[i].a = max(acc[i].a, cur[i]);
      } else {
        const int32_t L = cur[i];
        acc[i].add(L, !c && L >= window);
        cur[i] = c ? L + 1 : 0;
      }
    }
  };
  stream_rows<VEC>(col, ldx, t0, t1, step);

  if constexpr (AFTER) {
    // Runs still open at the period end keep their FULL length: read on until they all close.
    // (VALID counts only the period's own steps.)
    int t = t1;
    bool open = false;
#pragma unroll
    for (int i = 0; i < VEC; ++i) open = open || (cur[i] > 0);
    const float* pp = col + (int64_t)t1 * ldx;
    while (open && t < (int)T) {
      Vec<VEC> r;
      r.load(pp);
      open = false;
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        // a cell whose run has closed must not start a new one here (it belongs to a later period)
        bool c = (cur[i] > 0) && cmp<OP>(r.v[i], thr);
        if constexpr (FASTMAX) {
          cur[i] = c ? cur[i] + 1 : 0;
          acc[i].a = max(acc[i].a, cur[i]);
        } else {
          const int32_t L = cur[i];
          acc[i].add(L, !c && L >= window);
          cur[i] = c ? L + 1 : 0;
        }
        open = open || c;
      }
      pp += ldx;
      ++t;
    }
  }
  float res[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    if constexpr (!FASTMAX) acc[i].add(cur[i], cur[i] >= window);  // run closed by the period/series end
    res[i] = acc[i].result();
  }
  store_vec<VEC>(out + (int64_t)p * C + c0, res);
  if constexpr (VALID) store_vec<VEC>(valid + (int64_t)p * C + c0, nv);
}

// ------------------------------------------------------------------------------------------------
// windowed_max_run_sum of the excess over a threshold (indices/run_length.py:491-540 applied to
// `(x - thr).clip(0)`, indices/_threshold.py:2064-2073 `hot_spell_max_magnitude`): per period the
// largest sum of (x - thr) over a run of x > thr (x < thr: thr - x) at least `window` long, 0 if none.
// The excess is formed in float32 like the reference's `tasmax - thresh`; run sums are float64.
// ------------------------------------------------------------------------------------------------
template <int OP, int VEC, bool AFTER>
__global__ void __launch_bounds__(kThreads)
period_run_maxsum_kernel(const float* __restrict__ x, int64_t T, int64_t C, int64_t ldx,
                         const int32_t* __restrict__ poff, float thr, int32_t window, float* __restrict__ out) {
  const int64_t c0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  if (c0 >= C) return;
  const int p = blockIdx.y;
  const int t0 = poff[p], t1 = poff[p + 1];
  const float* col = x + c0;
  int32_t cur[VEC];
  double rs[VEC], best[VEC];
  bool skip[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { cur[i] = 0; rs[i] = 0.0; best[i] = 0.0; skip[i] = false; }
  auto excess = [&](float v) -> float {
    const float d = (OP == XC_OP_GT || OP == XC_OP_GE) ? (v - thr) : (thr - v);
    return (d > 0.f) ? d : 0.f;  // NaN -> 0: not part of a run (rle: da > 0)
  };
  if constexpr (AFTER) {
    if (t0 > 0) {
      Vec<VEC> r;
      r.load(col + (int64_t)(t0 - 1) * ldx);
#pragma unroll
      for (int i = 0; i < VEC; ++i) skip[i] = excess(r.v[i]) > 0.f;
    }
  }
  auto step = [&](const Vec<VEC>& r, bool only_open) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float e = excess(r.v[i]);
      bool in = e > 0.f;
      if constexpr (AFTER) {
        if (!only_open) {
          skip[i] = skip[i] && in;
          in = in && !skip[i];
        } else {
          in = in && (cur[i] > 0);
        }
      }
      if (in) {
        cur[i] += 1;
        rs[i] += (double)e;
      } else {
        if (cur[i] >= window) best[i] = fmax(best[i], rs[i]);
        cur[i] = 0;
        rs[i] = 0.0;
      }
    }
  };
  stream_rows<VEC>(col, ldx, t0, t1, [&](const Vec<VEC>& r) { step(r, false); });
  if constexpr (AFTER) {
    int t = t1;
    bool open = false;
#pragma unroll
    for (int i = 0; i < VEC; ++i) open = open || (cur[i] > 0);
    while (open && t < (int)T) {
      Vec<VEC> r;
      r.load(col + (int64_t)t * ldx);
      step(r, true);
      open = false;
#pragma unroll
      for (int i = 0; i < VEC; ++i) open = open || (cur[i] > 0);
      ++t;
    }
  }
  float res[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    if (cur[i] >= window) best[i] = fmax(best[i], rs[i]);
    res[i] = (float)best[i];
  }
  store_vec<VEC>(out + (int64_t)p * C + c0, res);
}

// ------------------------------------------------------------------------------------------------
// per-period reductions with optional fused transform
// ------------------------------------------------------------------------------------------------
template <int STAT, int TF, int OP, int VEC, bool VALID>
__global__ void __launch_bounds__(kThreads)
period_reduce_kernel(const float* __restrict__ x, int64_t C, int64_t ldx,
                     const int32_t* __restrict__ poff, float thr,
                     float* __restrict__ out, int32_t* __restrict__ valid) {
  const int64_t c0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  if (c0 >= C) return;
  const int p = blockIdx.y;
  const int t0 = poff[p], t1 = poff[p + 1];
  double s[VEC], q[VEC];
  float m[VEC];
  int32_t n[VEC], nv[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    s[i] = 0.0; q[i] = 0.0; n[i] = 0; nv[i] = 0;
    m[i] = (STAT == XC_STAT_MIN) ? INFINITY : -INFINITY;
  }
  stream_rows<VEC>(x + c0, ldx, t0, t1, [&](const Vec<VEC>& r) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float v = r.v[i];
      if constexpr (VALID) nv[i] += (v == v) ? 1 : 0;
      if constexpr (TF == XC_TF_EXCESS) {
        // (x - t).clip(0) / (t - x).clip(0) in float32 (indices/generic.py:1545-1549)
        float d = (OP == XC_OP_GT || OP == XC_OP_GE) ? (v - thr) : (thr - v);
        v = (d != d) ? d : fmaxf(d, 0.f);
      }
      if constexpr (TF == XC_TF_WHERE) v = cmp<OP>(v, thr) ? v : NAN;
      const bool ok = (v == v);
      n[i] += ok ? 1 : 0;
      if constexpr (STAT == XC_STAT_SUM || STAT == XC_STAT_MEAN || STAT == XC_STAT_STD ||
                    STAT == XC_STAT_VAR)
        s[i] += ok ? (double)v : 0.0;
      if constexpr (STAT == XC_STAT_STD || STAT == XC_STAT_VAR) q[i] += ok ? (double)v * (double)v : 0.0;
      if constexpr (STAT == XC_STAT_MIN) m[i] = fminf(m[i], v);  // fminf ignores NaN
      if constexpr (STAT == XC_STAT_MAX) m[i] = fmaxf(m[i], v);
    }
  });
  float res[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const double nn = (double)n[i];
    if constexpr (STAT == XC_STAT_SUM) res[i] = (float)s[i];
    if constexpr (STAT == XC_STAT_COUNT) res[i] = (float)n[i];
    if constexpr (STAT == XC_STAT_MEAN) res[i] = n[i] ? (float)(s[i] / nn) : NAN;
    if constexpr (STAT == XC_STAT_MIN || STAT == XC_STAT_MAX) res[i] = n[i] ? m[i] : NAN;
    if constexpr (STAT == XC_STAT_STD || STAT == XC_STAT_VAR) {
      if (n[i] == 0) {
        res[i] = NAN;
      } else {
        double mean = s[i] / nn;
        double var = q[i] / nn - mean * mean;
        var = var > 0.0 ? var : 0.0;
        res[i] = (STAT == XC_STAT_STD) ? (float)sqrt(var) : (float)var;
      }
    }
  }
  store_vec<VEC>(out + (int64_t)p * C + c0, res);
  if constexpr (VALID) store_vec<VEC>(valid + (int64_t)p * C + c0, nv);
}

inline bool can_vec4(const void* x, int64_t C, int64_t ldx, const void* o1, const void* o2) {
  return (C % 4 == 0) && (ldx % 4 == 0) && aligned16(x) && aligned16(o1) && (o2 == nullptr || aligned16(o2));
}

inline dim3 grid_for(int64_t C, int vec, int32_t P) {
  int64_t nvec = (C + vec - 1) / vec;
  return dim3((unsigned)((nvec + kThreads - 1) / kThreads), (unsigned)P, 1);
}

int32_t check_common(const void* x, int64_t T, int64_t C, int64_t ldx, const void* poff, int32_t P,
                     const void* out) {
  XC_REQUIRE(x != nullptr && out != nullptr && poff != nullptr, "null pointer argument");
  XC_REQUIRE(T > 0 && C > 0 && ldx >= C, "bad shape: T=%lld C=%lld ldx=%lld", (long long)T, (long long)C,
             (long long)ldx);
  XC_REQUIRE(T < 2147483647LL, "time axis too long");
  XC_REQUIRE(P > 0 && P <= 65535, "number of periods must be in [1, 65535], got %d", P);
  return XC_OK;
}


// ------------------------------------------------------------------------------------------------
// threshold count against an ARRAY threshold (indices/generic.py:301-361 with a DataArray threshold:
// numpy compares float32 data with a float64 array in float64, SURVEY.md A.1); thr_tstride = 0 for a
// per-cell threshold (lat, lon), C for one that also varies in time.
// ------------------------------------------------------------------------------------------------
template <int OP>
__global__ void __launch_bounds__(kThreads)
period_count_arr_kernel(const float* __restrict__ x, int64_t C, int64_t ldx, const int32_t* __restrict__ poff,
                        const double* __restrict__ thr, int64_t thr_tstride, int32_t* __restrict__ out) {
  const int64_t c = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (c >= C) return;
  const int p = blockIdx.y;
  const int t0 = poff[p], t1 = poff[p + 1];
  int32_t n = 0;
  const float* px = x + (int64_t)t0 * ldx + c;
  const double* pt = thr + (int64_t)t0 * thr_tstride + c;
#pragma unroll 4
  for (int t = t0; t < t1; ++t) {
    n += cmpd<OP>((double)ld_stream(px), *pt) ? 1 : 0;
    px += ldx;
    pt += thr_tstride;
  }
  out[(int64_t)p * C + c] = n;
}


// ------------------------------------------------------------------------------------------------
// fused multi-output pass: every count / run statistic / reduction that shares (x, periods)
// ------------------------------------------------------------------------------------------------
// One thread = 2 adjacent cells x one period (64-bit loads, kUnroll rows in flight); the state of NC
// conditions (run length, count, longest run), NR windowed run outputs, NM largest-run-sum outputs and NS
// conditional sums lives in registers next to the plain statistics -- about 25 registers per cell for the
// richest pass of the batch (tasmax), so that 4-5 CTAs stay resident per SM.  Per element and cell: 7
// instructions per condition, 3 per run output, ~10 per run sum, 6 per conditional sum, 8 for the plain
// statistics.  The template arguments are the (rounded-up) numbers of each kind: unused entries are
// computed and dropped (their slots are -1).
template <>
struct Vec<2> {
  float v[2];
  __device__ __forceinline__ void load(const float* p) {
    float2 q;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(q.x), "=f"(q.y) : "l"(p));
    v[0] = q.x; v[1] = q.y;
  }
};

// a[j] for a warp-uniform runtime j without dynamic register indexing (which would go through local memory)
template <int N, typename T>
__device__ __forceinline__ T pick_uniform(const T (&a)[N], int j) {
  T r = a[0];
#pragma unroll
  for (int k = 1; k < N; ++k) r = (j == k) ? a[k] : r;
  return r;
}

// Pipe balance (sm_100a issues one warp instruction per clock but the ALU pipe -- compares, selects, integer
// adds, min/max -- and the FMA pipe each take one every OTHER clock): run lengths and counters are kept as
// float32 (exact below 2^24 steps) so that their updates are FFMA / FADD on the FMA pipe,
//     cf = (sgn * v > thr) ? 1 : 0;   len' = cf * len + cf;   fin = len - cf * len;   n += cf
// leaving one FSET and one FMNMX per condition on the ALU pipe, and the run outputs sit at fixed places (two
// per leading condition) so that no select chain is needed to find their condition.  History (tasmax pass of
// the batch, quarter grid, HBM time 1.75 ms): integer state, 4 cells per thread 19.1 ms (255 registers);
// unit list + 2 cells 15.4 ms; float state 13.3 ms (ncu: ALU pipe 74 %, 18 FSEL + 18 ISETP per element in
// the select chains, long_scoreboard 50 % at 16 warps per SM).
// VEC / UNROLL: light passes (no run outputs) take 4 cells per thread, the others 2 cells and more rows in flight;
// grids that cannot be read 16 bytes at a time (cell count or row stride not a multiple of 4, unaligned buffers) take
// 1 cell per thread.
template <int NC, int NCR, int NM, int NS, int VEC, int UNROLL>
__global__ void __launch_bounds__(kThreads)
period_multi_kernel(const float* __restrict__ x, int64_t C, int64_t ldx, const int32_t* __restrict__ poff,
                    const XcMultiPlan plan, float* __restrict__ out, int64_t slot_stride) {
  constexpr int NR = 2 * NCR;
  constexpr int NC1 = NC > 0 ? NC : 1, NR1 = NR > 0 ? NR : 1, NM1 = NM > 0 ? NM : 1, NS1 = NS > 0 ? NS : 1;
  static_assert(NCR <= NC && (NM == 0 || NC > 0), "run outputs need their condition");
  const int64_t c0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  if (c0 >= C) return;
  const int p = blockIdx.y;
  const int t0 = poff[p], t1 = poff[p + 1];
  double s[VEC];
  float mn[VEC], mx[VEC], nok[VEC];
  float c_len[NC1][VEC], c_n[NC1][VEC], c_mx[NC1][VEC];
  float r_acc[NR1][VEC];
  double m_rs[NM1][VEC], m_best[NM1][VEC];
  double q[NS1][VEC];
  // run outputs: value added when a run of length L >= window closes = ra * L + rb  (sum: L, count: 1)
  float r_w[NR1], r_a[NR1], r_b[NR1];
#pragma unroll
  for (int k = 0; k < NR; ++k) {
    r_w[k] = (float)plan.runs[k].window;
    r_a[k] = plan.runs[k].kind == 0 ? 1.f : 0.f;
    r_b[k] = 1.f - r_a[k];
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    s[i] = 0.0; mn[i] = INFINITY; mx[i] = -INFINITY; nok[i] = 0.f;
#pragma unroll
    for (int j = 0; j < NC; ++j) { c_len[j][i] = 0.f; c_n[j][i] = 0.f; c_mx[j][i] = 0.f; }
#pragma unroll
    for (int k = 0; k < NR; ++k) r_acc[k][i] = 0.f;
#pragma unroll
    for (int k = 0; k < NM; ++k) { m_rs[k][i] = 0.0; m_best[k][i] = 0.0; }
#pragma unroll
    for (int k = 0; k < NS; ++k) q[k][i] = 0.0;
  }
  stream_rows<VEC, UNROLL>(x + c0, ldx, t0, t1, [&](const Vec<VEC>& r) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float v = r.v[i];
      const bool ok = (v == v);
      nok[i] += ok ? 1.f : 0.f;
      s[i] += ok ? (double)v : 0.0;
      mn[i] = fminf(mn[i], v);
      mx[i] = fmaxf(mx[i], v);
      float cf[NC1], fin[NC1];   // cf: condition as 1 / 0; fin: length of the run that ends at this step (0: none)
#pragma unroll
      for (int j = 0; j < NC; ++j) {
        cf[j] = (plan.cond[j].sgn * v > plan.cond[j].thr) ? 1.f : 0.f;
        const float L = c_len[j][i];
        fin[j] = __fmaf_rn(-cf[j], L, L);
        c_len[j][i] = __fmaf_rn(cf[j], L, cf[j]);
        c_n[j][i] += cf[j];
        c_mx[j][i] = fmaxf(c_mx[j][i], c_len[j][i]);
      }
#pragma unroll
      for (int k = 0; k < NR; ++k) {   // windows are >= 1: fin == 0 never qualifies
        const float L = fin[k >> 1];
        const float take = (L >= r_w[k]) ? 1.f : 0.f;
        r_acc[k][i] = __fmaf_rn(take, __fmaf_rn(r_a[k], L, r_b[k]), r_acc[k][i]);
      }
      if constexpr (NM > 0) {
        const float e = plan.msum[0].sgn * (v - plan.msum[0].thr0);   // float32 excess, like `tasmax - thresh`
        m_best[0][i] = (fin[0] >= (float)plan.msum[0].window) ? fmax(m_best[0][i], m_rs[0][i]) : m_best[0][i];
        m_rs[0][i] = (cf[0] != 0.f) ? m_rs[0][i] + (double)e : 0.0;
      }
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        if (plan.sums[k].mode == 0) {
          const float d = plan.sums[k].off_sgn * (v - plan.sums[k].off);     // (x - t) / (t - x) in float32
          q[k][i] += ok ? (double)fmaxf(d, 0.f) : 0.0;
        } else {
          q[k][i] += (plan.sums[k].sgn * v > plan.sums[k].thr) ? (double)v : 0.0;
        }
      }
    }
  });
  auto put_f = [&](int slot, const float (&v)[VEC]) {
    if (slot >= 0) store_vec<VEC>(out + (int64_t)slot * slot_stride + (int64_t)p * C + c0, v);
  };
  auto put_i = [&](int slot, const int32_t (&v)[VEC]) {
    if (slot >= 0) store_vec<VEC>(reinterpret_cast<int32_t*>(out) + (int64_t)slot * slot_stride + (int64_t)p * C + c0, v);
  };
  float rf[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) rf[i] = (float)s[i];
  put_f(plan.slot_sum, rf);
#pragma unroll
  for (int i = 0; i < VEC; ++i) rf[i] = (nok[i] != 0.f) ? (float)(s[i] / (double)nok[i]) : NAN;
  put_f(plan.slot_mean, rf);
#pragma unroll
  for (int i = 0; i < VEC; ++i) rf[i] = (nok[i] != 0.f) ? mn[i] : NAN;
  put_f(plan.slot_min, rf);
#pragma unroll
  for (int i = 0; i < VEC; ++i) rf[i] = (nok[i] != 0.f) ? mx[i] : NAN;
  put_f(plan.slot_max, rf);
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    int32_t ri[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) ri[i] = (int32_t)c_n[j][i];
    put_i(plan.cond[j].slot_n, ri);
#pragma unroll
    for (int i = 0; i < VEC; ++i) rf[i] = (c_mx[j][i] >= (float)plan.cond[j].wmax) ? c_mx[j][i] : 0.f;
    put_f(plan.cond[j].slot_max, rf);
  }
#pragma unroll
  for (int k = 0; k < NR; ++k) {      // runs closed by the period end
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float L = c_len[k >> 1][i];
      rf[i] = r_acc[k][i] + ((L >= r_w[k]) ? __fmaf_rn(r_a[k], L, r_b[k]) : 0.f);
    }
    put_f(plan.runs[k].slot, rf);
  }
  if constexpr (NM > 0) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float L = c_len[0][i];
      rf[i] = (float)((L >= (float)plan.msum[0].window) ? fmax(m_best[0][i], m_rs[0][i]) : m_best[0][i]);
    }
    put_f(plan.msum[0].slot, rf);
  }
#pragma unroll
  for (int k = 0; k < NS; ++k) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) rf[i] = (float)q[k][i];
    put_f(plan.sums[k].slot, rf);
  }
}

template <int NC, int NCR, int NM, int NS>
int32_t launch_multi(const float* x, int64_t C, int64_t ldx, const int32_t* poff, int32_t P, const XcMultiPlan& plan,
                     float* out, cudaStream_t st) {
  // 4 cells per thread only pays for the lightest passes (measured: conditional sums are bound by the
  // float32 -> float64 conversions on the XU pipe, more conditions by registers)
  if (!can_vec4(x, C, ldx, out, nullptr)) {
    period_multi_kernel<NC, NCR, NM, NS, 1, kUnroll><<<grid_for(C, 1, P), kThreads, 0, st>>>(x, C, ldx, poff, plan,
                                                                                           out, (int64_t)P * C);
  } else if constexpr (NCR == 0 && NM == 0 && NS == 0 && NC <= 2) {
    period_multi_kernel<NC, NCR, NM, NS, 4, 8><<<grid_for(C, 4, P), kThreads, 0, st>>>(x, C, ldx, poff, plan, out,
                                                                                        (int64_t)P * C);
  } else {
    period_multi_kernel<NC, NCR, NM, NS, 2, 12><<<grid_for(C, 2, P), kThreads, 0, st>>>(x, C, ldx, poff, plan, out,
                                                                                         (int64_t)P * C);
  }
  return launch_status("period_multi_kernel");
}

}  // namespace
}  // namespace xc

using namespace xc;

extern "C" int32_t xc_period_count_f32(const float* x, int64_t T, int64_t C, int64_t ldx,
                                       const int32_t* period_offsets, int32_t P, int32_t op, double thr,
                                       int32_t cmp_f64, int32_t* out_count, int32_t* valid_count,
                                       void* stream) {
  if (int32_t e = check_common(x, T, C, ldx, period_offsets, P, out_count)) return e;
  const float t32 = fold_threshold(op, thr, cmp_f64);
  const bool v4 = can_vec4(x, C, ldx, out_count, valid_count);
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch_op_nan(op, [&](auto OPC) -> int32_t {
    constexpr int OP = decltype(OPC)::value;
    auto go = [&](auto VECC, auto VALC) -> int32_t {
      constexpr int VEC = decltype(VECC)::value;
      constexpr bool VAL = decltype(VALC)::value;
      period_count_kernel<OP, VEC, VAL><<<grid_for(C, VEC, P), kThreads, 0, st>>>(
          x, C, ldx, period_offsets, t32, out_count, valid_count);
      return launch_status("period_count_kernel");
    };
    if (v4) return valid_count ? go(std::integral_constant<int, 4>{}, std::true_type{})
                               : go(std::integral_constant<int, 4>{}, std::false_type{});
    return valid_count ? go(std::integral_constant<int, 1>{}, std::true_type{})
                       : go(std::integral_constant<int, 1>{}, std::false_type{});
  });
}

namespace {
template <int OP, int RED, bool FASTMAX>
int32_t launch_runstat(const float* x, int64_t T, int64_t C, int64_t ldx, const int32_t* poff, int32_t P,
                       float t32, int32_t window, bool after, float* out, int32_t* valid, cudaStream_t st) {
  const bool v4 = can_vec4(x, C, ldx, out, valid);
  auto go = [&](auto VECC, auto VALC, auto AFTC) -> int32_t {
    constexpr int VEC = decltype(VECC)::value;
    constexpr bool VAL = decltype(VALC)::value;
    constexpr bool AFT = decltype(AFTC)::value;
    period_runstat_kernel<OP, RED, VEC, VAL, AFT, FASTMAX><<<grid_for(C, VEC, P), kThreads, 0, st>>>(
        x, T, C, ldx, poff, t32, window, out, valid);
    return launch_status("period_runstat_kernel");
  };
  auto go2 = [&](auto VECC) -> int32_t {
    if (valid) return after ? go(VECC, std::true_type{}, std::true_type{}) : go(VECC, std::true_type{}, std::false_type{});
    return after ? go(VECC, std::false_type{}, std::true_type{}) : go(VECC, std::false_type{}, std::false_type{});
  };
  return v4 ? go2(std::integral_constant<int, 4>{}) : go2(std::integral_constant<int, 1>{});
}
}  // namespace

extern "C" int32_t xc_period_runstat_f32(const float* x, int64_t T, int64_t C, int64_t ldx,
                                         const int32_t* period_offsets, int32_t P, int32_t op, double thr,
                                         int32_t cmp_f64, int32_t reducer, int32_t window,
                                         int32_t resample_before_rl, float* out, int32_t* valid_count,
                                         void* stream) {
  if (int32_t e = check_common(x, T, C, ldx, period_offsets, P, out)) return e;
  XC_REQUIRE(window >= 1, "window must be >= 1, got %d", window);
  XC_REQUIRE(reducer >= XC_RL_MAX && reducer <= XC_RL_STD, "unknown run-length reducer %d", reducer);
  const float t32 = fold_threshold(op, thr, cmp_f64);
  const bool after = resample_before_rl == 0;
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch_op_nan(op, [&](auto OPC) -> int32_t {
    constexpr int OP = decltype(OPC)::value;
#define XC_RS(RED, FAST) \
  return launch_runstat<OP, RED, FAST>(x, T, C, ldx, period_offsets, P, t32, window, after, out, valid_count, st)
    switch (reducer) {
      case XC_RL_MAX:
        if (window == 1) { XC_RS(XC_RL_MAX, true); }
        XC_RS(XC_RL_MAX, false);
      case XC_RL_MIN: XC_RS(XC_RL_MIN, false);
      case XC_RL_SUM: XC_RS(XC_RL_SUM, false);
      case XC_RL_COUNT: XC_RS(XC_RL_COUNT, false);
      case XC_RL_MEAN: XC_RS(XC_RL_MEAN, false);
      default: XC_RS(XC_RL_STD, false);
    }
#undef XC_RS
  });
}

namespace {
template <int STAT, int TF, int OP>
int32_t launch_reduce(const float* x, int64_t C, int64_t ldx, const int32_t* poff, int32_t P, float t32,
                      float* out, int32_t* valid, cudaStream_t st) {
  const bool v4 = can_vec4(x, C, ldx, out, valid);
  auto go = [&](auto VECC, auto VALC) -> int32_t {
    constexpr int VEC = decltype(VECC)::value;
    constexpr bool VAL = decltype(VALC)::value;
    period_reduce_kernel<STAT, TF, OP, VEC, VAL><<<grid_for(C, VEC, P), kThreads, 0, st>>>(x, C, ldx, poff, t32,
                                                                                         out, valid);
    return launch_status("period_reduce_kernel");
  };
  if (v4) return valid ? go(std::integral_constant<int, 4>{}, std::true_type{})
                       : go(std::integral_constant<int, 4>{}, std::false_type{});
  return valid ? go(std::integral_constant<int, 1>{}, std::true_type{})
               : go(std::integral_constant<int, 1>{}, std::false_type{});
}

template <int TF, int OP>
int32_t reduce_stat(int32_t stat, const float* x, int64_t C, int64_t ldx, const int32_t* poff, int32_t P, float t32,
                    float* out, int32_t* valid, cudaStream_t st) {
  switch (stat) {
    case XC_STAT_SUM: return launch_reduce<XC_STAT_SUM, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
    case XC_STAT_MEAN: return launch_reduce<XC_STAT_MEAN, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
    case XC_STAT_MIN: return launch_reduce<XC_STAT_MIN, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
    case XC_STAT_MAX: return launch_reduce<XC_STAT_MAX, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
    case XC_STAT_STD: return launch_reduce<XC_STAT_STD, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
    case XC_STAT_VAR: return launch_reduce<XC_STAT_VAR, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
    case XC_STAT_COUNT: return launch_reduce<XC_STAT_COUNT, TF, OP>(x, C, ldx, poff, P, t32, out, valid, st);
  }
  set_error("unknown reduction %d", stat);
  return XC_ERR_INVALID;
}
}  // namespace

extern "C" int32_t xc_period_reduce_f32(const float* x, int64_t T, int64_t C, int64_t ldx,
                                        const int32_t* period_offsets, int32_t P, int32_t stat,
                                        int32_t transform, int32_t op, double thr, float* out,
                                        int32_t* valid_count, void* stream) {
  if (int32_t e = check_common(x, T, C, ldx, period_offsets, P, out)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  if (transform == XC_TF_NONE)
    return reduce_stat<XC_TF_NONE, XC_OP_GT>(stat, x, C, ldx, period_offsets, P, 0.f, out, valid_count, st);
  // thresholds of the fused transforms are applied in float32 (float32 data op python float)
  const float t32 = (float)thr;
  if (transform == XC_TF_EXCESS) {
    XC_REQUIRE(op >= XC_OP_GT && op <= XC_OP_LE, "Operation `%d` not permitted for indice.", op);
    if (op == XC_OP_GT || op == XC_OP_GE)
      return reduce_stat<XC_TF_EXCESS, XC_OP_GT>(stat, x, C, ldx, period_offsets, P, t32, out, valid_count, st);
    return reduce_stat<XC_TF_EXCESS, XC_OP_LT>(stat, x, C, ldx, period_offsets, P, t32, out, valid_count, st);
  }
  if (transform == XC_TF_WHERE) {
    return dispatch_op(op, [&](auto OPC) -> int32_t {
      constexpr int OP = decltype(OPC)::value;
      return reduce_stat<XC_TF_WHERE, OP>(stat, x, C, ldx, period_offsets, P, t32, out, valid_count, st);
    });
  }
  set_error("unknown transform %d", transform);
  return XC_ERR_INVALID;
}

extern "C" int32_t xc_period_run_maxsum_f32(const float* x, int64_t T, int64_t C, int64_t ldx,
                                            const int32_t* period_offsets, int32_t P, int32_t op, double thr,
                                            int32_t window, int32_t resample_before_rl, float* out, void* stream) {
  if (int32_t e = check_common(x, T, C, ldx, period_offsets, P, out)) return e;
  XC_REQUIRE(window >= 1, "window must be >= 1, got %d", window);
  XC_REQUIRE(op >= XC_OP_GT && op <= XC_OP_LE, "Operation `%d` not permitted for indice.", op);
  const float t32 = (float)thr;
  const bool after = resample_before_rl == 0;
  const bool v4 = can_vec4(x, C, ldx, out, nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  auto go = [&](auto OPC, auto VECC, auto AFTC) -> int32_t {
    constexpr int OP = decltype(OPC)::value;
    constexpr int VEC = decltype(VECC)::value;
    constexpr bool AFT = decltype(AFTC)::value;
    period_run_maxsum_kernel<OP, VEC, AFT><<<grid_for(C, VEC, P), kThreads, 0, st>>>(x, T, C, ldx, period_offsets,
                                                                                   t32, window, out);
    return launch_status("period_run_maxsum_kernel");
  };
  auto go2 = [&](auto OPC) -> int32_t {
    if (v4) return after ? go(OPC, std::integral_constant<int, 4>{}, std::true_type{})
                         : go(OPC, std::integral_constant<int, 4>{}, std::false_type{});
    return after ? go(OPC, std::integral_constant<int, 1>{}, std::true_type{})
                 : go(OPC, std::integral_constant<int, 1>{}, std::false_type{});
  };
  return (op == XC_OP_GT || op == XC_OP_GE) ? go2(std::integral_constant<int, XC_OP_GT>{})
                                            : go2(std::integral_constant<int, XC_OP_LT>{});
}

extern "C" int32_t xc_period_multi_f32(const float* x, int64_t T, int64_t C, int64_t ldx,
                                       const int32_t* period_offsets, int32_t P, const XcMultiPlan* plan_host,
                                       void* out, int32_t n_slots, void* stream) {
  int32_t e = check_common(x, T, C, ldx, period_offsets, P, out);
  if (e) return e;
  XC_REQUIRE(plan_host != nullptr, "null pointer argument");
  XcMultiPlan pl = *plan_host;
  XC_REQUIRE(pl.n_cond >= 0 && pl.n_cond <= XC_MULTI_MAX_COND && pl.n_runs >= 0 && pl.n_runs <= XC_MULTI_MAX_RUNS &&
                 pl.n_runs % 2 == 0 && pl.n_msum >= 0 && pl.n_msum <= XC_MULTI_MAX_MSUM && pl.n_sums >= 0 &&
                 pl.n_sums <= XC_MULTI_MAX_SUMS,
             "plan holds at most %d conditions, %d run outputs (an even number), %d run sums and %d conditional sums",
             XC_MULTI_MAX_COND, XC_MULTI_MAX_RUNS, XC_MULTI_MAX_MSUM, XC_MULTI_MAX_SUMS);
  XC_REQUIRE(pl.n_runs / 2 <= pl.n_cond && (pl.n_msum == 0 || pl.n_cond > 0), "run outputs need their condition");
  auto slot_ok = [&](int32_t sl) { return sl >= -1 && sl < n_slots; };
  bool ok = slot_ok(pl.slot_sum) && slot_ok(pl.slot_mean) && slot_ok(pl.slot_min) && slot_ok(pl.slot_max);
  // entries beyond the declared counts are neutralised (the rounded-up instantiation computes and drops them)
  for (int j = 0; j < XC_MULTI_MAX_COND; ++j) {
    if (j >= pl.n_cond) { pl.cond[j].slot_n = pl.cond[j].slot_max = -1; pl.cond[j].wmax = 1; pl.cond[j].sgn = 0.f; pl.cond[j].thr = 0.f; }
    ok = ok && slot_ok(pl.cond[j].slot_n) && slot_ok(pl.cond[j].slot_max);
  }
  for (int k = 0; k < XC_MULTI_MAX_RUNS; ++k) {
    if (k >= pl.n_runs) { pl.runs[k].slot = -1; pl.runs[k].cond = k / 2; pl.runs[k].window = 1; pl.runs[k].kind = 0; }
    ok = ok && slot_ok(pl.runs[k].slot) && pl.runs[k].window >= 1 && (pl.runs[k].kind == 0 || pl.runs[k].kind == 1) &&
         pl.runs[k].cond == k / 2;
  }
  for (int k = 0; k < XC_MULTI_MAX_MSUM; ++k) {
    if (k >= pl.n_msum) { pl.msum[k].slot = -1; pl.msum[k].cond = 0; pl.msum[k].window = 1; }
    ok = ok && slot_ok(pl.msum[k].slot) && pl.msum[k].window >= 1 && pl.msum[k].cond == 0;
  }
  for (int k = 0; k < XC_MULTI_MAX_SUMS; ++k) {
    if (k >= pl.n_sums) { pl.sums[k].slot = -1; pl.sums[k].mode = 0; }
    ok = ok && slot_ok(pl.sums[k].slot) && (pl.sums[k].mode == 0 || pl.sums[k].mode == 1);
  }
  XC_REQUIRE(ok, "plan: output slot outside [-1, n_slots), window < 1 or run output not at its condition's place");
  cudaStream_t st = (cudaStream_t)stream;
  float* o = (float*)out;
  const int ncr = pl.n_runs / 2;
  int nc = pl.n_cond == 0 ? 0 : (pl.n_cond <= 2 ? 2 : (pl.n_cond <= 4 ? 4 : 6));
  const int nm = pl.n_msum;
  const int ns = pl.n_sums == 0 ? 0 : 3;
#define XC_MULTI(CN, R, M, S) \
  if (nc == CN && ncr == R && nm == M && ns == S) return launch_multi<CN, R, M, S>(x, C, ldx, period_offsets, P, pl, o, st)
#define XC_MULTI_C(CN)                                                                                   \
  XC_MULTI(CN, 0, 0, 0); XC_MULTI(CN, 0, 0, 3); XC_MULTI(CN, 1, 0, 0); XC_MULTI(CN, 1, 0, 3);            \
  XC_MULTI(CN, 2, 0, 0); XC_MULTI(CN, 2, 0, 3); XC_MULTI(CN, 0, 1, 0); XC_MULTI(CN, 0, 1, 3);            \
  XC_MULTI(CN, 1, 1, 0); XC_MULTI(CN, 1, 1, 3); XC_MULTI(CN, 2, 1, 0); XC_MULTI(CN, 2, 1, 3)
  XC_MULTI(0, 0, 0, 0); XC_MULTI(0, 0, 0, 3);
  XC_MULTI_C(2); XC_MULTI_C(4); XC_MULTI_C(6);
#undef XC_MULTI_C
#undef XC_MULTI
  set_error("plan shape not instantiated");
  return XC_ERR_UNSUPPORTED;
}

extern "C" int32_t xc_period_count_arr_f32(const float* x, int64_t T, int64_t C, int64_t ldx,
                                           const int32_t* period_offsets, int32_t P, int32_t op,
                                           const double* thr, int64_t thr_tstride, int32_t* out_count, void* stream) {
  int32_t e = check_common(x, T, C, ldx, period_offsets, P, out_count);
  if (e) return e;
  XC_REQUIRE(thr != nullptr, "null pointer argument");
  XC_REQUIRE(thr_tstride == 0 || thr_tstride >= C, "threshold time stride must be 0 (per cell) or >= C");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((unsigned)((C + kThreads - 1) / kThreads), (unsigned)P, 1);
  return dispatch_op(op, [&](auto OPC) -> int32_t {
    constexpr int OP = decltype(OPC)::value;
    period_count_arr_kernel<OP><<<grid, kThreads, 0, st>>>(x, C, ldx, period_offsets, thr, thr_tstride, out_count);
    return launch_status("period_count_arr_kernel");
  });
}
