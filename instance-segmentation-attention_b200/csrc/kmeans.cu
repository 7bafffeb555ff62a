// GPU embedding clustering: k-means++ seeding + batched-restart Lloyd + best-restart
// selection, all on the device with no host round trip.  Replaces
//   sklearn.cluster.KMeans(n_clusters=k, n_init=35, max_iter=500).fit_predict(X)
// as called by /root/reference/code/lib/prediction.py:72-74, using the same seeds stream
// (numpy RandomState draws are made on the host and handed over as `uniforms`) and the same
// iteration rule (E-step argmin |c|^2-2x.c with first-index ties, mean M-step, empty-cluster
// relocation, strict-then-tol stop, E-step re-run, best inertia unless same clustering).
//
// Arithmetic contract (bit-exact with oracle/kmeans_oracle.c, which documents the mapping to
// scikit-learn's sources):
//   * per-pair arithmetic in fp32, explicit round-to-nearest intrinsics, fixed fmaf order;
//   * every sum over points in exact 64-bit fixed point -> order independent, so atomics and
//     incremental M-step updates ("move the points whose label changed") are exact.
//
// Layout: X is feature-major [C][ld] (what the fg compaction of the NCHW embedding produces),
// so a warp reads 32 consecutive points of one feature per load; every restart keeps its
// labels as u8 [n_init][ld]; per-restart centre sums are int64 [n_init][k][C].
//
// Kernels:  km_prep_max / km_prep_sums / km_prep_center   (one pass each over X)
//           km_seed   one CTA per restart, greedy k-means++ (exact int64 prefix search)
//           km_lloyd  ONE persistent cooperative kernel for all restarts and all iterations:
//                     E-step tiles of every active restart -> grid barrier -> per-restart
//                     update CTA -> grid barrier; then E-step re-run, inertia, selection.
#include "isa_common.cuh"
#include "isa_tcgen05.cuh"
#include <math.h>

namespace {

constexpr int kMaxL = 8;
constexpr int kLloydThreads = 256;
constexpr int kMaxPPT = 4;                      // points per thread in the E-step (2 or 4)
constexpr int kMaxTile = kLloydThreads * kMaxPPT;   // points per work item (upper bound)
constexpr int kSeedThreads = 256;
constexpr int kMaxK = 254;
constexpr int kMaxInit = 64;
constexpr int kSeedMaxCtas = 512;

struct KmScales {
  int S_mean, S_x, S_d, S_t;
  double p_mean, p_x, p_d, p_t;       // 2^S
  double ip_mean, ip_x, ip_d, ip_t;   // 2^-S
};

struct KmWs {
  // header (zeroed)
  unsigned* maxabs_bits;   // [1]
  int* status;             // [1] 0 ok, 1 n<k, 2 non-finite
  unsigned* barrier;       // [1] grid barrier of the Lloyd kernel
  unsigned* seed_barrier;  // [1] grid barrier of the seeding kernel (separate counter: both start from 0)
  long long* colsum;       // [C]
  long long* tolsum;       // [1]
  long long* sums;         // [R][k][C]
  int* cnt;                // [R][k]
  long long* inertia_q;    // [R]
  int* changed;            // [R]
  int* state;              // [R] 0 active, 1 strict, 2 tol/max_iter
  int* n_iter;             // [R]
  long long* seed_pot;     // [k][R][kMaxL] potentials of the candidates of every k-means++ step (atomically summed)
  unsigned long long* seed_prof;   // [6] CTA 0's phase times of the seeding kernel in ns: search, pass 1, pass 2, grid barriers; its search segments, rounds
  size_t zero_bytes;
  // not zeroed
  float* mean;             // [C]
  float* Xc;               // [C][ld]
  float* closest;          // [R][ld]
  float* centers;          // [R][k][C]
  unsigned char* labels;   // [R][ld]
  unsigned char* acct;     // [R][ld]
  int* seed_idx;           // [R][k]
  long long* seed_tot;     // [R][kSeedMaxCtas] per-CTA totals of closest[] (fixed point)
  int* seed_cand;          // [R][kMaxL] candidate indices of the current step
  float* ub;               // [R][ld] Hamerly bounds of the packed-FP32 E-step: upper bound of the distance to the assigned centre
  float* lb;               // [R][ld] ... lower bound of the distance to every other centre
  float* delta;            // [R][k]  how far the last update moved every centre (rounded up)
  unsigned char* Xa;       // tensor-core E-step: Xc as bf16 hi / lo UMMA operand tiles, [half-tile of 128 points][hi | lo][128 x KP]
  float* xn;               // [ld] |x|_2 of every centred point, rounded up (error bound of the tensor-core distances)
  size_t total_bytes;
};

// Tensor-core E-step (km_lloyd_kernel<.., TC = true>): available for C <= 32 and k <= 128.
__host__ __device__ inline bool km_tc_ok(int C, int k) { return C <= 32 && k <= 128; }
__host__ __device__ inline int km_tc_kp(int C) { return C <= 16 ? 16 : 32; }                      // K of the MMAs (multiple of 16)
__host__ __device__ inline int km_tc_halftiles(int ld) { return ((ld + 255) / 256) * 2; }         // 128-point half tiles (even)
__host__ __device__ inline int km_tc_npad(int k) { return k <= 16 ? 16 : k <= 32 ? 32 : k <= 64 ? 64 : 128; }

KmWs km_carve(void* base, int ld, int C, int k, int R) {
  KmWs w;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* r = p ? p + off : nullptr;
    off += isa_align_up(bytes, 256);
    return r;
  };
  w.maxabs_bits = (unsigned*)take(4);
  w.status = (int*)take(4);
  w.barrier = (unsigned*)take(4);
  w.seed_barrier = (unsigned*)take(4);
  w.colsum = (long long*)take(8 * (size_t)C);
  w.tolsum = (long long*)take(8);
  w.sums = (long long*)take(8 * (size_t)R * k * C);
  w.cnt = (int*)take(4 * (size_t)R * k);
  w.inertia_q = (long long*)take(8 * (size_t)R);
  w.changed = (int*)take(4 * (size_t)R);
  w.state = (int*)take(4 * (size_t)R);
  w.n_iter = (int*)take(4 * (size_t)R);
  w.seed_pot = (long long*)take(8 * (size_t)k * R * kMaxL);
  w.seed_prof = (unsigned long long*)take(8 * 8);
  w.zero_bytes = off;
  w.mean = (float*)take(4 * (size_t)C);
  w.Xc = (float*)take(4 * (size_t)C * ld);
  w.closest = (float*)take(4 * (size_t)R * ld);
  w.centers = (float*)take(4 * (size_t)R * k * C);
  w.labels = (unsigned char*)take((size_t)R * ld);
  w.acct = (unsigned char*)take((size_t)R * ld);
  w.seed_idx = (int*)take(4 * (size_t)R * k);
  w.seed_tot = (long long*)take(8 * (size_t)R * kSeedMaxCtas);
  w.seed_cand = (int*)take(4 * (size_t)R * kMaxL);
  w.ub = (float*)take(4 * (size_t)R * ld);
  w.lb = (float*)take(4 * (size_t)R * ld);
  w.delta = (float*)take(4 * (size_t)R * k);
  w.Xa = (unsigned char*)take(km_tc_ok(C, k) ? (size_t)km_tc_halftiles(ld) * 128 * km_tc_kp(C) * 4 : 0);
  w.xn = (float*)take(4 * (size_t)ld);
  w.total_bytes = off;
  return w;
}

__host__ __device__ inline int ceil_log2_int(int v) {
  int b = 0;
  while ((1 << b) < v) ++b;
  return b;
}

// Same rule as isa_km_oracle_scales (oracle/kmeans_oracle.c).
__device__ inline KmScales km_scales(unsigned maxabs_bits, int n, int C) {
  const float maxabs = __uint_as_float(maxabs_bits);
  const int e_m = (maxabs > 0.f) ? (ilogbf(maxabs) + 1) : 0;
  int bits = 0;
  while (bits < 31 && (n >> bits) != 0) ++bits;
  const int e_c = e_m + 1;
  KmScales s;
  s.S_mean = 62 - e_m - bits;
  s.S_x = 62 - e_c - bits;
  s.S_d = 62 - (2 * e_c + 2 + ceil_log2_int(C)) - bits;
  s.S_t = 62 - 2 * e_c - bits - ceil_log2_int(C);
  s.p_mean = ldexp(1.0, s.S_mean); s.ip_mean = ldexp(1.0, -s.S_mean);
  s.p_x = ldexp(1.0, s.S_x);       s.ip_x = ldexp(1.0, -s.S_x);
  s.p_d = ldexp(1.0, s.S_d);       s.ip_d = ldexp(1.0, -s.S_d);
  s.p_t = ldexp(1.0, s.S_t);       s.ip_t = ldexp(1.0, -s.S_t);
  return s;
}

// llrint(ldexp((double)v, S)): the product by a power of two is exact.
__device__ __forceinline__ long long to_fixed(float v, double p2) { return __double2ll_rn(__dmul_rn((double)v, p2)); }

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& epoch) {
  epoch += 1;
  group_barrier(counter, epoch * gridDim.x);
}

// ------------------------------------------------------------------ prep
__global__ void km_prep_max_kernel(const float* __restrict__ X, const int* __restrict__ n_ptr, int ld, int C, int k, KmWs ws) {
  const int n = *n_ptr;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0 && (n < k || n <= 0)) atomicMax(ws.status, 1);
  const int f = blockIdx.y;
  unsigned m = 0;
  bool bad = false;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float a = fabsf(__ldg(X + (size_t)f * ld + i));
    if (!(a <= 3.0e38f)) bad = true;
    m = max(m, __float_as_uint(a));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(ws.maxabs_bits, m);
  if (bad) atomicMax(ws.status, 2);
}

__global__ void km_prep_sums_kernel(const float* __restrict__ X, const int* __restrict__ n_ptr, int ld, int C, KmWs ws) {
  const int n = *n_ptr;
  if (*ws.status) return;
  const KmScales sc = km_scales(*ws.maxabs_bits, n, C);
  const int f = blockIdx.y;
  long long s = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    s += to_fixed(__ldg(X + (size_t)f * ld + i), sc.p_mean);
  s = warp_sum_ll(s);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd((unsigned long long*)(ws.colsum + f), (unsigned long long)s);
}

__global__ void km_prep_center_kernel(const float* __restrict__ X, const int* __restrict__ n_ptr, int ld, int C, KmWs ws) {
  const int n = *n_ptr;
  if (*ws.status) return;
  const KmScales sc = km_scales(*ws.maxabs_bits, n, C);
  const int f = blockIdx.y;
  const float mean = __double2float_rn(__ddiv_rn(__dmul_rn(__ll2double_rn(ws.colsum[f]), sc.ip_mean), (double)n));
  if (blockIdx.x == 0 && threadIdx.x == 0) ws.mean[f] = mean;
  long long t = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float v = __fsub_rn(__ldg(X + (size_t)f * ld + i), mean);
    ws.Xc[(size_t)f * ld + i] = v;
    t += to_fixed(__fmul_rn(v, v), sc.p_t);
  }
  t = warp_sum_ll(t);
  if ((threadIdx.x & 31) == 0 && t) atomicAdd((unsigned long long*)ws.tolsum, (unsigned long long)t);
}

// centres handed in by the caller (array init): subtract the mean like KMeans.fit does.
__global__ void km_init_centers_kernel(const float* __restrict__ init, int R, int k, int C, KmWs ws) {
  if (*ws.status) return;
  const int total = R * k * C;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    ws.centers[i] = __fsub_rn(init[i], ws.mean[i % C]);
    if (i % C == 0) ws.seed_idx[i / C] = -1;
  }
}

// |x|_2 of every centred point, rounded up (xn^2 >= |x|^2 >= 0.9997 xn^2): the error bounds of the E-step filters need it
__global__ void km_prep_xn_kernel(const int* __restrict__ n_ptr, int ld, int C, KmWs ws) {
  const int n = *n_ptr;
  if (*ws.status) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ld) return;
  float nn = 0.f;
  if (i < n)
    for (int f = 0; f < C; ++f) { const float v = ws.Xc[(size_t)f * ld + i]; nn = __fmaf_rn(v, v, nn); }
  ws.xn[i] = __fmul_rn(__fsqrt_rn(nn), 1.0001f);
}

// Tensor-core operand of the points: every centred row split into bf16 hi + lo (x = hi + lo to ~16 mantissa bits) and
// written in the canonical K-major no-swizzle UMMA layout (8 x 16 B core matrices), one block of [hi | lo] per 128 points,
// so that a Lloyd work item of 256 points is ONE bulk copy.  Rows >= n and features >= C are zero.  Also |x|_2 (rounded up).
__global__ void km_prep_tc_kernel(const int* __restrict__ n_ptr, int ld, int C, int KP, KmWs ws) {
  const int n = *n_ptr;
  if (*ws.status) return;
  const int rows = km_tc_halftiles(ld) * 128;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  const int gs = (KP / 8) * 128;
  unsigned char* blk = ws.Xa + (size_t)(row >> 7) * (128 * KP * 4);
  const int r = row & 127;
  float nn = 0.f;
  for (int kc = 0; kc < KP / 8; ++kc) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int f = kc * 8 + i;
      v[i] = (row < n && f < C) ? ws.Xc[(size_t)f * ld + row] : 0.f;
      nn = __fmaf_rn(v[i], v[i], nn);
    }
    uint4 hi, lo;
    split2(v[0], v[1], hi.x, lo.x);
    split2(v[2], v[3], hi.y, lo.y);
    split2(v[4], v[5], hi.z, lo.z);
    split2(v[6], v[7], hi.w, lo.w);
    const int off = (r >> 3) * gs + kc * 128 + (r & 7) * 16;
    *reinterpret_cast<uint4*>(blk + off) = hi;
    *reinterpret_cast<uint4*>(blk + 128 * KP * 2 + off) = lo;
  }
}

// ------------------------------------------------------------------ seeding
// scikit-learn's k-means++ for float32 inputs (sklearn/cluster/_kmeans.py:180-283), decision for decision:
//   * candidate distances through the float64 upcast of _euclidean_distances (pairwise.py): d = -2 x.y + |x|^2 + |y|^2
//     in double (x = the candidate, y = the point), cast to fp32, clamped at 0;
//   * candidates = searchsorted(cumsum(closest_dist_sq), uniform * current_pot): numpy's cumsum of a float32 array is a
//     SEQUENTIAL float32 sum whose rounding drift (~1e-5 of the total) is as large as one point's share, so the picks
//     depend on it -- reproduced exactly, in parallel, by seq_cumsum_search_cta below;
//   * potentials (sums over points, BLAS-order dependent in scikit-learn) = the float32 rounding of the exact
//     fixed-point sum.
// Bit-exact with oracle/kmeans_oracle.c:isa_km_oracle_seed.

// squared distance of a point in (double) registers to a candidate in shared memory; both are zero padded beyond C
// (fma(0, 0, acc) == acc).  Products of two float32 values are exact in double, so fma == mul + add here.
template <int CP>
__device__ __forceinline__ float sqdist_upcast(const double (&x)[CP], double xx, const double* __restrict__ c, double cc) {
  double dot = 0.0;
#pragma unroll
  for (int f2 = 0; f2 < CP; f2 += 2) {
    const double2 cv = *reinterpret_cast<const double2*>(c + f2);
    dot = __fma_rn(cv.x, x[f2], dot);
    dot = __fma_rn(cv.y, x[f2 + 1], dot);
  }
  double d = __dmul_rn(-2.0, dot);
  d = __dadd_rn(d, cc);
  d = __dadd_rn(d, xx);
  const float r = __double2float_rn(d);
  return r > 0.f ? r : 0.f;
}

template <int CP>
__device__ __forceinline__ double sqnorm64(const double (&x)[CP]) {
  double s = 0.0;
#pragma unroll
  for (int f = 0; f < CP; ++f) s = __fma_rn(x[f], x[f], s);
  return s;
}

// float32 value of an exact fixed-point potential: (float)ldexp((double)q, -S_d)
__device__ __forceinline__ float pot_to_float(long long q, double ip_d) { return __double2float_rn(__dmul_rn(__ll2double_rn(q), ip_d)); }

// RandomState.choice(n, p=uniform): first i with fl64((i+1)/n) > u
__device__ inline int first_center_index(double u, int n) {
  long long i = __double2ll_rz(__dmul_rn(u, (double)n));
  if (i > n - 1) i = n - 1;
  if (i < 0) i = 0;
  while (i > 0 && __ddiv_rn((double)i, (double)n) > u) --i;
  while (i < n - 1 && __ddiv_rn((double)(i + 1), (double)n) <= u) ++i;
  return (int)i;
}

// warp sum of non-negative fixed-point values < 2^63 with three REDUX.SUMs on 21-bit limbs
__device__ __forceinline__ long long warp_sum_q(long long q) {
  const unsigned long long u = (unsigned long long)q;
  const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(u & 0x1FFFFFull));
  const unsigned mi = __reduce_add_sync(0xffffffffu, (unsigned)((u >> 21) & 0x1FFFFFull));
  const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(u >> 42));
  return (long long)((unsigned long long)lo + ((unsigned long long)mi << 21) + ((unsigned long long)hi << 42));
}

// ---- searchsorted on a SEQUENTIAL float32 running sum, computed in parallel and bit-exactly.
// S_i = fl32(S_{i-1} + x_i) with x_i >= 0 looks inherently serial (62 k dependent FADDs = 0.13 ms per draw), but while S
// stays inside one binade [2^e, 2^(e+1)) it lives on the grid u = 2^(e-23): S = m u with an integer m, and adding x moves
// m by round-to-nearest-even(x / u) -- an INTEGER increment that depends on the past only through the parity of m (ties).
// So a run of elements is a pair (increment if it starts on an even m, increment if it starts on an odd m), pairs
// compose associatively, and a binade is one parallel scan.  A CTA takes 8192 elements per round (32 per thread:
// sequential composition in registers, warp scan, cross-warp fold), keeps the prefix up to the first run in which m
// would leave the binade (or an element is too large for the grid), replays that single run with real FADDs and goes
// on in the new binade: ~log2(n) replays per search.  A threshold v is crossed in the first run whose final m reaches
// v / u; that run is replayed from its exact start value to get the index.
constexpr int kScanRun = 32;
constexpr unsigned kScanSat = 0x40000000u;        // saturation of the run increments (anything >= 2^24 is "left the binade")
constexpr unsigned kScanLimit = 1u << 24;

struct ScanShared {
  unsigned wsum[kSeedThreads / 32][2];
  int wbad[kSeedThreads / 32];
  int hit[kMaxL];
  float s;              // running sum after everything consumed so far
  int pos;              // first element of the current round
  int lane0;            // first thread of the round whose run is not consumed yet
  unsigned pending;     // thresholds not crossed yet
  unsigned nseg, nround;   // diagnostics: segments / rounds of all searches of this CTA
};

__device__ __forceinline__ unsigned scan_sat_add(unsigned a, unsigned b) {
  const unsigned s = a + b;                        // both <= 2^30
  return s > kScanSat ? kScanSat : s;
}

// The running sum s2 has reached the lowest pending threshold at element idx: record every threshold of `pend` that is
// crossed, take it out of *pending_word, and return {float bits of the next lowest threshold (rounded up: for a float s,
// (double)s >= v  <=>  s >= float_ru(v)), remaining thresholds}.  Out of line: it runs a handful of times per search.
__device__ __noinline__ uint2 scan_cross(float s2, int idx, unsigned pend, const double* v, int L, int* out, unsigned* pending_word) {
  double vmin = __longlong_as_double(0x7ff0000000000000ll);
  const double sd = (double)s2;
  for (int t = 0; t < L; ++t)
    if ((pend >> t) & 1u) {
      if (sd >= v[t]) {
        out[t] = idx;
        pend &= ~(1u << t);
        atomicAnd(pending_word, ~(1u << t));
      } else {
        vmin = fmin(vmin, v[t]);
      }
    }
  return make_uint2(__float_as_uint(__double2float_ru(vmin)), pend);
}

// out[t] = first i with (double)S_i >= v[t], else n - 1 (np.searchsorted(..., side='left') clipped).  Whole CTA.
// A round = 8192 elements, 32 per thread, loaded ONCE into registers; inside a round the runs are consumed in segments:
// quantise the not yet consumed runs on the grid of the current binade, scan, accept the prefix up to the first run that
// leaves the binade, let the thread that owns that run replay it with real FADDs from its registers (it knows its exact
// start value), and continue behind it on the new grid.  The thread owning the run that crosses a threshold resolves
// the index the same way.
__device__ void seq_cumsum_search_cta(const float* __restrict__ cl, int n, const double* v, int L, int* out, ScanShared& sh) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = kSeedThreads / 32;
  __syncthreads();
  if (tid == 0) { sh.s = 0.f; sh.pos = 0; sh.lane0 = 0; sh.pending = (1u << L) - 1u; }
  if (tid < L) out[tid] = n - 1;
  __syncthreads();
  while (true) {
    const int pos = sh.pos;
    if (pos >= n || !sh.pending) break;
    if (tid == 0) ++sh.nround;
    // ---- this thread's run of the round
    const int i0 = pos + tid * kScanRun;
    float xv[kScanRun];
    if (i0 + kScanRun <= n && ((reinterpret_cast<size_t>(cl + i0) & 15) == 0)) {
#pragma unroll
      for (int j4 = 0; j4 < kScanRun / 4; ++j4) {
        const float4 q = __ldcg(reinterpret_cast<const float4*>(cl + i0) + j4);
        xv[4 * j4] = q.x; xv[4 * j4 + 1] = q.y; xv[4 * j4 + 2] = q.z; xv[4 * j4 + 3] = q.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < kScanRun; ++j) xv[j] = (i0 + j < n) ? __ldcg(cl + i0 + j) : 0.f;
    }
    // real float32 adds over this thread's run (registers) from `s0`; the hot path is FADD + one compare per element
    auto replay = [&](float s0, unsigned pend) {
      float s2 = s0;
      double vmin = __longlong_as_double(0x7ff0000000000000ll);
      for (int t = 0; t < L; ++t)
        if ((pend >> t) & 1u) vmin = fmin(vmin, v[t]);
      float vf = __double2float_ru(vmin);
#pragma unroll
      for (int j = 0; j < kScanRun; ++j) {
        s2 = __fadd_rn(s2, xv[j]);                 // elements beyond n are zeros: they cannot cross anything
        if (s2 >= vf) {
          const uint2 r = scan_cross(s2, i0 + j, pend, v, L, out, &sh.pending);
          vf = __uint_as_float(r.x);
          pend = r.y;
        }
      }
      return s2;
    };
    // ---- segments of the round
    while (true) {
      __syncthreads();                                                         // state of the previous segment is visible
      const float S = sh.s;
      const int lane0 = sh.lane0;
      const unsigned pending = sh.pending;
      if (lane0 >= NW * 32 || pos + lane0 * kScanRun >= n || !pending) break;
      __syncthreads();                                                         // everyone has read the state
      if (tid == 0) ++sh.nseg;
      if (!(S >= 0x1p-100f)) {
        // no usable grid yet (zero / tiny running sum): the owner of the next run replays it
        if (tid == lane0) { sh.s = replay(S, pending); sh.lane0 = lane0 + 1; }
        continue;
      }
      const int e = (int)((__float_as_uint(S) >> 23) & 0xffu) - 127;
      const float scale = __uint_as_float((unsigned)(127 + 23 - e) << 23);   // 1 / u
      const float inv = __uint_as_float((unsigned)(127 - 23 + e) << 23);     // u
      const unsigned m = (unsigned)__fmul_rn(S, scale);                      // exact, in [2^23, 2^24)
      if (tid < L) sh.hit[tid] = 0x7fffffff;
      // (increment from an even start, increment from an odd start) of this thread's run on the grid u
      unsigned ie = 0, io = 0;
      bool big = false;
      if (tid >= lane0 && i0 < n) {
#pragma unroll
        for (int j = 0; j < kScanRun; ++j) {
          const float t = __fmul_rn(xv[j], scale);  // exact scaling (a denormal result rounds to 0: increment 0 either way)
          if (!(t < 8388607.f)) big = true;         // rint(t) must fit 23 bits; such an element (x >= ~S / 2) gets a real add
          else {
            // r = rint(t) without a conversion instruction: the mantissa of t + 2^23; fr = t - r in [-1/2, 1/2], exact
            const float tr = __fadd_rn(t, 8388608.f);
            const unsigned r = __float_as_uint(tr) & 0x7fffffu;
            const float fr = __fsub_rn(t, __fsub_rn(tr, 8388608.f));
            // m + t rounds to m + r unless it is a tie (|fr| = 1/2, r even) and m is odd: then to the even neighbour r +- 1
            const unsigned adj = (fr == 0.5f) ? 1u : ((fr == -0.5f) ? 0xffffffffu : 0u);
            ie += r + ((ie & 1u) ? adj : 0u);
            io += r + (((1u + io) & 1u) ? adj : 0u);
          }
        }
      }
      // inclusive warp scan of the pairs (the shuffled-in value is the EARLIER segment)
      unsigned pe = ie, po = io;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned ae = __shfl_up_sync(0xffffffffu, pe, o), ao = __shfl_up_sync(0xffffffffu, po, o);
        if (lane >= o) {
          const unsigned ne = scan_sat_add(ae, (ae & 1u) ? po : pe);
          const unsigned no = scan_sat_add(ao, ((1u + ao) & 1u) ? po : pe);
          pe = ne; po = no;
        }
      }
      if (lane == 31) { sh.wsum[warp][0] = pe; sh.wsum[warp][1] = po; }
      __syncthreads();                                                         // A
      unsigned mw = m;                                                         // m at the start of this warp's runs
      for (int w2 = 0; w2 < warp; ++w2) mw = scan_sat_add(mw, (mw & 1u) ? sh.wsum[w2][1] : sh.wsum[w2][0]);
      const unsigned m_after = scan_sat_add(mw, (mw & 1u) ? po : pe);
      unsigned m_before = __shfl_up_sync(0xffffffffu, m_after, 1);
      if (lane == 0) m_before = mw;
      const bool bad = (tid >= lane0) && (big || m_after >= kScanLimit);
      const unsigned badmask = __ballot_sync(0xffffffffu, bad);
      if (lane == 0) sh.wbad[warp] = badmask ? (__ffs(badmask) - 1) : 32;
      __syncthreads();                                                         // B
      int valid = NW * 32;                                                     // first thread whose run leaves the grid
      for (int w2 = NW - 1; w2 >= 0; --w2)
        if (sh.wbad[w2] < 32) valid = w2 * 32 + sh.wbad[w2];
      // thresholds crossed inside the accepted prefix: S_i >= v  <=>  m_i >= v / u
      for (int t = 0; t < L; ++t) {
        if (!((pending >> t) & 1u)) continue;
        const double need = __dmul_rn(v[t], (double)scale);
        const unsigned hm = __ballot_sync(0xffffffffu, tid >= lane0 && tid < valid && (double)m_after >= need);
        if (hm && lane == 0) atomicMin(&sh.hit[t], warp * 32 + (__ffs(hm) - 1));
      }
      __syncthreads();                                                         // C
      // owners: the runs that cross a threshold (only that threshold is resolved there), the run that leaves the grid
      unsigned mine = 0;
      for (int t = 0; t < L; ++t)
        if (sh.hit[t] == tid) mine |= 1u << t;
      if (mine) replay(__fmul_rn((float)m_before, inv), mine);
      if (tid == valid) {
        // thresholds already owned by an earlier run were taken out of `pending` by their owners (atomicAnd) or are
        // being taken out right now; this run only looks at those that no accepted run crosses
        unsigned rest = pending;
        for (int t = 0; t < L; ++t)
          if (sh.hit[t] != 0x7fffffff) rest &= ~(1u << t);
        sh.s = replay(valid == lane0 ? S : __fmul_rn((float)m_before, inv), rest);
        sh.lane0 = valid + 1;
      } else if (valid == NW * 32 && tid == NW * 32 - 1) {
        sh.s = __fmul_rn((float)m_after, inv);
        sh.lane0 = NW * 32;
      }
    }
    __syncthreads();
    if (tid == 0) { sh.pos = pos + NW * 32 * kScanRun; sh.lane0 = 0; }
    __syncthreads();
  }
  __syncthreads();
}

// Greedy k-means++ for ALL restarts in one cooperative kernel.  The points are partitioned over the CTAs
// (contiguous ranges, multiples of 32); every step of every restart is
//   search   CTA (r mod G) finds the L candidates of restart r: thresholds u * float32(potential) against the
//            sequential float32 running sum of closest[] (seq_cumsum_search_cta)                 -> grid barrier
//   pass 1   potential of every (restart, trial) candidate over the CTA's own points: warp REDUX -> CTA -> one
//            int64 atomic per (restart, trial) and CTA                                           -> grid barrier
//   pass 2   best trial per restart (lowest float32 potential, first wins), closest = min(closest, d(best)),
//            per-CTA totals for the next potential                                               -> grid barrier
// RES (tile-resident): the launch has at least ceil(ld / 256) CTAs, so every CTA owns at most 256 points = one point
// per thread: the point's features stay in REGISTERS (as doubles) and closest[] of all restarts in shared memory for
// the whole seeding (a copy goes to global memory for the searches), and warps without points skip the passes.
template <int CP, bool RES>
__global__ void __launch_bounds__(kSeedThreads, 2)
km_seed_coop_kernel(const int* __restrict__ n_ptr, int ld, int C, int k, int L, int R, const double* __restrict__ uniforms, KmWs ws) {
  extern __shared__ __align__(16) unsigned char seed_smem[];
  const int n = *n_ptr;
  if (*ws.status) return;
  const int G = gridDim.x, b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = kSeedThreads / 32;
  const KmScales sc = km_scales(*ws.maxabs_bits, n, C);
  const float* __restrict__ Xc = ws.Xc;
  const int per = 1 + (k - 1) * L;
  const int RL = R * L;

  double* s_cand = reinterpret_cast<double*>(seed_smem);                       // [R][L][CP] candidate rows (double)
  double* s_cc = s_cand + (size_t)RL * CP;                                     // [R*L] their squared norms
  double* s_v = s_cc + RL;                                                     // [kMaxL] thresholds of the restart being searched
  long long* s_pot = reinterpret_cast<long long*>(s_v + kMaxL);                // [NW][R*L]
  int* s_best = reinterpret_cast<int*>(s_pot + (size_t)NW * RL);               // [R]
  int* s_cidx = s_best + R;                                                    // [R*L] candidate indices of the current step
  float* s_cl = reinterpret_cast<float*>(s_cidx + RL);                         // RES: [R][kSeedThreads] closest[] of this CTA's points
  __shared__ ScanShared s_scan;
  __shared__ long long s_tot;

  const int PT = ((n + G - 1) / G + 31) / 32 * 32;      // points per CTA
  const int p_lo = min(n, b * PT), p_hi = min(n, p_lo + PT);
  unsigned epoch = 0;

  // ---- first centre of every restart (RandomState.choice), closest[] and per-CTA totals
  for (int r = threadIdx.x; r < R; r += kSeedThreads) {
    const int c0 = first_center_index(uniforms[(size_t)r * per], n);
    s_best[r] = c0;
    if (b == 0) ws.seed_idx[(size_t)r * k] = c0;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < R * CP; idx += kSeedThreads) {
    const int r = idx / CP, f = idx % CP;
    s_cand[(size_t)r * L * CP + f] = (f < C) ? (double)Xc[(size_t)f * ld + s_best[r]] : 0.0;
  }
  for (int idx = threadIdx.x; idx < NW * RL; idx += kSeedThreads) s_pot[idx] = 0;
  __syncthreads();
  for (int r = threadIdx.x; r < R; r += kSeedThreads) {
    const double* c = s_cand + (size_t)r * L * CP;
    double s = 0.0;
    for (int f = 0; f < CP; ++f) s = __fma_rn(c[f], c[f], s);
    s_cc[r * L] = s;
  }
  __syncthreads();
  // RES: this thread's point for the whole kernel
  const int my_i = p_lo + threadIdx.x;
  const bool my_ok = my_i < p_hi;
  const bool warp_ok = (p_lo + warp * 32) < p_hi;       // warps without points skip the passes
  double xr[CP];
  double xxr = 0.0;
  if (RES) {
#pragma unroll
    for (int f = 0; f < CP; ++f) xr[f] = (my_ok && f < C) ? (double)Xc[(size_t)f * ld + my_i] : 0.0;
    xxr = sqnorm64<CP>(xr);
  }
  if (RES) {
    if (warp_ok)
      for (int r = 0; r < R; ++r) {
        long long q = 0;
        if (my_ok) {
          const float d = sqdist_upcast<CP>(xr, xxr, s_cand + (size_t)r * L * CP, s_cc[r * L]);
          s_cl[r * kSeedThreads + threadIdx.x] = d;
          ws.closest[(size_t)r * ld + my_i] = d;
          q = to_fixed(d, sc.p_d);
        }
        q = warp_sum_q(q);
        if (lane == 0) s_pot[(size_t)warp * RL + r * L] += q;
      }
  } else
  for (int i0 = p_lo; i0 < p_hi; i0 += kSeedThreads) {
    const int i = i0 + threadIdx.x;
    const bool ok = i < p_hi;
    double x[CP];
#pragma unroll
    for (int f = 0; f < CP; ++f) x[f] = (ok && f < C) ? (double)Xc[(size_t)f * ld + i] : 0.0;
    const double xx = sqnorm64<CP>(x);
    for (int r = 0; r < R; ++r) {
      long long q = 0;
      if (ok) {
        const float d = sqdist_upcast<CP>(x, xx, s_cand + (size_t)r * L * CP, s_cc[r * L]);
        ws.closest[(size_t)r * ld + i] = d;
        q = to_fixed(d, sc.p_d);
      }
      q = warp_sum_q(q);
      if (lane == 0) s_pot[(size_t)warp * RL + r * L] += q;
    }
  }
  __syncthreads();
  for (int r = threadIdx.x; r < R; r += kSeedThreads) {
    long long t = 0;
    for (int w = 0; w < NW; ++w) t += s_pot[(size_t)w * RL + r * L];
    ws.seed_tot[(size_t)r * kSeedMaxCtas + b] = t;
  }
  grid_barrier(ws.seed_barrier, epoch);

  // CTA 0 keeps a coarse phase profile (ns): search, pass 1, pass 2, the three grid barriers
  if (threadIdx.x == 0) { s_scan.nseg = 0; s_scan.nround = 0; }
  unsigned long long t_s = 0, t_p1 = 0, t_p2 = 0, t_bar = 0, t_mark = gtime_ns();
  auto lap = [&](unsigned long long& acc) { const unsigned long long t = gtime_ns(); acc += t - t_mark; t_mark = t; };

  for (int c = 1; c < k; ++c) {
    // ---- search: CTA (r mod G) draws the L candidates of restart r
    for (int r = b; r < R; r += G) {
      __syncthreads();
      if (warp == 0) {
        long long tot = 0;
        for (int g = lane; g < G; g += 32) tot += __ldcg(ws.seed_tot + (size_t)r * kSeedMaxCtas + g);
        tot = warp_sum_ll(tot);
        if (lane == 0) s_tot = tot;
      }
      __syncthreads();
      if (threadIdx.x < L) {
        // rand_vals = random_state.uniform(size=L) * current_pot: float64 * float32 -> float64
        const float pot = pot_to_float(s_tot, sc.ip_d);
        s_v[threadIdx.x] = __dmul_rn(uniforms[(size_t)r * per + 1 + (c - 1) * L + threadIdx.x], (double)pot);
      }
      __syncthreads();
      seq_cumsum_search_cta(ws.closest + (size_t)r * ld, n, s_v, L, ws.seed_cand + (size_t)r * L, s_scan);
    }
    lap(t_s);
    epoch += 1;
    group_barrier_patient(ws.seed_barrier, epoch * gridDim.x);
    lap(t_bar);

    // ---- pass 1: potential of every candidate over this CTA's points
    for (int pair = threadIdx.x; pair < RL; pair += kSeedThreads) s_cidx[pair] = __ldcg(ws.seed_cand + pair);
    for (int idx = threadIdx.x; idx < NW * RL; idx += kSeedThreads) s_pot[idx] = 0;
    __syncthreads();
#pragma unroll 4
    for (int idx = threadIdx.x; idx < RL * CP; idx += kSeedThreads) {
      const int pair = idx / CP, f = idx % CP;
      s_cand[idx] = (f < C) ? (double)Xc[(size_t)f * ld + s_cidx[pair]] : 0.0;
    }
    __syncthreads();
    for (int pair = threadIdx.x; pair < RL; pair += kSeedThreads) {
      const double* cc = s_cand + (size_t)pair * CP;
      double s = 0.0;
      for (int f = 0; f < CP; ++f) s = __fma_rn(cc[f], cc[f], s);
      s_cc[pair] = s;
    }
    __syncthreads();
    if (RES) {
      if (warp_ok)
        for (int r = 0; r < R; ++r) {
          const float cl = my_ok ? s_cl[r * kSeedThreads + threadIdx.x] : 0.f;
#pragma unroll 4
          for (int t = 0; t < L; ++t) {
            long long q = 0;
            if (my_ok) q = to_fixed(fminf(cl, sqdist_upcast<CP>(xr, xxr, s_cand + (size_t)(r * L + t) * CP, s_cc[r * L + t])), sc.p_d);
            q = warp_sum_q(q);
            if (lane == 0) s_pot[(size_t)warp * RL + r * L + t] = q;   // one chunk per CTA: plain store
          }
        }
    } else
    for (int i0 = p_lo; i0 < p_hi; i0 += kSeedThreads) {
      const int i = i0 + threadIdx.x;
      const bool ok = i < p_hi;
      double x[CP];
#pragma unroll
      for (int f = 0; f < CP; ++f) x[f] = (ok && f < C) ? (double)Xc[(size_t)f * ld + i] : 0.0;
      const double xx = sqnorm64<CP>(x);
      for (int r = 0; r < R; ++r) {
        const float cl = ok ? ws.closest[(size_t)r * ld + i] : 0.f;
        for (int t = 0; t < L; ++t) {
          long long q = 0;
          if (ok) q = to_fixed(fminf(cl, sqdist_upcast<CP>(x, xx, s_cand + (size_t)(r * L + t) * CP, s_cc[r * L + t])), sc.p_d);
          q = warp_sum_q(q);
          if (lane == 0) s_pot[(size_t)warp * RL + r * L + t] += q;
        }
      }
    }
    __syncthreads();
    long long* pot_c = ws.seed_pot + (size_t)c * R * kMaxL;
    for (int pair = threadIdx.x; pair < RL; pair += kSeedThreads) {
      long long t = 0;
      for (int w = 0; w < NW; ++w) t += s_pot[(size_t)w * RL + pair];
      if (t) atomicAdd((unsigned long long*)(pot_c + (pair / L) * kMaxL + pair % L), (unsigned long long)t);
    }
    lap(t_p1);
    grid_barrier(ws.seed_barrier, epoch);
    lap(t_bar);

    // ---- best trial per restart (candidates_pot is float32; np.argmin: first lowest); pass 2: closest = min(closest,
    //      d(best)), new per-CTA totals
    for (int r = threadIdx.x; r < R; r += kSeedThreads) {
      int best = 0;
      float bp = 0.f;
      for (int t = 0; t < L; ++t) {
        const float pf = pot_to_float(__ldcg(pot_c + r * kMaxL + t), sc.ip_d);
        if (t == 0 || pf < bp) { bp = pf; best = t; }
      }
      s_best[r] = best;
      if (b == 0) ws.seed_idx[(size_t)r * k + c] = s_cidx[r * L + best];
    }
    for (int idx = threadIdx.x; idx < NW * RL; idx += kSeedThreads) s_pot[idx] = 0;
    __syncthreads();
    if (RES) {
      if (warp_ok)
        for (int r = 0; r < R; ++r) {
          long long q = 0;
          if (my_ok) {
            float* cl = s_cl + r * kSeedThreads + threadIdx.x;
            const int pair = r * L + s_best[r];
            const float nd = fminf(*cl, sqdist_upcast<CP>(xr, xxr, s_cand + (size_t)pair * CP, s_cc[pair]));
            *cl = nd;
            ws.closest[(size_t)r * ld + my_i] = nd;
            q = to_fixed(nd, sc.p_d);
          }
          q = warp_sum_q(q);
          if (lane == 0) s_pot[(size_t)warp * RL + r * L] = q;
        }
    } else
    for (int i0 = p_lo; i0 < p_hi; i0 += kSeedThreads) {
      const int i = i0 + threadIdx.x;
      const bool ok = i < p_hi;
      double x[CP];
#pragma unroll
      for (int f = 0; f < CP; ++f) x[f] = (ok && f < C) ? (double)Xc[(size_t)f * ld + i] : 0.0;
      const double xx = sqnorm64<CP>(x);
      for (int r = 0; r < R; ++r) {
        long long q = 0;
        if (ok) {
          float* cl = ws.closest + (size_t)r * ld + i;
          const int pair = r * L + s_best[r];
          const float nd = fminf(*cl, sqdist_upcast<CP>(x, xx, s_cand + (size_t)pair * CP, s_cc[pair]));
          *cl = nd;
          q = to_fixed(nd, sc.p_d);
        }
        q = warp_sum_q(q);
        if (lane == 0) s_pot[(size_t)warp * RL + r * L] += q;
      }
    }
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += kSeedThreads) {
      long long t = 0;
      for (int w = 0; w < NW; ++w) t += s_pot[(size_t)w * RL + r * L];
      ws.seed_tot[(size_t)r * kSeedMaxCtas + b] = t;
    }
    lap(t_p2);
    grid_barrier(ws.seed_barrier, epoch);
    lap(t_bar);
  }
  // centres of every restart = the picked rows (CTA 0 wrote seed_idx itself)
  if (b == 0) {
    if (threadIdx.x == 0) { ws.seed_prof[0] = t_s; ws.seed_prof[1] = t_p1; ws.seed_prof[2] = t_p2; ws.seed_prof[3] = t_bar;
                            ws.seed_prof[4] = 1000ull * s_scan.nseg; ws.seed_prof[5] = 1000ull * s_scan.nround; }
    __syncthreads();
    for (int idx = threadIdx.x; idx < R * k * C; idx += kSeedThreads) {
      const int rj = idx / C, f = idx % C;
      ws.centers[idx] = Xc[(size_t)f * ld + ws.seed_idx[rj]];
    }
  }
}

size_t seed_smem_bytes(int R, int L, int CP, bool res) {
  const size_t RL = (size_t)R * L;
  return RL * CP * 8 + RL * 8 + kMaxL * 8 + (size_t)(kSeedThreads / 32) * RL * 8 + (size_t)R * 4 + RL * 4 +
         (res ? (size_t)R * kSeedThreads * 4 : 0) + 16;
}

// ------------------------------------------------------------------ Lloyd
struct LloydParams {
  const int* n_ptr;
  int ld, C, k, R, max_iter;
  double tol_rel;
  KmWs ws;
  int* labels_out;      // [ld] int32
  float* centers_out;   // [k][C]
  double* inertia_out;  // [R]
  int* n_iter_out;      // [R]
  int* info;            // [16] status, best restart, n, total Lloyd iterations, then CTA 0's phase profile in us
};

// The packed-FP32 E-step with two points per thread skips, from this Lloyd iteration on, the points whose label provably
// cannot change (Hamerly bounds).  Measured on one B200 box, same process order (Lloyd loop of the four benchmark images,
// 49-52 k points, k = 16, 35 restarts, 3100-3700 restart-iterations): 9.73 / 9.59 / 11.18 / 8.71 ms without, 8.43 / 8.91 /
// 10.50 / 8.20 ms with bounds from iteration 32 (80 % of the point visits skipped; what is left is the wait for the slowest
// CTA, whose range holds the restarts that still move).  Planted clusters that converge in ~50 iterations: 9.26 -> 9.59 ms
// (49 k points), 17.0 -> 17.5 ms (131 k): the bound arrays and the list passes cost 3 % there.  From iteration 1 / 6 / 16
// the planted cases lose 10 / 8 / 4 % (loose bounds while every centre still moves) and the benchmark images gain no more.
constexpr int kBoundsFrom = 32;

typedef unsigned long long km_u64;
__device__ __forceinline__ void km_ffma2(km_u64& acc, km_u64 a, km_u64 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b)); }
__device__ __forceinline__ km_u64 km_pack2(float lo, float hi) {
  km_u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void km_unpack2(km_u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }

// E-step of one tile: labels of PPT points per thread against the centres in smem.  The dot products run on the
// packed FP32 pipe (fma.rn.f32x2 -> FFMA2, two IEEE fmas per instruction, same rounding as __fmaf_rn): two points
// of a thread share one accumulator pair, the centres sit in shared memory duplicated as {c, c} so one LDS.128
// (warp broadcast) feeds two features.  A scalar FFMA issues every other cycle per scheduler on sm_100.
template <int CP, int PPT>
__device__ __forceinline__ void estep_tile(const float* __restrict__ Xc, int ld, int n, int C, int k, int tile,
                                           const float* __restrict__ s_cdup, const float* __restrict__ s_csq, int (&lab)[PPT]) {
  static_assert(PPT % 2 == 0, "points are processed in pairs");
  constexpr int kTileP = kLloydThreads * PPT;
  const int base = tile * kTileP + threadIdx.x;
  km_u64 xp[PPT / 2][CP];
#pragma unroll
  for (int pp = 0; pp < PPT / 2; ++pp) {
    const int i0 = base + (2 * pp) * kLloydThreads, i1 = i0 + kLloydThreads;
#pragma unroll
    for (int f = 0; f < CP; ++f) {
      const float a = (f < C && i0 < n) ? Xc[(size_t)f * ld + i0] : 0.f;
      const float b = (f < C && i1 < n) ? Xc[(size_t)f * ld + i1] : 0.f;
      xp[pp][f] = km_pack2(a, b);
    }
  }
  float bv[PPT];
#pragma unroll
  for (int p = 0; p < PPT; ++p) { bv[p] = 0.f; lab[p] = 0; }
  for (int j = 0; j < k; ++j) {
    const float* __restrict__ c = s_cdup + (size_t)j * 2 * CP;
    km_u64 dot[PPT / 2];
#pragma unroll
    for (int pp = 0; pp < PPT / 2; ++pp) dot[pp] = 0ull;
#pragma unroll
    for (int f2 = 0; f2 < CP; f2 += 2) {
      const ulonglong2 cv = *reinterpret_cast<const ulonglong2*>(c + 2 * f2);   // {c[f2], c[f2]}, {c[f2+1], c[f2+1]}
#pragma unroll
      for (int pp = 0; pp < PPT / 2; ++pp) {
        // zero padding beyond C is exact: fma(0, 0, acc) == acc
        km_ffma2(dot[pp], xp[pp][f2], cv.x);
        km_ffma2(dot[pp], xp[pp][f2 + 1], cv.y);
      }
    }
    const float cs = s_csq[j];
#pragma unroll
    for (int pp = 0; pp < PPT / 2; ++pp) {
      float d0, d1;
      km_unpack2(dot[pp], d0, d1);
      const float v0 = __fmaf_rn(-2.f, d0, cs), v1 = __fmaf_rn(-2.f, d1, cs);
      if (j == 0 || v0 < bv[2 * pp]) { bv[2 * pp] = v0; lab[2 * pp] = j; }
      if (j == 0 || v1 < bv[2 * pp + 1]) { bv[2 * pp + 1] = v1; lab[2 * pp + 1] = j; }
    }
  }
}

// Two points given by their global indices (-1: none) against the centres in shared memory, same arithmetic as
// estep_tile; also returns the best and the second-best score of each point (for the Hamerly bounds).
template <int CP>
__device__ __forceinline__ void estep_pair(const float* __restrict__ Xc, int ld, int C, int k, int i0, int i1,
                                           const float* __restrict__ s_cdup, const float* __restrict__ s_csq, int (&lab)[2],
                                           float (&best)[2], float (&second)[2]) {
  km_u64 xp[CP];
#pragma unroll
  for (int f = 0; f < CP; ++f) {
    const float a = (f < C && i0 >= 0) ? Xc[(size_t)f * ld + i0] : 0.f;
    const float b = (f < C && i1 >= 0) ? Xc[(size_t)f * ld + i1] : 0.f;
    xp[f] = km_pack2(a, b);
  }
  lab[0] = lab[1] = 0;
  best[0] = best[1] = 0.f;
  second[0] = second[1] = 3.4e38f;
  for (int j = 0; j < k; ++j) {
    const float* __restrict__ c = s_cdup + (size_t)j * 2 * CP;
    km_u64 dot = 0ull;
#pragma unroll
    for (int f2 = 0; f2 < CP; f2 += 2) {
      const ulonglong2 cv = *reinterpret_cast<const ulonglong2*>(c + 2 * f2);
      km_ffma2(dot, xp[f2], cv.x);
      km_ffma2(dot, xp[f2 + 1], cv.y);
    }
    const float cs = s_csq[j];
    float d0, d1;
    km_unpack2(dot, d0, d1);
    const float v0 = __fmaf_rn(-2.f, d0, cs), v1 = __fmaf_rn(-2.f, d1, cs);
    if (j == 0 || v0 < best[0]) { if (j) second[0] = best[0]; best[0] = v0; lab[0] = j; } else if (v0 < second[0]) second[0] = v0;
    if (j == 0 || v1 < best[1]) { if (j) second[1] = best[1]; best[1] = v1; lab[1] = j; } else if (v1 < second[1]) second[1] = v1;
  }
}

__device__ __forceinline__ void load_centers(const float* __restrict__ gc, float* s_cent, float* s_csq, int k, int C, int CP,
                                             float* s_cdup = nullptr) {
  for (int idx = threadIdx.x; idx < k * CP; idx += kLloydThreads) {
    const int j = idx / CP, f = idx % CP;
    const float v = (f < C) ? __ldcg(gc + (size_t)j * C + f) : 0.f;
    s_cent[idx] = v;
    if (s_cdup) *reinterpret_cast<float2*>(s_cdup + 2 * idx) = make_float2(v, v);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < k; j += kLloydThreads) {
    float a = 0.f;
    for (int f = 0; f < C; ++f) a = __fmaf_rn(s_cent[j * CP + f], s_cent[j * CP + f], a);
    s_csq[j] = a;
  }
  __syncthreads();
}

// New centres of restart r from the exact fixed-point sums (empty clusters relocated first), centre shift, and the
// convergence decision of Lloyd iteration `it` (sklearn/cluster/_kmeans.py:705-740): run by ONE whole CTA.
template <int CP>
__device__ void lloyd_update_restart(const LloydParams& prm, const KmScales& sc, float tol_abs, int r, int it, int n, float* s_cent, float* s_csq) {
  const int C = prm.C, k = prm.k, ld = prm.ld;
  const KmWs& ws = prm.ws;
  const float* __restrict__ Xc = ws.Xc;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ float s_redf[kLloydThreads / 32];
  __shared__ int s_redi[kLloydThreads / 32];
  __shared__ int s_misc[4];
  long long* gs = ws.sums + (size_t)r * k * C;
  int* gc = ws.cnt + (size_t)r * k;
  float* cen = ws.centers + (size_t)r * k * C;
  unsigned char* labels = ws.labels + (size_t)r * ld;
  unsigned char* acct = ws.acct + (size_t)r * ld;
  // empty clusters (list fixed before any point moves): ascending list by ballot compaction
  __shared__ int s_empty[kMaxK + 2];
  __shared__ int s_nempty;
  if (warp == 0) {
    int m = 0;
    for (int j0 = 0; j0 < k; j0 += 32) {
      const int j = j0 + lane;
      const bool e = (j < k) && (__ldcg(gc + j) == 0);
      const unsigned bal = __ballot_sync(0xffffffffu, e);
      if (e) s_empty[m + __popc(bal & ((1u << lane) - 1u))] = j;
      m += __popc(bal);
    }
    if (lane == 0) s_nempty = m;
  }
  __syncthreads();
  if (s_nempty > 0) {
    // old centres are still in ws.centers; distances of every point to its assigned centre
    load_centers(cen, s_cent, s_csq, k, C, CP);
    __shared__ int s_taken[kMaxK + 2];
    for (int e = 0; e < s_nempty; ++e) {
      float bd = -1.f;
      int bi = 0x7fffffff;
      for (int i = threadIdx.x; i < n; i += kLloydThreads) {
        bool taken = false;
        for (int q = 0; q < e; ++q) taken |= (s_taken[q] == i);
        if (taken) continue;
        const float* c = s_cent + (int)labels[i] * CP;
        float acc = 0.f;
        for (int f = 0; f < C; ++f) { const float t = __fsub_rn(Xc[(size_t)f * ld + i], c[f]); acc = __fmaf_rn(t, t, acc); }
        if (acc > bd) { bd = acc; bi = i; }  // ascending i per thread: lowest index wins ties
      }
      // block arg-max on (distance desc, index asc)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(0xffffffffu, bd, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (od > bd || (od == bd && oi < bi)) { bd = od; bi = oi; }
      }
      if (lane == 0) { s_redf[warp] = bd; s_redi[warp] = bi; }
      __syncthreads();
      if (threadIdx.x == 0) {
        float fd = s_redf[0]; int fi = s_redi[0];
        for (int w = 1; w < kLloydThreads / 32; ++w)
          if (s_redf[w] > fd || (s_redf[w] == fd && s_redi[w] < fi)) { fd = s_redf[w]; fi = s_redi[w]; }
        s_misc[0] = fi;
        s_misc[1] = (e == 0 && !(fd > 0.f)) ? 1 : 0;  // max distance 0: relocation is pointless
        s_taken[e] = fi;
      }
      __syncthreads();
      if (s_misc[1] || s_misc[0] == 0x7fffffff) break;
      const int far = s_misc[0];
      const int j = s_empty[e];
      const int old = acct[far];
      for (int f = threadIdx.x; f < C; f += kLloydThreads) {
        const long long q = to_fixed(Xc[(size_t)f * ld + far], sc.p_x);
        gs[(size_t)old * C + f] -= q;
        gs[(size_t)j * C + f] = q;
      }
      __syncthreads();
      if (threadIdx.x == 0) { gc[old] -= 1; gc[j] = 1; acct[far] = (unsigned char)j; }
      __syncthreads();
    }
  }
  // new centres
  float* s_new = s_cent;  // reuse [k][CP] (old centres are read from global below)
  __syncthreads();
  for (int idx = threadIdx.x; idx < k * C; idx += kLloydThreads) {
    const int j = idx / C, f = idx % C;
    const int cj = gc[j];
    if (cj > 0) s_new[j * CP + f] = __double2float_rn(__ddiv_rn(__dmul_rn(__ll2double_rn(gs[idx]), sc.ip_x), (double)cj));
  }
  if (warp == 0) {
    // argmax of the counts, lowest index among equals (`gc[j] > gc[amax]` scanning upwards)
    int bc = -1, bj = 0x7fffffff;
    for (int j = lane; j < k; j += 32) {
      const int cj = gc[j];
      if (cj > bc) { bc = cj; bj = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int oc = __shfl_xor_sync(0xffffffffu, bc, o), oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (oc > bc || (oc == bc && oj < bj)) { bc = oc; bj = oj; }
    }
    if (lane == 0) s_misc[2] = bj;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < k * C; idx += kLloydThreads) {
    const int j = idx / C, f = idx % C;
    if (gc[j] <= 0) s_new[j * CP + f] = s_new[s_misc[2] * CP + f];
  }
  __syncthreads();
  for (int j = threadIdx.x; j < k; j += kLloydThreads) {
    float acc = 0.f;
    for (int f = 0; f < C; ++f) { const float t = __fsub_rn(s_new[j * CP + f], cen[(size_t)j * C + f]); acc = __fmaf_rn(t, t, acc); }
    s_csq[j] = __fsqrt_rn(acc);
    // upper bound of the true move |c' - c| (the fp32 chain errs by < (C + 2) 2^-24 relative) for the E-step's bounds
    ws.delta[(size_t)r * k + j] = __fadd_ru(__fmul_ru(s_csq[j], 1.0000153f), 1e-30f);
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < k * C; idx += kLloydThreads) cen[idx] = s_new[(idx / C) * CP + idx % C];
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int j = 0; j < k; ++j) tot = __fmaf_rn(s_csq[j], s_csq[j], tot);
    const int changed = __ldcg(ws.changed + r);
    ws.changed[r] = 0;
    int st = 0;
    if (!changed) st = 1;
    else if (tot <= tol_abs) st = 2;
    else if (it + 1 >= prm.max_iter) st = 2;
    if (st) { ws.state[r] = st; ws.n_iter[r] = it + 1; }
  }
  __syncthreads();
}

// Shared-memory layout of the tensor-core E-step (bytes from the start of its region, 128 B aligned pieces).
struct TcLayout {
  int kp, npad, nb, a_stage, b_part;
  size_t a, b, cent, csq, thr, lab, amb, moved, total;
};
__host__ __device__ inline TcLayout km_tc_layout(int C, int CP, int k) {
  TcLayout t;
  t.kp = km_tc_kp(C);
  t.npad = km_tc_npad(k);
  t.nb = 128 / t.npad;                                   // restarts per MMA batch: nb * npad = 128 accumulator columns per half
  t.a_stage = 256 * t.kp * 4;                            // 256 points x (hi + lo) x kp bf16
  t.b_part = 128 * t.kp * 2;                             // 128 centre rows x kp bf16 (one of hi / lo)
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t r = off; off += (bytes + 127) / 128 * 128; return r; };
  t.a = take(2 * (size_t)t.a_stage);
  t.b = take(2 * (size_t)t.b_part);
  t.cent = take((size_t)t.nb * k * CP * 4);
  t.csq = take((size_t)t.nb * t.npad * 4);
  t.thr = take((size_t)t.nb * 2 * 4);
  t.lab = take((size_t)t.nb * 256);
  t.amb = take((size_t)t.nb * 256 * 2);
  t.moved = take((size_t)t.nb * 256 * 4);
  t.total = off;
  return t;
}

template <int CP, int PPT, bool TC>
__global__ void __launch_bounds__(kLloydThreads, (PPT == 2 || TC) ? 2 : 1) km_lloyd_kernel(const LloydParams prm) {
  constexpr int kPPT = TC ? 1 : PPT;
  constexpr int kTile = kLloydThreads * kPPT;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int n = *prm.n_ptr;
  const int C = prm.C, k = prm.k, R = prm.R, ld = prm.ld;
  const KmWs& ws = prm.ws;
  const int status = *ws.status;
  if (status) {
    if (blockIdx.x == 0 && threadIdx.x < 16) prm.info[threadIdx.x] = threadIdx.x == 0 ? status : (threadIdx.x == 2 ? n : 0);
    return;
  }
  float* s_cent = reinterpret_cast<float*>(smem_raw);                       // [k][CP]
  float* s_csq = s_cent + k * CP;                                           // [k]
  float* s_cdup = s_csq + (k + 3) / 4 * 4;                                  // [k][CP] x {c, c} (16 B aligned); FFMA E-step only
  unsigned* s_moved = reinterpret_cast<unsigned*>(s_cdup + (TC ? 0 : (size_t)2 * k * CP));  // [kTile] (point in tile | old << 12 | new << 20)
  // tensor-core E-step: its own region behind the update's centres
  unsigned char* tc_base = smem_raw + (((size_t)(k * CP + (k + 3) / 4 * 4) * 4 + 127) / 128) * 128;
  const TcLayout tl = km_tc_layout(C, CP, k);
  __shared__ uint64_t s_afull[2], s_mma;
  __shared__ uint32_t s_tmem;
  __shared__ unsigned s_namb, s_chg;
  __shared__ int s_batch_r[8];
  __shared__ int s_nmoved;
  __shared__ int s_nneed;
  __shared__ float s_delta[kMaxK + 2], s_bmisc[4];
  __shared__ int s_active[kMaxInit];
  __shared__ int s_nactive;
  __shared__ long long s_redll[kLloydThreads / 32];
  __shared__ float s_redf[kLloydThreads / 32];
  __shared__ int s_redi[kLloydThreads / 32];
  __shared__ int s_misc[4];

  const KmScales sc = km_scales(*ws.maxabs_bits, n, C);
  const float tol_abs = __double2float_rn(__dmul_rn(__ddiv_rn(__dmul_rn(__ll2double_rn(*ws.tolsum), sc.ip_t),
                                                               __dmul_rn((double)n, (double)C)), prm.tol_rel));
  const int tiles = (n + kTile - 1) / kTile;
  const float* __restrict__ Xc = ws.Xc;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned epoch = 0;
  int total_iters = 0;

  // mode 0: Lloyd E-step with incremental M-step; mode 1: labels only (E-step re-run).
  // Incremental M-step: the points of a tile whose cluster changed are compacted into a shared list, then the
  // whole CTA walks (entry, feature) pairs densely and moves each exact fixed-point contribution with native
  // 64-bit global reductions (RED.ADD.64, fire and forget).  r1a did this per thread with 64-bit SHARED atomics
  // (CAS loops) inside divergent code: every warp with one changed lane paid 2*C serialized atomics, and the
  // E-steps took 9 of the kernel's 10 ms.
  auto run_estep = [&](int mode) {
   if constexpr (!TC) {
    const int total = s_nactive * tiles;
    // balanced contiguous ranges (sizes differ by at most one item; ceil-sized ranges left up to half the CTAs idle)
    const int it0 = (int)((long long)blockIdx.x * total / gridDim.x), it1 = (int)((long long)(blockIdx.x + 1) * total / gridDim.x);
    int cur = -1;
    for (int item = it0; item < it1; ++item) {
      const int r = s_active[item / tiles], tile = item % tiles;
      if (r != cur) {
        __syncthreads();
        load_centers(ws.centers + (size_t)r * k * C, s_cent, s_csq, k, C, CP, s_cdup);
        cur = r;
      }
      unsigned char* labels = ws.labels + (size_t)r * ld;
      unsigned char* acct = ws.acct + (size_t)r * ld;
      if (threadIdx.x == 0) s_nmoved = 0;
      __syncthreads();
      // previous labels / accounted clusters are fetched before the distance loop so their latency hides behind it
      int lprev[kPPT], aprev[kPPT];
#pragma unroll
      for (int p = 0; p < kPPT; ++p) {
        const int i = tile * kTile + p * kLloydThreads + threadIdx.x;
        lprev[p] = (i < n) ? labels[i] : 0;
        aprev[p] = (i < n && mode == 0) ? acct[i] : 255;
      }
      int lab[kPPT];
      estep_tile<CP, PPT>(Xc, ld, n, C, k, tile, s_cdup, s_csq, lab);
      bool any_changed = false;
#pragma unroll
      for (int p = 0; p < kPPT; ++p) {
        const int li = p * kLloydThreads + threadIdx.x;     // index inside the tile
        const int i = tile * kTile + li;
        bool moved = false;
        const int a = aprev[p];
        const int l = lab[p];
        if (i < n) {
          if (mode == 0) {
            moved = (l != a);
            if (moved) acct[i] = (unsigned char)l;
          }
          if (l != lprev[p]) { labels[i] = (unsigned char)l; any_changed = true; }
        }
        if (mode == 0) {
          const unsigned bal = __ballot_sync(0xffffffffu, moved);
          if (bal) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&s_nmoved, __popc(bal));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (moved) s_moved[base + __popc(bal & ((1u << lane) - 1u))] = (unsigned)li | ((unsigned)a << 12) | ((unsigned)l << 20);
          }
        }
      }
      const int any = __syncthreads_or(any_changed);        // also publishes s_moved / s_nmoved
      if (mode == 0) {
        if (any && threadIdx.x == 0) ws.changed[r] = 1;
        const int nm = s_nmoved;
        long long* gs = ws.sums + (size_t)r * k * C;
        int* gcnt = ws.cnt + (size_t)r * k;
        // (the guard changes no result; without it ptxas spills in the 24-feature instance at 128 registers)
        if (nm > 0)
        for (int idx = threadIdx.x; idx < nm * C; idx += kLloydThreads) {
          const int e = idx / C, f = idx - e * C;
          const unsigned ent = s_moved[e];
          const int li = ent & 0xfff, a = (ent >> 12) & 0xff, l = (ent >> 20) & 0xff;
          const long long q = to_fixed(Xc[(size_t)f * ld + tile * kTile + li], sc.p_x);
          if (a != 255) atomicAdd((unsigned long long*)(gs + a * C + f), (unsigned long long)(-q));
          atomicAdd((unsigned long long*)(gs + l * C + f), (unsigned long long)q);
          if (f == 0) {
            if (a != 255) atomicSub(gcnt + a, 1);
            atomicAdd(gcnt + l, 1);
          }
        }
      }
    }
   }
  };

  // ---- packed-FP32 E-step with Hamerly bounds (exact).  Per point and restart: U >= |x - c_a| (a = its label), L <= |x - c_j|
  // for every other centre, both shifted by how far the last update moved the centres.  If U^2 + 2 E < L^2, E = bound of the
  // fp32 score error (C + 4) 2^-23 (|c|^2 + 2 |x| |c|), the oracle's fp32 argmin is still a -- strictly, so the first-index
  // tie rule never decides -- and the point is skipped (~80 % of the point visits on the benchmark image).  The bounds of
  // ALL tiles of a CTA's range are tested first (independent loads in flight, next tile prefetched), the points that need
  // their distances are compacted into ONE shared list over the tiles, and the FFMA2 loop runs densely over that list.
  auto run_estep_bounds = [&](int mode) {
    if constexpr (!TC && PPT == 2) {
      constexpr int kCap = 2048;
      __shared__ unsigned s_list[kCap];                 // global index of a point that needs its distances
      __shared__ unsigned short s_prev[kCap];           // its previous label | accounted cluster << 8
      __shared__ unsigned s_mv[kCap + 512];             // moved points: global index
      __shared__ unsigned short s_mval[kCap + 512];     // ... old accounted cluster | new << 8
      __shared__ int s_chg;
      const int total = s_nactive * tiles;
      const float gam = (float)(C + 4) * 0x1p-23f;
      const int tid = threadIdx.x;
      // (Handing out chunks of items through a global counter instead of static ranges was measured: the barrier wait
      // drops from 2.7 to 1.5 ms but every chunk reloads its restart's centres and the loop gets slower, 9.6 vs 8.7 ms.)
      const int it0 = (int)((long long)blockIdx.x * total / gridDim.x), it1 = (int)((long long)(blockIdx.x + 1) * total / gridDim.x);
      if (tid == 0) { s_nneed = 0; s_nmoved = 0; s_chg = 0; }
      __syncthreads();
      {
       int item = it0;
       while (item < it1) {
        const int r = s_active[item / tiles];
        int run_end = (item / tiles + 1) * tiles;                        // items of this restart inside the range
        if (run_end > it1) run_end = it1;
        unsigned char* labels = ws.labels + (size_t)r * ld;
        unsigned char* acct = ws.acct + (size_t)r * ld;
        float* ub = ws.ub + (size_t)r * ld;
        float* lb = ws.lb + (size_t)r * ld;
        __syncthreads();
        load_centers(ws.centers + (size_t)r * k * C, s_cent, s_csq, k, C, CP, s_cdup);
        for (int j = tid; j < k; j += kLloydThreads) s_delta[j] = __ldcg(ws.delta + (size_t)r * k + j);
        __syncthreads();
        if (warp == 0) {
          float dm = 0.f, cm = 0.f;
          for (int j = lane; j < k; j += 32) { dm = fmaxf(dm, s_delta[j]); cm = fmaxf(cm, s_csq[j]); }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) { dm = fmaxf(dm, __shfl_xor_sync(0xffffffffu, dm, o)); cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, o)); }
          if (lane == 0) {
            const float cm2 = __fmul_ru(cm, 1.00001f);
            s_bmisc[0] = dm; s_bmisc[1] = cm2; s_bmisc[2] = __fsqrt_ru(cm2);
          }
        }
        __syncthreads();
        const float dmax = s_bmisc[0], cmax2 = s_bmisc[1], cmax = s_bmisc[2];

        // distances of the listed points, their labels / bounds / moves, then the exact M-step of everything that moved
        auto process_list = [&]() {
          __syncthreads();
          const int nl = s_nneed;
          bool changed = false;
          for (int base = 0; base < nl; base += 2 * kLloydThreads) {
            if (base + warp * 64 >= nl) break;
            const int e0 = base + 2 * tid, e1 = e0 + 1;
            const int ig0 = e0 < nl ? (int)s_list[e0] : -1, ig1 = e1 < nl ? (int)s_list[e1] : -1;
            int lab2[2];
            float best[2], second[2];
            estep_pair<CP>(Xc, ld, C, k, ig0, ig1, s_cdup, s_csq, lab2, best, second);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const int ig = q == 0 ? ig0 : ig1;
              bool moved = false;
              int a = 255;
              const int l = lab2[q];
              if (ig >= 0) {
                const unsigned pv = s_prev[q == 0 ? e0 : e1];
                const int lp = pv & 255;
                a = pv >> 8;
                if (mode == 0) {
                  const float xnv = ws.xn[ig];
                  const float xx_up = __fmul_ru(xnv, xnv), xx_lo = __fmul_rd(__fmul_rd(xnv, xnv), 0.9997f);
                  const float E = __fmaf_ru(xx_up, 0x1p-17f, __fmul_ru(gam, __fmaf_ru(__fmul_ru(2.f, xnv), cmax, cmax2)));
                  const float tu = __fadd_ru(__fadd_ru(xx_up, best[q]), E);
                  float L = 3.0e38f;
                  if (second[q] < 3.0e38f) {
                    const float tlo = __fsub_rd(__fadd_rd(xx_lo, second[q]), E);
                    L = tlo > 0.f ? __fsqrt_rd(tlo) : 0.f;
                  }
                  ub[ig] = tu > 0.f ? __fsqrt_ru(tu) : 0.f;
                  lb[ig] = L;
                  moved = (l != a);
                  if (moved) acct[ig] = (unsigned char)l;
                }
                if (l != lp) { labels[ig] = (unsigned char)l; changed = true; }
              }
              const unsigned bal = __ballot_sync(0xffffffffu, moved);
              if (bal) {
                int mb = 0;
                if (lane == 0) mb = atomicAdd(&s_nmoved, __popc(bal));
                mb = __shfl_sync(0xffffffffu, mb, 0);
                if (moved) {
                  const int slot = mb + __popc(bal & ((1u << lane) - 1u));
                  s_mv[slot] = (unsigned)ig;
                  s_mval[slot] = (unsigned short)(a | (l << 8));
                }
              }
            }
          }
          if (__any_sync(0xffffffffu, changed) && lane == 0) s_chg = 1;
          __syncthreads();
          if (mode == 0) {
            if (s_chg && tid == 0) ws.changed[r] = 1;
            const int nm = s_nmoved;
            long long* gs = ws.sums + (size_t)r * k * C;
            int* gcnt = ws.cnt + (size_t)r * k;
            for (int idx = tid; idx < nm * C; idx += kLloydThreads) {
              const int e = idx / C, f = idx - e * C;
              const int ig = (int)s_mv[e];
              const int a = s_mval[e] & 255, l = s_mval[e] >> 8;
              const long long qv = to_fixed(Xc[(size_t)f * ld + ig], sc.p_x);
              if (a != 255) atomicAdd((unsigned long long*)(gs + a * C + f), (unsigned long long)(-qv));
              atomicAdd((unsigned long long*)(gs + l * C + f), (unsigned long long)qv);
              if (f == 0) {
                if (a != 255) atomicSub(gcnt + a, 1);
                atomicAdd(gcnt + l, 1);
              }
            }
          }
          __syncthreads();
          if (tid == 0) { s_nneed = 0; s_nmoved = 0; s_chg = 0; }
          __syncthreads();
        };

        // ---- bound tests of the run's tiles (the next tile's values are fetched while this one is tested)
        int lpv[2], apv[2];
        float ubv[2], lbv[2], xnv[2];
        auto fetch = [&](int tile) {
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            const int i = tile * kTile + p * kLloydThreads + tid;
            lpv[p] = 255; apv[p] = 255; ubv[p] = 0.f; lbv[p] = 0.f; xnv[p] = 0.f;
            if (i < n) {
              lpv[p] = labels[i];
              if (mode == 0) { apv[p] = acct[i]; ubv[p] = ub[i]; lbv[p] = lb[i]; xnv[p] = ws.xn[i]; }
            }
          }
        };
        fetch(item % tiles);
        for (; item < run_end; ++item) {
          const int tile = item % tiles;
          __syncthreads();                                                // every append of the previous tile is done
          // ONE decision for the CTA (a warp that raced ahead and appended must not change what a slower warp reads)
          if (__syncthreads_or(tid == 0 && s_nneed + kTile > kCap)) process_list();
          int lp[2], ap[2];
          float u_[2], l_[2], x_[2];
#pragma unroll
          for (int p = 0; p < 2; ++p) { lp[p] = lpv[p]; ap[p] = apv[p]; u_[p] = ubv[p]; l_[p] = lbv[p]; x_[p] = xnv[p]; }
          if (item + 1 < run_end) fetch((item + 1) % tiles);
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            const int i = tile * kTile + p * kLloydThreads + tid;
            bool need = i < n, moved = false;
            if (need && mode == 0 && lp[p] != 255) {
              const float U = __fadd_ru(u_[p], s_delta[lp[p]]);
              const float L = fmaxf(__fsub_rd(l_[p], dmax), 0.f);
              const float E = __fmul_ru(gam, __fmaf_ru(__fmul_ru(2.f, x_[p]), cmax, cmax2));
              if (__fmaf_ru(U, U, __fmul_ru(2.0001f, E)) < __fmul_rd(L, L)) {
                need = false;
                ub[i] = U; lb[i] = L;
                moved = (lp[p] != ap[p]);                                 // a relocated point returns to its label's cluster
                if (moved) acct[i] = (unsigned char)lp[p];
              }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, need);
            if (bal) {
              int nb = 0;
              if (lane == 0) nb = atomicAdd(&s_nneed, __popc(bal));
              nb = __shfl_sync(0xffffffffu, nb, 0);
              if (need) {
                const int slot = nb + __popc(bal & ((1u << lane) - 1u));
                s_list[slot] = (unsigned)i;
                s_prev[slot] = (unsigned short)(lp[p] | (ap[p] << 8));
              }
            }
            const unsigned balm = __ballot_sync(0xffffffffu, moved);
            if (balm) {
              int mb = 0;
              if (lane == 0) mb = atomicAdd(&s_nmoved, __popc(balm));
              mb = __shfl_sync(0xffffffffu, mb, 0);
              if (moved) {
                const int slot = mb + __popc(balm & ((1u << lane) - 1u));
                s_mv[slot] = (unsigned)i;
                s_mval[slot] = (unsigned short)(ap[p] | (lp[p] << 8));
              }
            }
          }
        }
        process_list();
       }
      }
    }
  };

  // ---- tensor-core E-step (TC): the distances of 256 points to the centres of up to `nb` restarts are ONE batch of
  // tcgen05 MMAs (D[128 x nb*npad] per half tile, fp32 in tensor memory; bf16 hi/lo split: x c ~ xh ch + xh cl + xl ch, ~2^-16).
  // They are a FILTER, not the result: a point whose best and second-best scores are further apart than the error bound
  // of the tensor-core scores has the same argmin in the oracle's fp32 fmaf arithmetic; the few points inside the bound
  // are recomputed with exactly that arithmetic.  Labels stay bit-exact, ~95 % of the FFMA work moves to the tensor pipe.
  unsigned tc_seq = 0;                                    // work items issued so far by this CTA (mbarrier phases)
  uint32_t tmem = 0;
  if constexpr (TC) {
    if (threadIdx.x == 0) {
      mbar_init(&s_afull[0], 1); mbar_init(&s_afull[1], 1); mbar_init(&s_mma, 1);
      fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(&s_tmem, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tmem = s_tmem;
  }
  auto run_estep_tc = [&](int mode) {
    if constexpr (TC) {
      const int KP = tl.kp, NPAD = tl.npad, NB = tl.nb;
      const int gs = (KP / 8) * 128;
      unsigned char* tc_a = tc_base + tl.a;
      unsigned char* tc_b = tc_base + tl.b;
      float* tc_cent = reinterpret_cast<float*>(tc_base + tl.cent);       // [NB][k][CP]
      float* tc_csq = reinterpret_cast<float*>(tc_base + tl.csq);         // [NB][NPAD] (+huge beyond k)
      float* tc_thr = reinterpret_cast<float*>(tc_base + tl.thr);         // [NB][2]: ambiguity bound = thr0 * |x| + thr1
      unsigned char* tc_lab = tc_base + tl.lab;                           // [NB][256]
      unsigned short* tc_amb = reinterpret_cast<unsigned short*>(tc_base + tl.amb);   // point | slot << 8
      unsigned* tc_moved = reinterpret_cast<unsigned*>(tc_base + tl.moved);           // point | old << 8 | new << 16 | slot << 24
      const int tid = threadIdx.x;
      const int nact = s_nactive;
      const int nbat = (nact + NB - 1) / NB;
      const int total = nbat * tiles;
      const int it0 = (int)((long long)blockIdx.x * total / gridDim.x), it1 = (int)((long long)(blockIdx.x + 1) * total / gridDim.x);
      const uint32_t el = elect_one();
      auto issue_load = [&](int tile, unsigned seq) {
        const unsigned st = seq & 1u;
        mbar_arrive_expect_tx(&s_afull[st], (uint32_t)tl.a_stage);
        tma_bulk_g2s(tc_a + (size_t)st * tl.a_stage, ws.Xa + (size_t)tile * tl.a_stage, (uint32_t)tl.a_stage, &s_afull[st]);
      };
      if (it0 < it1 && tid == 0) issue_load(it0 % tiles, tc_seq);
      int cur_b = -1, nbq = 0;
      const int half = tid >> 7;                                           // which 128-point half of the tile this thread reads
      const uint32_t t_row = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)half * 128u;
      for (int item = it0; item < it1; ++item) {
        const int bi = item / tiles, tile = item % tiles;
        if (bi != cur_b) {
          // ---- centres of the batch: fp32 copy (exact path), |c|^2, bf16 hi / lo B operand, error-bound coefficients
          __syncthreads();
          cur_b = bi;
          nbq = nact - bi * NB < NB ? nact - bi * NB : NB;
          if (tid < 8) s_batch_r[tid] = tid < nbq ? s_active[bi * NB + tid] : 0;
          __syncthreads();
          for (int idx = tid; idx < nbq * k * CP; idx += kLloydThreads) {
            const int q = idx / (k * CP), rem = idx - q * (k * CP), j = rem / CP, f = rem - j * CP;
            tc_cent[idx] = (f < C) ? __ldcg(ws.centers + ((size_t)s_batch_r[q] * k + j) * C + f) : 0.f;
          }
          __syncthreads();
          for (int idx = tid; idx < NB * NPAD; idx += kLloydThreads) {
            const int q = idx / NPAD, j = idx - q * NPAD;
            float a = 3.0e38f;                                             // padded columns never win
            if (q < nbq && j < k) {
              a = 0.f;
              const float* c = tc_cent + ((size_t)q * k + j) * CP;
              for (int f = 0; f < C; ++f) a = __fmaf_rn(c[f], c[f], a);
            }
            tc_csq[idx] = a;
          }
          for (int idx = tid; idx < 128 * (KP / 8); idx += kLloydThreads) {
            const int row = idx / (KP / 8), kc = idx - row * (KP / 8);
            const int q = row / NPAD, j = row - q * NPAD;
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int f = kc * 8 + i;
              v[i] = (q < nbq && j < k && f < CP) ? tc_cent[((size_t)q * k + j) * CP + f] : 0.f;
            }
            uint4 hi, lo;
            split2(v[0], v[1], hi.x, lo.x);
            split2(v[2], v[3], hi.y, lo.y);
            split2(v[4], v[5], hi.z, lo.z);
            split2(v[6], v[7], hi.w, lo.w);
            const int off = (row >> 3) * gs + kc * 128 + (row & 7) * 16;
            *reinterpret_cast<uint4*>(tc_b + off) = hi;
            *reinterpret_cast<uint4*>(tc_b + tl.b_part + off) = lo;
          }
          __syncthreads();
          if (tid < nbq) {
            float cm2 = 0.f;
            for (int j = 0; j < k; ++j) cm2 = fmaxf(cm2, tc_csq[tid * NPAD + j]);
            const float cm = __fmul_rn(__fsqrt_rn(cm2), 1.0001f);
            // |score_tc - score_fp32| <= 2^-13 |x| |c| + 2^-22 |c|^2 (3x the analytic bound: dropped lo*lo terms 3 * 2^-18,
            // tensor-core accumulation, the fmaf chain's own rounding); ambiguous when the gap is within twice that
            tc_thr[2 * tid] = __fmul_rn(cm, 0x1p-12f);
            tc_thr[2 * tid + 1] = __fmul_rn(__fmul_rn(cm, cm), 0x1p-21f);
          }
          fence_proxy_async();
          __syncthreads();
        }
        if (item + 1 < it1 && tid == 0) issue_load((item + 1) % tiles, tc_seq + 1);
        const int i = tile * 256 + tid;
        // previous labels / accounted clusters: fetched before the MMA wait so that their latency hides behind it
        int lprev[8], aprev[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          lprev[q] = 0; aprev[q] = 255;
          if (q < nbq && i < n) {
            const size_t o = (size_t)s_batch_r[q] * ld + i;
            lprev[q] = ws.labels[o];
            if (mode == 0) aprev[q] = ws.acct[o];
          }
        }
        const float xnorm = (i < n) ? ws.xn[i] : 0.f;
        if (tid == 0) { s_nmoved = 0; s_namb = 0; s_chg = 0; }
        // ---- MMAs of the item (warp 0, one elected lane)
        if (warp == 0) {
          const unsigned st = tc_seq & 1u;
          mbar_wait(&s_afull[st], (tc_seq >> 1) & 1u);
          tc_fence_after();
          const uint32_t abase = smem_u32(tc_a + (size_t)st * tl.a_stage);
          const uint32_t idesc = make_idesc(128, nbq * NPAD);
          const uint64_t b_hi = make_desc(smem_u32(tc_b), 128, gs), b_lo = make_desc(smem_u32(tc_b + tl.b_part), 128, gs);
          for (int h = 0; h < 2; ++h) {
            const uint32_t ah = abase + (uint32_t)h * (128 * KP * 4);
            const uint64_t a_hi = make_desc(ah, 128, gs), a_lo = make_desc(ah + 128 * KP * 2, 128, gs);
            const uint32_t d = tmem + (uint32_t)h * 128u;
            for (int kk = 0; kk < KP / 16; ++kk) {
              const uint64_t ko = (uint64_t)((kk * 256) >> 4);
              umma_bf16_e(el, d, a_hi + ko, b_hi + ko, idesc, kk > 0 ? 1u : 0u);
              umma_bf16_e(el, d, a_hi + ko, b_lo + ko, idesc, 1u);
              umma_bf16_e(el, d, a_lo + ko, b_hi + ko, idesc, 1u);
            }
          }
          umma_commit_e(el, &s_mma);
        }
        __syncthreads();                                                    // the counters are reset before anyone appends
        mbar_wait(&s_mma, tc_seq & 1u);
        tc_fence_after();
        // ---- scores -> best / second best per restart; ambiguous (point, restart) pairs go to the exact list
        for (int q = 0; q < nbq; ++q) {
          float best = 3.4e38f, second = 3.4e38f;
          int bl = 0;
          const float* cs = tc_csq + q * NPAD;
          for (int c0 = 0; c0 < NPAD; c0 += 16) {
            uint32_t d[16];
            tmem_ld16_issue(t_row + (uint32_t)(q * NPAD + c0), d);
            tmem_ld16_wait(d);
#pragma unroll
            for (int u = 0; u < 16; ++u) {
              const float v = __fmaf_rn(-2.f, __uint_as_float(d[u]), cs[c0 + u]);
              if (v < best) { second = best; best = v; bl = c0 + u; }
              else if (v < second) second = v;
            }
          }
          tc_lab[q * 256 + tid] = (unsigned char)bl;
          const bool amb = (i < n) && (k > 1) && !(__fsub_rn(second, best) > __fmaf_rn(tc_thr[2 * q], xnorm, tc_thr[2 * q + 1]));
          const unsigned bal = __ballot_sync(0xffffffffu, amb);
          if (bal) {
            int base = 0;
            if (lane == 0) base = (int)atomicAdd(&s_namb, (unsigned)__popc(bal));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (amb) tc_amb[base + __popc(bal & ((1u << lane) - 1u))] = (unsigned short)(tid | (q << 8));
          }
        }
        tc_fence_before();
        __syncthreads();
        // ---- exact path for the ambiguous pairs: the oracle's fmaf chain, strict <, first index wins
        for (int e = tid; e < (int)s_namb; e += kLloydThreads) {
          const int ent = tc_amb[e], pt = ent & 255, q = ent >> 8;
          const int ip = tile * 256 + pt;
          float x[CP];
#pragma unroll
          for (int f = 0; f < CP; ++f) x[f] = (f < C) ? Xc[(size_t)f * ld + ip] : 0.f;
          const float* cq = tc_cent + (size_t)q * k * CP;
          float bv = 0.f;
          int bl = 0;
          for (int j = 0; j < k; ++j) {
            const float* c = cq + j * CP;
            float dot = 0.f;
#pragma unroll
            for (int f = 0; f < CP; ++f) dot = __fmaf_rn(x[f], c[f], dot);
            const float v = __fmaf_rn(-2.f, dot, tc_csq[q * NPAD + j]);
            if (j == 0 || v < bv) { bv = v; bl = j; }
          }
          tc_lab[q * 256 + pt] = (unsigned char)bl;
        }
        __syncthreads();
        // ---- labels, accounted clusters, list of moved points
        for (int q = 0; q < nbq; ++q) {
          const int l = tc_lab[q * 256 + tid];
          bool moved = false, changed = false;
          if (i < n) {
            const size_t o = (size_t)s_batch_r[q] * ld + i;
            if (mode == 0) {
              moved = (l != aprev[q]);
              if (moved) ws.acct[o] = (unsigned char)l;
            }
            if (l != lprev[q]) { ws.labels[o] = (unsigned char)l; changed = true; }
          }
          if (__any_sync(0xffffffffu, changed) && lane == 0) atomicOr(&s_chg, 1u << q);
          if (mode == 0) {
            const unsigned bal = __ballot_sync(0xffffffffu, moved);
            if (bal) {
              int base = 0;
              if (lane == 0) base = atomicAdd(&s_nmoved, __popc(bal));
              base = __shfl_sync(0xffffffffu, base, 0);
              if (moved) tc_moved[base + __popc(bal & ((1u << lane) - 1u))] = (unsigned)tid | ((unsigned)aprev[q] << 8) | ((unsigned)l << 16) | ((unsigned)q << 24);
            }
          }
        }
        __syncthreads();
        if (mode == 0) {
          if (tid < nbq && ((s_chg >> tid) & 1u)) ws.changed[s_batch_r[tid]] = 1;
          const int nm = s_nmoved;
          for (int idx = tid; idx < nm * C; idx += kLloydThreads) {
            const int e = idx / C, f = idx - e * C;
            const unsigned ent = tc_moved[e];
            const int pt = ent & 0xff, a = (ent >> 8) & 0xff, l = (ent >> 16) & 0xff, r = s_batch_r[ent >> 24];
            long long* gsum = ws.sums + (size_t)r * k * C;
            int* gcnt = ws.cnt + (size_t)r * k;
            const long long qv = to_fixed(Xc[(size_t)f * ld + tile * 256 + pt], sc.p_x);
            if (a != 255) atomicAdd((unsigned long long*)(gsum + a * C + f), (unsigned long long)(-qv));
            atomicAdd((unsigned long long*)(gsum + l * C + f), (unsigned long long)qv);
            if (f == 0) {
              if (a != 255) atomicSub(gcnt + a, 1);
              atomicAdd(gcnt + l, 1);
            }
          }
        }
        ++tc_seq;
        __syncthreads();                                                    // lists / labels of the item are consumed
      }
    }
  };

  auto rebuild_active = [&](int want_mode) {
    // want_mode 0: state==0 (still iterating); 1: finished without strict convergence; 2: all.
    // One warp reads the states in parallel (r1a walked them with thread 0: R dependent L2 round trips per iteration).
    __syncthreads();
    if (warp == 0) {
      int m = 0;
      for (int r0 = 0; r0 < R; r0 += 32) {
        const int r = r0 + lane;
        bool take = false;
        if (r < R) {
          const int st = __ldcg(ws.state + r);
          take = (want_mode == 0 && st == 0) || (want_mode == 1 && st == 2) || want_mode == 2;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, take);
        if (take) s_active[m + __popc(bal & ((1u << lane) - 1u))] = r;
        m += __popc(bal);
      }
      if (lane == 0) s_nactive = m;
    }
    __syncthreads();
  };

  for (int idx = blockIdx.x * kLloydThreads + threadIdx.x; idx < R * k; idx += gridDim.x * kLloydThreads) ws.delta[idx] = 0.f;
  // labels / acct start as "none" (255)
  for (size_t idx = (size_t)blockIdx.x * kLloydThreads + threadIdx.x; idx < (size_t)R * ld; idx += (size_t)gridDim.x * kLloydThreads) {
    ws.labels[idx] = 255;
    ws.acct[idx] = 255;
    ws.ub[idx] = __int_as_float(0x7f800000);      // no bounds yet: the first E-step computes every point
    ws.lb[idx] = 0.f;
  }
  grid_barrier(ws.barrier, epoch);

  // CTA 0 keeps a coarse phase profile (ns): E-step, barrier after it, update, barrier after it
  unsigned long long t_e = 0, t_b1 = 0, t_u = 0, t_b2 = 0, t_mark = gtime_ns();
  const unsigned long long t_start = t_mark;
  auto lap = [&](unsigned long long& acc) { const unsigned long long t = gtime_ns(); acc += t - t_mark; t_mark = t; };

  for (int it = 0; it < prm.max_iter; ++it) {
    rebuild_active(0);
    if (s_nactive == 0) break;
    ++total_iters;
    // the bounds pay once most points have settled: the first iterations (nearly every point moves, the bounds are loose)
    // take the plain path; the first bounded iteration starts from U = inf and computes every point
    if constexpr (TC) run_estep_tc(0); else if (PPT == 2 && it >= kBoundsFrom) run_estep_bounds(0); else run_estep(0);
    lap(t_e);
    grid_barrier(ws.barrier, epoch);
    lap(t_b1);

    // ---- per-restart update: one CTA per active restart
    for (int a = blockIdx.x; a < s_nactive; a += gridDim.x)
      lloyd_update_restart<CP>(prm, sc, tol_abs, s_active[a], it, n, s_cent, s_csq);
    lap(t_u);
    grid_barrier(ws.barrier, epoch);
    lap(t_b2);
  }
  const unsigned long long t_loop_end = gtime_ns();

  // ---- E-step re-run for restarts that did not converge strictly
  rebuild_active(1);
  if (s_nactive > 0) { if constexpr (TC) run_estep_tc(1); else run_estep(1); }
  grid_barrier(ws.barrier, epoch);

  // ---- inertia of every restart (direct-form distances, exact fixed-point sum)
  rebuild_active(2);
  {
    const int total = R * tiles;
    const int it0 = (int)((long long)blockIdx.x * total / gridDim.x), it1 = (int)((long long)(blockIdx.x + 1) * total / gridDim.x);
    int cur = -1;
    long long acc = 0;
    auto flush_inertia = [&](int r) {
      long long v = warp_sum_ll(acc);
      if (lane == 0) s_redll[warp] = v;
      __syncthreads();
      if (threadIdx.x == 0) {
        long long t = 0;
        for (int w = 0; w < kLloydThreads / 32; ++w) t += s_redll[w];
        if (t) atomicAdd((unsigned long long*)(ws.inertia_q + r), (unsigned long long)t);
      }
      __syncthreads();
      acc = 0;
    };
    for (int item = it0; item < it1; ++item) {
      const int r = item / tiles, tile = item % tiles;
      if (r != cur) {
        if (cur >= 0) flush_inertia(cur);
        __syncthreads();
        load_centers(ws.centers + (size_t)r * k * C, s_cent, s_csq, k, C, CP);
        cur = r;
      }
      const unsigned char* labels = ws.labels + (size_t)r * ld;
#pragma unroll
      for (int p = 0; p < kPPT; ++p) {
        const int i = tile * kTile + p * kLloydThreads + threadIdx.x;
        if (i < n) {
          const float* c = s_cent + (int)labels[i] * CP;
          float d = 0.f;
          for (int f = 0; f < C; ++f) { const float t = __fsub_rn(Xc[(size_t)f * ld + i], c[f]); d = __fmaf_rn(t, t, d); }
          acc += to_fixed(d, sc.p_d);
        }
      }
    }
    if (cur >= 0) flush_inertia(cur);
  }
  grid_barrier(ws.barrier, epoch);

  // ---- best restart: lowest inertia unless it is the same clustering (KMeans.fit, _kmeans.py:1534-1541)
  if (blockIdx.x == 0) {
    __shared__ int s_mapmin[256], s_mapmax[256];
    int best = 0;
    for (int r = 1; r < R; ++r) {
      if (__ldcg(ws.inertia_q + r) < __ldcg(ws.inertia_q + best)) {
        for (int j = threadIdx.x; j < 256; j += kLloydThreads) { s_mapmin[j] = 0x7fffffff; s_mapmax[j] = -1; }
        __syncthreads();
        const unsigned char* l1 = ws.labels + (size_t)r * ld;
        const unsigned char* l2 = ws.labels + (size_t)best * ld;
        for (int i = threadIdx.x; i < n; i += kLloydThreads) {
          const int a = l1[i], b = l2[i];
          if (s_mapmin[a] > b) atomicMin(&s_mapmin[a], b);
          if (s_mapmax[a] < b) atomicMax(&s_mapmax[a], b);
        }
        __syncthreads();
        const int bad = __syncthreads_or(threadIdx.x < 256 && s_mapmax[threadIdx.x] >= 0 && s_mapmin[threadIdx.x] != s_mapmax[threadIdx.x]);
        if (bad) best = r;  // not the same clustering -> take the better restart
      }
    }
    const unsigned char* lb = ws.labels + (size_t)best * ld;
    for (int i = threadIdx.x; i < n; i += kLloydThreads) prm.labels_out[i] = lb[i];
    for (int idx = threadIdx.x; idx < k * C; idx += kLloydThreads)
      prm.centers_out[idx] = __fadd_rn(ws.centers[(size_t)best * k * C + idx], ws.mean[idx % C]);
    for (int r = threadIdx.x; r < R; r += kLloydThreads) {
      prm.inertia_out[r] = __dmul_rn(__ll2double_rn(ws.inertia_q[r]), sc.ip_d);
      prm.n_iter_out[r] = ws.n_iter[r];
    }
    if (threadIdx.x == 0) {
      prm.info[0] = 0; prm.info[1] = best; prm.info[2] = n; prm.info[3] = total_iters;
      prm.info[4] = (int)(t_e / 1000); prm.info[5] = (int)(t_b1 / 1000); prm.info[6] = (int)(t_u / 1000); prm.info[7] = (int)(t_b2 / 1000);
      prm.info[8] = (int)((t_loop_end - t_start) / 1000); prm.info[9] = (int)((gtime_ns() - t_loop_end) / 1000);
      for (int q = 0; q < 6; ++q) prm.info[10 + q] = (int)(ws.seed_prof[q] / 1000);   // seeding kernel: search, pass 1, pass 2, barriers (us); search segments, rounds
    }
  }
  if constexpr (TC) {
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
  }
}


size_t lloyd_smem_bytes(int k, int C, int CP) {
  size_t fl = (size_t)3 * k * CP + (k + 3) / 4 * 4;
  return fl * 4 + (size_t)kMaxTile * 4 + 16;
}
size_t lloyd_tc_smem_bytes(int k, int C, int CP) {
  const size_t base = (((size_t)(k * CP + (k + 3) / 4 * 4) * 4 + 127) / 128) * 128;
  return base + km_tc_layout(C, CP, k).total + 128;
}

template <int CP, bool RES>
int launch_seed_v(const int* n_ptr, int ld, int C, int k, int L, int R, const double* uniforms, const KmWs& ws, int num_sms, cudaStream_t stream,
                  bool* launched) {
  const size_t smem = seed_smem_bytes(R, L, CP, RES);
  const void* fn = (const void*)km_seed_coop_kernel<CP, RES>;
  *launched = false;
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  if (smem > (size_t)di.max_smem_optin) {
    ISA_CHECK_ARG(RES, "kmeans: seeding kernel needs %zu B of shared memory", smem);
    return ISA_OK;   // resident variant does not fit: the caller falls back to the streaming variant
  }
  if (smem > 48 * 1024) ISA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  ISA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, kSeedThreads, smem));
  if (occ > 2) occ = 2;
  int grid;
  if (RES) {
    grid = (ld + kSeedThreads - 1) / kSeedThreads;      // one point per thread
    if (occ < 1 || grid > num_sms * occ || grid > kSeedMaxCtas) return ISA_OK;   // too many points to keep resident
  } else {
    ISA_CHECK_ARG(occ >= 1, "kmeans: seeding kernel does not fit on an SM (smem %zu)", smem);
    grid = num_sms * occ;
    const int want = (ld + 127) / 128;       // no point in CTAs with fewer than ~128 points
    if (grid > want) grid = want;
    if (grid > kSeedMaxCtas) grid = kSeedMaxCtas;
    if (grid < 1) grid = 1;
  }
  void* args[] = {(void*)&n_ptr, (void*)&ld, (void*)&C, (void*)&k, (void*)&L, (void*)&R, (void*)&uniforms, (void*)&ws};
  ISA_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kSeedThreads), args, smem, stream));
  *launched = true;
  return ISA_OK;
}

template <int CP>
int launch_seed(const int* n_ptr, int ld, int C, int k, int L, int R, const double* uniforms, const KmWs& ws, int num_sms, cudaStream_t stream) {
  bool launched = false;
  const int rc = launch_seed_v<CP, true>(n_ptr, ld, C, k, L, R, uniforms, ws, num_sms, stream, &launched);
  if (rc || launched) return rc;
  return launch_seed_v<CP, false>(n_ptr, ld, C, k, L, R, uniforms, ws, num_sms, stream, &launched);
}

// Tensor-core E-step (C <= 32, k <= 128): two CTAs per SM, 256 tensor-memory columns each.
template <int CP>
int launch_lloyd_tc(const LloydParams& prm, int num_sms, cudaStream_t stream) {
  if constexpr (CP <= 32) {
    const size_t smem = lloyd_tc_smem_bytes(prm.k, prm.C, CP);
    const void* fn = (const void*)km_lloyd_kernel<CP, 2, true>;
    ISA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    ISA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, kLloydThreads, smem));
    ISA_CHECK_ARG(occ >= 1, "kmeans: tensor-core Lloyd kernel does not fit on an SM (smem %zu)", smem);
    if (occ > 2) occ = 2;
    km_prep_tc_kernel<<<(km_tc_halftiles(prm.ld) * 128 + 255) / 256, 256, 0, stream>>>(prm.n_ptr, prm.ld, prm.C, km_tc_kp(prm.C), prm.ws);
    ISA_CUDA(cudaGetLastError());
    void* args[] = {(void*)&prm};
    ISA_CUDA(cudaLaunchCooperativeKernel(fn, dim3(num_sms * occ), dim3(kLloydThreads), args, smem, stream));
    return ISA_OK;
  } else {
    return ISA_ERR_UNSUPPORTED;
  }
}

template <int CP, int PPT>
int launch_lloyd_ppt(const LloydParams& prm, int num_sms, cudaStream_t stream) {
  const size_t smem = lloyd_smem_bytes(prm.k, prm.C, CP);
  const void* fn = (const void*)km_lloyd_kernel<CP, PPT, false>;
  ISA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   // static + dynamic may exceed 48 KB
  int occ = 0;
  ISA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, kLloydThreads, smem));
  ISA_CHECK_ARG(occ >= 1, "kmeans: Lloyd kernel does not fit on an SM (smem %zu)", smem);
  if (occ > 2) occ = 2;
  void* args[] = {(void*)&prm};
  ISA_CUDA(cudaLaunchCooperativeKernel(fn, dim3(num_sms * occ), dim3(kLloydThreads), args, smem, stream));
  return ISA_OK;
}

template <int CP>
int launch_lloyd(const LloydParams& prm, int num_sms, cudaStream_t stream) {
  // Tensor-core E-step from 33 centres on.  Measured on B200 (tools/bench_kmeans.py): k = 64, C = 32, 524 k points: 114 ms
  // against 135 ms for the packed-FP32 kernel (E-steps 60 / 80 ms); k = 16, C = 24: 10.3 against 8.9 ms (49 k points),
  // 19.2 against 16.7 ms (131 k): with 16 centres the per-item costs of the batch (operand conversion, MMA round trip,
  // tensor-memory reads, the exact pass) outweigh the 384 FFMAs per point they replace.
  if (CP <= 32 && km_tc_ok(prm.C, prm.k) && prm.k > 32) return launch_lloyd_tc<CP>(prm, num_sms, stream);
  // packed FP32: 2 points per thread and two CTAs per SM (one CTA's loads overlap the other's distance loop) unless the
  // embedding is too wide for 128 registers
  if constexpr (CP <= 32) return launch_lloyd_ppt<CP, 2>(prm, num_sms, stream);
  else return launch_lloyd_ppt<CP, 4>(prm, num_sms, stream);
}

int pick_cp(int C) { return C <= 8 ? 8 : C <= 16 ? 16 : C <= 24 ? 24 : C <= 32 ? 32 : 64; }

}  // namespace

extern "C" {

size_t isa_kmeans_workspace_bytes(int ld, int C, int k, int n_init) {
  if (ld <= 0 || C <= 0 || k <= 0 || n_init <= 0) return 0;
  return km_carve(nullptr, ld, C, k, n_init).total_bytes;
}

int isa_kmeans_fit(const float* X, const int* n_ptr, int ld, int C, int k, int n_init, int max_iter, double tol_rel,
                   int n_local_trials, const double* uniforms, const float* init_centers,
                   int* labels_out, float* centers_out, double* inertia_out, int* n_iter_out, int* seed_idx_out, int* info,
                   void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  ISA_CHECK_ARG(X && n_ptr && labels_out && centers_out && inertia_out && n_iter_out && info && workspace, "kmeans_fit: null pointer");
  ISA_CHECK_ARG(uniforms || init_centers, "kmeans_fit: need either the uniforms of the k-means++ stream or init_centers");
  ISA_CHECK_ARG(ld > 0 && C > 0 && C <= 64, "kmeans_fit: need 0 < C <= 64 (got C=%d, ld=%d)", C, ld);
  ISA_CHECK_ARG(k > 0 && k <= kMaxK, "kmeans_fit: need 0 < k <= %d (uint8 instance mask), got %d", kMaxK, k);
  ISA_CHECK_ARG(n_init > 0 && n_init <= kMaxInit, "kmeans_fit: need 0 < n_init <= %d, got %d", kMaxInit, n_init);
  ISA_CHECK_ARG(max_iter > 0, "kmeans_fit: max_iter must be positive");
  ISA_CHECK_ARG(n_local_trials > 0 && n_local_trials <= kMaxL, "kmeans_fit: n_local_trials %d not in 1..%d", n_local_trials, kMaxL);
  KmWs ws = km_carve(workspace, ld, C, k, n_init);
  if (workspace_bytes < ws.total_bytes) {
    isa_set_error("kmeans_fit: workspace %zu < required %zu bytes", workspace_bytes, ws.total_bytes);
    return ISA_ERR_WORKSPACE;
  }
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  ISA_CUDA(cudaMemsetAsync(workspace, 0, ws.zero_bytes, stream));
  int gx = (ld + 255) / 256;
  const int cap = (di.num_sms * 8 + C - 1) / C;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  dim3 grid(gx, C);
  km_prep_max_kernel<<<grid, 256, 0, stream>>>(X, n_ptr, ld, C, k, ws);
  km_prep_sums_kernel<<<grid, 256, 0, stream>>>(X, n_ptr, ld, C, ws);
  km_prep_center_kernel<<<grid, 256, 0, stream>>>(X, n_ptr, ld, C, ws);
  km_prep_xn_kernel<<<(ld + 255) / 256, 256, 0, stream>>>(n_ptr, ld, C, ws);
  ISA_CUDA(cudaGetLastError());
  const int CP = pick_cp(C);
  if (init_centers) {
    km_init_centers_kernel<<<(n_init * k * C + 255) / 256, 256, 0, stream>>>(init_centers, n_init, k, C, ws);
    ISA_CUDA(cudaGetLastError());
  } else {
    switch (CP) {
      case 8: rc = launch_seed<8>(n_ptr, ld, C, k, n_local_trials, n_init, uniforms, ws, di.num_sms, stream); break;
      case 16: rc = launch_seed<16>(n_ptr, ld, C, k, n_local_trials, n_init, uniforms, ws, di.num_sms, stream); break;
      case 24: rc = launch_seed<24>(n_ptr, ld, C, k, n_local_trials, n_init, uniforms, ws, di.num_sms, stream); break;
      case 32: rc = launch_seed<32>(n_ptr, ld, C, k, n_local_trials, n_init, uniforms, ws, di.num_sms, stream); break;
      default: rc = launch_seed<64>(n_ptr, ld, C, k, n_local_trials, n_init, uniforms, ws, di.num_sms, stream); break;
    }
    if (rc) return rc;
  }
  LloydParams prm;
  prm.n_ptr = n_ptr; prm.ld = ld; prm.C = C; prm.k = k; prm.R = n_init; prm.max_iter = max_iter; prm.tol_rel = tol_rel;
  prm.ws = ws; prm.labels_out = labels_out; prm.centers_out = centers_out; prm.inertia_out = inertia_out;
  prm.n_iter_out = n_iter_out; prm.info = info;
  switch (CP) {
    case 8: rc = launch_lloyd<8>(prm, di.num_sms, stream); break;
    case 16: rc = launch_lloyd<16>(prm, di.num_sms, stream); break;
    case 24: rc = launch_lloyd<24>(prm, di.num_sms, stream); break;
    case 32: rc = launch_lloyd<32>(prm, di.num_sms, stream); break;
    default: rc = launch_lloyd<64>(prm, di.num_sms, stream); break;
  }
  if (rc) return rc;
  if (seed_idx_out) ISA_CUDA(cudaMemcpyAsync(seed_idx_out, ws.seed_idx, sizeof(int) * (size_t)n_init * k, cudaMemcpyDeviceToDevice, stream));
  return ISA_OK;
}

}  // extern "C"
